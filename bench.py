#!/usr/bin/env python
"""bench.py -- headline benchmark of the EasySFM matching hot path on B200 (contract: see task brief §4).

Workload (BASELINE.json configs[3], the config the metric is quoted on): synthetic SURF-like descriptors,
1000 images x 8000 features x 64 fp32, all-pairs 2-NN + ratio 0.8 + mutual cross-check.  The whole triangle
is 499,500 image pairs = 3.2e13 comparisons (~1.5 min on one B200), so one *step* is a fixed slice of it:
  value : `pairs_per_step` consecutive pairs of this rank's block-cyclic shard of the triangle, descriptor bank
          already resident in HBM (device-resident throughput; only per-pair counts come back to the host);
  e2e   : the public call a user makes on HOST buffers -- scheduler.match_all_pairs(frames): esfm_bank_set_frame x M from
          PAGEABLE memory (what a cv::Mat is) + esfm_bank_commit + all M(M-1)/2 pairs + the compacted matches back on rank 0's
          host, all inside the timed region.  The triangle is FIXED (M frames, ~4 x pairs_per_step pairs), so at N GPUs this
          is the sharded job itself (strong scaling): NCCL broadcast of the bank, work-balanced pair deal, chunked NCCL return of
          the matches to rank 0.  `e2e.sha1` digests (counts, matches) of the last step: it must be equal at N = 1/2/4/8.
          `e2e_pinned` (N = 1) is the same step fed from page-locked frames (esfm_bank_set_frame_pinned).
  parity_sample : after the timed loop one timed step's matches are fetched and a seeded sample of its pairs is checked
          against the oracle (outside the timed region).
Both are reported as descriptor comparisons/s (rows_q * rows_t per pair, counted once even with cross-check).
`--impl reference` times the reference's own CPU path (cv2.BFMatcher knnMatch(k=2) + reverse knnMatch(k=1) as in
python_code/feature_match.py:26-39) on a bounded sample of the same pairs with all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_IMAGES = {"surf": 1000, "orb": 5000}
N_FEAT = {"surf": 8000, "orb": 4000}
RATIO = 0.8
CROSS_CHECK = True
SEED = {"surf": 4, "orb": 5}
SM_LANES_FP32 = 128      # FFMA lanes per SM per clock (verified: profiles/pipes_r1.txt)
POPC_LANES = 16          # POPC lanes per SM per clock (verified: profiles/pipes_r1.txt)


TC8_FLOP_PER_CMP = (256 + 32) * 2       # ORB on the tensor cores: 256 FP8 MACs + one K=32 augmented step, x 2
TC_FLOP_PER_CMP = (3 * 64 + 8) * 2   # 3xTF32 split over 64 dims + one K=8 augmented step (norms), x 2: tensor FLOPs executed per comparison


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    # fallback stated by /opt/skills/guides/B200_PROFILING.md: 6.65 TB/s copy, 1.59 PFLOP/s cuBLAS bf16 (burst)
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        hi = [x for x in sm if x >= 0.5 * max(sm)]
        return {"sm_mhz": float(np.median(hi)), "sm_max_mhz": float(max(smax)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


def make_bank_device(kind, n_images, n_feat, seed, dev):
    import torch
    from easysfm_b200 import synth
    if kind == "surf":
        return synth.surf_like_torch(n_images, n_feat, seed, dev)
    return synth.orb_like_torch(n_images, n_feat, seed, dev)


def cpu_reference_sample(host_bank, pairs, budget_s, cross_check):
    """Time the reference's cv2 calls on pairs from the same bank until ~budget_s of CPU work is done."""
    import cv2
    from oracle import cv2_oracle
    t_total, n_done, comps = 0.0, 0, 0
    while True:
        for (i, j) in pairs:
            Q, T = host_bank[i], host_bank[j]
            t_total += cv2_oracle.time_pair(Q, T, cross_check, repeats=1)
            n_done += 1
            comps += Q.shape[0] * T.shape[0]
            if t_total >= budget_s and n_done >= 4:
                return comps / t_total, n_done, t_total, cv2.getNumThreads()


def parity_sample(kind, results, step_pairs, raw, n_feat, row_bytes, np_dtype, cols, n_sample):
    """A seeded sample of one TIMED step's pairs against the oracle (test infrastructure used as the checker, outside the
    timed region): ORB bit-exact; SURF identical candidates => bit-identical distances, any differing query must be a
    float64-verified near-tie within the north star's 1e-5 relative tolerance (tests/util.justify_l2)."""
    import oracle
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import LazyDist64, justify_l2
    results.fetch()
    rng = np.random.default_rng(12345)
    sel = np.sort(rng.choice(len(step_pairs), min(n_sample, len(step_pairs)), replace=False))
    frame_cache = {}

    def frame(f):
        if f not in frame_cache:
            lo = int(f) * n_feat * row_bytes
            frame_cache[f] = raw[lo: lo + n_feat * row_bytes].cpu().numpy().view(np_dtype).reshape(n_feat, cols)
        return frame_cache[f]

    mismatches, near_ties, n_matches = 0, 0, 0
    for k in sel:
        q, t, got = results.pair_at(int(k))
        assert (q, t) == tuple(int(x) for x in step_pairs[k])
        Q, T = frame(q), frame(t)
        ref = oracle.match(Q, T, RATIO, CROSS_CHECK)
        n_matches += len(ref)
        same = len(got) == len(ref) and (got["queryIdx"] == ref["queryIdx"]).all() and (got["trainIdx"] == ref["trainIdx"]).all()
        if same and (got["distance"] == ref["distance"]).all():
            continue
        if kind == "orb":
            mismatches += 1
            continue
        try:
            near_ties += justify_l2(Q, T, RATIO, CROSS_CHECK, got, ref, D=LazyDist64(Q, T))
        except AssertionError:
            mismatches += 1
    return {"pairs": int(len(sel)), "mismatches": int(mismatches), "matches_checked": int(n_matches),
            "queries_differing_at_float64_near_ties": int(near_ties),
            "checker": "oracle.match (oracle/bf_oracle.c) on the last timed device-resident step; SURF tolerance 1e-5 relative"}


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, results, step_pairs, n_feat):
    """Writes what the caller of the timed path receives for one step as float32 .npy files (indices stay below 2^24, so they are
    exact): pairs [P, 2] (query frame, train frame) and match_counts [P] of every pair, and the matches of a seeded sample of the
    pairs (sample [S]: positions in the step, ascending; query_idx, train_idx, distance: their matches back to back in sample
    order).  The sample is sized for n_feat matches per pair, the most a cross-checked 2-NN can return, so which pairs are
    written depends only on the arguments and the files stay under DUMP_BYTES."""
    results.fetch()
    matches, off = results.all_matches()
    n_pairs = len(step_pairs)
    assert results.n_pairs == n_pairs
    n_sample = min(n_pairs, (DUMP_BYTES - 12 * n_pairs - 1024) // (12 * n_feat + 4))
    sample = np.sort(np.random.default_rng(2024).choice(n_pairs, n_sample, replace=False))
    picked = np.concatenate([matches[off[k]:off[k + 1]] for k in sample]) if n_sample else matches[:0]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"pairs": step_pairs, "match_counts": np.diff(off), "sample": sample,
              "query_idx": picked["queryIdx"], "train_idx": picked["trainIdx"], "distance": picked["distance"]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float32))


def run_reference(args, kind):
    """--impl reference: cv2.BFMatcher on the box's host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import cv2
    from easysfm_b200 import synth
    n_feat = N_FEAT[kind]
    pairs_per_step = args.ref_pairs_per_step
    n_frames = 2 * pairs_per_step * (args.steps + args.warmup) + 2
    n_frames = min(n_frames, 64)
    gen = synth.surf_like if kind == "surf" else synth.orb_like
    frames = gen(n_frames, n_feat, seed=SEED[kind])
    from oracle import cv2_oracle   # all host threads (cv2 default); setNumThreads(0) would DISABLE threading
    rng = np.random.default_rng(0)
    def step():
        comps = 0
        for _ in range(pairs_per_step):
            i, j = rng.choice(n_frames, 2, replace=False)
            cv2_oracle.time_pair(frames[i], frames[j], CROSS_CHECK, repeats=1)
            comps += frames[i].shape[0] * frames[j].shape[0]
        return comps
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    comps = 0
    for _ in range(args.steps):
        comps += step()
    dt = time.perf_counter() - t0
    value = comps / dt
    sample = f"{pairs_per_step} image pairs of {n_feat}x{n_feat} per step, {args.steps} steps"
    line = {
        "impl": "reference", "metric": "descriptor comparisons/sec, all-pairs 2-NN + ratio + cross-check", "value": value,
        "unit": "comparisons/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if kind == "surf" else "u8", "data": "synthetic",
        "config": workload_config(kind, pairs_per_step, None),
        "cpu_baseline": {"value": value, "unit": "comparisons/s", "cores": cv2.getNumThreads(), "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "comparisons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "pairs_per_s": value / (n_feat * n_feat),
    }
    print(json.dumps(line))
    return 0


def workload_config(kind, pairs_per_step, e2e_frames):
    name = {"surf": "synthetic SURF 64-d fp32, 1000 images x 8k features, all-pairs 2-NN + ratio 0.8 + cross-check (BASELINE configs[3])",
            "orb": "synthetic ORB 256-bit, 5000 images x 4k features, all-pairs Hamming 2-NN + ratio 0.8 + cross-check (BASELINE configs[4])"}[kind]
    cfg = {"workload": name, "step": f"{pairs_per_step} image pairs per GPU per step (a slice of the pair triangle)",
           "ratio": RATIO, "cross_check": CROSS_CHECK,
           "l2_flush": "inputs larger than L2: every step touches new frames of a bank (2.0 GB SURF / 0.64 GB ORB) >> 126 MB L2"}
    if e2e_frames:
        cfg["e2e_step"] = (f"all pairs of a fixed triangle of {e2e_frames} pageable host frames ({e2e_frames * (e2e_frames - 1) // 2} pairs), "
                           "matches returned to rank 0's host: the same job at every N (strong scaling)")
    return cfg


def bench_kind(args, kind, ctx, dev, rank, world, dist, steps, warmup, cpu_budget_s, engine=None, e2e_arm=True, dump_dir=None):
    """Returns the result dict for one descriptor kind (device-resident value, e2e, roofline, cpu baseline); with `dump_dir`,
    rank 0 also writes the last timed device-resident step's matches there (dump_outputs).
    `engine` selects the sweep kernel: SURF 'tc16' (tcgen05 FP16 split, slice keys) | 'tc' (tcgen05 3xTF32) | 'ffma' (exact-FP32 FMA pipe);
    ORB 'tc16' (tcgen05 FP8 dot product, FP16 accumulators, slice keys) | 'tc' (FP8 dot product delivering packed keys) | 'popc' (XOR + POPC);
    None = library default (tc16)."""
    import torch
    from easysfm_b200 import scheduler
    import easysfm_b200 as esfm
    if engine:
        (ctx.set_l2_engine if kind == "surf" else ctx.set_hamming_engine)(engine)
    engine = ctx.l2_engine() if kind == "surf" else ctx.hamming_engine()

    n_images, n_feat = N_IMAGES[kind], N_FEAT[kind]
    if args.images:
        n_images = args.images
    sms = ctx.sm_count
    pairs_per_step = args.pairs_per_step or sms * (16 if kind == "surf" else 64)
    e2e_frames = args.e2e_frames or int((1 + (1 + 8 * 4 * pairs_per_step) ** 0.5) / 2)  # M(M-1)/2 ~ 4 x pairs_per_step
    e2e_frames = max(2, min(e2e_frames, n_images))

    # ---- setup (untimed): bank generated on rank 0's GPU, replicated with one NCCL broadcast -------------
    t_setup = time.perf_counter()
    kind_id = esfm.KIND_F32X64 if kind == "surf" else esfm.KIND_B256
    bank = ctx.bank(kind_id, n_images)
    for f in range(n_images):
        bank.set_frame_rows(f, n_feat)
    bank.alloc_device()
    ptr, nbytes = bank.device_rows()
    raw = scheduler._wrap_device_bytes(ptr, nbytes, ctx.device)
    bcast_ms = None
    if rank == 0:
        data = make_bank_device(kind, n_images, n_feat, SEED[kind], dev)
        raw.copy_(data.reshape(-1).view(torch.uint8))
        del data
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dist.broadcast(raw, src=0)
        e1.record()
        torch.cuda.synchronize()
        bcast_ms = e0.elapsed_time(e1)
    torch.cuda.synchronize()
    bank.commit_device()

    # host copy (PAGEABLE numpy memory, like the reference's cv::Mat data) of the frames the e2e steps, the parity sample and
    # the CPU baseline read; rank 0 only
    n_host = min(n_images, e2e_frames * (steps + warmup) + 2)
    row_bytes = 256 if kind == "surf" else 32
    np_dtype, cols = (np.float32, 64) if kind == "surf" else (np.uint8, 32)
    host_bank = None
    if rank == 0 and (e2e_arm or cpu_budget_s > 0):
        host_raw = raw[: n_host * n_feat * row_bytes].cpu()
        host_bank = host_raw.numpy().view(np_dtype).reshape(n_host, n_feat, cols)

    pairs = scheduler.all_pairs(n_images)
    mine = scheduler.shard_pairs(len(pairs), rank, world, block=64)
    my_pairs = pairs[mine]
    need = (steps + warmup) * pairs_per_step
    if len(my_pairs) < need:
        reps = (need + len(my_pairs) - 1) // len(my_pairs)
        my_pairs = np.concatenate([my_pairs] * reps)
    setup_s = time.perf_counter() - t_setup

    def step_pairs(s):
        return my_pairs[s * pairs_per_step:(s + 1) * pairs_per_step]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident arm ---------------------------------------------------------------------------
    for s in range(warmup):
        bank.match_pairs(step_pairs(s), RATIO, CROSS_CHECK, device_resident=True).close()
    sampler = ClockSampler(ctx.device)
    sync_all()
    sampler.start()
    st0 = ctx.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    n_matches = 0
    r_last = None
    for s in range(warmup, warmup + steps):
        if r_last is not None:
            r_last.close()
        r_last = bank.match_pairs(step_pairs(s), RATIO, CROSS_CHECK, device_resident=True)
        n_matches += r_last.n_matches
    ev1.record()
    sync_all()
    clocks = sampler.stop()
    st1 = ctx.stats()
    ms = ev0.elapsed_time(ev1)
    comps_local = st1["comparisons"] - st0["comparisons"]
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_max = float(t.item())
        c = torch.tensor([float(comps_local)], dtype=torch.float64, device=dev)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        comps_all = float(c.item())
    else:
        ms_max, comps_all = ms, float(comps_local)
    value = comps_all / (ms_max * 1e-3)
    launches = st1["kernel_launches"] - st0["kernel_launches"]
    sweep_ms = (st1["sweep_ms_total"] - st0["sweep_ms_total"]) / max(1, st1["sweep_launches"] - st0["sweep_launches"])
    comps_per_launch = comps_local / max(1, st1["sweep_launches"] - st0["sweep_launches"])

    # ---- parity of what was just timed (outside the timed region): the LAST timed step's matches vs the oracle -----------
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_sample(kind, r_last, step_pairs(warmup + steps - 1), raw, n_feat, row_bytes, np_dtype, cols, args.parity_pairs)
    if rank == 0 and dump_dir:
        dump_outputs(dump_dir, r_last, step_pairs(warmup + steps - 1), n_feat)
    r_last.close()

    # ---- end-to-end arm: PAGEABLE host frames in, host matches out (on rank 0), through the public API -----------------
    dbg = os.environ.get("BENCH_E2E_DEBUG") == "1"
    e2e_pairs = e2e_frames * (e2e_frames - 1) // 2

    def e2e_window(s):
        return (s * e2e_frames) % max(1, n_host - e2e_frames + 1)

    def e2e_step(s):
        tm = {}
        frames = None
        if rank == 0:
            f0 = e2e_window(s)
            frames = [host_bank[f0 + k] for k in range(e2e_frames)]
        res = scheduler.match_all_pairs(frames, RATIO, CROSS_CHECK, ctx=ctx, reuse_staging=True, timing=tm)
        if dbg and rank == 0:
            st = ctx.stats()
            print("e2e step %d: upload+broadcast %.1f ms, match+return %.1f ms (rank 0 last sweep %.1f finalize %.1f), %d matches" % (
                s, 1e3 * tm["upload_broadcast_s"], 1e3 * tm["match_gather_s"], st["last_sweep_ms"], st["last_finalize_ms"],
                res.n_matches), file=sys.stderr)
        return res

    e2e = None
    if e2e_arm:
        res = None
        for s in range(warmup):
            res = e2e_step(s)     # (held until the next step returns, exactly like the timed steps: the pinned pools reach steady state)
        sync_all()
        st2 = ctx.stats()
        ev0.record()
        n_e2e_matches = 0
        for s in range(warmup, warmup + steps):
            res = e2e_step(s)
            if rank == 0:
                n_e2e_matches += res.n_matches
        ev1.record()
        sync_all()
        st3 = ctx.stats()
        e2e_ms = max(ev0.elapsed_time(ev1), 1e-9)
        if world > 1:
            t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        e2e_comps = float(steps) * e2e_pairs * n_feat * n_feat
        e2e = {"value": e2e_comps / (e2e_ms * 1e-3), "unit": "comparisons/s", "scaling": "strong",
               "h2d_bytes_per_step": int((st3["h2d_bytes"] - st2["h2d_bytes"]) / steps),                  # rank 0: the frames (+ pair lists)
               "d2h_bytes_per_step": int(n_e2e_matches * 16 / steps + e2e_pairs * 12),                    # matches + counts/offsets reaching rank 0's host
               "ms_per_step": e2e_ms / steps, "frames": e2e_frames, "pairs_per_step": e2e_pairs,
               "host_memory": "pageable (esfm_bank_set_frame: staged through pinned memory, upload overlapped frame by frame)",
               "return_path": "device->host on the one GPU" if world == 1 else
                              f"{world} ranks: NCCL broadcast of the bank, work-balanced deal, chunked NCCL send of the matches to rank 0, device->host there"}
        del res
        # one more (untimed) step on a FIXED window of the bank: its digest of (counts, matches) must be equal at every N
        res = e2e_step(0)
        if rank == 0:
            e2e["sha1"] = res.sha1()
            e2e["sha1_of"] = f"all {e2e_pairs} pairs of frames 0..{e2e_frames - 1} of the seeded synthetic bank (per-pair counts | matches in pair order)"
            e2e["matches_in_digest"] = res.n_matches
        del res
        if world == 1:
            # same step fed from page-locked frames (no staging copy): what a caller with a pinned descriptor arena gets
            pin = torch.empty((e2e_frames * n_feat * row_bytes,), dtype=torch.uint8, pin_memory=True)
            pin_np = pin.numpy().view(np_dtype).reshape(e2e_frames, n_feat, cols)
            def pinned_step(s):
                f0 = e2e_window(s)
                pin_np[:] = host_bank[f0:f0 + e2e_frames]      # (untimed part of a real pipeline: the extractor writes there)
                t0 = time.perf_counter()
                b = ctx.bank(kind_id, e2e_frames)
                for k in range(e2e_frames):
                    b.set_frame_pinned(k, pin_np[k])
                b.commit()
                r = b.match_all_pairs(RATIO, CROSS_CHECK)
                n = r.n_matches
                r.close(); b.close()
                return time.perf_counter() - t0
            for s in range(2):
                pinned_step(s)
            tp = sum(pinned_step(warmup + s) for s in range(steps))
            e2e["e2e_pinned"] = {"value": steps * e2e_pairs * n_feat * n_feat / tp, "unit": "comparisons/s", "ms_per_step": 1e3 * tp / steps,
                                 "note": f"esfm_bank_set_frame_pinned (host wall clock, {steps} steps)"}
            del pin, pin_np

    # ---- roofline of the dominant kernel (the sweep) -----------------------------------------------------
    peaks, peak_src = _peaks()
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    fp32_pipe_peak = sms * SM_LANES_FP32 * 2 * sm_max * 1e6 / 1e12
    if kind == "surf" and engine == "tc16":
        unit_ops, unit = 128.0, "TFLOP/s"                      # algorithmic: 64 FMA = 128 FLOP per comparison
        peak = float(peaks.get("bf16_tflops", 1590.0))         # kind::f16 operands: the measured dense 16-bit tensor rate
        bound = "tensor"
        kern = "sweep_win_kernel<ESFM_KIND_F32X64>"
    elif kind == "surf" and engine == "tc":
        unit_ops, unit = 128.0, "TFLOP/s"                      # algorithmic: 64 FMA = 128 FLOP per comparison
        peak = float(peaks.get("bf16_tflops", 1590.0)) / 2.0   # dense TF32 = half the measured dense bf16 rate
        bound = "tensor"
        kern = "sweep_l2_tc_kernel"
    elif kind == "surf":
        unit_ops, unit = 128.0, "TFLOP/s"                      # 64 FFMA = 128 FLOP per comparison
        peak = fp32_pipe_peak
        bound = "fp32-fma-pipe"
        kern = "sweep_l2_kernel"
    elif engine in ("tc", "tc16"):
        unit_ops, unit = 8.0, "TPOPC/s"                        # algorithmic: 8 x 32-bit POPC per comparison (north_star)
        peak = sms * POPC_LANES * sm_max * 1e6 / 1e12          # ... against the pipe the XOR+POPC design is bound by
        bound = "tensor"
        kern = "sweep_l2_tc_kernel<1, kTcKindB256Z>" if engine == "tc" else "sweep_win_kernel<ESFM_KIND_B256>"
    else:
        unit_ops, unit = 8.0, "TPOPC/s"                        # 8 x 32-bit POPC per comparison (algorithmic, north_star)
        peak = sms * POPC_LANES * sm_max * 1e6 / 1e12
        bound = "popc-pipe"
        kern = "sweep_hamming_kernel"
    achieved = comps_per_launch * unit_ops / (sweep_ms * 1e-3) / 1e12
    roofline = {"bound": bound, "kernel": kern, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak,
                "peak_source": ((f"dense 16-bit tensor peak = bf16_tflops of MEASURED_PEAKS.json ({peak_src}): the sweep's MMAs are kind::f16"
                                 if engine == "tc16" else
                                 f"dense TF32 tensor peak = bf16_tflops / 2 of MEASURED_PEAKS.json ({peak_src}: "
                                 f"{peaks.get('bf16_tflops', 1590.0):.0f} TFLOP/s bf16)") if kind == "surf" else
                                f"{sms} SMs x 16 POPC lanes x {sm_max:.0f} MHz: the pipe the north star's XOR + POPC design is bound by "
                                f"(sm_max_mhz {peak_src})") if bound == "tensor" else
                               f"{sms} SMs x {'128 FFMA lanes x 2 FLOP' if kind == 'surf' else '16 POPC lanes'} x {sm_max:.0f} MHz "
                               f"(sm_max_mhz {peak_src}; lanes/clk measured by csrc/microbench/pipes.cu, profiles/pipes_r1.txt)",
                "kernel_ms": sweep_ms, "comparisons_per_launch": comps_per_launch,
                "hbm_gbs_algorithmic": None, "traffic": None}
    if bound == "tensor" and kind == "orb":
        # ORB on the tensor cores: scaled FP8 operands whose exact fp32 dot product is the packed key 20480 + 2^15 hamming + column
        # (DESIGN.md 5.2b; $ESFM_ORB_Z=0: plain +-1 vectors, Hamming = (256 - dot) / 2).  `achieved`/`frac` stay in the north
        # star's algorithmic unit (8 POPC per comparison against the POPC-pipe peak: > 1 means faster than any XOR+POPC kernel
        # can be); `executed_tflops` / `frac_executed` are the FP8 tensor FLOPs actually issued over the dense FP8 peak
        # (= 2 x the measured dense bf16 rate).  The kernel is bound by its selection epilogue, not by the tensor pipe.
        fp8_peak = 2.0 * float(peaks.get("bf16_tflops", 1590.0))
        flop_per_cmp = 512.0 if engine == "tc16" else TC8_FLOP_PER_CMP      # tc16: 8 MMAs of K = 32, no augmented step
        roofline["executed_tflops"] = (comps_per_launch / (sweep_ms * 1e-3)) * flop_per_cmp / 1e12
        roofline["frac_executed"] = roofline["executed_tflops"] / fp8_peak
        roofline["tensor_peak_tflops"] = fp8_peak
        roofline["note"] = (("Hamming as an exact FP8 dot product on tcgen05 (kind::f8f6f4) with FP16 accumulators (-2 hamming), selection on packed halves: "
                             if engine == "tc16" else
                             "Hamming as an exact FP8 dot product on tcgen05 (kind::f8f6f4) that yields packed (distance, column) keys: ") +
                            ("512" if engine == "tc16" else "576") + " tensor FLOP per comparison; frac is the algorithmic 8-POPC rate over the POPC-pipe peak; "
                            "frac_executed is the tensor work over the dense FP8 peak (2 x the measured bf16 rate); the rest is the latency of the "
                            "selection epilogue (one tournament per 64 columns and row), not the tensor pipe")
        roofline["mma_bound_cmp_per_s"] = sms * sm_max * 1e6 * 16384 / ((8 if engine == "tc16" else 9) * 64.1)
        roofline["frac_of_mma_bound"] = (comps_per_launch / (sweep_ms * 1e-3)) / roofline["mma_bound_cmp_per_s"]
    if bound == "tensor" and kind == "surf" and engine == "tc16":
        # `achieved`/`frac`: ALGORITHMIC 128 FLOP per comparison over the dense 16-bit tensor peak.  Executed: 3 x 64 x 2 FLOP on kind::f16
        # + 16 on kind::tf32 = 13 MMA slots of 64 clk per 128 x 128 tile (h16_probe: 64.1 clk per MMA); `frac_of_mma_bound` = how close the
        # sweep is to that issue-rate ceiling.  What binds it is the selection epilogue's instruction issue, not the tensor pipe.
        roofline["executed_tflops"] = achieved * 400.0 / 128.0
        roofline["frac_executed"] = achieved * (384.0 / 128.0) / peak + achieved * (16.0 / 128.0) / (peak / 2.0)
        roofline["mma_bound_cmp_per_s"] = sms * sm_max * 1e6 * 16384 / (13 * 64.1)
        roofline["frac_of_mma_bound"] = (comps_per_launch / (sweep_ms * 1e-3)) / roofline["mma_bound_cmp_per_s"]
        roofline["frac_vs_tf32_peak"] = achieved / (peak / 2.0)
        roofline["frac_of_fp32_pipe_roofline"] = achieved / fp32_pipe_peak
        roofline["note"] = ("two-term FP16 split product (b.a + a.b + a.a over 64 dims on kind::f16, + one exact K=8 kind::tf32 step adding the norms) "
                            "on tcgen05: 13 MMA slots per tile instead of the 25 of 3xTF32; frac_vs_tf32_peak is the round-1 denominator (bf16 / 2)")
    if bound == "tensor" and kind == "surf" and engine == "tc":
        # `achieved`/`frac` use the ALGORITHMIC 128 FLOP per comparison (SURVEY 8d).  The tensor cores execute 3.125x that
        # (3xTF32 split over 64 dims + 8 augmented columns); `frac_executed` is that executed rate over the same peak (= tensor-pipe utilisation),
        # and `frac_of_fp32_pipe_roofline` compares the algorithmic rate with the FP32-FFMA pipe peak the FFMA engine is bound by.
        roofline["executed_tflops"] = achieved * TC_FLOP_PER_CMP / 128.0
        roofline["frac_executed"] = roofline["executed_tflops"] / peak
        roofline["frac_of_fp32_pipe_roofline"] = achieved / fp32_pipe_peak
        roofline["note"] = ("3xTF32 split product (lo.hi + hi.lo + hi.hi over 64 dims, + one K=8 step adding the norms) on tcgen05; "
                            f"{TC_FLOP_PER_CMP} tensor FLOP executed per 128 algorithmic FLOP")
    if kind == "orb" and engine == "popc":
        # The kernel compresses the 8 xor words with carry-save adders and issues only 4 POPC per comparison, so it can
        # exceed the algorithmic 8-POPC roofline; what binds it is instruction issue (~36 warp-instructions per 32
        # comparisons, 4 issue slots per clock per SM; profiles/sass_hamming_loop_r1.txt).
        roofline["note"] = "frac > 1 is real: 4 POPC + 16 LOP3 per comparison (Harley-Seal), not 8 POPC"
        issue_peak_cmp = sms * 4 * 32 / 35.8 * sm_max * 1e6
        roofline["frac_of_issue_bound"] = (comps_per_launch / (sweep_ms * 1e-3)) / issue_peak_cmp
    if clocks.get("sm_mhz"):
        roofline["frac_at_sampled_clock"] = achieved / (peak * clocks["sm_mhz"] / sm_max)
    # algorithmic HBM bytes: every pair reads both frames once + writes its matches
    # (SURF rows: 260 B in the FFMA engine's k-major bank; tensor-core engine: 544 B per train row = hi + lo images + augmented
    #  columns, 256 B per query row = the fp32 rows the sweep converts on the fly)
    bytes_per_pair = n_feat * ((((544 if engine == "tc" else 288) + 256) if engine in ("tc", "tc16") else 520) if kind == "surf"
                               else ((288 + 32) if engine in ("tc", "tc16") else 64))
    roofline["hbm_gbs_algorithmic"] = (comps_per_launch / (n_feat * n_feat)) * bytes_per_pair / (sweep_ms * 1e-3) / 1e9
    roofline["hbm_peak_gbs"] = peaks.get("hbm_gbs")
    # measured DRAM traffic of this kernel on this command (one ncu pass, committed under profiles/): far BELOW the per-pair
    # algorithmic bytes because pairs launched together share their train frame in L2 (capi.cu sorts a chunk by train frame)
    import glob
    tkey = {"surf": "surf_", "orb": "orb_"}[kind] + engine if engine in ("tc", "tc16") else kind
    for tpath in sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_traffic_r*.json")), reverse=True):    # newest round that has this kernel
        try:
            with open(tpath) as f:
                tr = json.load(f).get(tkey)
        except (OSError, ValueError):
            tr = None
        if tr:
            per_pair = (tr["dram_read_bytes_per_launch"] + tr["dram_write_bytes_per_launch"]) / tr["pairs_per_launch"]
            roofline["traffic"] = per_pair * (comps_per_launch / (n_feat * n_feat))
            roofline["traffic_source"] = f"profiles/{os.path.basename(tpath)} (dram__bytes_read.sum + dram__bytes_write.sum per launch)"
            roofline["algorithmic_bytes_per_launch"] = (comps_per_launch / (n_feat * n_feat)) * bytes_per_pair
            break

    # ---- CPU baseline (rank 0, N = 1 only): the reference's cv2 calls on a bounded sample ----------------
    cpu = None
    if rank == 0 and world == 1 and cpu_budget_s > 0:
        sample_pairs = [(i + 1, i) for i in range(0, min(n_host - 1, 64))]
        v, n_done, secs, cores = cpu_reference_sample(host_bank, sample_pairs, cpu_budget_s, CROSS_CHECK)
        cpu = {"value": v, "unit": "comparisons/s", "cores": cores, "kind": "reference",
               "sample": f"{n_done} image pairs of {n_feat}x{n_feat} ({secs:.1f} s of cv2.BFMatcher knnMatch(k=2) + reverse knnMatch(k=1))",
               "extrapolated_all_pairs_hours": (n_images * (n_images - 1) / 2) * (n_feat * n_feat) / v / 3600.0}

    out = {
        "metric": "descriptor comparisons/sec, all-pairs 2-NN + ratio + cross-check", "value": value, "unit": "comparisons/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_max / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if kind == "surf" else "u8", "data": "synthetic",
        "config": workload_config(kind, pairs_per_step, e2e_frames),
        "pairs_per_s": value / (n_feat * n_feat), "matches_per_step": n_matches / steps,
        "engine": engine, "e2e": e2e, "parity_sample": parity, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "cpu_baseline": cpu,
        "setup_s": setup_s, "bank_broadcast_ms": bcast_ms,
        "full_job_estimate_s": (n_images * (n_images - 1) / 2) * (n_feat * n_feat) / value,
    }
    bank.close()
    del host_bank, raw
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kind", default="surf", choices=["surf", "orb"], help="headline descriptor kind")
    ap.add_argument("--no-secondary", action="store_true", help="skip the second descriptor kind")
    ap.add_argument("--pairs-per-step", type=int, default=0)
    ap.add_argument("--images", type=int, default=0, help="override the number of images (smoke runs)")
    ap.add_argument("--cpu-budget-s", type=float, default=15.0)
    ap.add_argument("--ref-pairs-per-step", type=int, default=4)
    ap.add_argument("--l2-engine", default=None, choices=["tc16", "tc", "ffma"],
                    help="SURF sweep kernel: tcgen05 3xTF32 ('tc', library default) or exact-FP32 FMA pipe ('ffma')")
    ap.add_argument("--hamming-engine", default=None, choices=["tc16", "tc", "popc"],
                    help="ORB sweep kernel: tcgen05 FP8 +-1 dot product ('tc') or XOR + POPC ('popc'); default = library default")
    ap.add_argument("--no-alt-engine", action="store_true", help="skip the short run of the other engine of each kind")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of a sample of the timed step (runs under ncu)")
    ap.add_argument("--parity-pairs", type=int, default=20)
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames of the fixed e2e triangle (default: ~4 x pairs_per_step pairs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline kind's last timed device-resident step (rank 0's pairs) as DIR/<name>.npy, float32, < 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3

    if args.impl == "reference":
        return run_reference(args, args.kind)

    # stdout carries exactly ONE line (the JSON): anything libraries print to fd 1 (e.g. NCCL's version banner)
    # is routed to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    import easysfm_b200 as esfm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: easysfm_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # the library launches on torch's current (non-default) stream so torch.cuda.Event brackets its kernels
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = esfm.Context(local_rank, stream=stream.cuda_stream)

    engines = {"surf": args.l2_engine or ctx.l2_engine(), "orb": args.hamming_engine or ctx.hamming_engine()}
    other_engine = {"surf": {"tc16": "ffma", "tc": "ffma", "ffma": "tc16"}, "orb": {"tc16": "popc", "tc": "popc", "popc": "tc16"}}

    def alt_run(kind):
        # the other engine of this kind on the same workload, device-resident arm only (context, not the headline)
        a = bench_kind(args, kind, ctx, dev, rank, world, dist, args.steps, args.warmup, 0.0, engine=other_engine[kind][engines[kind]],
                       e2e_arm=False)
        (ctx.set_l2_engine if kind == "surf" else ctx.set_hamming_engine)(engines[kind])
        return {k: a[k] for k in ("engine", "value", "unit", "ms_per_step", "roofline", "clocks", "parity_sample")}

    primary = bench_kind(args, args.kind, ctx, dev, rank, world, dist, args.steps, args.warmup, args.cpu_budget_s,
                         engine=engines[args.kind], dump_dir=args.dump_outputs)
    if not args.no_alt_engine and world == 1:
        primary["alt_engine"] = alt_run(args.kind)
    if not args.no_secondary:
        other = "orb" if args.kind == "surf" else "surf"
        sec = bench_kind(args, other, ctx, dev, rank, world, dist, args.steps, args.warmup, args.cpu_budget_s / 2,
                         engine=engines[other])
        primary["secondary"] = {k: sec[k] for k in ("value", "unit", "ms_per_step", "dtype", "config", "pairs_per_s", "e2e", "parity_sample",
                                                    "engine", "roofline", "cpu_baseline", "gpu_launches", "clocks", "full_job_estimate_s")}
        if not args.no_alt_engine and world == 1:
            primary["secondary"]["alt_engine"] = alt_run(other)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    if rank == 0:
        os.write(json_fd, (json.dumps(primary) + "\n").encode())
    os.close(json_fd)
    return 0


if __name__ == "__main__":
    sys.exit(main())
