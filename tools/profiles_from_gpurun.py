"""Turn what a GPU session left under gpurun_out/ into the committed evidence under profiles/ (run here, after gpurun returned):
  bench.json            -> profiles/bench_<tag>.json
  launches.csv          -> profiles/launches_<tag>.csv + per-kernel shares printed + profiles/ncu_traffic_<tag>.json (DRAM bytes per launch
                           of the device-resident sweep launches: the `traffic` field of bench.py's roofline reads this file)
  prof_*.ncu-rep        -> profiles/ncu_<name>_<tag>.txt (tools/ncu_summary.py + ncu_brief.py) and ncu_<name>_source_<tag>.txt
usage: python tools/profiles_from_gpurun.py <tag>            e.g. r2"""
import collections, csv, json, os, shutil, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G, P = os.path.join(ROOT, "gpurun_out"), os.path.join(ROOT, "profiles")
tag = sys.argv[1] if len(sys.argv) > 1 else "rX"

if os.path.exists(os.path.join(G, "bench.json")) and os.path.getsize(os.path.join(G, "bench.json")) > 10:
    shutil.copy(os.path.join(G, "bench.json"), os.path.join(P, f"bench_{tag}.json"))
    d = json.load(open(os.path.join(G, "bench.json")))
    for name, x in (("primary", d), ("secondary", d.get("secondary") or {})):
        if x:
            print(f"{name}: value {x['value']:.4g} e2e {(x.get('e2e') or {}).get('value', float('nan')):.4g} engine {x.get('engine')} "
                  f"kernel_ms {x['roofline']['kernel_ms']:.2f} frac {x['roofline']['frac']:.3f} clocks {x.get('clocks')}")

lp = os.path.join(G, "launches.csv")
if os.path.exists(lp):
    shutil.copy(lp, os.path.join(P, f"launches_{tag}.csv"))
    rows = [r for r in csv.reader(open(lp)) if len(r) > 10]
    hdr = rows[0]
    ik, im, iv, iid, ig = (hdr.index(k) for k in ("Kernel Name", "Metric Name", "Metric Value", "ID", "Grid Size"))
    per = collections.OrderedDict()
    for r in rows[1:]:
        per.setdefault(r[iid], {"k": r[ik], "g": r[ig]})[r[im]] = float(r[iv].replace(",", ""))
    L = list(per.values())
    tot = collections.Counter()
    for x in L:
        tot[x["k"].split("(")[0][-44:]] += x.get("gpu__time_duration.sum", 0)
    s = sum(tot.values()) or 1
    for k, v in tot.most_common():
        print(f"{k:46s} {v / 1e6:9.2f} ms {100 * v / s:5.1f}%")
    # device-resident sweep launches = the ones followed by a finalize whose grid is pairs_per_step (148 * 16 SURF, 148 * 64 ORB)
    traffic = {}
    for key, name, fin_grid, pairs, alg in (("surf_tc16", "sweep_win_kernel<0>", "(2368, 1, 1)", 2368, 8000 * (288 + 256)),
                                            ("orb_tc16", "sweep_win_kernel<1>", "(9472, 1, 1)", 9472, 4000 * (288 + 32)),
                                            ("surf_tc", "sweep_l2_tc_kernel<0>", "(2368, 1, 1)", 2368, 8000 * (544 + 256)),
                                            ("orb_tc", "sweep_l2_tc_kernel<2>", "(9472, 1, 1)", 9472, 4000 * (288 + 32)),
                                            ("surf", "sweep_l2_kernel", "(2368, 1, 1)", 2368, 8000 * 520),
                                            ("orb", "sweep_hamming_kernel", "(9472, 1, 1)", 9472, 4000 * 64)):
        g = [a for a, b in zip(L, L[1:]) if name in a["k"] and "finalize" in b["k"] and b["g"] == fin_grid]
        if not g:
            continue
        # two-phase cross-check: every chunk has a main sweep and a (usually tiny) verification sweep, each followed by a finalize launch
        tmax = max(x.get("gpu__time_duration.sum", 0) for x in g)
        g = [x for x in g if x.get("gpu__time_duration.sum", 0) >= 0.5 * tmax]
        rd = sum(x.get("dram__bytes_read.sum", 0) for x in g) / len(g)
        wr = sum(x.get("dram__bytes_write.sum", 0) for x in g) / len(g)
        ns = sum(x.get("gpu__time_duration.sum", 0) for x in g) / len(g)
        traffic[key] = {"dram_read_bytes_per_launch": rd, "dram_write_bytes_per_launch": wr, "kernel_ns_under_ncu": ns, "launches_averaged": len(g),
                        "pairs_per_launch": pairs, "algorithmic_bytes_per_pair": alg, "bytes_per_pair": (rd + wr) / pairs,
                        "source": f"ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum on a short bench.py run (profiles/launches_{tag}.csv; device-resident launches only)"}
        print(key, f"{len(g)} launches, {rd / 1e6:.0f} MB read + {wr / 1e6:.0f} MB written, {ns / 1e6:.2f} ms under ncu")
    if traffic:
        json.dump(traffic, open(os.path.join(P, f"ncu_traffic_{tag}.json"), "w"), indent=1)
        print(f"(bench.py picks the newest profiles/ncu_traffic_r*.json that has the kernel)")

for f in sorted(os.listdir(G)) if os.path.isdir(G) else []:
    if f.startswith("prof_") and f.endswith(".ncu-rep"):
        name = f[len("prof_"):-len(".ncu-rep")]
        rep = os.path.join(G, f)
        with open(os.path.join(P, f"ncu_{name}_{tag}.txt"), "w") as out:
            out.write(f"# ncu --set full --clock-control none --import-source on: {f}\n")
            for tool in ("ncu_summary.py", "ncu_brief.py"):
                out.write(subprocess.run([sys.executable, os.path.join(ROOT, "tools", tool), rep] + (["sm__pipe_tensor", "l1tex__data_pipe_tc", "lts__throughput"] if tool == "ncu_summary.py" else []),
                                         capture_output=True, text=True).stdout)
        src = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv"], capture_output=True, text=True).stdout
        tmp = os.path.join("/tmp", f"{name}_src.csv")
        open(tmp, "w").write(src)
        top = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ncu_source_top.py"), tmp, "48"], capture_output=True, text=True).stdout
        with open(os.path.join(P, f"ncu_{name}_source_{tag}.txt"), "w") as out:
            out.write(f"# ncu source page of {f}, aggregated by 48-instruction SASS regions (tools/ncu_source_top.py)\n{top}")
        print(f"wrote profiles/ncu_{name}_{tag}.txt and ncu_{name}_source_{tag}.txt")
