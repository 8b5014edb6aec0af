"""Cost of recording star samples on the large field, and of the convergence statistics over resident chains.

    python scripts/bigfield_samples_probe.py [--repeats 3] [--runs 5] [--stat-iters 200]

C5 of bench.py (8192 x 8192, 1e5 stars, device mock data, bench.py's run parameters), one GPU.  Three engines on the same
field -- recording off, want=("q",), want=("q", "p"), stride 1 -- each keep their captured iteration graph; their timed runs
alternate.  Device time is the host clock from the start of run() to the end of its synchronising chain read-back, before
any sample rows are downloaded; the download is reported separately.  Then two of the engines run longer chains with
different seeds and bf.convergence_stats is timed over their resident q rows.  Prints one JSON line.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def load_bench():
    spec = importlib.util.spec_from_file_location("bench_for_probe", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(bench)
    finally:
        sys.argv = argv
    return bench


def card():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3, help="alternations of the three recording modes")
    ap.add_argument("--runs", type=int, default=5, help="timed runs per mode and repeat")
    ap.add_argument("--stat-iters", type=int, default=200, help="Metropolis iterations of the two chains of the statistics")
    args = ap.parse_args()

    import torch

    from hmc_stellar_toy_model_b200 import bigfield as bf

    bench = load_bench()
    rows = cols = 8192
    n = 100000
    t = bench.c5_truth(rows, cols, n, 77)
    run = t["run"]
    niter = 9   # bench.py's --c5-niter
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    modes = {"off": (), "q": ("q",), "qp": ("q", "p")}
    engines, D = {}, None
    for m in modes:
        strip = bf.BigFieldStrip(rows=rows, cols=cols, rank=0, world=1, device=0, max_stars=n, max_ghosts=1024,
                                 patch_radius=12, halo=24, **t["consts"])
        strip.set_stream(stream.cuda_stream)
        if D is None:
            D = strip.gen_mock_data(t["q_true"], seed=77, return_data=True)
        else:
            strip.set_data(D)
        engines[m] = bf.BigFieldRHMC([strip])

    def timed(m, it=niter, seed=1000):
        eng = engines[m]
        eng.strips[0].set_stars(t["q0"])
        torch.cuda.synchronize()
        stamp = {}
        samples = bf.BigFieldRHMC._samples

        def first_download(name, nrows, **kw):
            stamp.setdefault("dev", time.perf_counter())
            return samples(eng, name, nrows, **kw)

        eng._samples = first_download
        t0 = time.perf_counter()
        out = eng.run(it, seed=seed, want=modes[m], **run)
        t1 = time.perf_counter()
        del eng._samples
        return out, stamp.get("dev", t1) - t0, t1 - stamp.get("dev", t1)

    for m in modes:   # capture and warm every engine's graph
        for _ in range(2):
            timed(m)
    units = n * (niter + 1) * run["nsteps"]
    dev = {m: [] for m in modes}
    dl = {m: [] for m in modes}
    last = {}
    for _ in range(args.repeats):
        for m in modes:
            s_dev = s_dl = 0.0
            for _ in range(args.runs):
                out, a, b = timed(m)
                s_dev += a
                s_dl += b
            dev[m].append(units * args.runs / s_dev / 1e6)
            dl[m].append(s_dl / args.runs * 1e3)
            last[m] = out
    same = all(np.array_equal(last["off"][k], last[m][k]) for m in ("q", "qp") for k in ("E_chain", "V_chain", "A_chain"))
    med = {m: float(np.median(v)) for m, v in dev.items()}

    # two resident chains of stat-iters rows (different seeds), statistics over their q rows
    for m, seed in (("q", 1), ("qp", 2)):
        engines[m].strips[0].set_stars(t["q0"])
        engines[m].run(args.stat_iters - 1, seed=seed, want=("q",), **run)
    stats = {}
    for thin in (5, 1):
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            R, n_eff = bf.convergence_stats([engines["q"], engines["qp"]], thin_rate=thin, warm_up_num=0)
            ts.append((time.perf_counter() - t0) * 1e3)
        stats["thin%d_ms" % thin] = [round(x, 2) for x in ts]
        stats["thin%d_finite" % thin] = bool(np.all(np.isfinite(R)) and np.all(np.isfinite(n_eff)))
    print(json.dumps({
        "card": card(),
        "workload": {"rows": rows, "cols": cols, "stars": n, "niter": niter, "nsteps": run["nsteps"], "dt": run["dt"],
                     "runs_per_sample": args.runs, "repeats": args.repeats},
        "M_star_steps_per_s": {m: [round(x, 2) for x in v] for m, v in dev.items()},
        "recording_cost_pct": {m: round(100.0 * (1.0 - med[m] / med["off"]), 3) for m in ("q", "qp")},
        "sample_download_ms_per_run": {m: [round(x, 2) for x in v] for m, v in dl.items() if m != "off"},
        "convergence_stats": dict(stats, chains=2, rows=args.stat_iters, variables=3 * n),
        "chains_bit_identical_recording_on_off": same,
    }))


if __name__ == "__main__":
    main()
