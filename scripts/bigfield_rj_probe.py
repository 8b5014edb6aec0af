"""Reversible-jump chains on the large field (BigFieldRHMC.run_rj) against the within-model engine on the same field.

    python scripts/bigfield_rj_probe.py [--niter 49] [--repeats 3]

C5 of bench.py: 8192 x 8192, 1e5 mock stars, r = 12, bench.py's run parameters (10 leapfrog steps, dt = 0.05).  The chains start
from the field's find_peaks catalogue, max_stars = 2e5.  Three runs, each a captured iteration graph replayed niter + 1 times:
    rj     run_rj, P_move = [0.4, 0.3, 0.3]
    rj0    run_rj, P_move = [1, 0, 0]   (within-model only: what the enqueued-but-skipped jump phases and leg 2 cost)
    run    run()
Each timed run starts from the catalogue (set outside the timed window for run, inside run_rj's own re-store for the two rj runs)
and ends with the synchronising chain read-back; the three alternate.  Star-steps count the stars of every leapfrog step the
device ran: N for leg 1 and the edited N for leg 2 of a jump.  Prints one JSON line with the card's name and power limit.
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
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def star_steps(out, nsteps):
    """Stars times leapfrog steps the device ran: leg 1 of every iteration, leg 2 of every jump (N after the edit)."""
    N = out["N_chain"].astype(np.int64)
    mv = out["move_chain"]
    edited = N + np.where((mv == 1) | (mv == 3), 1, -1)
    return int(nsteps * (N.sum() + edited[mv != 0].sum()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--niter", type=int, default=49)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()

    import torch

    from hmc_stellar_toy_model_b200 import bigfield as bf

    card0 = card()
    bench = load_bench()
    rows = cols = 8192
    t = bench.c5_truth(rows, cols, 100000, 77)
    run = t["run"]
    ftc = bench.exp_constants()["flux_to_count"]
    fmin, fmax = 10 ** (0.4 * (22.5 - 20)) * ftc, 10 ** (0.4 * (22.5 - 15)) * ftc
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    strip = bf.BigFieldStrip(rows=rows, cols=cols, rank=0, world=1, device=0, max_stars=200000, max_ghosts=1, patch_radius=12,
                             halo=12, **t["consts"])
    strip.set_stream(stream.cuda_stream)
    strip.gen_mock_data(t["q_true"], seed=77)
    np.random.seed(78)
    cat = strip.find_peaks(ftc, 22.0)
    eng = bf.BigFieldRHMC([strip])
    rj_kw = dict(fmin=fmin, fmax=fmax, K_split=1.0, beta_a=2.0, beta_b=2.0, want=(), use_graph=True, seed=5,
                 **{k: run[k] for k in ("g_ff2", "delta", "counter_max", "f_pos")})

    def timed(mode):
        strip.set_stars(cat)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if mode == "run":
            out = eng.run(args.niter, run["nsteps"], run["dt"], seed=5, use_graph=True,
                          **{k: run[k] for k in ("g_ff2", "delta", "counter_max", "f_pos")})
        else:
            out = eng.run_rj(args.niter, run["nsteps"], run["dt"], P_move=[0.4, 0.3, 0.3] if mode == "rj" else [1.0, 0.0, 0.0],
                             **rj_kw)
        return out, time.perf_counter() - t0

    modes = ("rj", "rj0", "run")
    for m in modes:   # capture and warm every graph
        timed(m)
    L = args.niter + 1
    res = {m: [] for m in modes}
    last = {}
    for _ in range(args.repeats):
        for m in modes:
            out, s = timed(m)
            steps = star_steps(out, run["nsteps"]) if m != "run" else len(cat) * L * run["nsteps"]
            jumps = int(np.sum(out["move_chain"] != 0)) if m != "run" else 0
            res[m].append(dict(seconds=s, it_per_s=L / s, jump_it_per_s=jumps / s, M_star_steps_per_s=steps / s / 1e6))
            last[m] = out
    o = last["rj"]
    acc = {name: int(np.sum((o["move_chain"] == c) & (o["A_chain"] != 0))) for c, name in
           ((1, "birth"), (2, "death"), (3, "split"), (4, "merge"))}
    prop = {name: int(np.sum(o["move_chain"] == c)) for c, name in ((1, "birth"), (2, "death"), (3, "split"), (4, "merge"))}
    med = {m: {k: float(np.median([r[k] for r in v])) for k in v[0]} for m, v in res.items()}
    print(json.dumps({
        "card": card0, "card_after": card(),
        "workload": {"rows": rows, "cols": cols, "mock_stars": 100000, "catalogue": int(len(cat)), "max_stars": 200000,
                     "patch_radius": 12, "niter": args.niter, "nsteps": run["nsteps"], "dt": run["dt"], "repeats": args.repeats},
        "median": {m: {k: round(v, 3) for k, v in d.items()} for m, d in med.items()},
        "all": {m: [{k: round(x, 3) for k, x in r.items()} for r in v] for m, v in res.items()},
        "rj_proposed": prop, "rj_accepted": acc, "rj_accepted_within": int(np.sum((o["move_chain"] == 0) & (o["A_chain"] != 0))),
        "rj_N_first_last": [int(o["N_chain"][0]), int(o["n_final"])],
        "rj0_vs_run_time_pct": round(100.0 * (med["rj0"]["seconds"] / med["run"]["seconds"] - 1.0), 2),
        "rj0_same_decisions_as_run": bool(np.array_equal(last["rj0"]["A_chain"], last["run"]["A_chain"])),
        "rj0_vs_run_E_relerr": float(np.max(np.abs(last["rj0"]["E_chain"] - last["run"]["E_chain"]) /
                                            np.abs(last["run"]["E_chain"]))),
    }))


if __name__ == "__main__":
    main()
