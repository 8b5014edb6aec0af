"""K chains of one field in one large-field context (BigFieldStrip(chains=K)) against today's one-chain engine on the same field.

    python scripts/bigfield_chains_probe.py [--niter 9] [--repeats 3] [--c3-k 1,2,4,8,16,32,64] [--c5-k 1,2,4]

Fields and run parameters are bench.py's: C3 = 256 x 256 with 3277 mock stars, C5 = 8192 x 8192 with 1e5; r = 12, halo 24,
bench's c5_truth run (10 leapfrog steps, dt = 0.05), niter + 1 iterations, each run a captured iteration graph replayed
niter + 1 times.  Per field:
    one      today's one-chain engine on the path srhmc_big_create chooses (C3: the star-parallel scatter path, the bench arm;
             C5: the tile kernel)
    K        one context of K chains (every evaluation on the tile kernel), all started from the bench start catalogue
Every run starts from the catalogue (set outside the timed window) and ends with the synchronising chain read-back; the arms
alternate, `repeats` rounds, medians reported.  Aggregate star-steps/s = K N (niter + 1) nsteps / time.  Device memory of
each context: the growth of the device's used bytes (torch.cuda.mem_get_info) while it is created; the per-chain cost is the
slope over K.  Prints one JSON line with the card's name and power limit.
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


def probe_field(torch, bf, bench, rows, cols, nstars, ks, niter, repeats):
    t = bench.c5_truth(rows, cols, nstars, 77)
    run = t["run"]
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def strip_of(k, tile):
        if tile:   # K chains always evaluate on the tile kernel; the K = 1 arm is put there too
            os.environ.update(SRHMC_BIG_PATH="tile", SRHMC_BIG_STAR="0")
        s = bf.BigFieldStrip(rows=rows, cols=cols, rank=0, world=1, device=0, max_stars=nstars, max_ghosts=1024, patch_radius=12,
                             halo=24, chains=k, **t["consts"])
        s.set_stream(stream.cuda_stream)
        s.gen_mock_data(t["q_true"], seed=77)
        os.environ.pop("SRHMC_BIG_PATH", None)
        os.environ.pop("SRHMC_BIG_STAR", None)
        return s

    def used():
        torch.cuda.synchronize()
        free, total = torch.cuda.mem_get_info()
        return total - free

    base = used()
    one = strip_of(1, False)
    one_bytes = used() - base
    arms = {"one": bf.BigFieldRHMC([one])}
    mem = {}
    for k in ks:
        before = used()
        arms[k] = bf.BigFieldRHMC([strip_of(k, True)])
        mem[k] = used() - before
    L = niter + 1

    def timed(name):
        eng = arms[name]
        eng.strips[0].set_stars(t["q0"])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = eng.run(niter, seed=1000, use_graph=True, **run)
        return out, time.perf_counter() - t0

    names = ["one"] + list(ks)
    for m in names:   # capture and warm every graph
        timed(m)
    res = {m: [] for m in names}
    for _ in range(repeats):
        for m in names:
            _, s = timed(m)
            k = 1 if m == "one" else m
            res[m].append(dict(seconds=s, ms_per_iter=1e3 * s / L, M_star_steps_per_s=k * nstars * L * run["nsteps"] / s / 1e6))
    med = {str(m): {q: round(float(np.median([r[q] for r in v])), 3) for q in v[0]} for m, v in res.items()}
    out1, _ = timed("one")
    same = {}
    for k in ks:   # chain 0 of K chains against the one-chain engine (bit-equal only when both run the tile kernel)
        o, _ = timed(k)
        same[str(k)] = bool(np.array_equal(o["A_chain"][0] if k > 1 else o["A_chain"], out1["A_chain"]))
    del arms
    torch.cuda.synchronize()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return {"rows": rows, "cols": cols, "stars": nstars, "niter": niter, "nsteps": run["nsteps"], "dt": run["dt"],
            "one_path": "tile" if -(-rows // 64) * -(-cols // 64) >= 2 * sms else "scatter",
            "median": med, "all": {str(m): [{q: round(x, 4) for q, x in r.items()} for r in v] for m, v in res.items()},
            "mem_one_chain_context_MB": round(one_bytes / 2 ** 20, 1),
            "mem_K_context_MB": {str(k): round(v / 2 ** 20, 1) for k, v in mem.items()},
            "chain0_same_accepts_as_one": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--niter", type=int, default=9)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--c3-k", default="1,2,4,8,16,32,64")
    ap.add_argument("--c5-k", default="1,2,4")
    args = ap.parse_args()

    import torch

    from hmc_stellar_toy_model_b200 import bigfield as bf

    card0 = card()
    bench = load_bench()
    c3 = probe_field(torch, bf, bench, 256, 256, 3277, [int(x) for x in args.c3_k.split(",")], args.niter, args.repeats)
    c5 = probe_field(torch, bf, bench, 8192, 8192, 100000, [int(x) for x in args.c5_k.split(",")], args.niter, args.repeats)
    print(json.dumps({"card": card0, "card_after": card(), "c3": c3, "c5": c5}))


if __name__ == "__main__":
    main()
