"""Peak finding on one large field (BigFieldStrip.find_peaks, srhmc_big_find_peaks): an 8192 x 8192 field with 1e5 stars
generated on the device at the benchmark's large-field density, the windowed descent of every grid seed and the greedy
merge timed separately, and the recall of the catalogue against the truth list.  Prints one JSON line that carries the
card's name and power limit read in the same run.

    python scripts/bigfield_peaks_probe.py [--rows 8192] [--stars 100000]

Each time is a host clock around one call that ends in a stream synchronise; it includes the copies of the seeds to the
device and of the results back (24 bytes per seed each way).  The merge is timed on its own by passing the alive
descended seeds with Nstep = 0 (they stay alive where they are)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hmc_stellar_toy_model_b200 import bigfield as bf  # noqa: E402

FTC = 1.0 / (0.00546689 * 4.62)


def mag2flux(m):
    return 10 ** (0.4 * (22.5 - m))


def c5_truth(rows, cols, nstars, seed):
    """The star list of bench.py's large-field workload (power law alpha = 2 in mag [15, 20], positions U(1, size - 1))."""
    rng = np.random.RandomState(seed)
    alpha = 2.0
    fmin, fmax = mag2flux(20.0) * FTC, mag2flux(15.0) * FTC
    u = rng.random_sample(nstars)
    fl = np.exp(np.log(fmin ** (1 - alpha) + u * (fmax ** (1 - alpha) - fmin ** (1 - alpha))) / (1 - alpha))
    x = rng.random_sample(nstars) * (rows - 2.0) + 1.0
    y = rng.random_sample(nstars) * (cols - 2.0) + 1.0
    return np.stack([fl, x, y], axis=1)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as e:  # the numbers below are then reported without their card
        return "unknown (%s)" % type(e).__name__, "unknown"


def recall(q_true, cat, hit_px=1.0):
    from scipy.spatial import cKDTree

    mag = 22.5 - 2.5 * np.log10(q_true[:, 0] / FTC)
    near = cKDTree(q_true[:, 1:]).query(q_true[:, 1:], k=2)[0][:, 1]
    iso = (mag < 19.0) & (near > 6.0)
    d = cKDTree(cat[:, 1:]).query(q_true[:, 1:])[0] if len(cat) else np.full(len(q_true), np.inf)
    return dict(isolated_bright=int(iso.sum()), isolated_bright_found=int(np.sum(d[iso] < hit_px)),
                all_found=int(np.sum(d < hit_px)), truth=len(q_true))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--stars", type=int, default=100000)
    ap.add_argument("--nstep", type=int, default=1000)
    ap.add_argument("--radius", type=int, default=12)
    args = ap.parse_args()
    rows = cols = args.rows
    B = mag2flux(23.0) * FTC
    strip = bf.BigFieldStrip(rows=rows, cols=cols, rank=0, world=1, device=0, max_stars=1, max_ghosts=1,
                             patch_radius=args.radius, halo=args.radius, psf_fwhm_pix=1.4 / 0.4, B_count=B, f_lim=B,
                             f_low=mag2flux(25.0) * FTC, g0=0.035997054345069765, g1=0.4523523265306124,
                             g2=0.008141675878296745, g_xx=0.05, g_ff=4.0)
    q_true = c5_truth(rows, cols, args.stars, 77)
    strip.gen_mock_data(q_true, seed=77)
    f_lim, f_seed = mag2flux(22.0) * FTC, mag2flux(21.5) * FTC
    n_side = int(0.2 * rows) - 1
    seeds = bf.peak_seeds(rows, cols, 0.2, np.random.RandomState(78).randn(n_side * n_side, 2), f_seed)
    # warm-up of both kernels and of the allocator
    w = strip.descend_seeds(seeds[:8192], args.nstep, 0.1, 0.1, f_lim)
    strip.descend_seeds(w["q"][w["alive"]], 0, 0.1, 0.1, f_lim, merge=(1.0, 0.5, FTC))
    strip.synchronize()
    t0 = time.perf_counter()
    d = strip.descend_seeds(seeds, args.nstep, 0.1, 0.1, f_lim)
    strip.synchronize()
    t_descent = time.perf_counter() - t0
    qa = d["q"][d["alive"]]
    t0 = time.perf_counter()
    m = strip.descend_seeds(qa, 0, 0.1, 0.1, f_lim, merge=(1.0, 0.5, FTC))
    strip.synchronize()
    t_merge = time.perf_counter() - t0
    cat = qa[m["kept"]]
    name, power = card()
    rec = dict(probe="bigfield_peaks", rows=rows, cols=cols, stars=args.stars, patch_radius=args.radius, nstep=args.nstep,
               seeds=len(seeds), alive=int(d["alive"].sum()), steps_median=float(np.median(d["steps"])),
               steps_max=int(d["steps"].max()), seed_steps=int(d["steps"].sum()), descent_s=round(t_descent, 4),
               seeds_per_s=round(len(seeds) / t_descent, 1), merge_s=round(t_merge, 4), merge_rounds=m["rounds"],
               catalogue=int(m["n_kept"]), gpu=name, power_limit=power, **recall(q_true, cat))
    strip.close()
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
