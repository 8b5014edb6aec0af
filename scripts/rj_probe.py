"""Throughput of reversible-jump chains on the device (field_kernel MODE_RUN_RJ) against within-model chains of the same
fields (srhmc_run) and against the drop-in's host-side proposals on one field.

    python scripts/rj_probe.py [--fields 148] [--niter 50] [--nsteps 10]

F fields of 64 x 64 pixels, PSF cut at r = 12 (compact tables), about 150 start stars, N_max = 200, P_move = [0.4, 0.3,
0.3].  Kernel times are CUDA events of the launch; star-steps count N_l x the leapfrog steps iteration l actually ran (two
legs for an executed jump, none for a refused one).  A refusal is read from N alone (a death with no star, a merge with
fewer than two, a birth or split past N_max); a merge refused because every pair weight is zero cannot be told from a
rejection in the chains and is counted as run (it needs every pair of stars within 1e-6 of equal flux or so far apart
that the Gaussian kernel underflows).  Prints one JSON line with the card's name and power limit."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)

import stellar_oracle as so  # noqa: E402
from hmc_stellar_toy_model_b200 import RHMCContext  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fields", type=int, default=148)
    ap.add_argument("--niter", type=int, default=50)
    ap.add_argument("--nsteps", type=int, default=10)
    a = ap.parse_args()
    F, R, N0, NMAX = a.fields, 64, 150, 200
    S = so.Setup(num_rows=R, num_cols=R, g_xx=0.05, g_ff=4.0, g_ff2=4.0, use_prior=True, alpha=2.0)
    fmin, fmax = S.mag2flux_converter(20.0), S.mag2flux_converter(15.0)
    S.fmin, S.fmax = fmin, fmax
    vpc = float(S.prior_const())
    rng = np.random.RandomState(3)
    q = np.zeros((F, 3 * NMAX))
    D = np.zeros((F, R, R))
    for f in range(F):
        t = np.stack([so.pow_law_sample(2.0, fmin, fmax, rng.random_sample(N0)), rng.uniform(1, R - 1, N0),
                      rng.uniform(1, R - 1, N0)], axis=1)
        q[f, :3 * N0] = t.ravel()
        D[f] = rng.poisson(so.model_image(S, t.ravel()))
    kw = dict(psf_fwhm_pix=S.PSF_FWHM_pix, B_count=S.B_count, f_lim=S.f_lim, f_low=S.mag2flux_converter(S.mB + 2), g0=S.g0,
              g1=S.g1, g2=S.g2, g_xx=S.g_xx, g_ff=S.g_ff, use_prior=True, alpha=2.0, V_prior_const=vpc)
    P_move = [0.4, 0.3, 0.3]
    run_kw = dict(nstars=[N0] * F, f_pos=True, g_ff2=4.0, seed=11)
    rj_kw = dict(P_move=P_move, fmin=fmin, fmax=fmax, K_split=1.0, beta_a=2.0, beta_b=2.0)
    dt = 5e-3
    with RHMCContext(n_fields=F, num_rows=R, num_cols=R, max_stars=NMAX, patch_radius=12, **kw) as ctx:
        ctx.set_data(D)
        plan = ctx.launch_plan()
        ctx.run_rj(q, 2, 2, dt, **rj_kw, **run_kw)  # warm-up
        r = ctx.run_rj(q, a.niter, a.nsteps, dt, **rj_kw, **run_kw)
        ms_rj = r.kernel_ms
        ctx.run(q, 2, 2, dt, **run_kw)
        r0 = ctx.run(q, a.niter, a.nsteps, dt, **run_kw)
        ms_0 = r0.kernel_ms
    L = a.niter + 1
    jumps = int(np.sum(r.move_chain > 0))
    refused = 0
    star_steps = 0
    for f in range(F):
        for l in range(L):
            n = int(r.N_chain[f, l])
            if r.move_chain[f, l] == 0:
                star_steps += n * a.nsteps
            else:
                grow = r.move_chain[f, l] in (1, 3)
                n_after = n + 1 if grow else n - 1
                ok = not ((grow and n + 1 > NMAX) or (r.move_chain[f, l] == 2 and n == 0) or (r.move_chain[f, l] == 4 and n < 2))
                refused += 0 if ok else 1
                star_steps += (n + n_after) * a.nsteps if ok else 0
    # the drop-in's host proposals on one field (one launch per leg, V / H / T calls around the proposal)
    from hmc_stellar_toy_model_b200.sampler_RHMC import multi_gym

    gym = multi_gym(dt=0.0, Nsteps=0, g_xx=0.05, g_ff=4.0, g_ff2=4.0)
    gym.num_rows = gym.num_cols = R
    gym.fmin, gym.fmax, gym.use_prior, gym.alpha, gym.V_prior_const = fmin, fmax, True, 2.0, vpc
    gym.K_split, gym.beta_a, gym.beta_b = 1.0, 2.0, 2.0
    gym.D = D[0]
    q_mag = q[0, :3 * N0].reshape(-1, 3).copy()
    q_mag[:, 0] = gym.flux2mag_converter(q_mag[:, 0])
    np.random.seed(5)
    niter_host = 10
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        gym.run_RHMC(q_mag, f_pos=True, Niter=niter_host, Nsteps=a.nsteps, dt=dt, P_move=P_move, N_max=NMAX)
    host_s = time.perf_counter() - t0
    print(json.dumps(dict(
        card=card(), fields=F, rows=R, start_stars=N0, N_max=NMAX, niter=a.niter, nsteps=a.nsteps, P_move=P_move,
        compact_tables=plan["compact_tables"], threads=plan["threads"],
        rj_kernel_ms=round(ms_rj, 3), rj_iterations_per_s=round(F * L / (ms_rj * 1e-3), 1),
        rj_jump_iterations_per_s=round(jumps / (ms_rj * 1e-3), 1), rj_refused_jumps=refused,
        rj_star_steps_per_s=round(star_steps / (ms_rj * 1e-3), 1), accept_rate_rj=float(np.mean(r.A_chain)),
        n_final_mean=float(np.mean(r.n_final)), move0_kernel_ms=round(ms_0, 3),
        move0_star_steps_per_s=round(F * L * N0 * a.nsteps / (ms_0 * 1e-3), 1),
        host_dropin_one_field_iterations_per_s=round((niter_host + 1) / host_s, 2))))


if __name__ == "__main__":
    main()
