#!/usr/bin/env python
"""Benchmark of the RHMC leapfrog hot path (BASELINE.json: "RHMC star-gradient evals/sec").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload all|c2|c4|c5]
                    [--dump-outputs DIR]

One unit of the metric = one star advanced by one RHMC_single_step (reference sampler_RHMC.py:522-566).
One "step" = one resident pass of the hot path over one batch of synthetic input (every chain of the batch runs
(niter+1) Metropolis iterations x nsteps generalised-leapfrog steps on the device with no host round trip).

The JSON line printed by rank 0 has the headline workload at the top level and, with the default `--workload all`, the
other BASELINE configs under "workloads":

  top level   c2  BASELINE configs[1]: 11 magnitudes x 1000 independent one-star 32x32 chains per GPU (README:92-102 of
                  the reference; RHMC-single-full-inference-test.py constants), one launch per step; weak scaling.
  workloads.c4    BASELINE configs[3]: 8192 independent crowded 64x64 fields x 204 stars (RHMC-big-sim4.py constants)
                  sharded over the N GPUs with no communication; strong scaling.
  workloads.c5    BASELINE configs[4]: ONE 8192 x 8192 field with 1e5 stars tiled in N row strips; ghost stars, the
                  fixed-point max and the energy sums cross NVLink through the library's own peer-memory exchange
                  kernels; strong scaling.  At N > 1 a small tiled chain is first checked against the untiled run through
                  the same IPC path ("parity_check").
  workloads.c5_weak   the same engine with an 8192 x 8192 strip PER GPU (N > 1 only).
  workloads.c5_perstar  configs[4] with the per-star stop rule of the implicit loops (fixed_point_mode = 1: not the reference's
                      field-wide rule; no iteration count crosses the GPUs, three kernels and one exchange per leapfrog step).

Per record: `value` (inputs resident, device time from CUDA events on the launching stream), `e2e` (public API with
pinned HOST buffers, copies inside the timed region), `roofline`, `clocks`, `gpu_launches`, and at N = 1 `cpu_baseline`
(the NumPy oracle port of the reference on the box's host cores; the Python-2 reference itself cannot travel).

--dump-outputs DIR: after the timed steps of the headline record, rank 0 writes what the timed path computed in its last
step as DIR/<name>.npy (see dump_outputs), so that two builds run with the same arguments -- hence the same inputs and
seeds -- can be compared output for output.  With N > 1 GPUs that is rank 0's share of the work only.  DIR must lie
outside the repository: bench.py writes nothing inside it.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "RHMC star-gradient evals/sec (leapfrog steps x stars)"
UNIT = "star-steps/s"
MAGS = [15, 16, 17, 18, 19, 20, 21, 21.5, 21.6, 21.7, 21.75]  # reference README:98
# per-core speed of the oracle port against the py3-shimmed reference itself, both timed in the build container on the
# headline workload (the reference cannot travel to the GPU box): the port is the faster one, so the CPU arm is conservative
PORT_VS_REFERENCE = {"port_star_steps_per_s_per_core": 2170.0, "reference_star_steps_per_s_per_core": 1565.0, "ratio": 1.39}


# ----------------------------------------------------------------------------------------------- workloads
def exp_constants():
    """default_exp_setup / compute_factors of the reference (sampler_RHMC.py:161-201): the frozen constants."""
    flux_to_count = 1.0 / (0.00546689 * 4.62)
    B = 10 ** (0.4 * (22.5 - 23)) * flux_to_count
    return dict(flux_to_count=flux_to_count, B_count=B, f_lim=B, f_low=10 ** (0.4 * (22.5 - 25)) * flux_to_count,
                psf_fwhm_pix=1.4 / 0.4, g0=0.035997054345069765, g1=0.4523523265306124, g2=0.008141675878296745)


def psf_image(R, C, x, y, fwhm):
    sigma = fwhm / 2.354
    ci = np.arange(0.5, R)[:, None]
    cj = np.arange(0.5, C)[None, :]
    return np.exp(-((ci - x) ** 2 + (cj - y) ** 2) / (2 * sigma**2)) / (2 * np.pi * sigma**2)


def workload_c2(chains_per_mag, seed):
    """One star per 32x32 field, truth at the centre, model start = truth."""
    k = exp_constants()
    R = C = 32
    rng = np.random.RandomState(seed)
    F = chains_per_mag * len(MAGS)
    psf = psf_image(R, C, 16.0, 16.0, k["psf_fwhm_pix"])
    fl = np.repeat([10 ** (0.4 * (22.5 - m)) * k["flux_to_count"] for m in MAGS], chains_per_mag)
    D = rng.poisson(k["B_count"] + fl[:, None, None] * psf[None]).astype(np.float64)
    q0 = np.stack([fl, np.full(F, 16.0), np.full(F, 16.0)], axis=1)
    cfg = dict(n_fields=F, num_rows=R, num_cols=C, max_stars=1, g_xx=1.0, g_ff=1.0, use_prior=False,
               **{n: k[n] for n in ("psf_fwhm_pix", "B_count", "f_lim", "f_low", "g0", "g1", "g2")})
    run = dict(nsteps=10, dt=0.2, g_ff2=1.0, delta=1e-6, counter_max=1000, f_pos=True)
    flops_per_unit = 9 * R * C + 2 * R * C  # SURVEY 8d: F = 9 P^2 + 2 A with P^2 = A = R*C (full-image PSF)
    # pixels the kernel actually visits for a star at the image centre: rows with |i + .5 - x| <= wcut (ex_i >= 2^-46)
    # times the 24-column window of the one-star kernel (chain_kernels.cu: use_column_window)
    sigma = k["psf_fwhm_pix"] / 2.354
    wcut = np.sqrt(46 * np.log(2.0) * 2.0) * sigma
    rows_kept = int(min(R, np.floor(15.5 + wcut) + 1) - max(0, np.ceil(15.5 - wcut)))
    cols_kept = 24 if 144.0 / (2 * sigma**2) >= 46 * np.log(2.0) else C
    flops_executed = 9 * rows_kept * cols_kept + 2 * R * C
    return dict(name="c2_one_star_32x32", D=D, q0=q0, cfg=cfg, run=run, nstars=1, flops_per_unit=flops_per_unit,
                flops_executed_per_unit=flops_executed,
                desc="%d mags x %d one-star 32x32 chains" % (len(MAGS), chains_per_mag))


def c4_truth(n_fields, seed, nstars=204, size=64):
    """Truth and start state of crowded fields: power-law fluxes (alpha = 2) in mag [15, 20], positions U(1, size-1),
    start = truth with f x 1.05 and positions jittered by 0.1 px (SURVEY 8d, RHMC-big-sim4.py)."""
    k = exp_constants()
    rng = np.random.RandomState(seed)
    alpha = 2.0
    fmin = 10 ** (0.4 * (22.5 - 20)) * k["flux_to_count"]
    fmax = 10 ** (0.4 * (22.5 - 15)) * k["flux_to_count"]
    u = rng.random_sample((n_fields, nstars))
    fl = np.exp(np.log(fmin ** (1 - alpha) + u * (fmax ** (1 - alpha) - fmin ** (1 - alpha))) / (1 - alpha))
    x = rng.random_sample((n_fields, nstars)) * (size - 2.0) + 1.0
    y = rng.random_sample((n_fields, nstars)) * (size - 2.0) + 1.0
    q_true = np.stack([fl, x, y], axis=2).reshape(n_fields, 3 * nstars)
    q0 = np.stack([fl * 1.05, x + 0.1 * rng.randn(n_fields, nstars), y + 0.1 * rng.randn(n_fields, nstars)],
                  axis=2).reshape(n_fields, 3 * nstars)
    vpc = np.log(size * size) - np.log((1 - alpha) / (fmax ** (1 - alpha) - fmin ** (1 - alpha)))
    return k, q_true, q0, alpha, float(vpc)


def workload_c4(n_fields, seed, nstars=204, size=64, host_data=True):
    """Crowded 64x64 fields, 0.05 stars/px, RHMC-big-sim4.py constants (g_xx=.05, g_ff=4, g_ff2=4, dt=5e-2).
    host_data=False leaves D to the device-side mock-data generator (srhmc_gen_mock_data)."""
    k, q_true, q0, alpha, vpc = c4_truth(n_fields, seed, nstars, size)
    D = None
    if host_data:
        rng = np.random.RandomState(seed + 1)
        sigma = k["psf_fwhm_pix"] / 2.354
        ci = np.arange(0.5, size)
        D = np.empty((n_fields, size, size))
        for f in range(n_fields):
            fl, x, y = q_true[f, 0::3], q_true[f, 1::3], q_true[f, 2::3]
            ex = np.exp(-((ci[None, :] - x[:, None]) ** 2) / (2 * sigma**2))
            ey = np.exp(-((ci[None, :] - y[:, None]) ** 2) / (2 * sigma**2)) / (2 * np.pi * sigma**2)
            D[f] = rng.poisson(k["B_count"] + np.einsum("k,ki,kj->ij", fl, ex, ey))
    cfg = dict(n_fields=n_fields, num_rows=size, num_cols=size, max_stars=nstars, g_xx=0.05, g_ff=4.0, use_prior=True,
               alpha=alpha, V_prior_const=vpc, patch_radius=12,
               **{n: k[n] for n in ("psf_fwhm_pix", "B_count", "f_lim", "f_low", "g0", "g1", "g2")})
    run = dict(nsteps=10, dt=5e-2, g_ff2=4.0, delta=1e-6, counter_max=1000, f_pos=True)
    flops_per_unit = 9 * 625 + 2 * (size * size / nstars)
    return dict(name="c4_crowded_%dx%d_%dstars" % (size, size, nstars), D=D, q0=q0, q_true=q_true, cfg=cfg, run=run,
                nstars=nstars, flops_per_unit=flops_per_unit, flops_executed_per_unit=flops_per_unit,
                desc="%d crowded %dx%d fields x %d stars" % (n_fields, size, size, nstars))


def c5_truth(rows, cols, nstars, seed):
    """Star list of one large crowded field (BASELINE configs[4] shape: 1.49e-3 stars/px, flux power law alpha = 2 in
    mag [15, 20], prior on, repulsion off).  Every rank calls this with the same seed and gets the same list."""
    k = exp_constants()
    rng = np.random.RandomState(seed)
    alpha = 2.0
    fmin = 10 ** (0.4 * (22.5 - 20)) * k["flux_to_count"]
    fmax = 10 ** (0.4 * (22.5 - 15)) * k["flux_to_count"]
    u = rng.random_sample(nstars)
    fl = np.exp(np.log(fmin ** (1 - alpha) + u * (fmax ** (1 - alpha) - fmin ** (1 - alpha))) / (1 - alpha))
    x = rng.random_sample(nstars) * (rows - 2.0) + 1.0
    y = rng.random_sample(nstars) * (cols - 2.0) + 1.0
    q_true = np.stack([fl, x, y], axis=1)
    q0 = np.stack([fl * 1.05, x + 0.1 * rng.randn(nstars), y + 0.1 * rng.randn(nstars)], axis=1)
    vpc = np.log(float(rows) * cols) - np.log((1 - alpha) / (fmax ** (1 - alpha) - fmin ** (1 - alpha)))
    consts = dict(g_xx=0.05, g_ff=4.0, use_prior=True, alpha=alpha, V_prior_const=float(vpc),
                  **{n: k[n] for n in ("psf_fwhm_pix", "B_count", "f_lim", "f_low", "g0", "g1", "g2")})
    run = dict(nsteps=10, dt=5e-2, g_ff2=4.0, delta=1e-6, counter_max=1000, f_pos=True)
    return dict(q_true=q_true, q0=q0, consts=consts, run=run)


# ----------------------------------------------------------------------------------------------- CPU arm (oracle port)
def _cpu_worker(task):
    """One oracle chain (c2, c4) or a batch of patch-limited gradient evaluations (c5) on one host core.
    Returns (units, seconds)."""
    import stellar_oracle as so  # oracle/ is the checker and, here only, the CPU baseline

    wl_name, seed, niter = task
    if wl_name.startswith("c5"):
        # patch-limited restatement on a 768 x 768 crop at the configs[4] density: one gradient evaluation per unit
        # (the true reference renders a full 8192^2 PSF per star and cannot run this configuration at all)
        size, nst = 768, 879
        t = c5_truth(size, size, nst, seed)
        S = so.Setup(num_rows=size, num_cols=size, g_xx=0.05, g_ff=4.0, g_ff2=4.0, use_prior=True, alpha=2.0,
                     V_prior_const=t["consts"]["V_prior_const"])
        k = exp_constants()
        sigma = k["psf_fwhm_pix"] / 2.354
        lam = np.full((size, size), k["B_count"])
        for f, x, y in t["q_true"]:
            i0, i1 = max(0, int(x) - 12), min(size - 1, int(x) + 12)
            j0, j1 = max(0, int(y) - 12), min(size - 1, int(y) + 12)
            ex = np.exp(-((np.arange(i0, i1 + 1) + 0.5 - x) ** 2) / (2 * sigma**2))
            ey = np.exp(-((np.arange(j0, j1 + 1) + 0.5 - y) ** 2) / (2 * sigma**2)) / (2 * np.pi * sigma**2)
            lam[i0:i1 + 1, j0:j1 + 1] += f * ex[:, None] * ey[None, :]
        D = np.random.RandomState(seed).poisson(lam).astype(float)
        t0 = time.perf_counter()
        for _ in range(niter):
            so.patch_eval(S, D, t["q0"], rad=12)
        return niter * nst, time.perf_counter() - t0
    wl = workload_c2(1, seed) if wl_name.startswith("c2") else workload_c4(1, seed)
    idx = seed % wl["D"].shape[0]
    cfg, run = wl["cfg"], wl["run"]
    S = so.Setup(num_rows=cfg["num_rows"], num_cols=cfg["num_cols"], g_xx=cfg["g_xx"], g_ff=cfg["g_ff"],
                 g_ff2=run["g_ff2"], use_prior=cfg.get("use_prior", False), alpha=cfg.get("alpha", 2.0),
                 V_prior_const=cfg.get("V_prior_const", 0.0), D=wl["D"][idx])
    rng = np.random.RandomState(seed + 17)
    d = wl["q0"].shape[1]
    normals = rng.randn(niter + 1, d)
    lnu = np.log(rng.random_sample(niter + 1))
    t0 = time.perf_counter()
    so.run_rhmc(S, wl["q0"][idx], normals, lnu, niter, run["nsteps"], run["dt"], f_pos=True, delta=run["delta"],
                counter_max=run["counter_max"])
    return (niter + 1) * run["nsteps"] * wl["nstars"], time.perf_counter() - t0


def cpu_arm(wl_name, niter, cores, rounds=1):
    """All host cores, one independent chain per process.  Returns (units/s, wall seconds, units)."""
    ctx = mp.get_context("spawn")
    tasks = [(wl_name, 1000 + i, niter) for i in range(cores * rounds)]
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(wl_name, 1, 1)] * cores)  # start-up (imports) outside the timed region
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, tasks, chunksize=1)
        wall = time.perf_counter() - t0
    units = sum(r[0] for r in res)
    return units / wall, wall, units


def cpu_niter_for(wl_name, target_seconds=12.0):
    # reference speed measured at survey time: ~2.7k star-steps/s/core (1 star), ~2.1k (204 stars 64x64); the
    # patch-limited port does ~10k star-gradients/s/core on the large-field crop
    if wl_name.startswith("c2"):
        return max(20, int(target_seconds * 2500 / 10))
    if wl_name.startswith("c5"):
        return max(2, int(target_seconds * 10000 / 879))
    return max(1, int(target_seconds * 2000 / (10 * 204)))


def cpu_baseline_record(wl_name, target_seconds):
    cores = os.cpu_count() or 1
    niter = cpu_niter_for(wl_name, target_seconds)
    v, wall, units = cpu_arm(wl_name, niter, cores)
    if wl_name.startswith("c5"):
        sample = ("%d processes x %d gradient evaluations of a 768x768 crop (879 stars, 25x25 patches) of the same field "
                  "density, %.1f s wall; patch-limited NumPy restatement (oracle.patch_eval), gradient only -- the "
                  "reference itself renders a full-image PSF per star and cannot run 8192^2" % (cores, niter, wall))
    else:
        sample = ("%d processes x 1 chain x %d iterations x 10 steps of the same workload (%.1f s wall, NumPy oracle "
                  "port of the reference)" % (cores, niter + 1, wall))
    return {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
            "port_vs_reference": PORT_VS_REFERENCE}


# ----------------------------------------------------------------------------------------------- GPU helpers
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        time.sleep(0.3)   # nvidia-smi needs ~0.2 s before its first line: start it ahead of the timed region, not inside it
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, reasons, power = [], [], set(), []
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "power_w_max": max(power), "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 * 10**6   # array data written by --dump-outputs (plus one 128-byte .npy header per file)


def dump_outputs(path, rows, whole=None):
    """Write each array as <path>/<name>.npy: flags (uint8) as float32, everything else as float64.
    `rows` maps names to arrays sharing a leading axis (chains, fields or stars); when they would exceed DUMP_LIMIT_BYTES,
    a fixed seeded sample of that axis is kept in increasing order.  sample_index.npy holds the kept indices.
    `whole` maps names to small arrays written in full."""
    def conv(a):
        a = np.asarray(a)
        return a.astype(np.float32) if a.dtype in (np.uint8, np.bool_) else a.astype(np.float64)

    out = {k: conv(v) for k, v in (whole or {}).items()}
    n = len(next(iter(rows.values())))
    per_row = 8 + sum(conv(v[:1]).nbytes for v in rows.values())
    keep = min(n, max(0, DUMP_LIMIT_BYTES - sum(v.nbytes for v in out.values())) // per_row)
    idx = np.arange(n) if keep == n else np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
    out["sample_index"] = conv(idx)
    out.update({k: conv(np.asarray(v)[idx]) for k, v in rows.items()})
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def traffic_from_profile(wl_name):
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(path):
        with open(path) as fh:
            return json.load(fh).get(wl_name)
    return None


def bind_to_gpu_numa(local):
    """Best effort: run this rank's host threads (and therefore first-touch its pinned buffers) on the CPUs local to its
    GPU, so that eight ranks' device-to-host chain copies do not all land on one NUMA node."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out   # 00000000:1b:00.0 -> 0000:1b:00.0
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as fh:
            spec = fh.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return spec
    except Exception:
        pass
    return None


class Env:
    """Rank plumbing: torch only owns the process group, the current stream and the timing events."""

    def __init__(self):
        import torch

        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the RHMC path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.numa = bind_to_gpu_numa(self.local) if self.world > 1 else None
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        self._peak = {}

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def min_over_ranks(self, value):
        t = self.torch.tensor([float(value)], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return float(t.item())

    def fma_peak(self, prec):
        if prec not in self._peak:
            from hmc_stellar_toy_model_b200 import _capi

            self._peak[prec] = _capi.measure_fma_peak(self.local, prec)[0]
        return self._peak[prec]

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------- independent chains / fields
def bench_chains(env, wl, *, niter, steps, warmup, e2e_steps, want, precision, scaling, seed_base, field_id_base=0,
                 device_data_seed=None, parallelism="", min_seconds=0.0, dump_dir=None):
    """C2 / C4: F independent fields per rank in one RHMCContext, one resident launch per step.
    min_seconds (sub-records only): lengthen the timed region to at least this, so that the clock sampler (50 ms period) sees
    it -- `steps` in the record is the number actually timed.
    dump_dir: write the chains, final states and acceptance rates of the last timed launch there (dump_outputs)."""
    torch = env.torch
    from hmc_stellar_toy_model_b200 import RHMCContext, _capi

    rank, world, local = env.rank, env.world, env.local
    F, S = wl["q0"].shape
    L = niter + 1
    units_per_step = F * L * wl["run"]["nsteps"] * wl["nstars"]
    ctx = RHMCContext(device=local, precision=precision, **wl["cfg"])
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    R, C = wl["cfg"]["num_rows"], wl["cfg"]["num_cols"]

    # pinned host buffers for the e2e path
    pin_D = _capi.PinnedBuffer((F, R, C))
    if wl["D"] is not None:
        pin_D.array[...] = wl["D"]
    else:  # device-side mock data (counter-based Philox Poisson), copied back once so the e2e arm has HOST images
        pin_D.array[...] = ctx.gen_mock_data(wl["q_true"], seed=device_data_seed, field_id_base=field_id_base)
    pin_q0 = _capi.PinnedBuffer(wl["q0"].shape)
    pin_q0.array[...] = wl["q0"]
    shapes = {"q": ("q_chain", (F, L, S), np.float64), "p": ("p_chain", (F, L, S), np.float64),
              "E": ("E_chain", (F, L), np.float64), "V": ("V_chain", (F, L), np.float64),
              "T": ("T_chain", (F, L), np.float64), "A": ("A_chain", (F, L), np.uint8)}
    outs = {shapes[k][0]: _capi.PinnedBuffer(shapes[k][1], shapes[k][2]) for k in want}
    outs["q_final"] = _capi.PinnedBuffer((F, S))
    outs["accept_rate"] = _capi.PinnedBuffer((F,))
    out_arrays = {k: v.array for k, v in outs.items()}

    ctx.set_data(pin_D.array)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def make_args(seed):
        a, keep = ctx.make_run_args(pin_q0.array, niter, seed=seed + 104729 * rank + seed_base, out=out_arrays, want=want,
                                    field_id_base=field_id_base, **wl["run"])
        return a, keep

    # ---- value: inputs resident, kernel-only device time
    a, keep = make_args(1)
    ctx.run_upload(a)
    for w in range(warmup):
        a, keep = make_args(100 + w)
        ctx.run_launch(a)
    if min_seconds > 0 and warmup > 0:
        t_step = env.max_over_ranks([ctx.last_kernel_ms()])[0]
        steps = int(max(steps, min(64, np.ceil(1e3 * min_seconds / max(t_step, 1e-3)))))
    env.barrier()
    sampler = ClockSampler(local).start() if rank == 0 else None
    launches0 = ctx.launch_count
    kernel_ms = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.barrier()
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    for s in range(steps):
        flush.zero_()  # L2 flush between timed iterations (outside the kernel's own events)
        a, keep = make_args(1000 + s)
        ctx.run_launch(a)
        kernel_ms.append(ctx.last_kernel_ms())
    ev1.record(stream)
    env.barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = ctx.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    total_ms = float(sum(kernel_ms))
    region_ms = ev0.elapsed_time(ev1)
    if dump_dir is not None and rank == 0:
        ctx.run_download(a)   # the last timed launch's results, copied back after the timed region
        dump_outputs(dump_dir, out_arrays)

    # ---- e2e: public API, host buffers, copies inside the timed region
    e2e_steps = max(1, min(steps, e2e_steps))
    ctx.set_data(pin_D.array)
    a, keep = make_args(5)
    ctx.run_prepared(a)
    env.barrier()
    t0 = time.perf_counter()
    acc = None
    for s in range(e2e_steps):
        ctx.set_data(pin_D.array)              # H2D images
        a, keep = make_args(2000 + s)
        ctx.run_prepared(a)                    # H2D start state, launch, D2H chains, sync
        acc = float(out_arrays["accept_rate"].mean())
    env.barrier()
    t_e2e = time.perf_counter() - t0
    h2d = pin_D.nbytes + pin_q0.nbytes
    d2h = sum(v.nbytes for v in outs.values())

    # ---- e2e, summary return: the chains stay on the device and only their statistics come back (split-chain R-hat and
    #      n_eff per magnitude group through srhmc_run_stats, final state, acceptance rate) -- one-star batches only
    summary = None
    if wl["nstars"] == 1 and "q" in want:
        groups = len(MAGS) if F % len(MAGS) == 0 else 1
        small = {k: out_arrays[k] for k in ("q_chain", "q_final", "accept_rate")}
        Rhat = None
        env.barrier()
        ts = time.perf_counter()
        for s in range(e2e_steps):
            ctx.set_data(pin_D.array)          # H2D images
            a2, keep2 = ctx.make_run_args(pin_q0.array, niter, seed=3000 + s + seed_base, want=("q",), out=small,
                                          field_id_base=field_id_base, **wl["run"])
            ctx.run_upload(a2)                 # H2D start state
            ctx.run_launch(a2)                 # q_chain is recorded on the device ...
            Rhat, neff = ctx.run_stats(n_groups=groups)
            a2.q_chain = None                  # ... and stays there: only q_final + accept_rate are copied back
            ctx.run_download(a2)
        env.barrier()
        t_sum = time.perf_counter() - ts
        summary = {"t": t_sum, "d2h": int(outs["q_final"].nbytes + outs["accept_rate"].nbytes + 2 * Rhat.nbytes),
                   "rhat_max": float(np.nanmax(Rhat))}

    red = env.max_over_ranks([total_ms, t_e2e, region_ms, summary["t"] if summary else 0.0])
    total_ms, t_e2e, region_ms, t_sum = red
    rec = None
    if rank == 0:
        peak_tf = env.fma_peak(precision)
        ms_per_step = total_ms / steps
        value = world * units_per_step * steps / (total_ms * 1e-3)
        e2e_value = world * units_per_step * e2e_steps / t_e2e
        achieved_tf = wl["flops_per_unit"] * units_per_step / (ms_per_step * 1e-3) / 1e12
        peaks, peak_src = measured_peaks()
        chain_bytes = d2h + pin_D.nbytes * (precision / 64.0)
        frac_exec = achieved_tf * wl["flops_executed_per_unit"] / wl["flops_per_unit"] / peak_tf
        rec = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f64" if precision == 64 else "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "description": wl["desc"], "fields_per_gpu": F, "stars_per_field": wl["nstars"],
                       "niter": niter, "nsteps": wl["run"]["nsteps"], "dt": wl["run"]["dt"],
                       "units_per_step_per_gpu": units_per_step, "rng": "device Philox4x32-10",
                       "l2": "256 MB flush write between timed iterations; kernel is shared-memory resident",
                       "parallelism": parallelism},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "ms_per_step": 1e3 * t_e2e / e2e_steps,
                    "returns": "every chain array requested (%s) + final state + acceptance rate" % ",".join(want)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "fp64" if precision == 64 else "fp32",
                         "achieved": achieved_tf * wl["flops_executed_per_unit"] / wl["flops_per_unit"], "peak": peak_tf,
                         "unit": "TFLOP/s", "frac": frac_exec,
                         "counts": "flops of the pixels the kernel visits (flops_executed_per_unit); frac_full_image uses "
                                   "SURVEY 8d's full-image count, which credits pixels whose PSF weight is below 2^-46",
                         "peak_source": "FP%d FMA-chain microbenchmark on this GPU (srhmc_measure_fma_peak, "
                                        "profiles/fma_peak_method.md); nominal %s" % (precision, "37.2" if precision == 64 else "74.4"),
                         "flops_per_unit": wl["flops_per_unit"],
                         "flops_executed_per_unit": wl["flops_executed_per_unit"],
                         "achieved_full_image": achieved_tf, "frac_full_image": achieved_tf / peak_tf,
                         "frac_executed": frac_exec,
                         "traffic": traffic_from_profile(wl["name"]),
                         "note": "CUDA-core pipe bound: images stay in shared memory for the whole launch, "
                                 "no dense contraction, so neither the HBM nor the tensor roofline applies"},
            "roofline_hbm": {"bound": "hbm", "achieved": chain_bytes / (ms_per_step * 1e-3) / 1e9,
                             "peak": peaks["hbm_gbs"], "unit": "GB/s", "peak_source": peak_src,
                             "frac": chain_bytes / (ms_per_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                             "bytes_per_launch": int(chain_bytes)},
            "accept_rate": acc,
            "timed_region_ms": region_ms, "wall_s": t_wall,
        }
        if summary:
            rec["e2e_summary"] = {"value": world * units_per_step * e2e_steps / t_sum, "unit": UNIT,
                                  "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": summary["d2h"],
                                  "steps": e2e_steps, "ms_per_step": 1e3 * t_sum / e2e_steps, "rhat_max": summary["rhat_max"],
                                  "returns": "split-chain R-hat and n_eff per magnitude group computed on the device from "
                                             "the resident chains (srhmc_run_stats), final state, acceptance rate"}
        if env.numa:
            rec["config"]["host_affinity"] = "rank bound to the CPUs local to its GPU (%s)" % env.numa
    for b in list(outs.values()) + [pin_D, pin_q0]:
        b.free()
    del flush
    ctx.close()
    return rec


# ----------------------------------------------------------------------------------------------- one large tiled field
def _make_strip(env, bf, rows, cols, nstars_cap, consts, halo, rad, world=None, rank=None):
    world = env.world if world is None else world
    rank = env.rank if rank is None else rank
    lo, hi = bf.strip_bounds(rows, world)[rank]
    max_ghosts = max(1024, int(4 * nstars_cap * (halo + rad + 1) / max(1, hi - lo)))
    return bf.BigFieldStrip(rows=rows, cols=cols, rank=rank, world=world, device=env.local, max_stars=nstars_cap,
                            max_ghosts=max_ghosts, patch_radius=rad, halo=halo, **consts)


def tiled_parity_check(env, stream):
    """A small field tiled over the ranks through the REAL multi-process path (IPC-mapped mailboxes, the library's
    exchange kernels, graph replay) against the untiled run of the same field on this rank's GPU: same accept decisions,
    energies to 1e-10, final stars to 1e-9.  Returns "ok" or a description of the first difference."""
    from hmc_stellar_toy_model_b200 import bigfield as bf

    world = env.world
    rows, cols = 48 * world + 32, 96
    nst = int(rows * cols * 0.02)
    t = c5_truth(rows, cols, nst, 4242)
    rad, halo = 12, 20
    run = dict(t["run"], dt=2e-2, nsteps=4)
    niter = 7
    msg = "ok"
    try:
        one = _make_strip(env, bf, rows, cols, nst, t["consts"], halo, rad, world=1, rank=0)
        one.set_stream(stream.cuda_stream)
        Dfull = one.gen_mock_data(t["q_true"], seed=11, return_data=True)
        one.set_stars(t["q0"])
        a = bf.BigFieldRHMC([one]).run(niter, seed=5, **run)
        qa = one.get_stars()[0]
        ids_all = one.ids
        one.close()
        strip = _make_strip(env, bf, rows, cols, nst, t["consts"], halo, rad)
        strip.set_stream(stream.cuda_stream)
        Dloc = strip.gen_mock_data(t["q_true"], seed=11, return_data=True)   # per-rank generation: halo rows must agree
        if not np.array_equal(Dloc, Dfull[strip.row0:strip.row0 + strip.nrows]):
            msg = "device mock data of the strip differ from the untiled image"
        strip.set_stars(t["q0"])
        eng = bf.BigFieldRHMC([strip], bf.PeerComm([strip], env.dist))
        b = eng.run(niter, seed=5, **run)
        qb = strip.get_stars()[0]
        back = np.empty(int(ids_all.max()) + 1 if len(ids_all) else 0, dtype=np.int64)
        back[ids_all] = np.arange(len(ids_all))
        mine = qa[back[strip.ids]]
        if not np.array_equal(a["A_chain"], b["A_chain"]):
            msg = "accept decisions differ: untiled %s tiled %s" % (a["A_chain"].tolist(), b["A_chain"].tolist())
        elif not a["A_chain"].any():
            msg = "degenerate check: no accepted iteration"
        elif np.max(np.abs(b["E_chain"] - a["E_chain"]) / np.abs(a["E_chain"])) > 1e-10:
            msg = "E_chain differs by %.2e" % float(np.max(np.abs(b["E_chain"] - a["E_chain"]) / np.abs(a["E_chain"])))
        elif len(mine) and np.max(np.abs(qb - mine) / np.maximum(np.abs(mine), 1e-300)) > 1e-9:
            msg = "final stars differ by %.2e" % float(np.max(np.abs(qb - mine) / np.maximum(np.abs(mine), 1e-300)))
        strip.close()
    except Exception as e:  # reported, never fatal for the timing that follows
        msg = "check raised %s: %s" % (type(e).__name__, e)
    ok = env.min_over_ranks(1.0 if msg == "ok" else 0.0)
    if msg == "ok" and ok < 1.0:
        msg = "another rank reported a mismatch"
    return msg


def bench_bigfield(env, *, rows, cols, nstars, weak, niter, steps, warmup, e2e_steps, comm_kind, with_parity, precision=64,
                   replicas=False, label="c5_tiled_field", dt=None, fixed_point_mode=0, min_seconds=0.0, dump_dir=None):
    """C5: ONE large field, row strips over the ranks (strong), or one rows x cols strip per rank (weak).
    replicas=True (C3): every rank runs its own copy of the whole field, no communication.
    dump_dir: write the chain scalars of the last timed run and the final (q, p, dV/dq) of this rank's stars, in global
    star-id order, there (dump_outputs)."""
    torch = env.torch
    from hmc_stellar_toy_model_b200 import _capi
    from hmc_stellar_toy_model_b200 import bigfield as bf

    rank, world = env.rank, env.world
    n_ranks = world
    if replicas:
        rank, world, weak = 0, 1, False
    rows_g = rows * (world if weak else 1)
    nst_g = int(nstars * (world if weak else 1))
    rad, halo = 12, 24
    stream = torch.cuda.Stream()   # kernels, exchange kernels and the timing events all ride on this stream
    torch.cuda.set_stream(stream)
    parity = None
    if with_parity and world > 1 and comm_kind == "peer":
        parity = tiled_parity_check(env, stream)
    t = c5_truth(rows_g, cols, nst_g, 77)
    run = dict(t["run"], dt=dt) if dt else t["run"]
    strip = _make_strip(env, bf, rows_g, cols, nst_g, t["consts"], halo, rad, world=world, rank=rank)
    strip.set_stream(stream.cuda_stream)
    if precision == 32:
        strip.set_precision(32)
    if world == 1:
        comm = bf.NoComm()
    elif comm_kind == "nccl":
        comm = bf.TorchDistComm(env.dist)   # NCCL collectives issued by the caller between the phases (eager launches)
    else:
        comm = bf.PeerComm([strip], env.dist)  # the library's own exchange kernels over NVLink peer memory; graph replay
    eng = bf.BigFieldRHMC([strip], comm, fixed_point_mode=fixed_point_mode)

    # data: generated on the device (srhmc_big_mock_data: tile-kernel render + counter-based Philox Poisson; halo rows of
    # neighbouring strips agree bit for bit), read back once into pinned memory for the e2e arm
    pin_D = _capi.PinnedBuffer((strip.nrows, cols))
    pin_D.array[...] = strip.gen_mock_data(t["q_true"], seed=77, return_data=True)
    units = nst_g * (niter + 1) * run["nsteps"] * (n_ranks if replicas else 1)
    t_step = 0.0
    for w in range(warmup):
        strip.set_stars(t["q0"])
        torch.cuda.synchronize()
        t0w = time.perf_counter()
        eng.run(niter, seed=1000, **run)
        torch.cuda.synchronize()
        t_step = time.perf_counter() - t0w
    if min_seconds > 0 and warmup > 0:   # sub-records: a timed region the 50 ms clock sampler can see
        t_step = env.max_over_ranks([t_step])[0]
        steps = int(max(steps, min(400, np.ceil(min_seconds / max(t_step, 1e-6)))))
    env.barrier()
    sampler = ClockSampler(env.local).start() if env.rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    acc = 0.0
    launches = 0
    for s in range(steps):
        strip.set_stars(t["q0"])
        l0 = strip.launch_count
        env.barrier()
        ev0.record(stream)
        out = eng.run(niter, seed=1000, **run)  # same launch parameters: the captured iteration graph is reused
        ev1.record(stream)
        torch.cuda.synchronize()
        times.append(ev0.elapsed_time(ev1))
        launches += strip.launch_count - l0 + eng.replayed_launches
        acc = out["accept_rate"]
    clocks = sampler.stop() if sampler else None
    if dump_dir is not None and env.rank == 0:
        q, p, g = strip.get_stars()
        order = np.argsort(strip.ids)
        dump_outputs(dump_dir, {"star_id": strip.ids[order], "q_final": q[order], "p_final": p[order], "grad_final": g[order]},
                     {k: out[k] for k in ("E_chain", "V_chain", "T_chain", "A_chain", "accept_rate")})
    # e2e: host buffers in (data window + stars), final stars and the chain scalars out
    e2e_steps = max(1, min(steps, e2e_steps))
    t_e2e = 0.0
    for s in range(e2e_steps):
        env.barrier()
        t0 = time.perf_counter()
        strip.set_data_window(pin_D.array)
        strip.set_stars(t["q0"])
        eng.run(niter, seed=1000, **run)
        strip.get_stars()
        env.barrier()
        t_e2e += time.perf_counter() - t0
    total_ms, t_e2e = env.max_over_ranks([sum(times), t_e2e])
    rec = None
    if env.rank == 0:
        world = n_ranks
        peaks, peak_src = measured_peaks()
        ms_per_step = total_ms / steps
        value = units * steps / (total_ms * 1e-3)
        A = rows_g * cols / float(nst_g)
        # SURVEY 8d: the data strip read once per gradient + star state (FP32 build: float pixels for 9 of 10 evaluations)
        bytes_per_unit = (8.0 if precision == 64 else 4.0 + 4.0 / run["nsteps"]) * A + 96.0
        gbs = bytes_per_unit * units / world / (ms_per_step * 1e-3) / 1e9
        name = "%s_%dx%d_%dstars%s%s" % (label, rows_g, cols, nst_g, "" if precision == 64 else "_fp32",
                                         "_perstar" if fixed_point_mode else "")
        n_own = strip.n
        rec = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if (weak or replicas) else "strong",
            "vs_baseline": None, "dtype": "f64" if precision == 64 else "f32", "data": "synthetic",
            "config": {"workload": name, "rows": rows_g, "cols": cols, "stars": nst_g, "niter": niter,
                       "nsteps": run["nsteps"], "dt": run["dt"], "patch_radius": rad, "halo_rows": halo,
                       "rng": "device Philox4x32-10", "data_source": "device-side mock data (srhmc_big_mock_data)",
                       "fixed_point_mode": ("1: every star's implicit loops stop at the star's own convergence (NOT the reference's "
                                            "field-wide stop rule: per-step results within delta of it); three kernels and one "
                                            "exchange per leapfrog step" if fixed_point_mode else
                                            "0: the reference's field-wide stop rule, bit for bit"),
                       "l2": "every gradient streams this rank's %.0f MB data window from HBM (larger than the 126 MB L2 "
                             "when above it; no flush between launches)" % (pin_D.nbytes / 1e6),
                       "parallelism": ("replicas only: every one of the %d GPU(s) runs its own chain on the whole field "
                                       "(one field of this size does not shard), no communication" % world) if replicas else
                                      "row strips over %d GPU(s); per step: 1 exchange of boundary stars with the two "
                                      "neighbours, 2 max all-reduces; per iteration: 2 sum all-reduces of 8 doubles (%s)"
                                      % (world, "none: single GPU" if world == 1 else
                                         ("own kernels over NVLink peer memory, CUDA-graph replay" if comm_kind == "peer"
                                          else "NCCL via torch.distributed, eager"))},
            "clocks": clocks,
            "e2e": {"value": units * e2e_steps / t_e2e, "unit": UNIT,
                    "h2d_bytes_per_step": int(pin_D.nbytes + 32 * n_own),
                    "d2h_bytes_per_step": int(72 * n_own + 25 * (niter + 1)), "steps": e2e_steps,
                    "ms_per_step": 1e3 * t_e2e / e2e_steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                         "peak_source": peak_src, "bytes_per_unit": bytes_per_unit,
                         "traffic": traffic_from_profile(name) if world == 1 else None,
                         "note": ("the %.1f MB data image stays in the 126 MB L2, so HBM is not what bounds this field: a leapfrog "
                                  "step is a handful of dependent kernels over %d tiles (fewer CTAs than the GPU holds), i.e. "
                                  "launch- and latency-bound; the HBM figure is reported for the common denominator only"
                                  % (pin_D.nbytes / 1e6, ((rows_g + 63) // 64) * ((cols + 63) // 64))) if replicas else
                                 "per GPU, over the WHOLE leapfrog step (tile kernel + the per-star kernels + exchanges); "
                                 "algorithmic bytes = the data strip read once per gradient + star state"},
            "accept_rate": acc,
        }
        if parity is not None:
            rec["parity_check"] = parity
    pin_D.free()
    strip.close()
    torch.cuda.set_stream(torch.cuda.default_stream())
    return rec


# ----------------------------------------------------------------------------------------------- arms
def guarded(env, name, fn):
    """Run one secondary workload; an exception on any rank becomes an error record instead of ending the bench."""
    t0 = time.perf_counter()
    rec, err = None, None
    try:
        rec = fn()
    except Exception as e:
        err = "%s: %s" % (type(e).__name__, e)
        sys.stderr.write("bench.py: workload %s failed on rank %d\n%s\n" % (name, env.rank, traceback.format_exc()))
    try:
        env.torch.cuda.synchronize()
    except Exception:
        pass
    bad = -env.min_over_ranks(-1.0 if err else 0.0)
    if env.rank != 0:
        return None
    if err or bad > 0 or rec is None:
        return {"error": err or "failed on another rank", "wall_s": time.perf_counter() - t0}
    rec["wall_s_total"] = time.perf_counter() - t0
    return rec


def run_ours(args):
    env = Env()
    rank, world = env.rank, env.world
    which = args.workload
    cpu = {}
    if rank == 0 and world == 1 and not args.no_cpu:  # CPU baselines first, before the GPU is busy
        cpu["c2"] = cpu_baseline_record("c2", 12.0) if which in ("all", "c2") else None
        cpu["c4"] = cpu_baseline_record("c4", 6.0) if which in ("all", "c4") else None
        cpu["c5"] = cpu_baseline_record("c5", 6.0) if which in ("all", "c5") else None

    def c2(dump_dir=None):
        wl = workload_c2(args.chains_per_mag, 77 + rank)
        return bench_chains(env, wl, niter=args.niter, steps=args.steps, warmup=args.warmup, e2e_steps=args.e2e_steps,
                            want=("q", "p", "E", "V", "T", "A"), precision=args.precision, scaling="weak", seed_base=0,
                            parallelism="independent chains sharded across %d GPU(s), no communication" % world,
                            dump_dir=dump_dir)

    def c4(precision=None, dump_dir=None):
        total = args.fields
        per = max(1, total // world)
        wl = workload_c4(per, 5000 + rank, host_data=False)
        wl["desc"] = "%d crowded 64x64 fields x 204 stars in total, %d per GPU" % (per * world, per)
        if precision == 32:
            wl["name"] += "_fp32"
        return bench_chains(env, wl, niter=args.c4_niter, steps=args.sub_steps, warmup=3, e2e_steps=2, want=("E", "A"),
                            precision=args.precision if precision is None else precision, scaling="strong", seed_base=17,
                            field_id_base=rank * per, min_seconds=0.6 if which == "all" else 0.0,
                            device_data_seed=4, parallelism="%d independent fields split over %d GPU(s) (contiguous "
                            "blocks), no communication" % (per * world, world), dump_dir=dump_dir)

    def c5(weak, precision=None, fixed_point_mode=0, dump_dir=None):
        return bench_bigfield(env, rows=args.rows, cols=args.cols, nstars=args.stars, weak=weak, niter=args.c5_niter,
                              steps=max(10, args.sub_steps) if which == "all" else args.steps, warmup=3, e2e_steps=2,
                              comm_kind=args.comm, with_parity=not weak and precision is None and not fixed_point_mode,
                              precision=args.precision if precision is None else precision,
                              fixed_point_mode=fixed_point_mode or args.fixed_point_mode,
                              min_seconds=0.6 if which == "all" else 0.0, dump_dir=dump_dir)

    def c3(dump_dir=None):
        # BASELINE configs[2]: "RHMC-big-sim2/3/4 crowded field: hundreds to thousands of stars in one large image with the
        # full RHMC leapfrog loop" -- one 256 x 256 field at the sim4 / configs[3] density (0.05 stars per pixel: 3277 stars)
        return bench_bigfield(env, rows=256, cols=256, nstars=3277, weak=False, niter=args.c5_niter,
                              steps=max(10, args.sub_steps) if which == "all" else args.steps, warmup=3, e2e_steps=2,
                              comm_kind=args.comm, with_parity=False, precision=args.precision, replicas=True,
                              label="c3_crowded_field", min_seconds=0.6 if which == "all" else 0.0, dump_dir=dump_dir)

    dump = args.dump_outputs
    if which == "c4":
        out = c4(dump_dir=dump)
    elif which == "c3":
        out = c3(dump_dir=dump)
    elif which == "c5":
        out = c5(args.weak, dump_dir=dump)
    else:
        out = c2(dump_dir=dump)
    if rank == 0 and out is not None:
        out["cpu_baseline"] = cpu.get("c2" if which == "all" else which)
    def c2_fp32():
        wl = workload_c2(args.chains_per_mag, 77 + rank)
        wl["name"] = "c2_one_star_32x32_fp32"
        return bench_chains(env, wl, niter=args.niter, steps=args.sub_steps, warmup=3, e2e_steps=2,
                            want=("q", "p", "E", "V", "T", "A"), precision=32, scaling="weak", seed_base=0, min_seconds=0.6,
                            parallelism="independent chains sharded across %d GPU(s), no communication; FP32 pixel "
                            "arithmetic for the gradient-only evaluations, FP64 state and energies" % world)

    if which == "all":
        subs = {}
        subs["c2_fp32"] = guarded(env, "c2_fp32", c2_fp32)
        subs["c3"] = guarded(env, "c3", c3)
        subs["c4"] = guarded(env, "c4", c4)
        subs["c5"] = guarded(env, "c5", lambda: c5(False))
        subs["c5_perstar"] = guarded(env, "c5_perstar", lambda: c5(False, fixed_point_mode=1))
        if world > 1:
            subs["c5_weak"] = guarded(env, "c5_weak", lambda: c5(True))
        else:
            subs["c4_fp32"] = guarded(env, "c4_fp32", lambda: c4(32))
            subs["c5_fp32"] = guarded(env, "c5_fp32", lambda: c5(False, 32))
        if rank == 0:
            for k in ("c4", "c5"):
                if subs.get(k) is not None and "error" not in subs[k]:
                    subs[k]["cpu_baseline"] = cpu.get(k)
            out["workloads"] = subs
    if rank == 0:
        print(json.dumps(out))
        sys.stdout.flush()
    env.close()


def run_reference(args):
    """The reference's CPU implementation of the path (NumPy oracle port; the Python-2 reference itself cannot
    travel to the GPU box) on all host cores, same config/metric as the headline.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl_key = "c2" if args.workload == "all" else args.workload
    cores = os.cpu_count() or 1
    niter = max(10, cpu_niter_for(wl_key, 4.0))
    for _ in range(args.warmup):
        cpu_arm(wl_key, max(2, niter // 10), cores)
    t_total, units_total = 0.0, 0
    for _ in range(args.steps):
        v, wall, units = cpu_arm(wl_key, niter, cores)
        t_total += wall
        units_total += units
    value = units_total / t_total
    wl_name = {"c2": "c2_one_star_32x32", "c4": "c4_crowded_64x64_204stars", "c5": "c5_tiled_field_crop"}[wl_key]
    sample = "%d processes x 1 chain x %d iterations x 10 steps per step" % (cores, niter + 1)
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic",
           "config": {"workload": wl_name, "description": "%d mags x 1000 one-star 32x32 chains" % len(MAGS) if wl_key == "c2" else wl_name,
                      "stars_per_field": 1 if wl_key == "c2" else 204, "niter": niter, "nsteps": 10,
                      "dt": 0.2 if wl_key == "c2" else 5e-2, "rng": "np.random.RandomState draws injected into the oracle",
                      "sample": sample,
                      "parallelism": "%d host processes, one independent chain each" % cores},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                            "port_vs_reference": PORT_VS_REFERENCE},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "c2", "c3", "c4", "c5"],
                    help="all: the c2 headline plus c4 / c5 records under 'workloads'; c2|c4|c5: that workload alone")
    ap.add_argument("--rows", type=int, default=8192, help="c5: image rows (per GPU with --weak); BASELINE configs[4] is 8192 x 8192")
    ap.add_argument("--cols", type=int, default=8192)
    ap.add_argument("--stars", type=float, default=100000, help="c5: stars (per GPU with --weak); 1.49e-3 per pixel")
    ap.add_argument("--weak", action="store_true", help="c5 alone: grow the field with the GPU count")
    ap.add_argument("--fixed-point-mode", type=int, default=0, choices=[0, 1],
                    help="c5: 0 = the reference's field-wide stop rule (default), 1 = per-star stop rule")
    ap.add_argument("--comm", default="peer", choices=["peer", "nccl"],
                    help="c5 on several GPUs: the library's own peer-memory exchange kernels, or NCCL through torch.distributed")
    ap.add_argument("--chains-per-mag", type=int, default=1000)
    ap.add_argument("--fields", type=int, default=8192, help="c4: fields in total (BASELINE configs[3]: 8192), split over the GPUs")
    ap.add_argument("--niter", type=int, default=1000, help="c2: Metropolis iterations per chain")
    ap.add_argument("--c4-niter", type=int, default=9)
    ap.add_argument("--c5-niter", type=int, default=9)
    ap.add_argument("--sub-steps", type=int, default=3, help="timed steps of the secondary workloads under --workload all")
    ap.add_argument("--precision", type=int, default=64, choices=[64, 32])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the headline record's timed path computed in its last step as DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB: a fixed seeded sample of the chains when larger); DIR "
                         "must lie outside the repository.  With N > 1 GPUs only rank 0 writes, and only its own share: "
                         "its chains or fields (c2, c4) or the stars of its strip (c5)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "ours":
            ap.error("--dump-outputs writes the outputs of the CUDA path: use it with --impl ours")
        args.dump_outputs = os.path.realpath(args.dump_outputs)
        root = os.path.realpath(ROOT)
        if os.path.commonpath([args.dump_outputs, root]) == root:
            ap.error("--dump-outputs: %s is inside the repository; bench.py writes nothing there" % args.dump_outputs)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.workload == "c4":
            args.sub_steps = args.steps
            if args.niter != 1000:
                args.c4_niter = args.niter   # `--workload c4 --niter n` (profiling scripts)
        if args.workload == "c5" and args.niter != 1000:
            args.c5_niter = args.niter
        run_ours(args)


if __name__ == "__main__":
    main()
