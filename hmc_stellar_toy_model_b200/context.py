"""RHMCContext: numpy-in / numpy-out wrapper over the C ABI for a batch of independent fields.

The gym classes in sampler_RHMC.py / samplers.py (the reference's call surface) are built on this; it is also the
batch API the reference lacks (`Nchain == 1` everywhere upstream): F fields or chains advance in one launch.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _capi
from ._capi import Config, LsArgs, RjArgs, RunArgs, as_f64, bptr, check, dptr, iptr


@dataclass
class RunResult:
    q_chain: np.ndarray | None
    p_chain: np.ndarray | None
    E_chain: np.ndarray | None
    V_chain: np.ndarray | None
    T_chain: np.ndarray | None
    A_chain: np.ndarray | None
    q_final: np.ndarray
    accept_rate: np.ndarray
    kernel_ms: float


@dataclass
class RjRunResult(RunResult):
    """RunResult of a reversible-jump run plus its trans-dimensional record."""
    N_chain: np.ndarray = None      # [F, Ls] int32: star count at the start of each kept iteration
    move_chain: np.ndarray = None   # [F, Ls] uint8: 0 within, 1 birth, 2 death, 3 split, 4 merge
    n_final: np.ndarray = None      # [F] int32: star count after the last iteration
    overflow: np.ndarray = None     # [F] int32: first iteration whose proposal needed more than max_stars stars, or -1


RJ_DRAWS = 14  # doubles of one (field, iteration) draw record of run_rj


class RHMCContext:
    """Device context holding `n_fields` fields of `num_rows x num_cols` pixels with up to `max_stars` stars."""

    def __init__(self, *, n_fields, num_rows, num_cols, max_stars, psf_fwhm_pix, B_count, f_lim, f_low, g0, g1, g2,
                 g_xx, g_ff, use_prior=False, alpha=2.0, V_prior_const=0.0, use_Vc=False, Vc_r_pow=1.0,
                 precision=64, patch_radius=0, shared_data=False, fixed_point_mode=0, device=0,
                 enable_hessian=False):
        self._lib = _capi.load_library()
        cfg = Config(
            abi_version=_capi.ABI_VERSION, device=device, precision=precision, n_fields=n_fields, num_rows=num_rows,
            num_cols=num_cols, max_stars=max_stars, patch_radius=patch_radius, shared_data=int(bool(shared_data)),
            fixed_point_mode=fixed_point_mode, use_prior=int(bool(use_prior)), use_Vc=int(bool(use_Vc)),
            psf_fwhm_pix=psf_fwhm_pix, B_count=B_count, f_lim=f_lim, f_low=f_low, g0=g0, g1=g1, g2=g2, g_xx=g_xx,
            g_ff=g_ff, alpha=alpha, V_prior_const=V_prior_const, Vc_r_pow=Vc_r_pow,
            enable_hessian=int(bool(enable_hessian)), reserved0=0)
        self.cfg = cfg
        self._h = C.c_void_p()
        check(self._lib.srhmc_create(C.byref(cfg), C.byref(self._h)))
        self.F = n_fields
        self.S = 3 * max_stars
        self._run_args = None
        self._keep = None

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.srhmc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    # ------------------------------------------------------------------ plumbing
    def set_stream(self, cuda_stream_ptr):
        check(self._lib.srhmc_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def synchronize(self):
        check(self._lib.srhmc_synchronize(self._h))

    def last_kernel_ms(self):
        ms = C.c_float()
        check(self._lib.srhmc_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    @property
    def launch_count(self):
        return int(self._lib.srhmc_launch_count(self._h))

    def launch_plan(self):
        """How the CTA-per-field kernel was configured for this context (struct srhmc_launch_plan as a dict):
        threads, tile_rows, tile_cols, chunk_stars, image_in_smem, compact_tables, chain_kernel, int_image_bytes
        (meaningful after set_data) and smem_bytes."""
        plan = _capi.LaunchPlan()
        check(self._lib.srhmc_get_launch_plan(self._h, C.byref(plan)))
        return {name: int(getattr(plan, name)) for name, _ in plan._fields_}

    def chain_plan(self):
        """What a launch of one-star fields runs now on the warp-resident one-star kernel (struct srhmc_chain_plan as a
        dict): chain_kernel, window_cols, image_bytes, pixel_f32, blocks_per_sm, tab_stride and smem_bytes; meaningful
        after set_data."""
        plan = _capi.ChainPlan()
        check(self._lib.srhmc_get_chain_plan(self._h, C.byref(plan)))
        return {name: int(getattr(plan, name)) for name, _ in plan._fields_}

    def _nstars(self, nstars):
        if nstars is None:
            return None
        return np.ascontiguousarray(nstars, dtype=np.int32).reshape(self.F)

    # ------------------------------------------------------------------ data
    def set_data(self, D):
        D = as_f64(D)
        n_img = 1 if self.cfg.shared_data else self.F
        D = D.reshape(n_img, self.cfg.num_rows, self.cfg.num_cols)
        check(self._lib.srhmc_set_data(self._h, dptr(D), n_img))

    def gen_model(self, q, nstars=None):
        """Model image B + sum f PSF of every field, rendered on the device (base_class.gen_model,
        sampler_RHMC.py:101-117).  q [F, S] with f in counts -> [F, R, C]."""
        q = as_f64(q, (self.F, self.S))
        ns = self._nstars(nstars)
        out = np.empty((self.F, self.cfg.num_rows, self.cfg.num_cols))
        check(self._lib.srhmc_gen_model(self._h, dptr(q), iptr(ns), dptr(out)))
        return out

    def gen_mock_data(self, q_true, nstars=None, seed=0, field_id_base=0, return_data=True):
        """Poisson mock data of every field generated on the device and installed as the context's data
        (base_class.gen_mock_data, sampler_RHMC.py:77-99): counter-based Philox, pixel p of field i draws with the
        counter (field_id_base + i) * R * C + p, so sharded batches reproduce the unsharded images."""
        q = as_f64(q_true, (self.F, self.S))
        ns = self._nstars(nstars)
        out = np.empty((self.F, self.cfg.num_rows, self.cfg.num_cols)) if return_data else None
        check(self._lib.srhmc_gen_mock_data(self._h, dptr(q), iptr(ns), int(seed), int(field_id_base), dptr(out)))
        return out

    def find_peaks_descend(self, q_seed, nstep, dt_f_coeff, dt_xy_coeff, f_lim):
        """Independent gradient descent of every seed [n,3] on data image 0 (find_peaks, samplers.py:196-226).
        Returns (q [n,3], alive [n] bool, steps [n])."""
        q = np.array(as_f64(q_seed).reshape(-1, 3), copy=True)
        n = len(q)
        alive = np.zeros(n, dtype=np.uint8)
        steps = np.zeros(n, dtype=np.int32)
        check(self._lib.srhmc_find_peaks_descend(self._h, dptr(q), n, int(nstep), float(dt_f_coeff), float(dt_xy_coeff),
                                                 float(f_lim), bptr(alive), iptr(steps)))
        return q, alive.astype(bool), steps

    def run_stats(self, n_groups=1, thin_rate=5, warm_up_num=0):
        """(R, n_eff) [n_groups, S] of utils.convergence_stats over the q_chain of the last launched run, computed
        from the chains still resident on the device (no chain download needed)."""
        R = np.empty((int(n_groups), self.S))
        n_eff = np.empty((int(n_groups), self.S))
        check(self._lib.srhmc_run_stats(self._h, int(n_groups), int(thin_rate), int(warm_up_num), dptr(R), dptr(n_eff)))
        return R, n_eff

    # ------------------------------------------------------------------ a2-a4: V, dVdq, H
    def eval(self, q, nstars=None, f_pos=False, g_ff2=1.0, beta=1.0):
        q = as_f64(q, (self.F, self.S))
        ns = self._nstars(nstars)
        V = np.empty(self.F)
        grad = np.zeros((self.F, self.S))
        H = np.zeros((self.F, self.S))
        Hg = np.zeros((self.F, self.S))
        check(self._lib.srhmc_eval(self._h, dptr(q), iptr(ns), int(bool(f_pos)), float(g_ff2), float(beta),
                                   dptr(V), dptr(grad), dptr(H), dptr(Hg)))
        return V, grad, H, Hg

    # ------------------------------------------------------------------ a4: H alone
    def metric(self, q, g_ff2=1.0):
        """H and dH/df for a flat array of [f, x, y] triples of any length (no image involved)."""
        q = as_f64(q).ravel()
        n = q.size // 3
        H = np.zeros(3 * n)
        Hg = np.zeros(3 * n)
        check(self._lib.srhmc_metric(self._h, dptr(q), n, float(g_ff2), dptr(H), dptr(Hg)))
        return H, Hg

    # ------------------------------------------------------------------ a5/a6: T, dtaudq, dtaudp
    def kinetic(self, q, p, nstars=None, g_ff2=1.0):
        q = as_f64(q, (self.F, self.S))
        p = as_f64(p, (self.F, self.S))
        ns = self._nstars(nstars)
        T = np.empty(self.F)
        dq = np.zeros((self.F, self.S))
        dp = np.zeros((self.F, self.S))
        check(self._lib.srhmc_kinetic(self._h, dptr(q), dptr(p), iptr(ns), float(g_ff2), dptr(T), dptr(dq), dptr(dp)))
        return T, dq, dp

    def kinetic_diag(self, p, H_diag):
        """T(p, H_diag) for an explicit diagonal (any length)."""
        p = as_f64(p).ravel()
        H = as_f64(H_diag).ravel()
        assert p.size == H.size
        T = np.empty(1)
        check(self._lib.srhmc_kinetic_diag(self._h, dptr(p), dptr(H), p.size, dptr(T)))
        return float(T[0])

    # ------------------------------------------------------------------ a7: RHMC_single_step
    def step(self, q, p, nsteps, dt, delta=1e-6, counter_max=1000, g_ff2=1.0, beta=1.0, nstars=None,
             return_counts=False):
        q = np.array(as_f64(q, (self.F, self.S)), copy=True)
        p = np.array(as_f64(p, (self.F, self.S)), copy=True)
        ns = self._nstars(nstars)
        counts = np.zeros((self.F, 2), dtype=np.int32)
        check(self._lib.srhmc_step(self._h, dptr(q), dptr(p), iptr(ns), int(nsteps), float(dt), float(delta),
                                   int(counter_max), float(g_ff2), float(beta), iptr(counts)))
        return (q, p, counts) if return_counts else (q, p)

    # ------------------------------------------------------------------ a8: run_RHMC move-0 leg
    def make_run_args(self, q0, niter, nsteps, dt, *, nstars=None, delta=1e-6, counter_max=1000, f_pos=True,
                      g_ff2=1.0, beta=1.0, schedule_g_ff2=None, schedule_beta=None, normals=None, lnu=None, seed=0,
                      chain_stride=1, want=("q", "p", "E", "V", "T", "A"), out=None, field_id_base=0,
                      field_id_stride=1, field_ids=None):
        """Build the argument block (and the host arrays it points at).  `out` may supply preallocated
        (e.g. pinned) output arrays keyed like RunResult fields."""
        F, S, L = self.F, self.S, int(niter) + 1
        rows = (L + chain_stride - 1) // chain_stride
        keep = {}
        keep["q0"] = as_f64(q0, (F, S))
        keep["nstars"] = self._nstars(nstars)
        keep["sg"] = None if schedule_g_ff2 is None else as_f64(schedule_g_ff2).ravel()
        keep["sb"] = None if schedule_beta is None else as_f64(schedule_beta).ravel()
        keep["normals"] = None if normals is None else as_f64(normals, (F, L, S))
        keep["lnu"] = None if lnu is None else as_f64(lnu, (F, L))
        keep["field_ids"] = None if field_ids is None else np.ascontiguousarray(field_ids, dtype=np.int32).reshape(F)
        out = dict(out or {})

        def buf(key, shape, dtype=np.float64):
            if key in out and out[key] is not None:
                a = out[key]
                assert a.shape == shape and a.dtype == dtype and a.flags.c_contiguous
                return a
            return np.zeros(shape, dtype=dtype)

        keep["q_chain"] = buf("q_chain", (F, rows, S)) if "q" in want else None
        keep["p_chain"] = buf("p_chain", (F, rows, S)) if "p" in want else None
        keep["E_chain"] = buf("E_chain", (F, rows)) if "E" in want else None
        keep["V_chain"] = buf("V_chain", (F, rows)) if "V" in want else None
        keep["T_chain"] = buf("T_chain", (F, rows)) if "T" in want else None
        keep["A_chain"] = buf("A_chain", (F, rows), np.uint8) if "A" in want else None
        keep["q_final"] = buf("q_final", (F, S))
        keep["accept_rate"] = buf("accept_rate", (F,))
        a = RunArgs(
            q0=dptr(keep["q0"]), nstars=iptr(keep["nstars"]), niter=int(niter), nsteps=int(nsteps), dt=float(dt),
            delta=float(delta), counter_max=int(counter_max), f_pos=int(bool(f_pos)), g_ff2=float(g_ff2),
            beta=float(beta), g_ff2_schedule=dptr(keep["sg"]), n_g_ff2=0 if keep["sg"] is None else keep["sg"].size,
            beta_schedule=dptr(keep["sb"]), n_beta=0 if keep["sb"] is None else keep["sb"].size,
            normals=dptr(keep["normals"]), lnu=dptr(keep["lnu"]), seed=int(seed), chain_stride=int(chain_stride),
            reserved=0, q_chain=dptr(keep["q_chain"]), p_chain=dptr(keep["p_chain"]), E_chain=dptr(keep["E_chain"]),
            V_chain=dptr(keep["V_chain"]), T_chain=dptr(keep["T_chain"]), A_chain=bptr(keep["A_chain"]),
            q_final=dptr(keep["q_final"]), accept_rate=dptr(keep["accept_rate"]),
            field_id_base=int(field_id_base), field_id_stride=int(field_id_stride), field_ids=iptr(keep["field_ids"]))
        return a, keep

    def _result(self, keep):
        return RunResult(keep["q_chain"], keep["p_chain"], keep["E_chain"], keep["V_chain"], keep["T_chain"],
                         keep["A_chain"], keep["q_final"], keep["accept_rate"], self.last_kernel_ms())

    def run(self, q0, niter, nsteps, dt, **kw):
        """All (niter+1) x nsteps leapfrog steps of every field in ONE resident launch."""
        a, keep = self.make_run_args(q0, niter, nsteps, dt, **kw)
        check(self._lib.srhmc_run(self._h, C.byref(a)))
        return self._result(keep)

    def run_prepared(self, a):
        """srhmc_run on an argument block from make_run_args (upload + launch + download + synchronize)."""
        check(self._lib.srhmc_run(self._h, C.byref(a)))

    # split phases, for callers that keep inputs resident (bench.py `value`)
    def run_upload(self, a):
        check(self._lib.srhmc_run_upload(self._h, C.byref(a)))

    def run_launch(self, a):
        check(self._lib.srhmc_run_launch(self._h, C.byref(a)))

    def run_download(self, a):
        check(self._lib.srhmc_run_download(self._h, C.byref(a)))

    def run_rj(self, q0, niter, nsteps, dt, *, P_move, fmin, fmax, K_split=1.0, beta_a=2.0, beta_b=2.0, draws=None,
               **run_kw):
        """Reversible-jump chains (multi_gym.run_RHMC with birth/death and split/merge moves): every iteration of every
        field in ONE launch, the star counts changing on the device.  run_kw as for run(); nstars gives the start counts
        (default max_stars).  draws [F, niter+1, 14] replaces the device records (philox_rj_draws).  alpha and
        V_prior_const are the context's.  Returns RjRunResult; chain rows are zero past 3 * N_chain of their row."""
        F, L = self.F, int(niter) + 1
        a, keep = self.make_run_args(q0, niter, nsteps, dt, **run_kw)
        rows = (L + a.chain_stride - 1) // a.chain_stride
        dr = None if draws is None else as_f64(draws, (F, L, RJ_DRAWS))
        out = dict(N_chain=np.zeros((F, rows), dtype=np.int32), move_chain=np.zeros((F, rows), dtype=np.uint8),
                   n_final=np.zeros(F, dtype=np.int32), overflow=np.zeros(F, dtype=np.int32))
        rj = RjArgs(P_move=(C.c_double * 3)(*[float(x) for x in P_move]), fmin=float(fmin), fmax=float(fmax),
                    K_split=float(K_split), beta_a=float(beta_a), beta_b=float(beta_b), draws=dptr(dr),
                    N_chain=iptr(out["N_chain"]), move_chain=bptr(out["move_chain"]), n_final=iptr(out["n_final"]),
                    overflow=iptr(out["overflow"]))
        check(self._lib.srhmc_run_rj(self._h, C.byref(a), C.byref(rj)))
        return RjRunResult(keep["q_chain"], keep["p_chain"], keep["E_chain"], keep["V_chain"], keep["T_chain"],
                           keep["A_chain"], keep["q_final"], keep["accept_rate"], self.last_kernel_ms(), **out)

    def philox_rj_draws(self, seed, niter, beta_a=2.0, beta_b=2.0, field_id_base=0, field_id_stride=1):
        """The draw records [F, niter+1, 14] run_rj consumes for `seed` (see rj_draws.cuh for the layout)."""
        draws = np.zeros((self.F, int(niter) + 1, RJ_DRAWS))
        check(self._lib.srhmc_philox_rj_draws(self._h, int(seed), int(niter), int(field_id_base), int(field_id_stride),
                                              float(beta_a), float(beta_b), dptr(draws)))
        return draws

    # ------------------------------------------------------------------ a9: run_single_RHMC(implicit)
    def run_single(self, q0, p0, nsteps, dt, delta=1e-6, counter_max=100, f_pos=False, g_ff2=1.0, beta=1.0,
                   nstars=None):
        F, S, rows = self.F, self.S, int(nsteps) + 1
        q0 = as_f64(q0, (F, S))
        p0 = as_f64(p0, (F, S))
        ns = self._nstars(nstars)
        qc = np.zeros((F, rows, S))
        pc = np.zeros((F, rows, S))
        E = np.zeros((F, rows))
        V = np.zeros((F, rows))
        T = np.zeros((F, rows))
        check(self._lib.srhmc_run_single(self._h, dptr(q0), dptr(p0), iptr(ns), int(nsteps), float(dt), float(delta),
                                         int(counter_max), int(bool(f_pos)), float(g_ff2), float(beta), dptr(qc),
                                         dptr(pc), dptr(E), dptr(V), dptr(T)))
        return qc, pc, E, V, T

    # ------------------------------------------------------------------ a10/a11: lightsource_gym family
    LS_HMC, LS_DIAG, LS_HESS, LS_TRIAL = 0, 1, 2, 3

    def hessian(self, q, p=None, f_lim=0.0, d2_only=False, nstars=None):
        """RHMC_efficient_computation: (d1, d2, d3, dqdt, dpdt, E), or d2 alone when d2_only."""
        F, S = self.F, self.S
        q = as_f64(q, (F, S))
        ns = self._nstars(nstars)
        d2 = np.zeros((F, S))
        if d2_only:
            check(self._lib.srhmc_hessian(self._h, dptr(q), None, iptr(ns), float(f_lim), 1, None, dptr(d2), None, None,
                                          None, None))
            return d2
        p = as_f64(p, (F, S))
        d1, d3, dq, dp = (np.zeros((F, S)) for _ in range(4))
        E = np.zeros(F)
        check(self._lib.srhmc_hessian(self._h, dptr(q), dptr(p), iptr(ns), float(f_lim), 0, dptr(d1), dptr(d2), dptr(d3),
                                      dptr(dq), dptr(dp), dptr(E)))
        return d1, d2, d3, dq, dp, E

    def eval_background(self, q, background, nstars=None):
        """V and dV/dq on a per-pixel background image (lightsource_gym.V_single / dVdq_single)."""
        q = as_f64(q, (self.F, self.S))
        bg = as_f64(background, (self.F, self.cfg.num_rows, self.cfg.num_cols))
        ns = self._nstars(nstars)
        V = np.zeros(self.F)
        grad = np.zeros((self.F, self.S))
        check(self._lib.srhmc_eval_background(self._h, dptr(q), iptr(ns), dptr(bg), dptr(V), dptr(grad)))
        return V, grad

    def ls_run(self, variant, q0, dt, normals, steps, lnu, f_lim=0.0, factor1=0.0, background=None, zero_xy=False,
               nstars=None):
        """One lightsource_gym chain per field with injected draws -> dict(q_chain, E_chain, dE_chain, A_chain,
        q_final, accept_count)."""
        F, S = self.F, self.S
        steps = np.ascontiguousarray(steps, dtype=np.int32).reshape(F, -1)
        niter = steps.shape[1]
        L = niter + 1
        q0 = as_f64(q0, (F, S))
        dt = as_f64(dt).ravel()
        normals = as_f64(normals, (F, L, S))
        lnu = as_f64(lnu, (F, niter))
        ns = self._nstars(nstars)
        bg = None if background is None else as_f64(background, (F, self.cfg.num_rows, self.cfg.num_cols))
        out = dict(q_chain=np.zeros((F, L, S)), E_chain=np.zeros((F, L)), dE_chain=np.zeros((F, L)),
                   A_chain=np.zeros((F, niter), dtype=np.uint8), q_final=np.zeros((F, S)), accept_count=np.zeros(F))
        a = LsArgs(variant=int(variant), niter=niter, q0=dptr(q0), nstars=iptr(ns), dt=dptr(dt), n_dt=dt.size,
                   zero_xy_momentum=int(bool(zero_xy)), f_lim=float(f_lim), factor1=float(factor1),
                   normals=dptr(normals), steps=iptr(steps), lnu=dptr(lnu), background=dptr(bg),
                   q_chain=dptr(out["q_chain"]), E_chain=dptr(out["E_chain"]), dE_chain=dptr(out["dE_chain"]),
                   A_chain=bptr(out["A_chain"]), q_final=dptr(out["q_final"]), accept_count=dptr(out["accept_count"]))
        check(self._lib.srhmc_ls_run(self._h, C.byref(a)))
        return out

    def device_math(self, which, x):
        """Diagnostic: the kernels' exp_neg (0), log_pos (1) or rcp_fast (2) evaluated on the device."""
        x = as_f64(x).ravel()
        y = np.empty_like(x)
        check(self._lib.srhmc_test_device_math(self._h, int(which), dptr(x), dptr(y), x.size))
        return y

    # ------------------------------------------------------------------ device RNG replay
    def philox_draws(self, seed, niter, field_id_base=0, field_id_stride=1):
        L = int(niter) + 1
        normals = np.zeros((self.F, L, self.S))
        lnu = np.zeros((self.F, L))
        check(self._lib.srhmc_philox_draws_ids(self._h, int(seed), int(niter), int(field_id_base),
                                               int(field_id_stride), dptr(normals), dptr(lnu)))
        return normals, lnu
