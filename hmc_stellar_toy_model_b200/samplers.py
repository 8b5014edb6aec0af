"""Drop-in for the reference's samplers.py `lightsource_gym`: same class, method names, argument meaning and
attributes, with the sampler loops running in the sm_100a kernels of libstellar_rhmc.so (csrc/ls_kernel.cuh).

    from hmc_stellar_toy_model_b200.samplers import *        # instead of `from samplers import *`

What runs where
  device (C ABI)  dVdq, V, E, K, dVdq_single, V_single, E_single, RHMC_efficient_computation, and the whole chain loops
                  of HMC_random, RHMC_random_diag and RHMC_random (ONE resident launch per chain); HMC_find_best_dt
                  keeps its search loop on the host (as SURVEY.md 8a says) and runs every acceptance-rate trial
                  (Niter_per_trial random-length trajectories) as one launch; the seed descent of find_peaks is one
                  launch for all seeds.
  host (set-up)   mock data, Fisher factors, mass_matrix / F / G / dlnDetdq / dpMpdq scalars, random draws -- taken from
                  the global np.random stream in exactly the reference's order (p_sample, then per iteration
                  p_sample, randint, random; samplers.py:507,520,529,562), so seeded scripts reproduce the reference;
                  find_peaks' seed grid and greedy merge (bigfield.BigFieldStrip.find_peaks runs both stages on the
                  device for images too large for this path).
  not provided    RHMC_GMM (unrelated toy density), display_data.

The reference's behavioural quirks are reproduced on the device (see csrc/ls_kernel.cuh).  No CPU fallback.
"""
from __future__ import annotations

import numpy as np

from .context import RHMCContext
from .utils import *  # noqa: F401,F403  (samplers.py:1 star-imports utils)
from .utils import factors, gauss_PSF, mag2flux, poisson_realization

__all__ = ["lightsource_gym"]


class lightsource_gym(object):
    """samplers.lightsource_gym (samplers.py:3-1237)."""

    device = 0

    def __init__(self):
        self.D = None
        self.M = None
        (self.num_rows, self.num_cols, self.flux_to_count, self.PSF_FWHM_pix, self.B_count,
         self.arcsec_to_pix) = self.default_exp_setup()
        self.Nchain = None
        self.Niter = None
        self.thin_rate = None
        self.Nwarmup = None
        self.q_chain = None
        self.p_chain = None
        self.V_chain = None
        self.E_chain = None
        self.dE_chain = None
        self.A_chain = None
        self.dt = None
        self.f_lim = 0.
        self._ctx = None
        self._ctx_key = None
        self._ctx_data = None

    # ------------------------------------------------------------------ set-up (host)
    def default_exp_setup(self):
        """samplers.py:1206-1237."""
        arcsec_to_pix = 0.4
        PSF_FWHM_pix = 1.4 / arcsec_to_pix
        flux_to_count = 1. / (0.00546689 * 4.62)
        self.mB = 23
        B_count = mag2flux(self.mB) * flux_to_count
        num_rows = num_cols = 48
        return num_rows, num_cols, flux_to_count, PSF_FWHM_pix, B_count, arcsec_to_pix

    def gen_mock_data(self, q_true=None, return_data=False):
        """q_true rows are [f, x, y] in flux counts (samplers.py:44-66)."""
        data = np.ones((self.num_rows, self.num_cols), dtype=float) * self.B_count
        for f, x, y in np.asarray(q_true, dtype=float):
            data += f * gauss_PSF(self.num_rows, self.num_cols, x, y, FWHM=self.PSF_FWHM_pix)
        data = poisson_realization(data)
        if return_data:
            return data
        self.D = data

    def compute_factors(self):
        """Uses the CURRENT image size, unlike base_class (samplers.py:69-75)."""
        self.factor0, self.factor1, self.factor2 = factors(self.num_rows, self.num_cols, self.num_rows / 2.,
                                                           self.num_cols / 2., self.PSF_FWHM_pix)

    def p_sample(self):
        return np.random.randn(self.d)

    # ------------------------------------------------------------------ device plumbing
    def _device_ctx(self, n_stars):
        key = (int(self.num_rows), int(self.num_cols), int(n_stars), float(self.PSF_FWHM_pix), float(self.B_count),
               int(self.device))
        if self._ctx is None or key != self._ctx_key:
            if self._ctx is not None:
                self._ctx.close()
            R, C, N, fwhm, B, dev = key
            # the metric constants are unused by this family; the context just needs valid numbers
            self._ctx = RHMCContext(n_fields=1, num_rows=R, num_cols=C, max_stars=N, psf_fwhm_pix=fwhm, B_count=B,
                                    f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, g_xx=1.0, g_ff=1.0,
                                    enable_hessian=True, device=dev)
            self._ctx_key = key
            self._ctx_data = None
        if self.D is None:
            raise ValueError("gym.D is not set: call gen_mock_data() or assign the data image first")
        D = np.ascontiguousarray(self.D, dtype=np.float64)
        from .sampler_RHMC import base_class  # the gyms share the "is gym.D still the device image?" test

        if self._ctx_data is None or not base_class._same_image(D, self._ctx_data):
            self._ctx.set_data(D)
            self._ctx_data = D.copy()
        return self._ctx

    @staticmethod
    def _flat(q):
        return np.ascontiguousarray(q, dtype=float).ravel()

    # ------------------------------------------------------------------ physics (device)
    def dVdq(self, objs_flat):
        q = self._flat(objs_flat)
        _, grad, _, _ = self._device_ctx(q.size // 3).eval(q[None])
        return grad[0]

    def V(self, objs_flat):
        q = self._flat(objs_flat)
        V, _, _, _ = self._device_ctx(q.size // 3).eval(q[None])
        return float(V[0])

    def K(self, p, mass_matrix=None):
        p = self._flat(p)
        ctx = self._device_ctx(max(1, p.size // 3))
        if mass_matrix is None:
            # identity mass: p.p/2 = T(p, ones) because ln|1| = 0
            return ctx.kinetic_diag(p, np.ones_like(p))
        return ctx.kinetic_diag(p, self._flat(mass_matrix))

    def E(self, q, p, mass_matrix=None):
        q = self._flat(q)
        for l in range(q.size // 3):
            if q[3 * l] < self.f_lim:
                return np.inf
        return self.V(q) + self.K(p, mass_matrix)

    def _single(self, q_single, model_data):
        """One evaluation of the single-star problem on a model_data background (samplers.py:77-127)."""
        V, grad = self._device_ctx(1).eval_background(self._flat(q_single)[None], np.asarray(model_data, float)[None])
        return float(V[0]), grad[0]

    def dVdq_single(self, q_single, model_data, f_only=True, return_all=False):
        V, g = self._single(q_single, model_data)
        if return_all:
            return g[0], g[1], g[2]
        if f_only:
            return g[0]
        return g[1], g[2]

    def V_single(self, q_single, model_data):
        V, _ = self._single(q_single, model_data)
        return V

    def E_single(self, q_single, p_single, model_data):
        p = self._flat(p_single)
        return self.V_single(q_single, model_data) + self.K(p)

    def mass_matrix(self, q):
        q = self._flat(q)
        M = np.zeros_like(q)
        M[0::3] = self.G(q[0::3])
        M[1::3] = self.F(q[0::3])
        M[2::3] = self.F(q[0::3])
        return M

    def F(self, f, dFdf=False):
        x1 = f * self.factor1
        return (x1, self.factor1) if dFdf else x1

    def G(self, f, dGdf=False):
        x1 = 1. / f
        return (x1, -1 / f ** 2) if dGdf else x1

    def dlnDetdq(self, q):
        q = self._flat(q)
        out = np.zeros_like(q)
        f = q[0::3]
        out[0::3] = 0.5 * ((-1 / f ** 2) / (1. / f) + 2 * self.factor1 / (f * self.factor1))
        return out

    def dpMpdq(self, q, p):
        q, p = self._flat(q), self._flat(p)
        out = np.zeros_like(q)
        f = q[0::3]
        G, dG, Fm, dF = 1. / f, -1 / f ** 2, f * self.factor1, self.factor1
        out[0::3] = -0.5 * (dG * p[0::3] ** 2 / G ** 2 + (p[1::3] ** 2 + p[2::3] ** 2) * dF / Fm ** 2)
        return out

    def RHMC_efficient_computation(self, q_tmp, p_tmp, debug=True, dVdqq_only=False):
        """(dqdt, dpdt, E), or dVdqq when dVdqq_only (samplers.py:828-927)."""
        q = self._flat(q_tmp)
        ctx = self._device_ctx(q.size // 3)
        if dVdqq_only:
            return ctx.hessian(q[None], d2_only=True)[0]
        d1, d2, d3, dqdt, dpdt, E = ctx.hessian(q[None], self._flat(p_tmp)[None], f_lim=self.f_lim)
        if np.isinf(E[0]):
            return np.inf, np.inf, np.inf
        if debug:
            print("q_tmp", q)
            print("dqdt", dqdt[0])
            print("p_tmp", p_tmp)
            print("dpdt", dpdt[0])
            print("dVdq", d1[0])
            print("dVdqq", d2[0])
            print("dVdqqq", d3[0])
        return dqdt[0], dpdt[0], float(E[0])

    def leap_frog(self, p_old, q_old, dt):
        p_half = p_old - dt * self.dVdq(q_old) / 2.
        q_new = q_old + dt * p_half
        p_new = p_half - dt * self.dVdq(q_new) / 2.
        return p_new, q_new

    # ------------------------------------------------------------------ chain loops (device-resident)
    def _set_f_lim(self, f_lim, f_lim_default):
        self.f_lim = mag2flux(self.mB - 1.) * self.flux_to_count if f_lim_default else f_lim

    def _draws(self, Niter, steps_min, steps_max, initial=True):
        """The reference's draw sequence: [p_sample()] then per iteration p_sample(), randint, random."""
        normals = np.zeros((Niter + 1, self.d))
        steps = np.zeros(Niter, dtype=np.int32)
        lnu = np.zeros(Niter)
        if initial:
            normals[0] = self.p_sample()
        for i in range(1, Niter + 1):
            normals[i] = self.p_sample()
            steps[i - 1] = np.random.randint(low=steps_min, high=steps_max, size=1)[0]
            lnu[i - 1] = np.log(np.random.random(1))[0]
        return normals, steps, lnu

    def _store(self, out, Niter):
        self.q_chain = np.zeros((self.Nchain, Niter + 1, self.d))
        self.E_chain = np.zeros((self.Nchain, Niter + 1, 1))
        self.dE_chain = np.zeros((self.Nchain, Niter + 1, 1))
        self.A_chain = np.zeros((self.Nchain, Niter, 1))
        self.q_chain[0] = out["q_chain"][0]
        self.E_chain[0, :, 0] = out["E_chain"][0]
        self.dE_chain[0, :, 0] = out["dE_chain"][0]
        self.A_chain[0, :, 0] = out["A_chain"][0]

    def _setup_run(self, Nchain, Niter, thin_rate, Nwarmup):
        assert Nchain == 1  # like the reference (samplers.py:472,682,941)
        self.Nchain, self.Niter, self.thin_rate, self.Nwarmup = Nchain, Niter, thin_rate, Nwarmup

    def HMC_random(self, q_model_0=None, Nchain=1, Niter=1000, thin_rate=0, Nwarmup=0, steps_min=10, steps_max=50,
                   f_lim=0., f_lim_default=False):
        """Identity-mass random-length HMC with the per-coordinate self.dt (samplers.py:460-572)."""
        self._setup_run(Nchain, Niter, thin_rate, Nwarmup)
        assert self.d is not None
        self._set_f_lim(f_lim, f_lim_default)
        if q_model_0 is None:
            q_model_0 = self.q_seed
        q0 = np.array(q_model_0, dtype=float).reshape((self.d,))
        normals, steps, lnu = self._draws(Niter, steps_min, steps_max)
        ctx = self._device_ctx(self.d // 3)
        out = ctx.ls_run(ctx.LS_HMC, q0[None], self.dt, normals[None], steps[None], lnu[None], f_lim=self.f_lim)
        self._store(out, Niter)
        print("Chain %d Acceptance rate: %.2f%%" % (0, np.sum(self.A_chain[0, :] * 100) / float(self.Niter)))

    def RHMC_random_diag(self, q_model_0, Nchain=1, Niter=1000, thin_rate=0, Nwarmup=0, steps_min=10, steps_max=50,
                         f_lim=0., f_lim_default=False, dt_global=1e-2, save_traj=False):
        """Diagonal-mass RHMC, M(f) = [1/f, f factor1, f factor1] (samplers.py:668-825)."""
        if save_traj:
            raise NotImplementedError("save_traj keeps per-step host arrays; not part of the device-resident path")
        self._setup_run(Nchain, Niter, thin_rate, Nwarmup)
        self._set_f_lim(f_lim, f_lim_default)
        if q_model_0 is None:
            q_model_0 = self.q_seed
        self.Nobjs = q_model_0.shape[0]
        self.d = int(np.prod(q_model_0.shape))
        q0 = np.array(q_model_0, dtype=float).reshape((self.d,))
        normals, steps, lnu = self._draws(Niter, steps_min, steps_max)
        ctx = self._device_ctx(self.Nobjs)
        out = ctx.ls_run(ctx.LS_DIAG, q0[None], [dt_global], normals[None], steps[None], lnu[None], f_lim=self.f_lim,
                         factor1=self.factor1)
        self._store(out, Niter)
        print("Chain %d Acceptance rate: %.2f%%" % (0, np.sum(self.A_chain[0, :] * 100) / float(self.Niter)))

    def RHMC_random(self, q_model_0=None, Nchain=1, Niter=1000, thin_rate=0, Nwarmup=0, steps_min=10, steps_max=50,
                    f_lim=0., f_lim_default=False, dt_RHMC_xy=1., dt_RHMC_f=0.1, debug=True):
        """Hessian-metric RHMC (samplers.py:930-1105).  `debug` printing of every intermediate is not reproduced.
        Like the reference, the state advances IN PLACE: q_model_0 is left at the chain's last state and a
        rejected proposal is not undone."""
        self._setup_run(Nchain, Niter, thin_rate, Nwarmup)
        self.Nobjs = q_model_0.shape[0]
        self.d = self.Nobjs * 3
        dt_RHMC = np.asarray([dt_RHMC_f, dt_RHMC_xy, dt_RHMC_xy] * self.Nobjs, dtype=float)
        self._set_f_lim(f_lim, f_lim_default)
        q_flat = q_model_0.reshape((self.d,))
        # draws: every iteration 0..Niter takes a p_sample; iterations >= 1 also a randint and a uniform
        normals = np.zeros((Niter + 1, self.d))
        steps = np.zeros(Niter, dtype=np.int32)
        lnu = np.zeros(Niter)
        states = {}
        for i in range(Niter + 1):
            normals[i] = self.p_sample()
            if i > 0:
                steps[i - 1] = np.random.randint(low=steps_min, high=steps_max, size=1)[0]
                lnu[i - 1] = np.log(np.random.random(1))[0]
                if (i % 100) == 0:
                    states[i] = np.random.get_state()
        ctx = self._device_ctx(self.Nobjs)
        out = ctx.ls_run(ctx.LS_HESS, np.array(q_flat, dtype=float)[None], dt_RHMC, normals[None], steps[None],
                         lnu[None], f_lim=self.f_lim)
        self._store(out, Niter)
        # the reference abandons a chain whose acceptance is below 50% at a multiple of 100 iterations
        # (samplers.py:1098-1101) and stops drawing there: put the global stream where it would have been left
        acc = np.cumsum(out["A_chain"][0].astype(float))
        for i in range(100, Niter + 1, 100):
            if acc[i - 1] * 100 / float(i) < 50:
                np.random.set_state(states[i])
                break
        q_flat[...] = out["q_final"][0]  # the reference's in-place `q_tmp += ...` mutates the caller's array
        self.R_accept = np.sum(self.A_chain[0, :] * 100) / float(self.Niter)
        print("Chain %d Acceptance rate: %.2f%%" % (0, self.R_accept))

    def HMC_find_best_dt(self, q_model_0=None, steps_min=10, steps_max=50, Niter_per_trial=10, Ntrial=10,
                         dt_f_coeff=1., dt_xy_coeff=10., default=False, A_target_f=0.9, A_target_xy=0.5):
        """Per-star step-size search: coarse division by 10, then bisection on the acceptance rate of single-star
        HMC trials (samplers.py:257-456).  The search logic is the reference's; each trial is one device launch."""
        if q_model_0 is None:
            q_model_0 = self.q_seed
        self.Nobjs = q_model_0.shape[0]
        self.d = self.Nobjs * 3
        self.dt = np.zeros(self.d)
        if default:
            for i in range(self.Nobjs):
                f0 = q_model_0[i][0]
                self.dt[3 * i:3 * i + 3] = np.array([dt_f_coeff * f0, dt_xy_coeff / f0, dt_xy_coeff / f0])
            return
        ctx = self._device_ctx(1)

        def trial(dt, k, q_start, model_data):
            """Acceptance rate of Niter_per_trial trajectories; draws in the reference's order (:340-366)."""
            normals = np.zeros((Niter_per_trial + 1, 3))
            steps = np.zeros(Niter_per_trial, dtype=np.int32)
            lnu = np.zeros(Niter_per_trial)
            for i in range(1, Niter_per_trial + 1):
                normals[i] = np.random.randn(3)
                steps[i - 1] = np.random.randint(low=steps_min, high=steps_max, size=1)[0]
                lnu[i - 1] = np.log(np.random.random(1))[0]
            out = ctx.ls_run(ctx.LS_TRIAL, q_start[None], dt, normals[None], steps[None], lnu[None],
                             background=model_data[None], zero_xy=(k == 0))
            return out["accept_count"][0] / float(Niter_per_trial)

        for l in range(self.Nobjs):
            f0, x0, y0 = q_model_0[l]
            dt_xy = dt_xy_coeff / f0
            dt_f = dt_f_coeff * f0
            model_data = self.gen_mock_data(q_model_0, return_data=True)
            model_data -= f0 * gauss_PSF(self.num_rows, self.num_cols, x0, y0, FWHM=self.PSF_FWHM_pix)
            q_start = np.array([f0, x0, y0], dtype=float)
            for k in range(2):
                if k == 0:
                    dt = np.array([dt_f, 0, 0])
                    A_target = A_target_f
                else:
                    dt = np.array([dt_f, dt_xy, dt_xy])
                    A_target = A_target_xy
                # coarse finding
                while True:
                    A_rate = trial(dt, k, q_start, model_data)
                    if A_rate < A_target:
                        if k == 0:
                            dt = dt / 10.
                        else:
                            dt = np.array([dt[0], dt[1] / 10., dt[2] / 10.])
                    else:
                        break
                # fine finding
                counter = 0
                dt_left = dt
                dt_right = 10. * dt
                if k == 1:
                    dt_right[0] = dt_f
                while counter < Ntrial:
                    counter += 1
                    dt = (dt_left + dt_right) / 2.
                    if k == 1:
                        dt[0] = dt_f
                    A_rate = trial(dt, k, q_start, model_data)
                    if np.abs(A_rate - A_target) < 1e-2:
                        break
                    elif A_rate > A_target:
                        dt_left = dt
                    else:
                        dt_right = dt
                if k == 0:
                    dt_f = dt[0]
                else:
                    dt_xy = dt[1] * 10
            self.dt[3 * l:3 * l + 3] = np.array([dt_f, dt_xy, dt_xy])

    def find_peaks(self, linear_pix_density=0.2, dr_tol=1., dmag_tol=0.5, mag_lim=None, Nstep=1000, dt_f_coeff=1e-1,
                   dt_xy_coeff=1e-1, no_perturb=False):
        """Likely star positions (samplers.py:129-254): seeds on a jittered grid (np.random.randn in the reference's
        order), independent gradient descent of all seeds in ONE device launch, then the greedy merge of near-duplicates
        on the host.  Result in self.q_seed."""
        if self.num_rows is None or self.D is None:
            print("The image must be specified first.")
            assert False
        if mag_lim is None:
            mag_lim = self.mB - 1.
        f_lim = mag2flux(mag_lim) * self.flux_to_count
        f_seed = mag2flux(mag_lim - 0.5) * self.flux_to_count
        n_row = int(linear_pix_density * self.num_rows) - 1
        n_col = int(linear_pix_density * self.num_cols) - 1
        spacing = 1 / float(linear_pix_density)
        q_seed = np.zeros((n_row * n_col, 3), dtype=float)
        for i in range(n_row):
            for j in range(n_col):
                x = spacing * (i + 0.5 + 0.1 * np.random.randn())
                y = spacing * (j + 0.5 + 0.1 * np.random.randn())
                q_seed[i * n_row + j] = np.array([f_seed, x, y])  # row count as stride, as upstream (samplers.py:176)
        if no_perturb:
            self.q_seed = q_seed
            return
        q_seed, alive, _ = self._device_ctx(1).find_peaks_descend(q_seed, Nstep, dt_f_coeff, dt_xy_coeff, f_lim)
        q_seed = q_seed[alive]
        if q_seed.shape[0] == 0:
            self.q_seed = q_seed
            print("No peaks were found.")
            return
        kept = []
        while True:  # greedy reduction (samplers.py:234-252)
            ref = q_seed[0]
            kept.append(ref)
            q_seed = q_seed[1:, :]
            dist_sq = (q_seed[:, 1] - ref[1]) ** 2 + (q_seed[:, 2] - ref[2]) ** 2
            dmag = np.abs(flux2mag(ref[0] / self.flux_to_count) - flux2mag(q_seed[:, 0] / self.flux_to_count))
            q_seed = q_seed[np.logical_or(dist_sq > dr_tol ** 2, dmag > dmag_tol)]
            if q_seed.shape[0] == 0:
                break
        self.q_seed = np.vstack(kept)

    def display_data(self, *args, **kwargs):
        return None
