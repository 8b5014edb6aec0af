"""Drop-in for the reference's sampler_RHMC.py: same classes, method names, argument meaning and attributes, with the
RHMC hot path running in the sm_100a kernels of libstellar_rhmc.so.

    from hmc_stellar_toy_model_b200.sampler_RHMC import *      # instead of `from sampler_RHMC import *`

What runs where
  device (C ABI)  V, dVdq, H/H_xx/H_ff, T, dphidq, dtaudq, dtaudp, RHMC_single_step, the move-0 leg of
                  multi_gym.run_RHMC (ONE resident launch for all (Niter+1) x Nsteps leapfrog steps), and
                  single_gym.run_single_RHMC(solver="implicit") (one resident launch per trajectory).
  host (set-up)   unit conversions, mock-data generation, the frozen Fisher constants, random draws.  The legacy
                  global np.random stream is consumed in exactly the reference's order (sampler_RHMC.py:1021-1075:
                  randn(3N), one uniform for np.random.choice, one uniform for the accept test, per iteration), so a
                  script that seeds np.random reproduces the reference's chain step for step.
  host + device   reversible-jump moves (birth/death, split/merge; sampler_RHMC.py:1084-1445): by default the
                  trans-dimensional proposal bookkeeping stays on the host as upstream (the legacy np.random stream, byte
                  for byte), every RHMC leg / V / H / T around it runs on the device (one launch per leg).
  device (opt-in) gym.device_seed = <int> (new capability): the whole reversible-jump run is ONE launch of the
                  crowded-field kernel (RHMCContext.run_rj), proposals included, drawing counter-based Philox; the global
                  np.random stream is not touched.
  not provided    matplotlib diagnostics (no-ops here), the "naive"/"leap_frog" solvers and run_single_HMC (unused by
                  any script, labelled broken upstream).

There is no CPU fallback: every numeric method needs the CUDA library and a B200.
"""
from __future__ import annotations

import numpy as np

from .context import RHMCContext
from .utils import *  # noqa: F401,F403  (the reference star-imports utils into this namespace, sampler_RHMC.py:25)
from .utils import factors, gauss_PSF, gen_pow_law_sample, mag2flux, flux2mag, poisson_realization

__all__ = ["base_class", "single_gym", "multi_gym"]


class base_class(object):
    """State container + physics of the reference's base_class (sampler_RHMC.py:27-566)."""

    #: CUDA device ordinal and pixel precision (64: parity build, 32: float pixels) used by this gym's context.
    device = 0
    precision = 64

    def __init__(self, dt=1., g_xx=10, g_ff=10, g_ff2=2):
        self.D = None
        self.M = None
        (self.num_rows, self.num_cols, self.flux_to_count, self.PSF_FWHM_pix, self.B_count,
         self.arcsec_to_pix) = self.default_exp_setup()
        self.dt = dt
        self.g_xx = g_xx
        self.g_ff = g_ff
        self.g_ff2 = g_ff2
        self.compute_factors()
        self.vmin = None
        self.vmax = None
        self.use_prior = False
        self.alpha = 2.
        self.use_Vc = False
        self.beta = 1.
        self.f_expnt = None
        self.Vc_r_pow = 1.
        self.V_prior_const = None
        self.K_split = 1.
        self.beta_a = 2.
        self.beta_b = 2.
        self.move_types = {0: "within", 1: "birth", 2: "death", 3: "split", 4: "merge"}
        self._ctx = None
        self._ctx_key = None
        self._ctx_data = None

    # ------------------------------------------------------------------ set-up (host; sampler_RHMC.py:77-227)
    def default_exp_setup(self):
        """SDSS-like constants (sampler_RHMC.py:169-201): 0.4"/pix, 1.4" seeing, mB = 23, 48x48 image."""
        arcsec_to_pix = 0.4
        PSF_FWHM_pix = 1.4 / arcsec_to_pix
        flux_to_count = 1. / (0.00546689 * 4.62)
        self.mB = 23
        B_count = mag2flux(self.mB) * flux_to_count
        self.f_lim = mag2flux(self.mB) * flux_to_count
        num_rows = num_cols = 48
        return num_rows, num_cols, flux_to_count, PSF_FWHM_pix, B_count, arcsec_to_pix

    def compute_factors(self):
        self.g0, self.g1, self.g2 = factors(self.num_rows, self.num_cols, self.num_rows / 2., self.num_cols / 2.,
                                            self.PSF_FWHM_pix)

    def mag2flux_converter(self, mag):
        return mag2flux(mag) * self.flux_to_count

    def flux2mag_converter(self, flux):
        return flux2mag(flux / self.flux_to_count)

    def gen_model(self, q_model):
        model = np.ones((self.num_rows, self.num_cols), dtype=float) * self.B_count
        for mag, x, y in np.asarray(q_model, dtype=float):
            model += self.mag2flux_converter(mag) * gauss_PSF(self.num_rows, self.num_cols, x, y,
                                                               FWHM=self.PSF_FWHM_pix)
        return model

    def gen_mock_data(self, q_true=None, return_data=False, device_seed=None):
        """sampler_RHMC.py:77-99.  By default the image is built like upstream (host PSFs, np.random.poisson from the
        global legacy stream, so a seeded script gets the reference's image).  device_seed=<int> (new capability) renders
        and Poisson-samples on the GPU with counter-based Philox instead; the global np.random stream is not touched."""
        if device_seed is None:
            data = poisson_realization(self.gen_model(q_true))
        else:
            q = self.format_q(np.array(q_true, dtype=float, copy=True))
            ctx = self._device_ctx(q.size // 3, need_data=False)
            data = ctx.gen_mock_data(q.reshape(1, -1), seed=device_seed)[0]
            self._ctx_data = data.copy()  # the context already holds this image
        if return_data:
            return data
        self.D = data

    def gen_noise_profile(self, q_true, N_trial=1000, sig_fac=10, device_seed=None):
        """Residual histogram of N_trial Poisson realisations of the truth image (sampler_RHMC.py:118-145).  By default the
        realisations come from the global np.random stream like upstream; device_seed=<int> (new capability) draws all
        N_trial images in one device launch (counter-based Philox, one context of N_trial fields sharing the truth stars)."""
        truth = self.gen_model(q_true)
        if device_seed is None:
            res = np.vstack([poisson_realization(truth) - truth for _ in range(N_trial)]).ravel()
        else:
            q = self.format_q(np.array(q_true, dtype=float, copy=True))
            ctx = RHMCContext(n_fields=int(N_trial), num_rows=int(self.num_rows), num_cols=int(self.num_cols),
                              max_stars=max(1, q.size // 3), psf_fwhm_pix=float(self.PSF_FWHM_pix), B_count=float(self.B_count),
                              f_lim=float(self.f_lim), f_low=float(self.mag2flux_converter(self.mB + 2)), g0=float(self.g0),
                              g1=float(self.g1), g2=float(self.g2), g_xx=float(self.g_xx), g_ff=float(self.g_ff),
                              device=int(self.device))
            try:
                nst = np.full(int(N_trial), q.size // 3, dtype=np.int32)
                qq = np.zeros((int(N_trial), 3 * max(1, q.size // 3)))
                qq[:, :q.size] = q
                draws = ctx.gen_mock_data(qq, nstars=nst, seed=int(device_seed))
            finally:
                ctx.close()
            res = (draws - truth[None]).ravel()
        sig = np.sqrt(self.B_count)
        bins = np.arange(-sig_fac * sig, sig_fac * sig, sig / 5.)
        hist, _ = np.histogram(res, bins=bins, density=True)
        self.hist_noise = hist
        self.centers_noise = (bins[1:] + bins[:-1]) / 2.

    def u_sample(self, d):
        return np.random.randn(d)

    def format_q(self, q):
        """(Nobjs, 3) [mag, x, y] -> flat [f, x, y, ...]; converts IN PLACE like the reference (:209-217)."""
        for i in range(q.shape[0]):
            q[i, 0] = self.mag2flux_converter(q[i, 0])
        return q.reshape((q.size,))

    def reverse_format_q(self, q):
        q = np.copy(q.reshape((self.Nobjs, 3)))
        for i in range(self.Nobjs):
            q[i, 0] = self.flux2mag_converter(q[i, 0])
        return q

    # ------------------------------------------------------------------ device plumbing
    def _prior_const(self):
        """gym.V_prior_const, computed on first use from fmin/fmax like sampler_RHMC.py:320-321.  The reference does
        this even when the prior is off (and crashes if fmin/fmax are unset); without a prior the constant never
        reaches V, so it is simply left unset here."""
        if self.V_prior_const is None:
            fmin, fmax = getattr(self, "fmin", None), getattr(self, "fmax", None)
            if fmin is None or fmax is None:
                if self.use_prior:
                    raise TypeError("use_prior needs gym.fmin/gym.fmax or gym.V_prior_const (sampler_RHMC.py:320-321)")
                return 0.0
            self.V_prior_const = np.log(self.num_rows * self.num_cols) - np.log(
                (1 - self.alpha) / (fmax ** (1 - self.alpha) - fmin ** (1 - self.alpha)))
        return float(self.V_prior_const)

    def _device_ctx(self, n_stars, need_data=True):
        """The context matching the gym's attributes as they are NOW (scripts mutate them between calls)."""
        key = (int(self.num_rows), int(self.num_cols), int(n_stars), float(self.PSF_FWHM_pix), float(self.B_count),
               float(self.f_lim), float(self.mag2flux_converter(self.mB + 2)), float(self.g0), float(self.g1),
               float(self.g2), float(self.g_xx), float(self.g_ff), bool(self.use_prior), float(self.alpha),
               self._prior_const(), bool(self.use_Vc), float(self.Vc_r_pow), int(self.precision), int(self.device))
        if self._ctx is None or key != self._ctx_key:
            if self._ctx is not None:
                self._ctx.close()
            (R, C, N, fwhm, B, f_lim, f_low, g0, g1, g2, g_xx, g_ff, use_prior, alpha, vpc, use_Vc, vc_pow, prec,
             dev) = key
            self._ctx = RHMCContext(n_fields=1, num_rows=R, num_cols=C, max_stars=N, psf_fwhm_pix=fwhm, B_count=B,
                                    f_lim=f_lim, f_low=f_low, g0=g0, g1=g1, g2=g2, g_xx=g_xx, g_ff=g_ff,
                                    use_prior=use_prior, alpha=alpha, V_prior_const=vpc, use_Vc=use_Vc,
                                    Vc_r_pow=vc_pow, precision=prec, device=dev)
            self._ctx_key = key
            self._ctx_data = None
        if need_data:
            if self.D is None:
                raise ValueError("gym.D is not set: call gen_mock_data() or assign the data image first")
            D = np.ascontiguousarray(self.D, dtype=np.float64)
            if D.shape != (self.num_rows, self.num_cols):
                raise ValueError("gym.D has shape %s, expected (%d, %d)" % (D.shape, self.num_rows, self.num_cols))
            if self._ctx_data is None or not self._same_image(D, self._ctx_data):
                self._ctx.set_data(D)
                self._ctx_data = D.copy()
        return self._ctx

    @staticmethod
    def _same_image(D, cached):
        """Is gym.D still the image the context holds?  Scripts assign and mutate gym.D freely, so small images (every
        reference script: <= 64 x 64) are compared in full; for large ones a full compare on every V / dVdq call would cost
        more than the call, so shape, both diagonals, the border and a strided sample stand in for it."""
        if D.shape != cached.shape:
            return False
        if D.size <= 16384:
            return np.array_equal(D, cached)
        step = max(1, D.size // 4096)
        return (np.array_equal(D.ravel()[::step], cached.ravel()[::step]) and np.array_equal(D[0], cached[0])
                and np.array_equal(D[-1], cached[-1]) and np.array_equal(D[:, 0], cached[:, 0])
                and np.array_equal(D[:, -1], cached[:, -1]) and D.sum() == cached.sum())

    def _nobjs(self, q):
        return int(np.size(q)) // 3

    # ------------------------------------------------------------------ physics (device; sampler_RHMC.py:229-492)
    def H(self, q, grad=False):
        q = np.asarray(q, dtype=float).ravel()
        H, Hg = self._device_ctx(self._nobjs(q), need_data=False).metric(q, self.g_ff2)
        return (H, Hg) if grad else H  # (H_diag, H_grad_diag) as sampler_RHMC.py:248-258

    def H_xx(self, f, grad=False):
        H, Hg = self._device_ctx(1, need_data=False).metric(np.array([f, 0., 0.]), self.g_ff2)
        return (float(H[1]), float(Hg[1])) if grad else float(H[1])  # (value, grad) as sampler_RHMC.py:280

    def H_ff(self, f, grad=False):
        H, Hg = self._device_ctx(1, need_data=False).metric(np.array([f, 0., 0.]), self.g_ff2)
        return (float(H[0]), float(Hg[0])) if grad else float(H[0])  # (value, grad) as sampler_RHMC.py:292

    def V(self, q, f_pos=False):
        q = np.asarray(q, dtype=float).ravel()
        V, _, _, _ = self._device_ctx(self._nobjs(q)).eval(q[None], f_pos=f_pos, g_ff2=self.g_ff2, beta=self.beta)
        return float(V[0])

    def T(self, p, H_diag):
        """(p^T H^-1 p + log|H|)/2 for the diagonal H given (sampler_RHMC.py:353-363)."""
        p = np.asarray(p, dtype=float).ravel()
        # any live context can reduce a diagonal of any length; do not rebuild one just because N changed
        ctx = self._ctx if self._ctx is not None else self._device_ctx(max(1, self._nobjs(p)), need_data=False)
        return ctx.kinetic_diag(p, H_diag)

    def dVdq(self, q):
        q = np.asarray(q, dtype=float).ravel()
        _, grad, _, _ = self._device_ctx(self._nobjs(q)).eval(q[None], g_ff2=self.g_ff2, beta=self.beta)
        return grad[0]

    def dphidq(self, q):
        """dV/dq + (1/2) d ln|H| / dq on the flux slots (sampler_RHMC.py:448-465)."""
        q = np.asarray(q, dtype=float).ravel()
        _, grad, H, Hg = self._device_ctx(self._nobjs(q)).eval(q[None], g_ff2=self.g_ff2, beta=self.beta)
        out = grad[0].copy()
        out[0::3] += (Hg[0][0::3] / H[0][0::3] + 2. * Hg[0][1::3] / H[0][1::3]) / 2.
        return out

    def dtaudq(self, q, p):
        q = np.asarray(q, dtype=float).ravel()
        _, dq, _ = self._device_ctx(self._nobjs(q), need_data=False).kinetic(q[None], np.asarray(p, float)[None],
                                                                              g_ff2=self.g_ff2)
        return dq[0]

    def dtaudp(self, q, p):
        q = np.asarray(q, dtype=float).ravel()
        _, _, dp = self._device_ctx(self._nobjs(q), need_data=False).kinetic(q[None], np.asarray(p, float)[None],
                                                                              g_ff2=self.g_ff2)
        return dp[0]

    def dVdq_RHMC(self, q, p):
        raise NotImplementedError("dVdq_RHMC serves only the naive/leap_frog solvers, which are not part of the "
                                  "B200 path (SURVEY.md section 2)")

    def RHMC_single_step(self, q_tmp, p_tmp, delta=1e-6, counter_max=1000):
        """One generalised (implicit) leapfrog step with reflections (sampler_RHMC.py:522-566) -> new (q, p)."""
        q = np.asarray(q_tmp, dtype=float).ravel()
        p = np.asarray(p_tmp, dtype=float).ravel()
        qn, pn = self._device_ctx(self._nobjs(q)).step(q[None], p[None], 1, self.dt, delta=delta,
                                                       counter_max=counter_max, g_ff2=self.g_ff2, beta=self.beta)
        return qn[0], pn[0]

    # ------------------------------------------------------------------ plotting (out of scope: no-ops)
    def display_image(self, *args, **kwargs):
        return None

    def diagnostics_first(self, *args, **kwargs):
        return None

    def diagnostics_all(self, *args, **kwargs):
        return None


class single_gym(base_class):
    """Single-trajectory energy tests (sampler_RHMC.py:569-881)."""

    def __init__(self, Nsteps=100, dt=0.1, g_xx=1., g_ff=1., g_ff2=1.):
        # the reference forwards g_ff2 = 1. whatever the argument (sampler_RHMC.py:578)
        base_class.__init__(self, dt=dt, g_xx=g_xx, g_ff=g_ff, g_ff2=1.)
        self.Nsteps = Nsteps
        self.q_chain = None
        self.p_chain = None
        self.E_chain = None
        self.V_chain = None
        self.T_chain = None

    def run_single_HMC(self, q_model_0=None, f_pos=False):
        raise NotImplementedError("run_single_HMC is the reference's self-described 'incorrect and naive' demo "
                                  "(sampler_RHMC.py:627); it is not part of the B200 path")

    def run_single_RHMC(self, q_model_0=None, f_pos=False, solver="naive", delta=1e-6, p_initial=None,
                        counter_max=100):
        """One long implicit-leapfrog trajectory; fills q_chain, p_chain [Nsteps+1, 3N] and V/T/E_chain
        [Nsteps+1] (differences from the initial values; row 0 zeros) like sampler_RHMC.py:649-783."""
        if solver != "implicit":
            raise NotImplementedError("only solver='implicit' runs on the B200 path (the reference labels "
                                      "'leap_frog' as not working and 'naive' is first order)")
        self.Nobjs = q_model_0.shape[0]
        self.d = self.Nobjs * 3
        q0 = self.format_q(q_model_0)
        ctx = self._device_ctx(self.Nobjs)
        if p_initial is None:
            H_diag, _ = ctx.metric(q0, self.g_ff2)
            p_initial = self.u_sample(self.d) * np.sqrt(H_diag)
        p0 = np.asarray(p_initial, dtype=float)
        qc, pc, E, V, T = ctx.run_single(q0[None], p0[None], self.Nsteps, self.dt, delta=delta,
                                         counter_max=counter_max, f_pos=f_pos, g_ff2=self.g_ff2, beta=self.beta)
        self.q_chain, self.p_chain = qc[0], pc[0]
        self.E_chain, self.V_chain, self.T_chain = E[0], V[0], T[0]


class multi_gym(base_class):
    """Full RHMC inference (sampler_RHMC.py:883-1198)."""

    def __init__(self, Nsteps=100, dt=0.1, g_xx=1., g_ff=1., g_ff2=1.):
        base_class.__init__(self, dt=dt, g_xx=g_xx, g_ff=g_ff, g_ff2=g_ff2)
        self.Nsteps = Nsteps
        self.q_chain = None
        self.p_chain = None
        self.E_chain = None
        self.V_chain = None
        self.T_chain = None
        self.A_chain = None
        self.fmin = None
        self.fmax = None
        #: None: reversible-jump runs draw from the global np.random stream with the proposals on the host (reference
        #: order).  An int: they run entirely on the device with counter-based Philox draws keyed by this seed.
        self.device_seed = None

    def run_RHMC(self, q_model_0, f_pos=True, delta=1e-6, Niter=100, Nsteps=100, dt=1e-1, save_traj=False,
                 counter_max=1000, verbose=False, q_true=None, schedule_g_ff2=None, N_max=50,
                 P_move=[1., 0., 0.], schedule_beta=None):
        """Same contract as sampler_RHMC.py:937-1198 for within-model moves: chains of Niter+1 rows, row l holding
        the state, momenta and energies at the START of iteration l and A_chain[l] its accept decision."""
        if save_traj:
            assert False  # not supported upstream either (sampler_RHMC.py:966-968)
        self.dt = dt
        self.Niter = Niter
        self.Nsteps = Nsteps
        self.save_traj = save_traj
        self.P_move = P_move
        self.N_max = N_max
        self.Nobjs = q_model_0.shape[0]
        self.d = self.Nobjs * 3
        if self.Nobjs > N_max:
            raise ValueError("N_max = %d is smaller than the %d model stars" % (N_max, self.Nobjs))
        q0 = self.format_q(q_model_0)
        L = Niter + 1

        if float(P_move[1]) != 0.0 or float(P_move[2]) != 0.0:
            if self.device_seed is not None:
                return self._run_RHMC_rj_device(q0, f_pos, delta, counter_max, schedule_g_ff2, schedule_beta)
            return self._run_RHMC_rj(q0, f_pos, delta, counter_max, verbose, schedule_g_ff2, schedule_beta)

        # the reference's draws, in the reference's order (sampler_RHMC.py:1022, 1046, 1075)
        normals = np.empty((L, self.d))
        lnu = np.empty(L)
        for l in range(L):
            normals[l] = self.u_sample(self.d)
            np.random.choice([0, 1, 2], p=self.P_move, size=1)
            lnu[l] = np.log(np.random.random(1))[0]

        ctx = self._device_ctx(self.Nobjs)
        sg = None if schedule_g_ff2 is None else np.asarray(schedule_g_ff2, dtype=float)
        sb = None if schedule_beta is None else np.asarray(schedule_beta, dtype=float)
        r = ctx.run(q0[None], Niter, Nsteps, dt, delta=delta, counter_max=counter_max, f_pos=f_pos,
                    g_ff2=self.g_ff2, beta=self.beta, schedule_g_ff2=sg, schedule_beta=sb,
                    normals=normals[None], lnu=lnu[None])
        # the schedules leave their last applied value on the gym (sampler_RHMC.py:1011-1016)
        if sg is not None and sg.size:
            self.g_ff2 = sg[min(L, sg.size) - 1]
        if sb is not None and sb.size:
            self.beta = sb[min(L, sb.size) - 1]

        self.q_chain = np.zeros((L, N_max * 3))
        self.p_chain = np.zeros((L, N_max * 3))
        self.q_chain[:, :self.d] = r.q_chain[0]
        self.p_chain[:, :self.d] = r.p_chain[0]
        self.E_chain, self.V_chain, self.T_chain = r.E_chain[0], r.V_chain[0], r.T_chain[0]
        self.A_chain = r.A_chain[0].astype(bool)
        self.move_chain = np.zeros(L, dtype=int)
        self.N_chain = np.full(L, self.Nobjs, dtype=int)
        self.kernel_ms = r.kernel_ms

        if verbose:
            for l in range(0, L, 50):
                print("/---- Completed iteration %d" % l)
                print("N_objs: %d\n" % self.Nobjs)
                self.R_accept_report(idx_iter=l, run_window=10)
                print("\n\n")
        print("Finished. Final report.")
        self.R_accept_report(idx_iter=-1, running=False)

    # ------------------------------------------------------------------ reversible-jump leg (SURVEY.md 8f, next #1)
    # The trans-dimensional proposals are host-side bookkeeping exactly as upstream (sampler_RHMC.py:1084-1181,
    # 1200-1445, same np.random / scipy BETA call order); every RHMC leg, V, H and T run on the device through ONE
    # context sized for N_max stars with the live count passed per call.
    def _rj_ctx(self):
        return self._device_ctx(self.N_max)

    def _pad(self, v):
        out = np.zeros((1, 3 * self.N_max))
        out[0, :v.size] = v
        return out

    def _rj_steps(self, q, p, nsteps, delta, counter_max):
        n = q.size // 3
        if n == 0 or nsteps == 0:
            return np.array(q, dtype=float), np.array(p, dtype=float)
        qn, pn = self._rj_ctx().step(self._pad(q), self._pad(p), nsteps, self.dt, delta=delta, counter_max=counter_max,
                                     g_ff2=self.g_ff2, beta=self.beta, nstars=[n])
        return qn[0, :q.size].copy(), pn[0, :p.size].copy()

    def _rj_VH(self, q, f_pos):
        n = q.size // 3
        V, _, H, _ = self._rj_ctx().eval(self._pad(q), nstars=[n], f_pos=f_pos, g_ff2=self.g_ff2, beta=self.beta)
        return float(V[0]), H[0, :q.size].copy()

    def _run_RHMC_rj(self, q0, f_pos, delta, counter_max, verbose, schedule_g_ff2, schedule_beta):
        Niter, Nsteps, N_max = self.Niter, self.Nsteps, self.N_max
        L = Niter + 1
        self.q_chain = np.zeros((L, N_max * 3))
        self.p_chain = np.zeros((L, N_max * 3))
        self.E_chain = np.zeros(L)
        self.V_chain = np.zeros(L)
        self.T_chain = np.zeros(L)
        self.A_chain = np.zeros(L, dtype=bool)
        self.move_chain = np.zeros(L, dtype=int)
        self.N_chain = np.zeros(L, dtype=int)
        q_tmp = np.copy(q0)
        for l in range(L):
            if schedule_g_ff2 is not None and l < schedule_g_ff2.size:
                self.g_ff2 = schedule_g_ff2[l]
            if schedule_beta is not None and l < schedule_beta.size:
                self.beta = schedule_beta[l]
            V_initial, H_diag = self._rj_VH(q_tmp, f_pos)
            p_tmp = self.u_sample(self.d) * np.sqrt(H_diag)
            T_initial = self.T(p_tmp, H_diag) if self.d else 0.0
            E_initial = V_initial + T_initial
            self.q_chain[l, :self.Nobjs * 3] = q_tmp
            self.p_chain[l, :self.Nobjs * 3] = p_tmp
            self.V_chain[l], self.E_chain[l], self.T_chain[l] = V_initial, E_initial, T_initial
            self.N_chain[l] = self.Nobjs
            move_type = np.random.choice([0, 1, 2], p=self.P_move, size=1)[0]
            if move_type == 0:
                self.move_chain[l] = 0
                q_tmp, p_tmp = self._rj_steps(q_tmp, p_tmp, Nsteps, delta, counter_max)
                V_final, H_diag = self._rj_VH(q_tmp, f_pos)
                dE = V_final + self.T(p_tmp, H_diag) - E_initial
                lnu = np.log(np.random.random(1))
                if (dE < 0) or (lnu < -dE):
                    self.A_chain[l] = 1
                else:
                    q_tmp = np.copy(self.q_chain[l, :self.Nobjs * 3])
            else:
                grow = bool(np.random.choice([True, False], p=[0.5, 0.5]))
                if move_type == 1:
                    self.move_chain[l] = 1 if grow else 2
                else:
                    self.move_chain[l] = 3 if grow else 4
                q_tmp, p_tmp = self._rj_steps(q_tmp, p_tmp, Nsteps, delta, counter_max)
                p_tmp = -p_tmp
                if move_type == 1:
                    q_tmp, p_tmp, factor = self.birth_death_move(q_tmp, p_tmp, birth_death=grow)
                else:
                    q_tmp, p_tmp, factor = self.split_merge_move(q_tmp, p_tmp, split_merge=grow)
                if self.Nobjs > N_max:
                    raise ValueError("the proposal needs %d stars but N_max = %d" % (self.Nobjs, N_max))
                q_tmp, p_tmp = self._rj_steps(q_tmp, p_tmp, Nsteps, delta, counter_max)
                p_tmp = -p_tmp
                V_final, H_diag = self._rj_VH(q_tmp, f_pos)
                dE = V_final + (self.T(p_tmp, H_diag) if p_tmp.size else 0.0) - E_initial
                ln_alpha0 = -dE + factor
                lnu = np.log(np.random.random(1))
                if (ln_alpha0 > 0) or (lnu < ln_alpha0):
                    self.A_chain[l] = 1
                else:
                    if grow:
                        self.Nobjs -= 1
                        self.d -= 3
                    else:
                        self.Nobjs += 1
                        self.d += 3
                    q_tmp = np.copy(self.q_chain[l, :self.Nobjs * 3])
            if verbose and ((l % 50) == 0):
                print("/---- Completed iteration %d" % l)
                print("N_objs: %d\n" % self.Nobjs)
                self.R_accept_report(idx_iter=l, run_window=10)
                print("\n\n")
        print("Finished. Final report.")
        self.R_accept_report(idx_iter=-1, running=False)

    def _run_RHMC_rj_device(self, q0, f_pos, delta, counter_max, schedule_g_ff2, schedule_beta):
        """The reversible-jump run as one device launch (RHMCContext.run_rj); same attributes, shapes and dtypes as
        _run_RHMC_rj."""
        if self.fmin is None or self.fmax is None:
            raise TypeError("reversible-jump moves need gym.fmin and gym.fmax (sampler_RHMC.py:1200-1210)")
        sg = None if schedule_g_ff2 is None else np.asarray(schedule_g_ff2, dtype=float)
        sb = None if schedule_beta is None else np.asarray(schedule_beta, dtype=float)
        r = self._rj_ctx().run_rj(self._pad(q0), self.Niter, self.Nsteps, self.dt, nstars=[self.Nobjs], delta=delta,
                                  counter_max=counter_max, f_pos=f_pos, g_ff2=self.g_ff2, beta=self.beta,
                                  schedule_g_ff2=sg, schedule_beta=sb, seed=int(self.device_seed), P_move=self.P_move,
                                  fmin=self.fmin, fmax=self.fmax, K_split=self.K_split, beta_a=self.beta_a,
                                  beta_b=self.beta_b)
        if r.overflow[0] >= 0:
            raise ValueError("the proposal of iteration %d needs %d stars but N_max = %d"
                             % (r.overflow[0], self.N_max + 1, self.N_max))
        L = self.Niter + 1
        if sg is not None and sg.size:
            self.g_ff2 = sg[min(L, sg.size) - 1]
        if sb is not None and sb.size:
            self.beta = sb[min(L, sb.size) - 1]
        self.q_chain, self.p_chain = r.q_chain[0], r.p_chain[0]
        self.E_chain, self.V_chain, self.T_chain = r.E_chain[0], r.V_chain[0], r.T_chain[0]
        self.A_chain = r.A_chain[0].astype(bool)
        self.move_chain = r.move_chain[0].astype(int)
        self.N_chain = r.N_chain[0].astype(int)
        self.Nobjs = int(r.n_final[0])
        self.d = 3 * self.Nobjs
        self.kernel_ms = r.kernel_ms
        print("Finished. Final report.")
        self.R_accept_report(idx_iter=-1, running=False)

    # ------------------------------------------------------------------ trans-dimensional proposals
    # Same proposal densities, acceptance terms and consumption order of the legacy np.random stream as the reference's
    # birth_death_move / split_merge_move (sampler_RHMC.py:1200-1445), written as: draw -> star table edit -> log ratio.
    # Star state is handled as an (N, 3) table of (flux, row, col); every metric the proposal needs comes from ONE
    # srhmc_metric call and the kinetic terms from srhmc_kinetic_diag on the device.
    def _stars_metric(self, *stars):
        """Diagonal metric of a few individual stars in one device call -> one length-3 array per star."""
        flat = np.concatenate([np.asarray(s, dtype=float).ravel() for s in stars])
        H, _ = self._rj_ctx().metric(flat, self.g_ff2)
        return [H[3 * i:3 * i + 3] for i in range(len(stars))]

    def _kinetic_sum(self, moms, metrics):
        """Sum of the kinetic terms T(p, H) of several stars in one device reduction (T is additive over stars)."""
        return self.T(np.concatenate(moms), np.concatenate(metrics))

    def _resize(self, table_q, table_p, log_ratio, d_stars):
        self.Nobjs += d_stars
        self.d += 3 * d_stars
        return table_q.reshape(-1), table_p.reshape(-1), log_ratio

    def birth_death_move(self, q_tmp, p_tmp, birth_death=None):
        """Birth (True) or death (False) proposal; returns (q, p, factor) (sampler_RHMC.py:1200-1273)."""
        if (birth_death is None) or (self.alpha is None) or (self.fmin is None) or (self.fmax is None):
            assert False
        self._prior_const()
        table_q = np.asarray(q_tmp, dtype=float).reshape(-1, 3)
        table_p = np.asarray(p_tmp, dtype=float).reshape(-1, 3)
        if birth_death:
            # draws: row, column, flux from the prior, three normals for the newborn's momentum
            row = np.random.random() * (self.num_rows - 2.) + 1.
            col = np.random.random() * (self.num_cols - 2.) + 1.
            flux = gen_pow_law_sample(self.alpha, self.fmin, self.fmax, 1)[0]
            newborn = np.array([flux, row, col])
            (metric_new,) = self._stars_metric(newborn)
            mom_new = self.u_sample(3) * np.sqrt(metric_new)
            log_ratio = self.alpha * np.log(flux) - 3 / 2. + self.T(mom_new, metric_new) + self.V_prior_const
            return self._resize(np.vstack([table_q, newborn]), np.vstack([table_p, mom_new]), log_ratio, +1)
        victim = np.random.randint(0, self.Nobjs, size=1)[0]
        (metric_old,) = self._stars_metric(table_q[victim])
        log_ratio = (-self.alpha * np.log(table_q[victim, 0]) + 3 / 2. - self.T(table_p[victim], metric_old)
                     - self.V_prior_const)
        return self._resize(np.delete(table_q, victim, axis=0), np.delete(table_p, victim, axis=0), log_ratio, -1)

    def _merge_weights(self, table_q, pdf):
        """Probability of choosing the ordered pair (i, j) for a merge: Beta density of the flux share f_j / (f_i + f_j)
        (zero for equal fluxes, i.e. the diagonal) times the Gaussian split kernel at their separation."""
        flux, rows, cols = table_q[:, 0], table_q[:, 1], table_q[:, 2]
        share = flux / (flux.reshape((-1, 1)) + flux)
        w = pdf(share, self.beta_a, self.beta_b)
        w[np.abs(share - 0.5) < 1e-6] = 0.
        sep_sq = (rows.reshape((-1, 1)) - rows) ** 2 + (cols.reshape((-1, 1)) - cols) ** 2
        w = w * (np.exp(-sep_sq / (2. * self.K_split ** 2)) / (2. * np.pi * self.K_split ** 2))
        return w / np.sum(w)

    def split_merge_move(self, q_tmp, p_tmp, split_merge=None):
        """Split (True) or merge (False) proposal; returns (q, p, factor) (sampler_RHMC.py:1276-1445)."""
        from scipy.stats import beta as BETA  # utils.py:18-21 of the reference

        if split_merge is None:
            assert False
        table_q = np.array(np.asarray(q_tmp, dtype=float).reshape(-1, 3), copy=True)
        table_p = np.array(np.asarray(p_tmp, dtype=float).reshape(-1, 3), copy=True)
        kernel_norm = np.log(2 * np.pi * self.K_split ** 2)
        if split_merge:
            # draws: parent, offset of the pair, flux share, three normals per child
            parent = np.random.randint(0, self.Nobjs, size=1)[0]
            flux_p, row_p, col_p = table_q[parent]
            off_r, off_c = np.random.randn(2) * self.K_split
            share = BETA.rvs(self.beta_a, self.beta_b, size=1)[0]
            z_one, z_two = self.u_sample(3), self.u_sample(3)
            child_one = np.array([share * flux_p, row_p + (1 - share) * off_r, col_p + (1 - share) * off_c])
            child_two = np.array([(1 - share) * flux_p, row_p - share * off_r, col_p - share * off_c])
            m_one, m_two, m_parent = self._stars_metric(child_one, child_two, table_q[parent])
            mom_one, mom_two = z_one * np.sqrt(m_one), z_two * np.sqrt(m_two)
            T_children = self._kinetic_sum([mom_one, mom_two], [m_one, m_two])
            T_parent = self.T(table_p[parent], m_parent)
            log_ratio = ((-3 / 2.) + np.log(flux_p) - BETA.logpdf(share, self.beta_a, self.beta_b) + kernel_norm
                         + ((off_r ** 2 + off_c ** 2) / (2 * self.K_split ** 2)) + T_children - T_parent)
            table_q[parent], table_p[parent] = child_one, mom_one
            return self._resize(np.vstack([table_q, child_two]), np.vstack([table_p, mom_two]), log_ratio, +1)
        # merge: one draw picks the ordered pair, three normals give the merged star's momentum
        n = self.Nobjs
        pick = np.random.choice(range(n ** 2), p=self._merge_weights(table_q, BETA.pdf).ravel())
        one, two = pick // n, pick % n
        share = table_q[one, 0] / (table_q[one, 0] + table_q[two, 0])
        gap_sq = (table_q[one, 1] - table_q[two, 1]) ** 2 + (table_q[one, 2] - table_q[two, 2]) ** 2
        flux_m = table_q[one, 0] + table_q[two, 0]
        merged = np.array([flux_m, share * table_q[one, 1] + (1 - share) * table_q[two, 1],
                           share * table_q[one, 2] + (1 - share) * table_q[two, 2]])
        m_one, m_two, m_merged = self._stars_metric(table_q[one], table_q[two], merged)
        T_pair = self._kinetic_sum([table_p[one], table_p[two]], [m_one, m_two])
        mom_merged = self.u_sample(3) * np.sqrt(m_merged)
        T_merged = self.T(mom_merged, m_merged)
        log_ratio = ((3 / 2.) - np.log(flux_m) + BETA.logpdf(share, self.beta_a, self.beta_b) - kernel_norm
                     - (gap_sq / (2 * self.K_split ** 2)) - T_pair + T_merged)
        keep = np.ones(n, dtype=bool)
        keep[[one, two]] = False
        return self._resize(np.vstack([table_q[keep], merged]), np.vstack([table_p[keep], mom_merged]), log_ratio, -1)

    def R_accept_report(self, idx_iter, cumulative=True, running=True, run_window=10):
        """Acceptance rate so far broken down by move type (sampler_RHMC.py:1447-1473)."""
        def report(A_chain, move_chain):
            for i in range(5):
                ibool = move_chain == i
                Ntot = np.sum(ibool)
                if Ntot > 0:
                    Naccept = np.sum(A_chain[ibool])
                    print("%10s: %.2f%% (%d / %d)" % (self.move_types[i], Naccept / float(Ntot) * 100, Naccept, Ntot))
        if cumulative:
            print("/--Acceptance rate (cumulative)")
            report(self.A_chain[:idx_iter], self.move_chain[:idx_iter])
        if running:
            print("/--Acceptance rate (running: %d)" % run_window)
            report(self.A_chain[idx_iter - run_window:idx_iter], self.move_chain[idx_iter - run_window:idx_iter])
