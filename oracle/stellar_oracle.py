"""CPU oracle for the RHMC leapfrog hot path  --  TEST INFRASTRUCTURE ONLY.

A NumPy float64 restatement of the reference algorithm
(jaekor91/HMC-stellar-toy-model), written from its behaviour, each function
citing the reference file:line it follows.  It is the *checker* for the CUDA
kernels: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
`--impl reference` legs may import it.  The product package never does, and has
no CPU fallback.

Parity pin: the reference has no tests or golden vectors of its own ("parity
unpinned" upstream, SURVEY.md section 4), so this oracle is pinned against the
reference itself executed in the build container through oracle/ref_shim.py:
tests/golden/make_golden.py records the reference's outputs as fixtures and
tests/test_oracle_golden.py checks this file against them (and against the live
reference when SRHMC_REFERENCE_DIR names a checkout).  The arithmetic follows the
reference's operation order so agreement is at the 1e-15 level, not just 1e-10.

Conventions (SURVEY.md section 8 / appendix A): q is a flat float64 array
[f1, x1, y1, f2, ...] with f in counts; x indexes image rows (axis 0), y
columns; pixel (i, j) has its centre at (i + 0.5, j + 0.5); D is float64 [R, C].

The cost structure deliberately mirrors the reference (one full-image PSF per
star, rendered twice per gradient, Python loops over stars) so that timing this
module on host cores is a fair stand-in for the reference's own CPU speed.
"""
from __future__ import annotations

import copy
import math
from dataclasses import dataclass, field

import numpy as np

FWHM_TO_SIGMA = 2.354  # utils.py:480 (not 2.3548)


# --------------------------------------------------------------------------- L1
def mag2flux(mag):
    """utils.py:24-25."""
    return 10 ** (0.4 * (22.5 - mag))


def flux2mag(flux):
    """utils.py:27-28."""
    return 22.5 - 2.5 * np.log10(flux)


def gauss_psf(num_rows, num_cols, x, y, fwhm):
    """Normalised circular Gaussian over the whole image (utils.py:475-486).

    x runs along axis 0.  Same elementwise operation order as the reference:
    square, add, negate, divide by 2*sigma^2, exp, divide by (pi*2)*sigma^2.
    """
    sigma = fwhm / FWHM_TO_SIGMA
    ci = np.arange(0.5, num_rows)[:, None]
    cj = np.arange(0.5, num_cols)[None, :]
    return np.exp(-(np.square(ci - x) + np.square(cj - y)) / (2 * sigma**2)) / (np.pi * 2 * sigma**2)


def psf_factors(num_rows, num_cols, x, y, fwhm):
    """Isolated-star Fisher constants g0, g1, g2 (utils.py:623-644)."""
    li = np.arange(0, num_rows)[:, None] * np.ones((1, num_cols))
    var = (fwhm / FWHM_TO_SIGMA) ** 2
    psf = gauss_psf(num_rows, num_cols, x, y, fwhm)
    psf_sq = np.square(psf)
    g0 = np.sum(psf_sq)
    g1 = np.sum(psf * (x - li - 0.5) ** 2) / float(var**2)
    g2 = np.sum(psf_sq * (x - li - 0.5) ** 2) / float(var**2)
    return g0, g1, g2


def scheduler(val_init, val_final, niter=10):
    """Exponential schedule from val_init to val_final (utils.py:649-660)."""
    c = np.exp(np.log(val_final / float(val_init)) / float(niter - 1))
    return c ** np.arange(0, niter, 1) * val_init


def pow_law_sample(alpha, fmin, fmax, u):
    """Inverse-CDF power-law draw given uniforms u (utils.py:460-471)."""
    alpha = float(alpha)
    lmbda = fmin ** (1 - alpha) + u * (fmax ** (1 - alpha) - fmin ** (1 - alpha))
    return np.exp(np.log(lmbda) / (1 - alpha))


# ------------------------------------------------------------------ experiment
@dataclass
class Setup:
    """Everything the reference keeps as attributes on a gym object.

    Defaults follow base_class.__init__ / default_exp_setup
    (sampler_RHMC.py:28-75, 169-201).  g0..g2 are frozen at the default 48x48
    image exactly as the reference does (compute_factors runs in __init__ and is
    never re-run when scripts shrink the image; SURVEY.md section 5).
    """

    num_rows: int = 48
    num_cols: int = 48
    dt: float = 1.0
    g_xx: float = 10.0
    g_ff: float = 10.0
    g_ff2: float = 2.0
    use_prior: bool = False
    alpha: float = 2.0
    V_prior_const: float | None = None
    fmin: float | None = None
    fmax: float | None = None
    use_Vc: bool = False
    beta: float = 1.0
    Vc_r_pow: float = 1.0
    f_expnt: np.ndarray | None = None
    # experimental constants
    mB: float = 23
    flux_to_count: float = field(default=1.0 / (0.00546689 * 4.62))
    PSF_FWHM_pix: float = field(default=1.4 / 0.4)
    B_count: float = 0.0
    f_lim: float = 0.0
    g0: float = 0.0
    g1: float = 0.0
    g2: float = 0.0
    D: np.ndarray | None = None

    def __post_init__(self):
        if self.B_count == 0.0:
            self.B_count = mag2flux(self.mB) * self.flux_to_count
        if self.f_lim == 0.0:
            self.f_lim = mag2flux(self.mB) * self.flux_to_count
        if self.g0 == 0.0:
            self.g0, self.g1, self.g2 = psf_factors(
                self.num_rows, self.num_cols, self.num_rows / 2.0, self.num_cols / 2.0, self.PSF_FWHM_pix
            )

    # sampler_RHMC.py:147-159
    def mag2flux_converter(self, mag):
        return mag2flux(mag) * self.flux_to_count

    def flux2mag_converter(self, flux):
        return flux2mag(flux / self.flux_to_count)

    def clone(self, **changes):
        other = copy.copy(self)
        for k, v in changes.items():
            setattr(other, k, v)
        return other

    def prior_const(self):
        """Lazy V_prior_const of sampler_RHMC.py:320-321."""
        if self.V_prior_const is None:
            self.V_prior_const = np.log(self.num_rows * self.num_cols) - np.log(
                (1 - self.alpha) / (self.fmax ** (1 - self.alpha) - self.fmin ** (1 - self.alpha))
            )
        return self.V_prior_const


def format_q(S: Setup, q_mag):
    """(N,3) [mag,x,y] -> flat [f,x,y,...] in counts (sampler_RHMC.py:209-217)."""
    q = np.array(q_mag, dtype=float, copy=True)
    for i in range(q.shape[0]):
        q[i, 0] = S.mag2flux_converter(q[i, 0])
    return q.reshape((q.size,))


def model_image(S: Setup, q_flat):
    """B + sum_k f_k PSF_k  (gen_model, sampler_RHMC.py:101-116, flux input)."""
    lam = np.ones((S.num_rows, S.num_cols), dtype=float) * S.B_count
    for k in range(q_flat.size // 3):
        f, x, y = q_flat[3 * k : 3 * k + 3]
        lam += f * gauss_psf(S.num_rows, S.num_cols, x, y, S.PSF_FWHM_pix)
    return lam


# --------------------------------------------------------------------------- L2
def h_ff(S: Setup, f):
    """Flux metric element and the reference's derivative formula
    (sampler_RHMC.py:283-292; the derivative ignores g_ff2 -- kept as is)."""
    c = (S.B_count / S.g0) / S.g_ff
    return 1.0 / (f / S.g_ff2 + c), -1.0 / (f + c) ** 2


def h_xx(S: Setup, f):
    """Position metric element with the faint clamp at mag mB+2
    (sampler_RHMC.py:260-280)."""
    f_low = S.mag2flux_converter(S.mB + 2)
    low = f < f_low
    if low:
        f = f_low
    inner = 1.0 / (S.g1 * f) + S.B_count / (S.g2 * f**2)
    val = S.g_xx * inner**-1
    if low:
        grad = 0
    else:
        grad = S.g_xx * (1.0 / (S.g1 * f**2) + 2 * S.B_count / (S.g2 * f**3)) * inner**-2
    return val, grad


def metric(S: Setup, q, grad=False):
    """Diagonal H and dH/df per star (sampler_RHMC.py:229-258)."""
    n = q.size // 3
    H = np.zeros(q.size)
    dH = np.zeros(q.size)
    for k in range(n):
        f = q[3 * k]
        H[3 * k], dH[3 * k] = h_ff(S, f)
        v, g = h_xx(S, f)
        H[3 * k + 1] = H[3 * k + 2] = v
        dH[3 * k + 1] = dH[3 * k + 2] = g
    return (H, dH) if grad else H


def _inverse_distance(q):
    """Pairwise 1/R with the diagonal forced to 1e-32 (sampler_RHMC.py:334-346)."""
    n = q.size // 3
    qq = np.copy(q.reshape((n, 3)))
    X = qq[:, 1]
    Y = qq[:, 2]
    R = np.sqrt((X - X.reshape((n, 1))) ** 2 + (Y - Y.reshape((n, 1))) ** 2)
    R[np.abs(R) < 1e-10] = 1e32
    return 1.0 / R, X, Y


def potential(S: Setup, q, f_pos=False, rad=0):
    """V(q): Poisson negative log-likelihood + prior + repulsion
    (sampler_RHMC.py:294-351).  +inf outside the support.  rad > 0: the
    likelihood and prior come from patch_eval (every PSF cut to (2 rad + 1)^2
    pixels), the repulsion term is unchanged."""
    n = q.size // 3
    if f_pos:
        for k in range(n):
            if q[3 * k] < S.f_lim:
                return np.inf
    for k in range(n):
        x, y = q[3 * k + 1 : 3 * k + 3]
        if (x < -1) or (x > S.num_rows + 1) or (y < -1) or (y > S.num_cols + 1):
            return np.inf
    if rad > 0:
        V = patch_eval(S, S.D, q, rad)[0]
    else:
        v_prior = 0.0
        vpc = S.prior_const() if (S.V_prior_const is not None or S.fmin is not None) else 0.0
        lam = np.ones_like(S.D) * S.B_count
        for k in range(n):
            f, x, y = q[3 * k : 3 * k + 3]
            lam += f * gauss_psf(S.num_rows, S.num_cols, x, y, S.PSF_FWHM_pix)
            if S.use_prior:
                v_prior += S.alpha * np.log(f) + vpc
        V = np.sum(lam - S.D * np.log(lam))
        if S.use_prior:
            V += v_prior
    if S.use_Vc:
        inv_r, _, _ = _inverse_distance(q)
        V += 0.5 * S.beta * np.sum(inv_r**S.Vc_r_pow)
    return V


def kinetic(p, H):
    """T = (sum p^2/H + sum ln|H|)/2  (sampler_RHMC.py:353-363)."""
    return (np.sum(p**2 / H) + np.sum(np.log(np.abs(H)))) / 2.0


def grad_potential(S: Setup, q, rad=0):
    """dV/dq as residual-weighted PSF reductions (sampler_RHMC.py:365-425).
    rad > 0: the pixel part comes from patch_eval (PSFs cut to (2 rad + 1)^2
    pixels); the prior and repulsion terms are unchanged."""
    n = q.size // 3
    if rad > 0:
        g = patch_eval(S, S.D, q, rad)[1].ravel()
    else:
        g = np.zeros(q.size)
        lam = np.ones_like(S.D) * S.B_count
        for k in range(n):
            f, x, y = q[3 * k : 3 * k + 3]
            lam += f * gauss_psf(S.num_rows, S.num_cols, x, y, S.PSF_FWHM_pix)
        rho = (S.D / lam) - 1.0
        li = np.arange(0, S.num_rows)[:, None] * np.ones((1, S.num_cols), dtype=int)
        mj = np.arange(0, S.num_cols)[None, :] * np.ones((S.num_rows, 1), dtype=int)
        var = (S.PSF_FWHM_pix / FWHM_TO_SIGMA) ** 2
        for k in range(n):
            f, x, y = q[3 * k : 3 * k + 3]
            psf = gauss_psf(S.num_rows, S.num_cols, x, y, S.PSF_FWHM_pix)
            g[3 * k] = -np.sum(rho * psf)
            g[3 * k + 1] = -np.sum(rho * (li - x + 0.5) * psf) * f / var
            g[3 * k + 2] = -np.sum(rho * (mj - y + 0.5) * psf) * f / var
    if S.use_Vc:
        inv_r, X, Y = _inverse_distance(q)
    for k in range(n):
        f, x, y = q[3 * k : 3 * k + 3]
        if S.use_prior:
            g[3 * k] += S.alpha / f
        if S.use_Vc:
            w = inv_r[k, :] ** (S.Vc_r_pow + 2)
            g[3 * k + 1] += S.beta * np.sum(w * (X - x)) * S.Vc_r_pow
            g[3 * k + 2] += S.beta * np.sum(w * (Y - y)) * S.Vc_r_pow
    return g


def patch_eval(S: Setup, D, q, rad=12):
    """V(q) and the PIXEL part of dV/dq (no alpha/f term) with every PSF truncated to the (2 rad + 1)^2 pixel patch
    centred on the pixel containing the star -- the restatement of sampler_RHMC.py:294-351 / 365-425 that fields too
    large for full-image PSFs are checked against (rad = 12 is within 3e-13 of the full-image result, SURVEY 8d).
    q is [n, 3] in counts; D is the data image."""
    q = np.asarray(q, dtype=float).reshape(-1, 3)
    R, C = D.shape
    sig2 = (S.PSF_FWHM_pix / FWHM_TO_SIGMA) ** 2
    norm = 1.0 / (2.0 * np.pi * sig2)
    lam = np.full((R, C), S.B_count)
    boxes = []
    for f, x, y in q:
        mi = int(min(max(np.floor(x), 0), R - 1))
        mj = int(min(max(np.floor(y), 0), C - 1))
        i0, i1, j0, j1 = max(0, mi - rad), min(R - 1, mi + rad), max(0, mj - rad), min(C - 1, mj + rad)
        dx = np.arange(i0, i1 + 1) + 0.5 - x
        dy = np.arange(j0, j1 + 1) + 0.5 - y
        ex = np.exp(-(dx * dx) / (2.0 * sig2))
        ey = np.exp(-(dy * dy) / (2.0 * sig2)) * norm
        lam[i0:i1 + 1, j0:j1 + 1] += f * ex[:, None] * ey[None, :]
        boxes.append((i0, i1, j0, j1, dx, dy, ex, ey))
    V = float(np.sum(lam - D * np.log(lam)))
    if S.use_prior:
        vpc = S.prior_const() if (S.V_prior_const is not None or S.fmin is not None) else 0.0
        V += float(np.sum(S.alpha * np.log(q[:, 0]) + vpc))
    rho = D / lam - 1.0
    g = np.zeros_like(q)
    for k, (i0, i1, j0, j1, dx, dy, ex, ey) in enumerate(boxes):
        w = rho[i0:i1 + 1, j0:j1 + 1] * ex[:, None] * ey[None, :]
        g[k, 0] = -np.sum(w)
        g[k, 1] = -np.sum(w * dx[:, None]) * q[k, 0] / sig2
        g[k, 2] = -np.sum(w * dy[None, :]) * q[k, 0] / sig2
    return V, g


def dphidq(S: Setup, q, rad=0):
    """grad V + half the log-det gradient on flux slots (sampler_RHMC.py:448-465)."""
    g = grad_potential(S, q, rad=rad)
    H, dH = metric(S, q, grad=True)
    for k in range(q.size // 3):
        g[3 * k] += ((dH[3 * k] / H[3 * k]) + (2 * dH[3 * k + 1] / H[3 * k + 1])) / 2.0
    return g


def dtaudq(S: Setup, q, p):
    """-p_f^2 H_ff'/(2 H_ff^2) on flux slots only (sampler_RHMC.py:467-483)."""
    g = np.zeros_like(q)
    H, dH = metric(S, q, grad=True)
    for k in range(q.size // 3):
        g[3 * k] = ((p[3 * k] ** 2) * (-dH[3 * k] / H[3 * k] ** 2)) / 2.0
    return g


def dtaudp(S: Setup, q, p):
    """p / H(q)  (sampler_RHMC.py:485-492)."""
    return p / metric(S, q)


def _per_star_fixed_point(x, update, delta, counter_max):
    """x <- update(x) for every star [3 slots] until that star's own max |x - x'| <= delta or counter_max iterations
    (srhmc_config.fixed_point_mode = 1).  A star's update reads only its own slots, so the stars still iterating see
    the same values as if each ran alone.  Returns x and the largest per-star iteration count."""
    n = x.size // 3
    cnt = np.zeros(n, dtype=int)
    live = cnt < counter_max
    while live.any():
        x_new = update(x)
        more = np.max(np.abs(x - x_new).reshape(n, 3), axis=1) > delta
        x = np.where(np.repeat(live, 3), x_new, x)
        cnt += live
        live &= more & (cnt < counter_max)
    return x, int(cnt.max(initial=0))


def rhmc_step(S: Setup, q, p, delta=1e-6, counter_max=1000, counters=None, rad=0, per_star=False):
    """One generalised (implicit) leapfrog step with reflections
    (base_class.RHMC_single_step, sampler_RHMC.py:522-566; SURVEY appendix A4).
    `counters`, if a list, receives the two fixed-point iteration counts.
    rad > 0: PSFs cut to (2 rad + 1)^2 pixels (see potential).  per_star: each
    star's two fixed-point loops stop on their own (fixed_point_mode = 1); the
    counts are then the maxima over the stars."""
    h = S.dt / 2.0
    p = p - h * dphidq(S, q, rad=rad)

    rho0 = np.copy(p)
    if per_star:
        p, cnt_p = _per_star_fixed_point(p, lambda pp: rho0 - h * dtaudq(S, q, pp), delta, counter_max)
    else:
        dp, cnt_p = np.inf, 0
        while (dp > delta) and (cnt_p < counter_max):
            p_new = rho0 - h * dtaudq(S, q, p)
            dp = np.max(np.abs(p - p_new))
            p = np.copy(p_new)
            cnt_p += 1

    sig0 = np.copy(q)
    if per_star:
        q, cnt_q = _per_star_fixed_point(q, lambda qq: sig0 + h * (dtaudp(S, sig0, p) + dtaudp(S, qq, p)), delta,
                                         counter_max)
    else:
        dq, cnt_q = np.inf, 0
        while (dq > delta) and (cnt_q < counter_max):
            q_new = sig0 + h * (dtaudp(S, sig0, p) + dtaudp(S, q, p))
            dq = np.max(np.abs(q - q_new))
            q = np.copy(q_new)
            cnt_q += 1

    p = p - h * dtaudq(S, q, p)
    p = p - h * dphidq(S, q, rad=rad)

    for k in range(q.size // 3):
        f, x, y = q[3 * k : 3 * k + 3]
        if f < S.f_lim:
            p[3 * k] *= -1.0
        if (x < 0) or (x > S.num_rows - 1):
            p[3 * k + 1] *= -1.0
        if (y < 0) or (y > S.num_cols - 1):
            p[3 * k + 2] *= -1.0
    if counters is not None:
        counters.append((cnt_p, cnt_q))
    return q, p


# --------------------------------------------------------------------------- L3
@dataclass
class Chains:
    q: np.ndarray
    p: np.ndarray
    E: np.ndarray
    V: np.ndarray
    T: np.ndarray
    A: np.ndarray | None = None


def run_rhmc(S: Setup, q0_flat, normals, lnu, niter, nsteps, dt, f_pos=True, delta=1e-6,
             counter_max=1000, schedule_g_ff2=None, schedule_beta=None, rad=0):
    """Within-model RHMC chain (multi_gym.run_RHMC move 0, sampler_RHMC.py:1009-1083;
    SURVEY appendix A5) with injected draws: normals[l] replaces
    np.random.randn(3N) of iteration l and lnu[l] replaces log(np.random.random(1)).
    Row l of every chain array is the state at the START of iteration l; there are
    niter+1 iterations and the outcome of the last is never stored.  rad > 0: PSFs
    cut to (2 rad + 1)^2 pixels (see potential)."""
    S = S.clone(dt=dt)
    d = q0_flat.size
    out = Chains(
        q=np.zeros((niter + 1, d)), p=np.zeros((niter + 1, d)), E=np.zeros(niter + 1),
        V=np.zeros(niter + 1), T=np.zeros(niter + 1), A=np.zeros(niter + 1, dtype=bool),
    )
    q = np.copy(q0_flat)
    for l in range(niter + 1):
        if schedule_g_ff2 is not None and l < schedule_g_ff2.size:
            S.g_ff2 = schedule_g_ff2[l]
        if schedule_beta is not None and l < schedule_beta.size:
            S.beta = schedule_beta[l]
        H = metric(S, q)
        p = normals[l] * np.sqrt(H)
        v0 = potential(S, q, f_pos=f_pos, rad=rad)
        t0 = kinetic(p, H)
        e0 = v0 + t0
        out.q[l], out.p[l], out.V[l], out.E[l], out.T[l] = q, p, v0, e0, t0
        for _ in range(nsteps):
            q, p = rhmc_step(S, q, p, delta=delta, counter_max=counter_max, rad=rad)
        H = metric(S, q)
        e1 = potential(S, q, f_pos=f_pos, rad=rad) + kinetic(p, H)
        dE = e1 - e0
        if (dE < 0) or (lnu[l] < -dE):
            out.A[l] = True
        else:
            q = np.copy(out.q[l])
    return out


def run_single_rhmc(S: Setup, q0_flat, p0, nsteps, dt, f_pos=False, delta=1e-6, counter_max=100, rad=0):
    """One long implicit-solver trajectory recording V-V0, T-T0 every step
    (single_gym.run_single_RHMC, solver="implicit", sampler_RHMC.py:649-783;
    SURVEY appendix A6).  Row 0 keeps q0, p0 and zeros for the energies.
    rad > 0: PSFs cut to (2 rad + 1)^2 pixels (see potential)."""
    S = S.clone(dt=dt)
    d = q0_flat.size
    out = Chains(q=np.zeros((nsteps + 1, d)), p=np.zeros((nsteps + 1, d)), E=np.zeros(nsteps + 1),
                 V=np.zeros(nsteps + 1), T=np.zeros(nsteps + 1))
    q = np.copy(q0_flat)
    p = np.copy(p0)
    H = metric(S, q)
    out.q[0], out.p[0] = q, p
    v0 = potential(S, q, f_pos=f_pos, rad=rad)
    t0 = kinetic(p, H)
    for i in range(1, nsteps + 1):
        q, p = rhmc_step(S, q, p, delta=delta, counter_max=counter_max, rad=rad)
        H = metric(S, q)
        out.q[i], out.p[i] = q, p
        out.V[i] = potential(S, q, f_pos=f_pos, rad=rad) - v0
        out.T[i] = kinetic(p, H) - t0
        out.E[i] = out.V[i] + out.T[i]
    return out


# ------------------------------------------------- samplers.lightsource_gym side
@dataclass
class LightSetup:
    """State of samplers.lightsource_gym (samplers.py:13-42, 1206-1237)."""

    num_rows: int = 48
    num_cols: int = 48
    mB: float = 23
    flux_to_count: float = field(default=1.0 / (0.00546689 * 4.62))
    PSF_FWHM_pix: float = field(default=1.4 / 0.4)
    B_count: float = 0.0
    f_lim: float = 0.0
    factor0: float = 0.0
    factor1: float = 0.0
    factor2: float = 0.0
    D: np.ndarray | None = None

    def __post_init__(self):
        if self.B_count == 0.0:
            self.B_count = mag2flux(self.mB) * self.flux_to_count

    def compute_factors(self):
        """samplers.py:69-75 (uses the CURRENT image size, unlike base_class)."""
        self.factor0, self.factor1, self.factor2 = psf_factors(
            self.num_rows, self.num_cols, self.num_rows / 2.0, self.num_cols / 2.0, self.PSF_FWHM_pix)

    def clone(self, **changes):
        other = copy.copy(self)
        for k, v in changes.items():
            setattr(other, k, v)
        return other


def ls_model(L: LightSetup, q):
    lam = np.ones_like(L.D) * L.B_count
    for k in range(q.size // 3):
        f, x, y = q[3 * k : 3 * k + 3]
        lam += f * gauss_psf(L.num_rows, L.num_cols, x, y, L.PSF_FWHM_pix)
    return lam


def ls_potential(L: LightSetup, q):
    """samplers.py:1137-1150."""
    lam = ls_model(L, q)
    return -np.sum(L.D * np.log(lam) - lam)


def ls_grad(L: LightSetup, q):
    """samplers.py:1108-1134."""
    g = np.zeros(q.size)
    lam = ls_model(L, q)
    rho = (L.D / lam) - 1.0
    li = np.arange(0, L.num_rows)[:, None] * np.ones((1, L.num_cols), dtype=int)
    mj = np.arange(0, L.num_cols)[None, :] * np.ones((L.num_rows, 1), dtype=int)
    var = (L.PSF_FWHM_pix / FWHM_TO_SIGMA) ** 2
    for k in range(q.size // 3):
        f, x, y = q[3 * k : 3 * k + 3]
        psf = gauss_psf(L.num_rows, L.num_cols, x, y, L.PSF_FWHM_pix)
        g[3 * k] = -np.sum(rho * psf)
        g[3 * k + 1] = -np.sum(rho * (li - x + 0.5) * psf) * f / var
        g[3 * k + 2] = -np.sum(rho * (mj - y + 0.5) * psf) * f / var
    return g


def ls_kinetic(p, mass=None):
    """samplers.py:1163-1173."""
    if mass is None:
        return np.dot(p, p) / 2.0
    return (np.sum(p**2 / mass) + np.log(np.abs(np.prod(mass)))) / 2.0


def ls_energy(L: LightSetup, q, p, mass=None):
    """samplers.py:1152-1161."""
    for k in range(q.size // 3):
        if q[3 * k] < L.f_lim:
            return np.inf
    return ls_potential(L, q) + ls_kinetic(p, mass)


def ls_mass_matrix(L: LightSetup, q):
    """M = [1/f, f*factor1, f*factor1] per star (samplers.py:574-625)."""
    M = np.zeros_like(q)
    for k in range(q.size // 3):
        f = q[3 * k]
        M[3 * k] = 1.0 / f
        M[3 * k + 1 : 3 * k + 3] = f * L.factor1
    return M


def ls_dlndet(L: LightSetup, q):
    """samplers.py:636-649."""
    out = np.zeros_like(q)
    for k in range(q.size // 3):
        f = q[3 * k]
        G, dG = 1.0 / f, -1 / f**2
        F, dF = f * L.factor1, L.factor1
        out[3 * k] = 0.5 * (dG / G + 2 * dF / F)
    return out


def ls_dpmp(L: LightSetup, q, p):
    """samplers.py:651-664."""
    out = np.zeros_like(q)
    for k in range(q.size // 3):
        f = q[3 * k]
        pf, px, py = p[3 * k : 3 * k + 3]
        G, dG = 1.0 / f, -1 / f**2
        F, dF = f * L.factor1, L.factor1
        out[3 * k] = -0.5 * (dG * pf**2 / G**2 + (px**2 + py**2) * dF / F**2)
    return out


def ls_efficient(L: LightSetup, q, p, dVdqq_only=False, parts=False):
    """First/second/third diagonal derivatives of V and the Hessian-metric flow
    (lightsource_gym.RHMC_efficient_computation, samplers.py:828-927)."""
    n = q.size // 3
    if not dVdqq_only:
        for k in range(n):
            if q[3 * k] < L.f_lim:
                return np.inf, np.inf, np.inf
    d1 = np.zeros(q.size)
    d2 = np.zeros(q.size)
    d3 = np.zeros(q.size)
    lam = ls_model(L, q)
    rho0 = L.D / lam
    rho1 = 1 - rho0
    rho2 = rho0 / lam
    rho3 = rho2 / lam
    li = (np.arange(0, L.num_rows) + 0.5)[:, None] * np.ones((1, L.num_cols))
    mj = (np.arange(0, L.num_cols) + 0.5)[None, :] * np.ones((L.num_rows, 1))
    var = (L.PSF_FWHM_pix / FWHM_TO_SIGMA) ** 2
    for k in range(n):
        f, x, y = q[3 * k : 3 * k + 3]
        psf = gauss_psf(L.num_rows, L.num_cols, x, y, L.PSF_FWHM_pix)
        psf_sq = psf**2
        psf_cube = psf_sq * psf
        ax = psf * (li - x) / var
        ax_sq = ax**2
        axx = (ax * (li - x) - psf) / var
        axxx = (axx * (li - x) - 2 * ax) / var
        ay = psf * (mj - y) / var
        ay_sq = ay**2
        ayy = (ay * (mj - y) - psf) / var
        ayyy = (ayy * (mj - y) - 2 * ay) / var
        d1[3 * k : 3 * k + 3] = np.array([
            np.sum(rho1 * psf), f * np.sum(rho1 * ax), f * np.sum(rho1 * ay)])
        d2[3 * k : 3 * k + 3] = np.array([
            np.sum(rho2 * psf_sq),
            f**2 * np.sum(rho2 * ax_sq) + f * np.sum(rho1 * axx),
            f**2 * np.sum(rho2 * ay_sq) + f * np.sum(rho1 * ayy)])
        d3[3 * k : 3 * k + 3] = np.array([
            -2 * np.sum(rho3 * psf_cube),
            -f**3 * np.sum(rho3 * ax_sq * ax) + 3 * f**2 * np.sum(rho2 * ax * axx) + f * np.sum(rho1 * axxx),
            -f**3 * np.sum(rho3 * ay_sq * ay) + 3 * f**2 * np.sum(rho2 * ay * ayy) + f * np.sum(rho1 * ayyy)])
    if dVdqq_only:
        return d2
    dqdt = p / d2
    dpdt = -d3 * ((1.0 / d2) - dqdt**2) / 2.0 - d1
    K = np.sum((p**2) / d2) / 2.0 + np.log(np.prod(d2)) / 2.0
    V = -np.sum(L.D * np.log(lam) - lam)
    if parts:
        return dqdt, dpdt, K + V, d1, d2, d3
    return dqdt, dpdt, K + V


@dataclass
class LsChains:
    """Chain outputs of the lightsource_gym samplers, plus diagnostics of the branches the chain took.  HMC_random /
    RHMC_random_diag: `flips` the iterations (1-based) whose trajectory ended in the flip branch, `flip_steps` one
    (iteration, step, flagged, new) entry per leapfrog step that took the flip branch, with the number of flux momenta
    flipped (the flags are never cleared inside an iteration) and the number that crossed f_lim in that step.
    RHMC_random: `breaks` the (iteration, step) pairs where a trajectory stopped on an infinite energy, `abandoned` the
    iteration at which the chain was given up for its acceptance rate (None if it was not)."""
    q: np.ndarray
    E: np.ndarray
    dE: np.ndarray
    A: np.ndarray
    flips: list = field(default_factory=list)
    flip_steps: list = field(default_factory=list)
    breaks: list = field(default_factory=list)
    abandoned: int | None = None


def ls_hmc_random(L: LightSetup, q0, dt, normals, steps, lnu, niter, f_lim=0.0):
    """Identity-mass random-length HMC (lightsource_gym.HMC_random,
    samplers.py:460-572) with injected draws: normals[0] is the initial p_sample,
    normals[i], steps[i-1], lnu[i-1] belong to iteration i >= 1.  Reference quirks
    kept: the flip set `iflip` is never cleared inside an iteration and the final
    half step in the flip branch leaves p_tmp untouched (samplers.py:531-554)."""
    L = L.clone(f_lim=f_lim)
    d = q0.size
    n = d // 3
    out = LsChains(q=np.zeros((niter + 1, d)), E=np.zeros(niter + 1), dE=np.zeros(niter + 1),
                   A=np.zeros(niter))
    out.q[0] = q0
    out.E[0] = ls_energy(L, q0, normals[0])
    e_prev = out.E[0]
    q = np.copy(q0)
    for i in range(1, niter + 1):
        q_init = q
        p = normals[i]
        e0 = ls_energy(L, q, p)
        out.E[i] = e0
        out.dE[i] = e0 - e_prev
        p_half = p - dt * ls_grad(L, q) / 2.0
        iflip = np.zeros(d, dtype=bool)
        flip = False
        for z in range(int(steps[i - 1])):
            flip = False
            q = q + dt * p_half
            for k in range(n):
                if q[3 * k] < L.f_lim:
                    iflip[3 * k] = True
                    flip = True
            if flip:
                new = sum(q[3 * k] < L.f_lim for k in range(n))
                out.flip_steps.append((i, z, int(np.sum(iflip)), int(new)))
                keep = -p_half[iflip]
                p_half = p_half - dt * ls_grad(L, q)
                p_half[iflip] = keep
            else:
                p_half = p_half - dt * ls_grad(L, q)
        if flip:
            out.flips.append(i)
        else:
            p = p_half + dt * ls_grad(L, q) / 2.0
        e1 = ls_energy(L, q, p)
        dE = e1 - e0
        e_prev = e0
        if (dE < 0) or (lnu[i - 1] < -dE):
            out.A[i - 1] = 1
            out.q[i] = q
        else:
            out.q[i] = q_init
            q = q_init
    return out


def ls_rhmc_random_diag(L: LightSetup, q0, dt_global, normals, steps, lnu, niter, f_lim=0.0):
    """Diagonal-mass RHMC (lightsource_gym.RHMC_random_diag, samplers.py:668-825).
    Quirk kept: dpMpdq is always evaluated with the iteration's INITIAL momentum
    p_tmp (samplers.py:781-800)."""
    L = L.clone(f_lim=f_lim)
    d = q0.size
    n = d // 3
    out = LsChains(q=np.zeros((niter + 1, d)), E=np.zeros(niter + 1), dE=np.zeros(niter + 1),
                   A=np.zeros(niter))
    M = ls_mass_matrix(L, q0)
    p_init = normals[0] * np.sqrt(M)
    out.q[0] = q0
    out.E[0] = ls_energy(L, q0, p_init, M)
    e_prev = out.E[0]
    q = np.copy(q0)

    def force(qq, pp):
        return ls_grad(L, qq) + ls_dlndet(L, qq) + ls_dpmp(L, qq, pp)

    for i in range(1, niter + 1):
        q_init = q
        M = ls_mass_matrix(L, q_init)
        p = normals[i] * np.sqrt(M)
        e0 = ls_energy(L, q, p, M)
        out.E[i] = e0
        out.dE[i] = e0 - e_prev
        p_half = p - dt_global / 2.0 * force(q, p)
        iflip = np.zeros(d, dtype=bool)
        flip = False
        for z in range(int(steps[i - 1])):
            flip = False
            M = ls_mass_matrix(L, q)
            q = q + dt_global * p_half / M
            for k in range(n):
                if q[3 * k] < L.f_lim:
                    iflip[3 * k] = True
                    flip = True
            if flip:
                new = sum(q[3 * k] < L.f_lim for k in range(n))
                out.flip_steps.append((i, z, int(np.sum(iflip)), int(new)))
                keep = -p_half[iflip]
                p_half = p_half - dt_global * force(q, p)
                p_half[iflip] = keep
            else:
                p_half = p_half - dt_global * force(q, p)
        if flip:
            out.flips.append(i)
        else:
            p = p_half + dt_global * force(q, p) / 2.0
        M = ls_mass_matrix(L, q)
        e1 = ls_energy(L, q, p, M)
        dE = e1 - e0
        e_prev = e0
        if (dE < 0) or (lnu[i - 1] < -dE):
            out.A[i - 1] = 1
            out.q[i] = q
        else:
            out.q[i] = q_init
            q = q_init
    return out


def ls_rhmc_random(L: LightSetup, q0, dt, normals, steps, lnu, niter, f_lim=0.0):
    """Hessian-metric RHMC (lightsource_gym.RHMC_random, samplers.py:930-1105) with injected draws: normals[i] is the
    p_sample of iteration i (0..niter); steps[i-1], lnu[i-1] belong to iteration i >= 1.  Quirks kept: the position
    test `(x < 0) or (x < num_rows)` (:1038-1043) flags every in-image star, the flags are never cleared inside an
    iteration, flagged momenta are sign-flipped instead of kicked, the state advances in place so a rejection does
    not restore it (:1031), and a chain below 50% acceptance at a multiple of 100 iterations is abandoned."""
    L = L.clone(f_lim=f_lim)
    d = q0.size
    n = d // 3
    out = LsChains(q=np.zeros((niter + 1, d)), E=np.zeros(niter + 1), dE=np.zeros(niter + 1), A=np.zeros(niter))
    q = np.array(q0, dtype=float)
    p = np.zeros(d)
    e_prev = 0.0
    for i in range(niter + 1):
        d2 = ls_efficient(L, q, p, dVdqq_only=True)
        p = normals[i] * np.sqrt(d2)
        dqdt, dpdt, E = ls_efficient(L, q, p)
        if i == 0:
            out.q[0] = q
            out.E[0] = E
            e_prev = E
            continue
        e0 = E
        out.E[i] = e0
        out.dE[i] = e0 - e_prev
        nst = int(steps[i - 1])
        p_half = p + dt * dpdt / 2.0
        flag = np.zeros(d, dtype=bool)
        for z in range(nst):
            dqdt, dpdt, E = ls_efficient(L, q, p_half)
            if E == np.inf:
                out.breaks.append((i, z))
                break
            q += dt * dqdt
            for k in range(n):
                if q[3 * k] < L.f_lim:
                    flag[3 * k] = True
                if (q[3 * k + 1] < 0) or (q[3 * k + 1] < L.num_rows):
                    flag[3 * k + 1] = True
                if (q[3 * k + 2] < 0) or (q[3 * k + 2] < L.num_rows):
                    flag[3 * k + 2] = True
            dt_tmp = dt / 2.0 if z == nst - 1 else dt
            dqdt, dpdt, E = ls_efficient(L, q, p_half)
            neg = -p_half
            p_half = p_half + dt_tmp * dpdt
            p_half[flag] = neg[flag]
        _, _, e1 = ls_efficient(L, q, p_half)
        dE = e1 - e0
        e_prev = e0
        if (dE < 0) or (lnu[i - 1] < -dE):
            out.A[i - 1] = 1
        out.q[i] = q
        if (i % 100) == 0 and np.sum(out.A[:i]) * 100 / float(i) < 50:
            out.abandoned = i
            break
    return out


def ls_single(L: LightSetup, q_single, model_data):
    """V_single and the full dVdq_single on a model_data background (samplers.py:77-127)."""
    f, x, y = q_single
    psf = gauss_psf(L.num_rows, L.num_cols, x, y, L.PSF_FWHM_pix)
    lam = model_data + f * psf
    rho = (L.D / lam) - 1.0
    li = np.arange(0, L.num_rows)[:, None] * np.ones((1, L.num_cols), dtype=int)
    mj = np.arange(0, L.num_cols)[None, :] * np.ones((L.num_rows, 1), dtype=int)
    var = (L.PSF_FWHM_pix / FWHM_TO_SIGMA) ** 2
    g = np.array([-np.sum(rho * psf), -np.sum(rho * (li - x + 0.5) * psf) * f / var,
                  -np.sum(rho * (mj - y + 0.5) * psf) * f / var])
    return -np.sum(L.D * np.log(lam) - lam), g



def ls_find_peaks(L: LightSetup, jitter, linear_pix_density=0.2, dr_tol=1.0, dmag_tol=0.5, mag_lim=None, Nstep=1000,
                  dt_f_coeff=1e-1, dt_xy_coeff=1e-1, no_perturb=False, return_all=False):
    """lightsource_gym.find_peaks (samplers.py:129-254): seeds on a jittered grid, independent gradient descent of every
    seed on a pure-background model until V changes by less than 1e-9 relative (seeds fainter than f_lim disappear),
    then greedy merging of seeds closer than dr_tol pixels and dmag_tol magnitudes.  `jitter` [Nobjs_row*Nobjs_col, 2]
    are the np.random.randn draws in the reference's order (x then y per seed, row-major over the grid).
    return_all: also the per-seed descent results (q, alive, steps) before the merge."""
    if mag_lim is None:
        mag_lim = L.mB - 1.0
    f_lim = mag2flux(mag_lim) * L.flux_to_count
    f_seed = mag2flux(mag_lim - 0.5) * L.flux_to_count
    n_row = int(linear_pix_density * L.num_rows) - 1
    n_col = int(linear_pix_density * L.num_cols) - 1
    spacing = 1 / float(linear_pix_density)
    q_seed = np.zeros((n_row * n_col, 3))
    t = 0
    for i in range(n_row):
        for j in range(n_col):
            # samplers.py:176: the flat index uses the ROW count as stride (harmless for square grids)
            q_seed[i * n_row + j] = [f_seed, spacing * (i + 0.5 + 0.1 * jitter[t, 0]), spacing * (j + 0.5 + 0.1 * jitter[t, 1])]
            t += 1
    if no_perturb:
        return q_seed
    model_data = np.ones((L.num_rows, L.num_cols)) * L.B_count
    alive = np.ones(len(q_seed), dtype=bool)
    steps = np.zeros(len(q_seed), dtype=int)
    for idx in range(len(q_seed)):
        f, x, y = q_seed[idx]
        V_prev, _ = ls_single(L, [f, x, y], model_data)
        for i in range(Nstep):
            _, g = ls_single(L, [f, x, y], model_data)
            dt_f, dt_xy = f * dt_f_coeff, dt_xy_coeff / f
            f -= g[0] * dt_f
            x -= g[1] * dt_xy
            y -= g[2] * dt_xy
            steps[idx] = i + 1
            if f < f_lim:
                alive[idx] = False
                break
            V_cur, _ = ls_single(L, [f, x, y], model_data)
            if np.abs((V_cur - V_prev) / V_prev) < 1e-9:
                break
            V_prev = V_cur
        q_seed[idx] = [f, x, y]
    descended = q_seed.copy()
    merged = merge_peaks(L, q_seed[alive], dr_tol, dmag_tol)
    return (merged, descended, alive, steps) if return_all else merged


def merge_peaks(L: LightSetup, q_seed, dr_tol=1.0, dmag_tol=0.5):
    """Greedy reduction of find_peaks (samplers.py:234-252): keep the first seed, drop every later one within dr_tol
    pixels AND dmag_tol magnitudes of it, repeat on the rest."""
    if q_seed.shape[0] == 0:
        return q_seed
    final = []
    while True:
        ref = q_seed[0]
        final.append(ref)
        q_seed = q_seed[1:, :]
        dist_sq = (q_seed[:, 1] - ref[1]) ** 2 + (q_seed[:, 2] - ref[2]) ** 2
        mag_seed = flux2mag(q_seed[:, 0] / L.flux_to_count)
        mag_ref = flux2mag(ref[0] / L.flux_to_count)
        q_seed = q_seed[np.logical_or(dist_sq > dr_tol**2, np.abs(mag_ref - mag_seed) > dmag_tol)]
        if q_seed.shape[0] == 0:
            break
    return np.vstack(final)


def ls_trial(L: LightSetup, q_start, model_data, dt, normals, steps, lnu, zero_xy):
    """One acceptance-rate trial of HMC_find_best_dt (samplers.py:327-370): single-star HMC on model_data whose
    leapfrog kicks all three momenta with the scalar FLUX gradient (dVdq_single's default f_only=True).
    normals[i], steps[i-1], lnu[i-1] belong to iteration i = 1..n.  Returns the number of accepted proposals."""
    q = np.array(q_start, dtype=float)
    acc = 0
    with np.errstate(invalid="ignore", divide="ignore"):
        for i in range(1, len(steps) + 1):
            q_init = q
            p = np.array(normals[i], dtype=float)
            if zero_xy:
                p[1:] = 0
            e0 = ls_single(L, q, model_data)[0] + np.dot(p, p) / 2.0
            p_half = p - dt * ls_single(L, q, model_data)[1][0] / 2.0
            for _ in range(int(steps[i - 1])):
                q = q + dt * p_half
                p_half = p_half - dt * ls_single(L, q, model_data)[1][0]
            p = p_half + dt * ls_single(L, q, model_data)[1][0] / 2.0
            e1 = ls_single(L, q, model_data)[0] + np.dot(p, p) / 2.0
            dE = e1 - e0
            if (dE < 0) or (lnu[i - 1] < -dE):
                acc += 1
            else:
                q = q_init
    return acc



# --------------------------------------------------------------------------- mock data (SURVEY 8f row 3)
def philox4x32_10(seed, c0, c1, c2, c3):
    """Philox4x32-10 (Salmon et al. 2011) of the counter (c0, c1, c2, c3) under the 64-bit key `seed`; vectorised over
    NumPy arrays.  Same constants and round structure as csrc/common.cuh (the device generator of the chains and of
    the mock data); returns four uint32 arrays."""
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    mask = np.uint64(0xFFFFFFFF)
    c = [np.asarray(v, dtype=np.uint64) & mask for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
        k0 = (k0 + 0x9E3779B9) & 0xFFFFFFFF
        k1 = (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return [v.astype(np.uint32) for v in c]


def philox_u01(a, b):
    """53-bit uniform in (0, 1) from two Philox words (csrc/common.cuh u01)."""
    m = ((a.astype(np.uint64) >> np.uint64(5)) << np.uint64(26)) | (b.astype(np.uint64) >> np.uint64(6))
    return (m.astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def poisson_philox(lam, seed, index_base=0):
    """One Poisson variate per element of `lam` (utils.poisson_realization, utils.py:488-496, calls np.random.poisson
    once per pixel) with the sampling algorithm of NumPy's legacy generator -- multiplication method for lam < 10,
    Hoermann's PTRS transformed rejection (1993) for lam >= 10 (NumPy is an un-vendored, unpinned dependency of the
    reference: restated from the published algorithm) -- driven by counter-based Philox uniforms exactly as
    csrc/poisson.cuh consumes them: element i uses the counters (idx_lo, attempt, idx_hi, 3), idx = index_base + i,
    two uniforms per attempt."""
    from scipy.special import gammaln

    lam = np.asarray(lam, dtype=float)
    flat = lam.ravel()
    out = np.zeros(flat.size)
    idx = np.uint64(index_base) + np.arange(flat.size, dtype=np.uint64)
    lo, hi = idx & np.uint64(0xFFFFFFFF), idx >> np.uint64(32)

    def uniforms(sel, attempt):
        r = philox4x32_10(seed, lo[sel], np.uint64(attempt), hi[sel], np.uint64(3))
        return philox_u01(r[0], r[1]), philox_u01(r[2], r[3])

    # multiplication method
    small = np.nonzero((flat > 0) & (flat < 10.0))[0]
    if small.size:
        enlam = np.exp(-flat[small])
        prod = np.ones(small.size)
        k = np.zeros(small.size)
        live = np.arange(small.size)
        attempt = 0
        while live.size:
            u, v = uniforms(small[live], attempt)
            prod[live] *= u
            done1 = ~(prod[live] > enlam[live])
            cont = live[~done1]
            k[cont] += 1
            prod[cont] *= v[~done1]
            done2 = ~(prod[cont] > enlam[cont])
            k[cont[~done2]] += 1
            live = cont[~done2]
            attempt += 1
        out[small] = k
    # PTRS
    big = np.nonzero(flat >= 10.0)[0]
    if big.size:
        L = flat[big]
        slam, loglam = np.sqrt(L), np.log(L)
        b = 0.931 + 2.53 * slam
        a = -0.059 + 0.02483 * b
        invalpha = 1.1239 + 1.1328 / (b - 3.4)
        vr = 0.9277 - 3.6224 / (b - 2.0)
        res = np.zeros(big.size)
        live = np.arange(big.size)
        attempt = 0
        while live.size:
            U, V = uniforms(big[live], attempt)
            U = U - 0.5
            us = 0.5 - np.abs(U)
            k = np.floor((2.0 * a[live] / us + b[live]) * U + L[live] + 0.43)
            acc = (us >= 0.07) & (V <= vr[live])
            rej = ~acc & ((k < 0.0) | ((us < 0.013) & (V > us)))
            rest = ~acc & ~rej
            with np.errstate(invalid="ignore", divide="ignore"):
                lhs = np.log(V) + np.log(invalpha[live]) - np.log(a[live] / (us * us) + b[live])
                rhs = -L[live] + k * loglam[live] - gammaln(np.where(k >= 0, k, 0.0) + 1.0)
            acc = acc | (rest & (lhs <= rhs))
            res[live[acc]] = k[acc]
            live = live[~acc]
            attempt += 1
        out[big] = res
    return out.reshape(lam.shape)


# --------------------------------------------------------------------------- chain statistics (SURVEY 8f row 4)
def variogram(chains, var_num, t_lag):
    """BDA3 (11.7) variogram of `chains` (list of [n, D] arrays) at lag t (utils.py:170-188)."""
    m = len(chains)
    n = chains[0].shape[0]
    V_t = 0.0
    for i in range(m):
        c = chains[i][:, var_num]
        V_t += np.sum(np.square(c[t_lag:] - c[:-t_lag]))
    return V_t / float(m * (n - t_lag))


def convergence_stats(q_chain, thin_rate=5, warm_up_num=0):
    """Split-chain Gelman-Rubin R and effective sample size per variable (utils.convergence_stats, utils.py:86-167),
    with the reference's Python-2 integer division `n = L_chain/2` (utils.py:111) and its quirks kept: W is the mean of
    the within-chain standard DEVIATIONS (np.std, utils.py:120), and the first autocorrelation is tested twice
    (utils.py:144).  q_chain [Nchain, Niter, D]."""
    Nchain, Niter, D = q_chain.shape
    assert Nchain > 1
    chains = []
    n = 0
    for m in range(Nchain):
        c = q_chain[m, warm_up_num:, :][::thin_rate, :]
        L_chain = c.shape[0]
        if L_chain % 2:
            c = c[: L_chain - 1]
        n = L_chain // 2
        chains.append(c[:n])
        chains.append(c[n:])
    m = len(chains)
    W = np.mean(np.array([np.std(c, ddof=1, axis=0) for c in chains]), axis=0)
    mean_within = np.array([np.mean(c, axis=0) for c in chains])
    mean_all = np.mean(mean_within, axis=0)
    B = np.sum(np.square(mean_within - mean_all), axis=0) * n / float(m - 1)
    var = W * (n - 1) / float(n) + B / float(n)
    R = np.sqrt(var / W)
    n_eff = np.zeros(D)
    for i in range(D):
        rho_t1 = 1.0 - variogram(chains, i, 1) / (2 * var[i])
        rho_t2 = 1.0 - variogram(chains, i, 2) / (2 * var[i])
        if rho_t1 < 5e-2:
            sum_rho = 0
        else:
            rho_t = [rho_t1, rho_t2]
            t = 1
            while t < n - 2:
                rho_t.append(1 - variogram(chains, i, t + 2) / (2 * var[i]))
                if (t % 2) == 1 and (rho_t[t] + rho_t[t + 1]) < 0:
                    break
                t += 1
            sum_rho = np.sum(rho_t[:t])
            if sum_rho < 0:
                sum_rho = 0
        n_eff[i] = m * n / (1 + 2 * sum_rho)
    return R, n_eff


def acceptance_rate(decision_chain, start=None, end=None):
    """Fraction of accepted proposals per chain (utils.acceptance_rate, utils.py:192-209); decision_chain [Nchain, Niter, 1]."""
    _, Niter, _ = decision_chain.shape
    if start is None and end is None:
        return np.sum(decision_chain, axis=(1, 2)) / Niter
    Niter = (end - start) if end > 0 else (Niter - start)
    return np.sum(decision_chain[:, start:end, :], axis=(1, 2)) / Niter


def star_steps(niter_plus_one: int, nsteps: int, nstars: int) -> int:
    """Units of BASELINE.json's metric produced by one run_rhmc call."""
    return niter_plus_one * nsteps * nstars


__all__ = [n for n in dir() if not n.startswith("_") and n not in ("np", "math", "copy", "dataclass", "field", "annotations")]
