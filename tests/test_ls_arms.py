"""Every launch arm of the lightsource-family kernel (ls_kernel<double, MR, MC>, ls_kernel.cuh) against the float64 oracle.
configure() (stellar_rhmc.cu) picks the arm from the image shape, the star count and whether the context keeps the 1/Lambda
image of the Hessian path (enable_hessian): 128 / 256 / 512 threads, the (2,4) / (2,2) / (1,2) register tile, one or several
table chunks, and the data image in shared or in global memory.  Each row below chooses its shape to land on one arm, first
asserts that it did (RHMCContext.launch_plan), then compares the variants it runs with the oracle: the Hessian reductions
(hessian(), RHMC_efficient_computation), V and dV/dq on a background image (eval_background, V_single / dVdq_single), the
chains of HMC_random, RHMC_random_diag and RHMC_random with injected draws, and the step-size trial of HMC_find_best_dt.

The rows also reach the branches where the reference's quirks show: a star just above f_lim so that trajectories end in
the flip branch while the other stars keep being kicked; a Hessian-metric chain whose energy becomes infinite in the middle
of a trajectory; a chain abandoned for its acceptance rate at iteration 100; stars just outside the image; a wide image with
a star whose y is not below num_rows; trajectories of length 0.  The oracle records which of these it took (LsChains.flips,
breaks, abandoned) and each row asserts that its edges were reached.  The last test checks that the rows together still
cover every arm."""
import contextlib
import functools
import io
from dataclasses import dataclass, field

import numpy as np
import pytest

import stellar_oracle as so
from helpers import first_divergence, relerr

RTOL = 1e-10
F2C = so.LightSetup().flux_to_count
F_EDGE = so.mag2flux(22.0) * F2C  # the scripts' f_lim (one-star-inference-single.py): flip rows start a star just above it



def FLIP_STARS(n):
    """Stars of a flip row's field that are as faint as f_lim: two, so that a flip step can find an older flag set."""
    return 1 if n < 3 else 2

# every plan a test asserted, with what it ran: the last test checks that together they cover every arm
PLANS = []


@dataclass(frozen=True)
class Row:
    R: int
    C: int
    N: int
    hess: bool
    expect: dict = field(hash=False)
    variants: str = ""         # hess bg hmc diag rhmc trial
    nstars: tuple = ()         # one entry per field; () = one field with N stars
    shared: bool = False
    mags: tuple = (19.0, 20.5)  # magnitude range of the stars
    edges: str = ""            # flip: a star just above f_lim (hmc, diag); div: f_lim crossed inside a trajectory (rhmc);
                               # outside: stars just outside the image; wide: a star with num_rows <= y < num_cols
    niter: int = 10
    noise: bool = True          # False: the data image is the model image itself (crowded rows: no negative curvature)


ROWS = {
    "a": Row(16, 16, 3, True, dict(threads=128, tile=(1, 2), chunks=1, image_in_smem=1), "hess bg hmc diag rhmc",
             edges="div"),
    "b": Row(8, 40, 2, True, dict(threads=256, tile=(1, 2), chunks=1), "hess bg hmc diag rhmc", edges="wide"),
    "c": Row(24, 40, 6, True, dict(threads=256, tile=(2, 2), chunks=1), "hess bg hmc diag", edges="flip outside"),
    "d": Row(40, 24, 6, True, dict(threads=256, tile=(2, 2), chunks=1), "hess bg hmc diag rhmc",
             edges="flip sticky outside"),
    "e": Row(48, 48, 3, True, dict(threads=256, tile=(2, 4), chunks=1), "hess bg hmc diag rhmc", edges="div"),
    "f": Row(40, 56, 12, True, dict(tile=(2, 4), chunks=1), "hess bg hmc diag rhmc", edges="flip"),
    "g": Row(48, 48, 300, True, dict(threads=512, tile=(2, 2), chunks=12), "hess bg hmc", mags=(17.5, 19.0), niter=3,
             noise=False),
    "h": Row(48, 48, 300, False, dict(threads=512, tile=(2, 2), chunks=7), "bg hmc", mags=(20.0, 21.5), edges="flip",
             niter=3),
    "i": Row(32, 32, 300, True, dict(threads=512, tile=(1, 2), chunks=4), "hess bg hmc", mags=(15.0, 16.5), niter=3,
             noise=False),
    "j": Row(96, 96, 20, True, dict(chunks=1, image_in_smem=0), "hess bg hmc diag rhmc", niter=4),
    "k": Row(96, 96, 150, True, dict(chunks=4, image_in_smem=0), "hess bg hmc", mags=(20.0, 21.5), niter=3),
    "l": Row(100, 100, 20, False, dict(chunks=1, image_in_smem=1), "bg hmc diag", edges="flip", niter=4),
    "m": Row(128, 128, 1, False, dict(image_in_smem=0), "bg hmc diag trial", niter=4),
    "n": Row(32, 32, 30, True, dict(chunks=1), "hess bg hmc diag rhmc", nstars=(30, 0, 1, 17), edges="flip"),
    "n-shared": Row(32, 32, 30, True, dict(chunks=1), "hess bg hmc diag", nstars=(30, 0, 1, 17), shared=True,
                    edges="flip", noise=False),
}


def _rows(variant):
    return [name for name, r in ROWS.items() if variant in r.variants.split()]


def _setup(row, D=None):
    L = so.LightSetup(num_rows=row.R, num_cols=row.C, D=D)
    L.compute_factors()
    return L


@functools.lru_cache(maxsize=None)
def _inputs(name):
    """Per field: the data image, a start state near the true stars, a background image for eval_background, and the chain
    draws (normals, trajectory lengths with some zeros, ln u)."""
    row = ROWS[name]
    rng = np.random.RandomState(sum(map(ord, name)))
    counts = list(row.nstars) or [row.N]
    L = _setup(row)

    def stars(n):
        f = so.mag2flux(rng.uniform(row.mags[0], row.mags[1], n)) * F2C
        x, y = rng.uniform(1, row.R - 1, n), rng.uniform(1, row.C - 1, n)
        if "outside" in row.edges.split():  # star 1 just above the first row, star 2 just below the last column
            x[1], y[2] = -0.6, row.C + 0.7
        if "wide" in row.edges.split():     # star 0 at num_rows <= y < num_cols, star 1 at y < num_rows
            y[0], y[1] = 0.6 * row.C, 0.4 * row.R
        if "flip" in row.edges.split() and n >= 2:  # stars as faint as f_lim: their chains cross it
            f[: FLIP_STARS(n)] = F_EDGE
        return np.stack([f, x, y], axis=1)

    def image(t):
        lam = so.ls_model(L.clone(D=np.zeros((row.R, row.C))), t.ravel())
        return rng.poisson(lam).astype(float) if row.noise else lam

    truth = stars(row.N)
    shared_D = image(truth) if row.shared else None
    S = 3 * row.N
    D, q = [], np.zeros((len(counts), S))
    for fi, n in enumerate(counts):
        t = truth[:n] if row.shared else stars(n)
        D.append(shared_D if row.shared else image(t))
        q0 = t * np.array([1.03, 1.0, 1.0]) + np.concatenate([np.zeros((n, 1)), 0.1 * rng.randn(n, 2)], axis=1)
        q[fi, : 3 * n] = q0.ravel()
    ii, jj = np.meshgrid(np.arange(row.R), np.arange(row.C), indexing="ij")
    bg = np.stack([L.B_count * (1.0 + 0.3 * np.sin(ii / 5.0 + fi) * np.cos(jj / 7.0)) + 2.0 for fi in range(len(counts))])
    niter = row.niter
    normals = rng.randn(len(counts), niter + 1, S)
    steps = rng.randint(0, 7, size=(len(counts), niter)).astype(np.int32)
    steps[:, 1] = 0
    lnu = np.log(rng.random_sample((len(counts), niter)))
    return counts, D, q, bg, normals, steps, lnu


def _field(name, fi):
    counts, D, q, *_ = _inputs(name)
    n = counts[fi]
    return _setup(ROWS[name], D[fi]), n, q[fi, : 3 * n]


def _q_flip(name):
    """Start state of the hmc / diag chains: in flip rows the first star of every field with two or more stars starts 1 %
    above f_lim = F_EDGE."""
    counts, _, q, *_ = _inputs(name)
    q = q.copy()
    if "flip" in ROWS[name].edges.split():
        for fi, n in enumerate(counts):
            if n >= 2:
                q[fi, 0 : 3 * FLIP_STARS(n) : 3] = 1.01 * F_EDGE
    return q


def _hmc_dt(name):
    """HMC_find_best_dt(default=True, dt_f_coeff=0.05, dt_xy_coeff=2) of the start state, padded to max_stars."""
    row = ROWS[name]
    q = _q_flip(name)[0].reshape(-1, 3)
    f = np.where(q[:, 0] > 0, q[:, 0], 400.0)
    return np.stack([0.05 * f, 2.0 / f, 2.0 / f], axis=1).ravel()[: 3 * row.N]


DIAG_DT = 5e-2
HESS_DT_F, HESS_DT_XY = 0.1, 0.3  # dt_RHMC_f default of RHMC_random, dt_RHMC_xy of the scripts


def _hess_dt(N):
    return np.tile([HESS_DT_F, HESS_DT_XY, HESS_DT_XY], N)


def _hess_flim(name, fi):
    """f_lim of the rhmc chain: 0, or in div rows 1 % below the faintest start flux."""
    _, n, q = _field(name, fi)
    return 0.99 * np.min(q[0::3]) if ("div" in ROWS[name].edges.split() and n) else 0.0


# ------------------------------------------------------------------------------------------------ oracle, once per module
def _oracle_bg(L, q, bg):
    """V_single / dVdq_single generalised to N stars: V and dV/dq of the stars on a per-pixel background image."""
    lam = np.array(bg, dtype=float)
    psfs = []
    for k in range(q.size // 3):
        psfs.append(so.gauss_psf(L.num_rows, L.num_cols, q[3 * k + 1], q[3 * k + 2], L.PSF_FWHM_pix))
        lam = lam + q[3 * k] * psfs[-1]
    rho = L.D / lam - 1.0
    li = np.arange(L.num_rows)[:, None] + 0.5
    mj = np.arange(L.num_cols)[None, :] + 0.5
    var = (L.PSF_FWHM_pix / so.FWHM_TO_SIGMA) ** 2
    g = np.zeros(q.size)
    for k, psf in enumerate(psfs):
        f, x, y = q[3 * k : 3 * k + 3]
        g[3 * k : 3 * k + 3] = [-np.sum(rho * psf), -np.sum(rho * (li - x) * psf) * f / var,
                                -np.sum(rho * (mj - y) * psf) * f / var]
    return -np.sum(L.D * np.log(lam) - lam), g


def _momentum(name, fi):
    """The momentum of the hessian() rows: p ~ N(0, |d2|)."""
    L, n, q = _field(name, fi)
    rng = np.random.RandomState(100 + fi)
    return rng.randn(3 * n) * np.sqrt(np.abs(so.ls_efficient(L, q, np.zeros(3 * n), dVdqq_only=True)))


def _oracle_hess(name):
    out = []
    for fi in range(len(_inputs(name)[0])):
        L, n, q = _field(name, fi)
        out.append(so.ls_efficient(L, q, _momentum(name, fi), parts=True))
    return out


def _oracle_bgv(name):
    counts, _, _, bg, *_ = _inputs(name)
    return [_oracle_bg(_field(name, fi)[0], _field(name, fi)[2], bg[fi]) for fi in range(len(counts))]


def _oracle_chain(name, variant):
    counts, _, _, _, normals, steps, lnu = _inputs(name)
    out = []
    qf = _q_flip(name)
    for fi, n in enumerate(counts):
        L, _, q = _field(name, fi)
        Z, st, lu, niter = normals[fi, :, : 3 * n], steps[fi], lnu[fi], ROWS[name].niter
        if variant == "hmc":
            out.append(so.ls_hmc_random(L, qf[fi, : 3 * n], _hmc_dt(name)[: 3 * n], Z, st, lu, niter, f_lim=F_EDGE))
        elif variant == "diag":
            out.append(so.ls_rhmc_random_diag(L, qf[fi, : 3 * n], DIAG_DT, Z, st, lu, niter, f_lim=F_EDGE))
        else:
            out.append(so.ls_rhmc_random(L, q, _hess_dt(n), Z, st, lu, niter, f_lim=_hess_flim(name, fi)))
    return out


@pytest.fixture(scope="module")
def oracle():
    """oracle(kind, row): the oracle's results for a row, computed on first use and kept for the module."""
    cache = {}

    def get(kind, name):
        if (kind, name) not in cache:
            cache[kind, name] = (_oracle_hess(name) if kind == "hess" else _oracle_bgv(name) if kind == "bg"
                                 else _oracle_chain(name, kind))
        return cache[kind, name]

    return get


# ------------------------------------------------------------------------------------------------ device side
def _ctx(name, variant, hess=None):
    from hmc_stellar_toy_model_b200 import RHMCContext

    row = ROWS[name]
    counts, D, *_ = _inputs(name)
    L = _setup(row)
    ctx = RHMCContext(n_fields=len(counts), num_rows=row.R, num_cols=row.C, max_stars=row.N, psf_fwhm_pix=L.PSF_FWHM_pix,
                      B_count=L.B_count, f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, g_xx=1.0, g_ff=1.0,
                      shared_data=row.shared, enable_hessian=row.hess if hess is None else hess)
    ctx.set_data(D[0] if row.shared else np.stack(D))
    _check_plan(ctx, row, name, variant)
    return ctx


def _check_plan(ctx, row, name, variant):
    """Record the context's plan and assert the row's expectations of it."""
    plan = ctx.launch_plan()
    PLANS.append(dict(plan, row=name, variant=variant, hess=bool(ctx.cfg.enable_hessian), ragged=bool(row.nstars),
                      shared_data=bool(ctx.cfg.shared_data), chunks=-(-max(row.N, 1) // plan["chunk_stars"])))
    got = dict(threads=plan["threads"], tile=(plan["tile_rows"], plan["tile_cols"]), chunks=PLANS[-1]["chunks"],
               image_in_smem=plan["image_in_smem"])
    for key, want in row.expect.items():
        assert got[key] == want, (name, key, got)
    assert plan["compact_tables"] == 0 and plan["smem_bytes"] <= 232448, plan


def _ns(name):
    row = ROWS[name]
    return list(row.nstars) if row.nstars else None


def _close(a, b, tol):
    """Relative to the per-coordinate scale, with a floor at 1e-3 of the largest value of each coordinate type."""
    a, b = np.asarray(a).reshape(-1, 3), np.asarray(b).reshape(-1, 3)
    if not b.size:
        return True
    scale = np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b), axis=0, keepdims=True))
    return float(np.max(np.abs(a - b) / scale)) < tol


def _same_nonfinite(a, b):
    """Same positions of inf (with sign) and NaN."""
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return (np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.isinf(a), np.isinf(b))
            and np.array_equal(a[np.isinf(b)], b[np.isinf(b)]))


def _check_energy_product(d2):
    """The kernel computes ln|prod d2| as sum ln|d2| (DESIGN 4.3), the oracle as np.log(np.prod(d2)): they agree where the
    product is a finite nonzero double, so a row must stay there."""
    prod = np.prod(d2)
    assert np.isfinite(prod) and prod != 0.0, prod


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("hess"))
def test_hessian_arm(name, oracle):
    """RHMC_efficient_computation: d1, d2, d3, dq/dt, dp/dt and E; d2_only gives the same d2 bit for bit.  One star below
    f_lim, the last of its field (outside chunk 0 in the multi-chunk rows), makes E, dq/dt and dp/dt of its field
    infinite; the same f_lim with that star above it changes nothing."""
    counts, _, q, *_ = _inputs(name)
    p = np.zeros_like(q)
    for fi, n in enumerate(counts):
        p[fi, : 3 * n] = _momentum(name, fi)
    with _ctx(name, "hess") as ctx:
        d1, d2, d3, dq, dp, E = ctx.hessian(q, p, nstars=_ns(name))
        only = ctx.hessian(q, d2_only=True, nstars=_ns(name))
        PLANS.append(dict(PLANS[-1], variant="d2_only"))
        f_lim = 0.5 * min(np.min(q[fi, 0 : 3 * n : 3]) for fi, n in enumerate(counts) if n)
        q_low = q.copy()
        for fi, n in enumerate(counts):
            if n:
                q_low[fi, 3 * (n - 1)] = 0.5 * f_lim
        _, _, _, dql, dpl, El = ctx.hessian(q_low, p, f_lim=f_lim, nstars=_ns(name))
        Ef = ctx.hessian(q, p, f_lim=f_lim, nstars=_ns(name))[5]
    assert np.array_equal(d2, only)
    for fi, n in enumerate(counts):
        odq, odp, oE, o1, o2, o3 = oracle("hess", name)[fi]
        _check_energy_product(o2)
        assert _close(d1[fi, : 3 * n], o1, 1e-9) and _close(d2[fi, : 3 * n], o2, 1e-9), fi
        assert _close(d3[fi, : 3 * n], o3, 1e-8), fi
        assert _close(dq[fi, : 3 * n], odq, 1e-9) and _close(dp[fi, : 3 * n], odp, 1e-8), fi
        assert relerr(E[fi], oE) < RTOL, (fi, E[fi], oE)
        assert not np.any(d1[fi, 3 * n:]) and not np.any(d2[fi, 3 * n:])
        assert relerr(Ef[fi], oE) < RTOL, fi
        if n:
            L, _, _ = _field(name, fi)
            assert so.ls_efficient(L.clone(f_lim=f_lim), q_low[fi, : 3 * n], p[fi, : 3 * n]) == (np.inf, np.inf, np.inf)
            assert El[fi] == np.inf and np.all(dql[fi, : 3 * n] == np.inf) and np.all(dpl[fi, : 3 * n] == np.inf), fi
        else:
            assert relerr(El[fi], oE) < RTOL


@pytest.mark.gpu
@pytest.mark.parametrize("shift, negatives", [((0.0, 3.0), 1), ((3.0, 3.0), 2)])
def test_hessian_sign_of_the_curvature_product(shift, negatives):
    """Row "a" with its first star moved off its light by three pixels, where the data have a deficit against the model: the
    moved axes get a negative curvature d2.  With one negative d2 the product is negative, so the reference's
    np.log(np.prod(d2)) and E are NaN, and the kernel's sum of ln|d2| must give NaN too; with two the product is positive
    and E agrees to 1e-10."""
    L, n, q = _field("a", 0)
    q = q.copy()
    q[1:3] += shift
    p = np.random.RandomState(8).randn(3 * n) * np.sqrt(np.abs(so.ls_efficient(L, q, np.zeros(3 * n), dVdqq_only=True)))
    with np.errstate(invalid="ignore"):
        odq, odp, oE, o1, o2, o3 = so.ls_efficient(L, q, p, parts=True)
    assert np.sum(o2 < 0) == negatives and np.isfinite(np.prod(o2)) and np.prod(o2) * (-1) ** negatives > 0, o2
    with _ctx("a", "hess") as ctx:
        d1, d2, d3, dq, dp, E = ctx.hessian(q[None], p[None])
    assert _close(d1[0], o1, 1e-9) and _close(d2[0], o2, 1e-9) and _close(d3[0], o3, 1e-8)
    assert _close(dq[0], odq, 1e-9) and _close(dp[0], odp, 1e-8)
    if negatives % 2:
        assert np.isnan(oE) and np.isnan(E[0]), (oE, E[0])
    else:
        assert relerr(E[0], oE) < RTOL, (E[0], oE)


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("bg"))
def test_background_arm(name, oracle):
    counts, _, q, bg, *_ = _inputs(name)
    with _ctx(name, "bg") as ctx:
        V, g = ctx.eval_background(q, bg, nstars=_ns(name))
    for fi, n in enumerate(counts):
        Vo, go = oracle("bg", name)[fi]
        assert relerr(V[fi], Vo) < RTOL, (fi, V[fi], Vo)
        assert _close(g[fi, : 3 * n], go, 1e-9), fi
        assert not np.any(g[fi, 3 * n:])


def _check_chain(r, fi, n, out, niter):
    """A_chain exactly, q_chain to 1e-9, E_chain to 1e-10 (same infinities), dE_chain to 1e-7 absolute (same NaN / inf),
    q_final and the accept count."""
    assert np.array_equal(r["A_chain"][fi].astype(bool), out.A.astype(bool)), (fi, r["A_chain"][fi], out.A)
    assert first_divergence(r["q_chain"][fi][:, : 3 * n], out.q, 1e-9) == -1, fi
    E, dE = r["E_chain"][fi], r["dE_chain"][fi]
    assert _same_nonfinite(E, out.E) and _same_nonfinite(dE, out.dE), (fi, E, out.E)
    fin = np.isfinite(out.E)
    assert relerr(E[fin], out.E[fin]) < RTOL, fi
    fin = np.isfinite(out.dE)
    assert np.max(np.abs(dE[fin] - out.dE[fin]), initial=0.0) < 1e-7, fi
    last = out.abandoned if out.abandoned is not None else niter
    assert relerr(r["q_final"][fi, : 3 * n], out.q[last]) < 1e-9, fi
    assert r["accept_count"][fi] == np.sum(out.A), fi


def _check_oracle_energies(out):
    """The oracle's energies are finite (so its np.log(np.prod(d2)) neither overflowed nor met a negative product) until
    the chain's fluxes fall below f_lim, and +inf from there on: RHMC_random restores nothing, so such a chain stays
    stuck, and a trajectory that meets an infinite energy stops (out.breaks)."""
    E = out.E
    bad = ~np.isfinite(E)
    first = int(np.argmax(bad)) if bad.any() else len(E)
    assert np.all(E[first:] == np.inf), E
    assert first == len(E) or out.breaks, E


@pytest.mark.gpu
@pytest.mark.parametrize("name, variant", [(name, v) for name in ROWS for v in ("hmc", "diag", "rhmc")
                                           if v in ROWS[name].variants.split()])
def test_chain_arm(name, variant, oracle):
    from hmc_stellar_toy_model_b200 import RHMCContext as R

    row = ROWS[name]
    counts, _, q, _, normals, steps, lnu = _inputs(name)
    outs = oracle(variant, name)
    with _ctx(name, variant) as ctx:
        if variant == "hmc":
            r = ctx.ls_run(R.LS_HMC, _q_flip(name), _hmc_dt(name), normals, steps, lnu, f_lim=F_EDGE, nstars=_ns(name))
        elif variant == "diag":
            r = ctx.ls_run(R.LS_DIAG, _q_flip(name), [DIAG_DT], normals, steps, lnu, f_lim=F_EDGE,
                           factor1=_setup(row).factor1, nstars=_ns(name))
        else:
            flims = {_hess_flim(name, fi) for fi in range(len(counts))}
            assert len(flims) == 1, flims
            r = ctx.ls_run(R.LS_HESS, q, _hess_dt(row.N), normals, steps, lnu, f_lim=flims.pop(), nstars=_ns(name))
    for fi, n in enumerate(counts):
        out = outs[fi]
        _check_oracle_energies(out)
        _check_chain(r, fi, n, out, row.niter)
    if "flip" in row.edges.split() and variant in ("hmc", "diag"):
        assert any(o.flip_steps for o in outs), "no trajectory took the flip branch"
    if "sticky" in row.edges.split() and variant in ("hmc", "diag"):
        assert any(flagged > new for o in outs for _, _, flagged, new in o.flip_steps), "no flip step kept an older flag"
    if "div" in row.edges.split() and variant == "rhmc":
        assert outs[0].breaks, "no trajectory met an infinite energy"


# ------------------------------------------------------------------------------------------------ single-row edges
ABANDON = Row(16, 16, 1, True, dict(threads=128, tile=(1, 2), chunks=1, image_in_smem=1), "rhmc trial", mags=(19.0, 19.0),
              niter=130)


@functools.lru_cache(maxsize=None)
def _abandon_inputs():
    rng = np.random.RandomState(77)
    L = _setup(ABANDON)
    t = np.array([so.mag2flux(19.0) * F2C, 8.3, 7.6])
    D = rng.poisson(so.ls_model(L.clone(D=np.zeros((16, 16))), t)).astype(float)
    n = ABANDON.niter
    return L.clone(D=D), t * np.array([1.02, 1.0, 1.0]), rng.randn(n + 1, 3), rng.randint(3, 9, n).astype(np.int32), \
        np.log(rng.random_sample(n))


ABANDON_DT = np.array([0.1, 1.8, 1.8])  # about 30 % acceptance


@pytest.mark.gpu
def test_hessian_chain_abandoned_at_iteration_100():
    """RHMC_random gives up a chain below 50 % acceptance at iteration 100: its later rows stay zero on both sides; the
    trajectories before that are compared like every other chain.  Also runs niter = 0."""
    from hmc_stellar_toy_model_b200 import RHMCContext

    L, q0, Z, steps, lnu = _abandon_inputs()
    out = so.ls_rhmc_random(L, q0, ABANDON_DT, Z, steps, lnu, ABANDON.niter)
    assert out.abandoned == 100 and 0 < np.sum(out.A[:100]) < 50 and not out.breaks, out.abandoned
    _check_oracle_energies(out)
    with RHMCContext(n_fields=1, num_rows=16, num_cols=16, max_stars=1, psf_fwhm_pix=L.PSF_FWHM_pix, B_count=L.B_count,
                     f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, g_xx=1.0, g_ff=1.0, enable_hessian=True) as ctx:
        ctx.set_data(L.D)
        _check_plan(ctx, ABANDON, "abandon", "rhmc")
        r = ctx.ls_run(ctx.LS_HESS, q0[None], ABANDON_DT, Z[None], steps[None], lnu[None])
        r0 = ctx.ls_run(ctx.LS_HESS, q0[None], ABANDON_DT, Z[None, :1], np.zeros((1, 0), np.int32), np.zeros((1, 0)))
    _check_chain(r, 0, 1, out, ABANDON.niter)
    assert not np.any(r["q_chain"][0, 101:]) and not np.any(r["E_chain"][0, 101:]) and not np.any(r["A_chain"][0, 100:])
    o0 = so.ls_rhmc_random(L, q0, ABANDON_DT, Z[:1], steps[:0], lnu[:0], 0)
    assert r0["q_chain"].shape == (1, 1, 3) and r0["A_chain"].shape == (1, 0)
    assert np.array_equal(r0["q_chain"][0, 0], q0) and relerr(r0["E_chain"][0, 0], o0.E[0]) < RTOL
    assert np.array_equal(r0["q_final"][0], q0) and r0["accept_count"][0] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["m", "abandon"])
def test_trial_arm(name):
    """The step-size trial of HMC_find_best_dt (single star on a model_data background, every momentum kicked by the
    scalar flux gradient) with both zero_xy values, on the one-star rows."""
    from hmc_stellar_toy_model_b200 import RHMCContext

    if name == "abandon":
        L, q, *_ = _abandon_inputs()
        row = ABANDON
    else:
        row = ROWS[name]
        L, _, q = _field(name, 0)
    rng = np.random.RandomState(4)
    n = 30
    normals, steps, lnu = rng.randn(n + 1, 3), rng.randint(0, 12, n), np.log(rng.random_sample(n))
    psf = so.gauss_psf(row.R, row.C, q[1], q[2], L.PSF_FWHM_pix)
    model_data = L.D - q[0] * psf * 0.9 + 3.0
    with RHMCContext(n_fields=1, num_rows=row.R, num_cols=row.C, max_stars=1, psf_fwhm_pix=L.PSF_FWHM_pix,
                     B_count=L.B_count, f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, g_xx=1.0, g_ff=1.0,
                     enable_hessian=row.hess) as ctx:
        ctx.set_data(L.D)
        _check_plan(ctx, row, name, "trial")
        for zero_xy, dt in ((True, np.array([q[0] * 0.06, 0.0, 0.0])), (False, np.array([q[0] * 0.05, 2e-3, 2e-3]))):
            out = ctx.ls_run(ctx.LS_TRIAL, q[None], dt, normals[None], steps[None], lnu[None],
                             background=model_data[None], zero_xy=zero_xy)
            ref = so.ls_trial(L, q, model_data, dt, normals, steps, lnu, zero_xy)
            assert int(out["accept_count"][0]) == ref, (zero_xy, out["accept_count"][0], ref)
            assert 0 < ref < n, ref


@pytest.mark.gpu
def test_hessian_context_too_large_fails_cleanly():
    """With the 1/Lambda image a 128x128 field does not fit the CTA: srhmc_create fails cleanly (row "m" runs the same
    shape without it)."""
    from hmc_stellar_toy_model_b200 import RHMCContext, _capi

    L = so.LightSetup(num_rows=128, num_cols=128)
    with pytest.raises(_capi.SrhmcError) as e:
        RHMCContext(n_fields=1, num_rows=128, num_cols=128, max_stars=1, psf_fwhm_pix=L.PSF_FWHM_pix, B_count=L.B_count,
                    f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, g_xx=1.0, g_ff=1.0, enable_hessian=True)
    assert e.value.code == -4  # SRHMC_ERR_TOO_LARGE


@pytest.mark.gpu
def test_lightsource_entry_points_reject_patch_radius():
    """The lightsource family sums over the whole image: a context with a patch radius is refused instead of running
    patch-limited sums the reference never computes."""
    from hmc_stellar_toy_model_b200 import RHMCContext, _capi

    L, n, q = _field("a", 0)
    with RHMCContext(n_fields=1, num_rows=16, num_cols=16, max_stars=n, psf_fwhm_pix=L.PSF_FWHM_pix, B_count=L.B_count,
                     f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, g_xx=1.0, g_ff=1.0, patch_radius=5,
                     enable_hessian=True) as ctx:
        ctx.set_data(L.D)
        calls = [lambda: ctx.hessian(q[None], d2_only=True),
                 lambda: ctx.eval_background(q[None], L.D[None]),
                 lambda: ctx.ls_run(ctx.LS_HMC, q[None], np.ones(3 * n), np.zeros((1, 2, 3 * n)), np.ones((1, 1)),
                                    np.zeros((1, 1)))]
        for call in calls:
            with pytest.raises(_capi.SrhmcError, match="patch_radius") as e:
                call()
            assert e.value.code == -1


# ------------------------------------------------------------------------------------------------ zero flux
ZERO = Row(32, 32, 4, True, dict(threads=256, tile=(2, 2), chunks=1, image_in_smem=1), "zero")


@functools.lru_cache(maxsize=None)
def _zero_inputs():
    """Two real stars and two placeholders with f = 0 and f = 1e-310 (subnormal)."""
    rng = np.random.RandomState(5)
    L = _setup(ZERO)
    t = np.array([so.mag2flux(19.0) * F2C, 10.3, 12.8, 0.0, 20.4, 9.7, 1e-310, 6.2, 24.1,
                  so.mag2flux(19.6) * F2C, 22.7, 21.9])
    D = rng.poisson(so.ls_model(L.clone(D=np.zeros((32, 32))), t)).astype(float)
    return L.clone(D=D), t.copy()


@pytest.mark.gpu
def test_zero_flux_star():
    """A star with f = 0 (and one with a subnormal f) has the finite flux gradient -sum(rho PSF) of the reference's dVdq /
    dVdq_single, through every path of the lightsource family: eval_background, the crowded-field evaluation the gym's dVdq
    runs on a one-chunk context, hessian() (d1, d2, d3: at f = 0 the position d2 is 0, so dq/dt and E are not finite in the
    reference either) and an HMC_random chain that starts there."""
    from hmc_stellar_toy_model_b200 import RHMCContext

    L, q = _zero_inputs()
    g_ref, V_ref = so.ls_grad(L, q), so.ls_potential(L, q)
    bg = np.full((32, 32), L.B_count) + np.linspace(0.0, 3.0, 32)[:, None]
    Vb_ref, gb_ref = _oracle_bg(L, q, bg)
    _, _, _, o1, o2, o3 = so.ls_efficient(L, q, np.zeros_like(q), parts=True)
    assert np.all(np.isfinite(g_ref)) and np.all(np.isfinite(o1)) and o2[4] == 0.0
    rng = np.random.RandomState(6)
    niter = 5
    Z, steps, lnu = rng.randn(niter + 1, 12), rng.randint(0, 6, niter).astype(np.int32), np.log(rng.random_sample(niter))
    dt = np.tile([20.0, 5e-3, 5e-3], 4)
    out = so.ls_hmc_random(L, q, dt, Z, steps, lnu, niter)
    with RHMCContext(n_fields=1, num_rows=32, num_cols=32, max_stars=4, psf_fwhm_pix=L.PSF_FWHM_pix, B_count=L.B_count,
                     f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, g_xx=1.0, g_ff=1.0, enable_hessian=True) as ctx:
        ctx.set_data(L.D)
        _check_plan(ctx, ZERO, "zero", "bg")
        Vb, gb = ctx.eval_background(q[None], bg[None])
        V, g, _, _ = ctx.eval(q[None])
        d1, d2, d3, _, _, _ = ctx.hessian(q[None], np.zeros((1, 12)))
        r = ctx.ls_run(ctx.LS_HMC, q[None], dt, Z[None], steps[None], lnu[None])
    assert np.all(np.isfinite(gb)) and np.all(np.isfinite(g)), (gb, g)
    assert relerr(Vb[0], Vb_ref) < RTOL and _close(gb[0], gb_ref, 1e-9)
    assert relerr(V[0], V_ref) < RTOL and _close(g[0], g_ref, 1e-9)
    assert _close(d1[0], o1, 1e-9) and _close(d2[0], o2, 1e-9) and _close(d3[0], o3, 1e-8)
    _check_chain(r, 0, 4, out, niter)


# ------------------------------------------------------------------------------------------------ gym replays
def _quiet():
    return contextlib.redirect_stdout(io.StringIO())


def _draws(seed, d, niter, steps_min, steps_max):
    """samplers.lightsource_gym._draws from a seeded np.random: p_sample, then per iteration p_sample, randint, random."""
    np.random.seed(seed)
    normals, steps, lnu = np.zeros((niter + 1, d)), np.zeros(niter, np.int32), np.zeros(niter)
    normals[0] = np.random.randn(d)
    for i in range(1, niter + 1):
        normals[i] = np.random.randn(d)
        steps[i - 1] = np.random.randint(low=steps_min, high=steps_max, size=1)[0]
        lnu[i - 1] = np.log(np.random.random(1))[0]
    return normals, steps, lnu


@pytest.mark.gpu
def test_gym_replays_three_stars_default_image():
    """HMC_random, RHMC_random_diag and RHMC_random of the default 48x48 gym on three stars, draws rebuilt from the same
    seeds: per-star dt vectors, factor1 at 48x48 and the Hessian chain beyond one star."""
    from hmc_stellar_toy_model_b200.samplers import lightsource_gym, mag2flux

    gym = lightsource_gym()
    assert (gym.num_rows, gym.num_cols) == (48, 48)
    np.random.seed(31)
    q0 = np.array([[mag2flux(19.0) * gym.flux_to_count, 14.2, 30.7], [mag2flux(19.5) * gym.flux_to_count, 31.6, 12.3],
                   [mag2flux(20.0) * gym.flux_to_count, 28.1, 33.9]])
    gym.gen_mock_data(q_true=q0)
    gym.HMC_find_best_dt(q0, default=True, dt_f_coeff=0.05, dt_xy_coeff=2.0)
    gym.compute_factors()
    L = so.LightSetup(D=gym.D)
    L.compute_factors()
    assert gym.factor1 == L.factor1
    f_lim = mag2flux(22.0) * gym.flux_to_count
    niter, smin, smax = 12, 3, 10
    with _quiet():
        np.random.seed(1)
        gym.HMC_random(np.copy(q0), Nchain=1, Niter=niter, steps_max=smax, steps_min=smin, f_lim=f_lim)
    _check_plan(gym._ctx, GYM, "gym", "hmc")
    # the drop-in's per-star step sizes are HMC_find_best_dt(default=True)'s: (0.05 f, 2 / f, 2 / f) of each star
    f = q0[:, 0]
    assert np.allclose(gym.dt, np.stack([0.05 * f, 2.0 / f, 2.0 / f], axis=1).ravel(), rtol=1e-15, atol=0)
    out = so.ls_hmc_random(L, q0.ravel(), gym.dt, *_draws(1, 9, niter, smin, smax), niter, f_lim=f_lim)
    _compare_gym(gym, out)
    with _quiet():
        np.random.seed(2)
        gym.RHMC_random_diag(np.copy(q0), Nchain=1, Niter=niter, steps_max=smax, steps_min=smin, f_lim=f_lim,
                             dt_global=0.2)
    out = so.ls_rhmc_random_diag(L, q0.ravel(), 0.2, *_draws(2, 9, niter, smin, smax), niter, f_lim=f_lim)
    _compare_gym(gym, out)
    with _quiet():
        np.random.seed(3)
        gym.RHMC_random(np.copy(q0), Nchain=1, Niter=niter, steps_max=smax, steps_min=smin, f_lim=f_lim,
                        dt_RHMC_xy=0.3, dt_RHMC_f=0.3, debug=False)
    out = so.ls_rhmc_random(L, q0.ravel(), np.full(9, 0.3), *_draws(3, 9, niter, smin, smax), niter, f_lim=f_lim)
    _check_oracle_energies(out)
    _compare_gym(gym, out)


GYM = Row(48, 48, 3, True, dict(threads=256, tile=(2, 4), chunks=1, image_in_smem=1))


def _compare_gym(gym, out):
    assert np.array_equal(gym.A_chain[0, :, 0].astype(bool), out.A.astype(bool)), (gym.A_chain[0, :, 0], out.A)
    assert 0 < np.sum(out.A) < len(out.A), out.A  # both branches of the Metropolis test
    assert first_divergence(gym.q_chain[0], out.q, 1e-9) == -1
    assert relerr(gym.E_chain[0, :, 0], out.E) < RTOL


# ------------------------------------------------------------------------------------------------ oracle restatements (CPU)
def _five_stars():
    rng = np.random.RandomState(9)
    L = _setup(Row(24, 40, 5, True, {}))
    q = np.array([900.0, 6.3, 9.2, 400.0, 15.8, 30.4, 1500.0, 11.1, 21.7, 250.0, 20.2, 4.4, 700.0, -0.8, 17.3])
    D = rng.poisson(so.ls_model(L.clone(D=np.zeros((24, 40))), q)).astype(float)
    return L.clone(D=D), q * np.array([1.05, 1.0, 1.0] * 5) + np.array([0, 0.2, -0.1] * 5)


def _fd(fun, q, i, h):
    qp, qm = q.copy(), q.copy()
    qp[i] += h
    qm[i] -= h
    return (fun(qp) - fun(qm)) / (2.0 * h)


def _steps(q):
    return np.where(np.arange(q.size) % 3 == 0, 1e-4 * np.abs(q), 1e-4)


def test_oracle_lightsource_gradient_vs_finite_differences():
    """ls_grad is the derivative of ls_potential on a 5-star 24x40 field with one star off the image; ls_efficient's d1 is
    ls_grad."""
    L, q = _five_stars()
    g = so.ls_grad(L, q)
    h = _steps(q)
    fd = np.array([_fd(lambda x: so.ls_potential(L, x), q, i, h[i]) for i in range(q.size)])
    assert _close(g, fd, 1e-6)
    _, _, _, d1, _, _ = so.ls_efficient(L, q, np.ones_like(q), parts=True)
    assert _close(d1, g, 1e-12)


def test_oracle_lightsource_curvatures_vs_finite_differences():
    """ls_efficient's d2 is the diagonal derivative of its d1 on the same field, and its flux d3 that of d2.  Its position
    d3 is RHMC_efficient_computation's (samplers.py:828-927), which the kernel reproduces: the derivative of d2_x is
    -2 f^3 S3 + 3 f^2 S2 + f S1 with S3 = sum(rho3 ax^3), and the reference's first term is -f^3 S3.  The finite
    differences agree with d3 once the missing -f^3 S3 is added, and differ from it without."""
    L, q = _five_stars()
    _, _, _, d1, d2, d3 = so.ls_efficient(L, q, np.ones_like(q), parts=True)
    h = _steps(q)
    part = lambda x, j: so.ls_efficient(L, x, np.ones_like(x), parts=True)[j]
    fd2 = np.array([_fd(lambda x: part(x, 3)[i], q, i, h[i]) for i in range(q.size)])
    fd3 = np.array([_fd(lambda x: part(x, 4)[i], q, i, h[i]) for i in range(q.size)])
    assert _close(d2, fd2, 1e-6)
    rho3 = L.D / so.ls_model(L, q) ** 3
    var = (L.PSF_FWHM_pix / so.FWHM_TO_SIGMA) ** 2
    li = np.arange(L.num_rows)[:, None] + 0.5
    mj = np.arange(L.num_cols)[None, :] + 0.5
    missing = np.zeros_like(q)
    for k in range(q.size // 3):
        f, x, y = q[3 * k : 3 * k + 3]
        psf = so.gauss_psf(L.num_rows, L.num_cols, x, y, L.PSF_FWHM_pix)
        missing[3 * k + 1] = -f**3 * np.sum(rho3 * (psf * (li - x) / var) ** 3)
        missing[3 * k + 2] = -f**3 * np.sum(rho3 * (psf * (mj - y) / var) ** 3)
    assert _close(d3 + missing, fd3, 1e-5)
    assert not _close(d3, fd3, 1e-2)


# ------------------------------------------------------------------------------------------------ coverage of the arms
@pytest.mark.gpu
def test_rows_cover_every_arm():
    """The union of the plans the tests above asserted (runs after them) covers every launch arm of the kernel."""
    assert PLANS, "run the whole module: the plans are recorded by the tests above"
    seen = lambda key, pls=PLANS: {pl[key] for pl in pls}
    assert seen("threads") >= {128, 256, 512}
    assert {(pl["tile_rows"], pl["tile_cols"]) for pl in PLANS} >= {(2, 4), (2, 2), (1, 2)}
    for hess in (False, True):
        pls = [pl for pl in PLANS if pl["hess"] == hess]
        assert {pl["chunks"] == 1 for pl in pls} == {True, False}, hess
        assert seen("image_in_smem", pls) == {0, 1}, hess
    assert seen("variant") >= {"hess", "d2_only", "bg", "hmc", "diag", "rhmc", "trial"}
    assert any(pl["ragged"] for pl in PLANS) and any(pl["shared_data"] for pl in PLANS)
