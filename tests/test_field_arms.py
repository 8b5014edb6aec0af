"""Every launch arm of the crowded-field kernel (field_kernel<T, MR, MC, MODE, V3>, field_kernel.cuh) against the float64
oracle.  configure() (stellar_rhmc.cu) picks the arm from the image shape, the star count, the precision and the patch
radius: 128 / 256 / 512 threads, the (2,4) / (2,2) / (1,2) register tile, one or several table chunks, the data image in
shared or in global memory, and the compact or the chunked tables.  Each arm compiles to different code, so each row below
chooses its shape to land on one arm, first asserts that it did (RHMCContext.launch_plan), then compares V, dV/dq, H and
H', leapfrog steps with their fixed-point counts, chains and long trajectories with the oracle.  If a change of
configure() moves a shape to another arm, the plan assertion fails instead of the coverage quietly going away; the last
test checks that the rows together still cover every arm.

Rows "o" and "p" are FP32 fields whose column count is 2 mod 4: the compact path reads four image pixels with one 16-byte
load, which such rows would start 8 bytes off, so configure() gives them the chunked tables."""
import functools
from dataclasses import dataclass, field

import numpy as np
import pytest

import stellar_oracle as so
from helpers import first_divergence, golden, relerr, setup_from

RTOL = 1e-10  # FP64: V, H, q
F32_TOL = 1e-4  # FP32: relative to the per-coordinate scale

# every plan a test asserted, with what it ran: the last test checks that together they cover every arm
PLANS = []


@dataclass(frozen=True)
class Row:
    R: int
    C: int
    N: int
    prec: int
    rad: int
    expect: dict = field(hash=False)
    modes: str = ""
    vc: bool = False           # repulsion on for eval / step (always off for run / single)
    nstars: tuple = ()         # one entry per field; () = one field with N stars
    shared: bool = False
    fp_mode: int = 0


ROWS = {
    "a": Row(16, 16, 5, 64, 0, dict(threads=128, tile=(1, 2), chunks=1, image_in_smem=1, compact=0), "eval step run single",
             vc=True),
    "b": Row(64, 4, 3, 64, 0, dict(threads=128, tile=(2, 4), compact=0), "eval step", vc=True),
    "c": Row(16, 16, 5, 64, 3, dict(threads=128, compact=1), "eval step run"),
    "d": Row(48, 40, 7, 64, 0, dict(threads=256, tile=(2, 4), chunks=1, compact=0), "eval step single"),
    "e": Row(48, 48, 300, 64, 0, dict(threads=512, tile=(2, 2), chunks=7, compact=0), "eval step"),
    "f": Row(32, 32, 300, 64, 0, dict(threads=512, tile=(1, 2), chunks=3, compact=0), "eval step"),
    "g": Row(128, 128, 40, 64, 0, dict(chunks=1, image_in_smem=0, compact=0), "eval step run"),
    "h": Row(112, 112, 150, 64, 0, dict(chunks=3, image_in_smem=0, compact=0), "eval step"),
    "i": Row(112, 112, 100, 64, 12, dict(image_in_smem=0, compact=1), "eval step run", nstars=(100, 0, 1, 37)),
    "j": Row(64, 64, 204, 64, 14, dict(compact=0), "eval step"),
    "k": Row(64, 63, 120, 64, 12, dict(compact=0), "eval step"),
    "l": Row(20, 40, 9, 64, 12, dict(compact=0), "eval step"),
    "m": Row(64, 64, 600, 64, 12, dict(chunks=7, compact=0), "eval"),
    "n": Row(48, 48, 150, 64, 4, dict(threads=256, compact=1), "eval step run"),
    "o": Row(64, 66, 120, 32, 12, dict(compact=0), "eval step"),
    "p": Row(40, 26, 9, 32, 12, dict(compact=0), "eval"),
    "q": Row(64, 64, 204, 32, 12, dict(compact=1), "eval step"),
    "r": Row(160, 160, 200, 32, 0, dict(chunks=3, image_in_smem=0, compact=0), "eval"),
    "s": Row(168, 168, 40, 32, 12, dict(image_in_smem=0, compact=1), "eval"),
    "t": Row(32, 32, 30, 64, 0, dict(compact=0), "eval step run", vc=True, nstars=(30, 0, 7, 30), shared=True),
    "u-compact": Row(64, 64, 120, 64, 12, dict(compact=1), "step", fp_mode=1),
    "u-chunked": Row(48, 40, 7, 64, 0, dict(compact=0), "step", fp_mode=1),
}


def _rows(mode):
    return [name for name, r in ROWS.items() if mode in r.modes.split()]


def _setup(row, vc):
    return so.Setup(num_rows=row.R, num_cols=row.C, dt=5e-2, g_xx=0.05, g_ff=4.0, g_ff2=4.0, use_prior=True, alpha=2.0,
                    V_prior_const=0.7, use_Vc=vc, beta=1e-3, Vc_r_pow=3.0)


@functools.lru_cache(maxsize=None)
def _inputs(name):
    """Per field: the data image, a start state near the true stars and a momentum draw; plus the run's draws."""
    row = ROWS[name]
    rng = np.random.RandomState(sum(map(ord, name)))
    S = _setup(row, False)
    counts = list(row.nstars) or [row.N]
    fmin, fmax = S.mag2flux_converter(20.0), S.mag2flux_converter(15.0)

    def stars(n):
        f = so.pow_law_sample(2.0, fmin, fmax, rng.random_sample(n))
        return np.stack([f, rng.uniform(1, row.R - 1, n), rng.uniform(1, row.C - 1, n)], axis=1)

    def image(q_true):
        return rng.poisson(so.model_image(S, q_true.ravel())).astype(float)

    truth = stars(row.N)
    shared_D = image(truth) if row.shared else None
    D, q, p = [], np.zeros((len(counts), 3 * row.N)), np.zeros((len(counts), 3 * row.N))
    for f, n in enumerate(counts):
        t = truth[:n] if row.shared else stars(n)
        D.append(shared_D if row.shared else image(t))
        q0 = t * np.array([1.05, 1.0, 1.0]) + np.concatenate([np.zeros((n, 1)), 0.1 * rng.randn(n, 2)], axis=1)
        q[f, : 3 * n] = q0.ravel()
        p[f, : 3 * n] = rng.randn(3 * n) * np.sqrt(so.metric(S, q0.ravel())) if n else 0.0
    L = 4
    normals = rng.randn(len(counts), L, 3 * row.N)
    lnu = np.log(rng.random_sample((len(counts), L)))
    return counts, D, q, p, normals, lnu


def _field_setup(name, f, vc):
    row = ROWS[name]
    return _setup(row, vc).clone(D=_inputs(name)[1][f])


# ------------------------------------------------------------------------------------------------ oracle, once per module
def _oracle_eval(name):
    row = ROWS[name]
    counts, _, q, _, _, _ = _inputs(name)
    out = []
    for f, n in enumerate(counts):
        S, qq = _field_setup(name, f, row.vc), q[f, : 3 * n]
        H, dH = so.metric(S, qq, grad=True)
        out.append((so.potential(S, qq, True, rad=row.rad), so.grad_potential(S, qq, rad=row.rad), H, dH))
    return out


def _oracle_step(name):
    """States after 1 and after 3 leapfrog steps, with the fixed-point counts of the last step of each."""
    row = ROWS[name]
    counts, _, q, p, _, _ = _inputs(name)
    out = []
    for f, n in enumerate(counts):
        if n == 0:
            out.append(None)
            continue
        S, qq, pp = _field_setup(name, f, row.vc), q[f, : 3 * n], p[f, : 3 * n]
        states = []
        for s in range(3):
            cnt = []
            qq, pp = so.rhmc_step(S, qq, pp, 1e-6, 1000, counters=cnt, rad=row.rad, per_star=row.fp_mode == 1)
            if s in (0, 2):
                states.append((qq, pp, cnt[0]))
        out.append(states)
    return out


NITER, NSTEPS = 3, 5  # run: 4 iterations of 5 leapfrog steps


def _oracle_run(name):
    row = ROWS[name]
    counts, _, q, _, normals, lnu = _inputs(name)
    out = []
    for f, n in enumerate(counts):
        S = _field_setup(name, f, False)
        if n == 0:  # no state: every row of the chain holds the pixel potential
            out.append(so.potential(S, np.zeros(0), True, rad=row.rad))
            continue
        out.append(so.run_rhmc(S, q[f, : 3 * n], normals[f, :, : 3 * n], lnu[f], NITER, NSTEPS, S.dt, f_pos=True,
                               rad=row.rad))
    return out


SINGLE_STEPS = 10


def _oracle_single(name):
    row = ROWS[name]
    counts, _, q, p, _, _ = _inputs(name)
    S = _field_setup(name, 0, False)
    n = counts[0]
    return so.run_single_rhmc(S, q[0, : 3 * n], p[0, : 3 * n], SINGLE_STEPS, S.dt, f_pos=True, rad=row.rad)


@pytest.fixture(scope="module")
def oracle():
    """oracle(kind, row): the oracle's results for a row, computed on first use and kept for the module."""
    kinds = dict(eval=_oracle_eval, step=_oracle_step, run=_oracle_run, single=_oracle_single)
    cache = {}

    def get(kind, name):
        if (kind, name) not in cache:
            cache[kind, name] = kinds[kind](name)
        return cache[kind, name]

    return get


# ------------------------------------------------------------------------------------------------ device side
def _ctx(name, mode, vc):
    from test_gpu_parity import make_ctx

    row = ROWS[name]
    counts, D, _, _, _, _ = _inputs(name)
    ctx = make_ctx(_setup(row, vc), n_fields=len(counts), max_stars=row.N, precision=row.prec, patch_radius=row.rad,
                   shared_data=row.shared, fixed_point_mode=row.fp_mode)
    ctx.set_data(D[0] if row.shared else np.stack(D))
    _check_plan(ctx, name, mode)
    return ctx


def _check_plan(ctx, name, mode):
    row = ROWS[name]
    plan = ctx.launch_plan()
    PLANS.append(dict(plan, row=name, mode=mode, precision=row.prec, rad=row.rad, shared_data=row.shared,
                      fixed_point_mode=row.fp_mode))
    got = dict(threads=plan["threads"], tile=(plan["tile_rows"], plan["tile_cols"]),
               chunks=-(-row.N // plan["chunk_stars"]), image_in_smem=plan["image_in_smem"], compact=plan["compact_tables"])
    for key, want in row.expect.items():
        assert got[key] == want, (name, key, got)
    assert plan["chain_kernel"] == 0 and plan["smem_bytes"] <= 232448, plan


def _grad_err(a, b, prec):
    """FP64: element-wise with a floor at 1e-3 of the per-coordinate scale (test_gpu_parity.grad_relerr); FP32: relative to
    the per-coordinate scale, as test_gpu_parity.test_fp32_build_within_1e4."""
    a, b = np.asarray(a).reshape(-1, 3), np.asarray(b).reshape(-1, 3)
    if not a.size:
        return 0.0
    if prec == 64:
        scale = np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b), axis=0, keepdims=True))
    else:
        scale = np.max(np.abs(b), axis=0, keepdims=True)
    return float(np.max(np.abs(a - b) / scale))


def _scale_err(a, b):
    return _grad_err(a, b, 32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("eval"))
def test_eval_arm(name, oracle):
    row = ROWS[name]
    counts, _, q, _, _, _ = _inputs(name)
    with _ctx(name, "eval", row.vc) as ctx:
        V, grad, H, Hg = ctx.eval(q, nstars=list(counts) if row.nstars else None, f_pos=True, g_ff2=4.0, beta=1e-3)
    tol = RTOL if row.prec == 64 else F32_TOL
    for f, n in enumerate(counts):
        Vo, go, Ho, dHo = oracle("eval", name)[f]
        assert relerr(V[f], Vo) < tol, (f, V[f], Vo)
        assert _grad_err(grad[f, : 3 * n], go, row.prec) < tol, f
        assert relerr(H[f, : 3 * n], Ho) < RTOL and np.allclose(Hg[f, : 3 * n], dHo, rtol=RTOL, atol=0), f
        assert np.all(grad[f, 3 * n:] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("step"))
def test_step_arm(name, oracle):
    row = ROWS[name]
    counts, _, q, p, _, _ = _inputs(name)
    ns = list(counts) if row.nstars else None
    with _ctx(name, "step", row.vc) as ctx:
        res = [ctx.step(q, p, k, 5e-2, g_ff2=4.0, beta=1e-3, nstars=ns, return_counts=True) for k in (1, 3)]
    for f, n in enumerate(counts):
        want = oracle("step", name)[f]
        for (qk, pk, cnt), state in zip(res, want or [None, None]):
            if n == 0:
                assert tuple(cnt[f]) == (0, 0)
                continue
            qo, po, co = state
            if row.prec == 64:
                assert relerr(qk[f, : 3 * n], qo) < RTOL, f
                assert _grad_err(pk[f, : 3 * n], po, 64) < 1e-9, f
                assert tuple(cnt[f]) == co, (f, tuple(cnt[f]), co)
            else:
                assert relerr(qk[f, : 3 * n], qo) < F32_TOL, f
                assert _grad_err(pk[f, : 3 * n], po, 32) < F32_TOL, f


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("run"))
def test_run_arm(name, oracle):
    row = ROWS[name]
    counts, _, q, _, normals, lnu = _inputs(name)
    with _ctx(name, "run", False) as ctx:
        r = ctx.run(q, NITER, NSTEPS, 5e-2, nstars=list(counts) if row.nstars else None, normals=normals, lnu=lnu,
                    g_ff2=4.0, beta=1e-3, f_pos=True)
    for f, n in enumerate(counts):
        out = oracle("run", name)[f]
        if n == 0:
            assert relerr(r.E_chain[f], np.full(NITER + 1, out)) < RTOL
            continue
        assert np.array_equal(r.A_chain[f].astype(bool), out.A), f
        assert first_divergence(r.q_chain[f][:, : 3 * n], out.q, 1e-9) == -1, f
        assert relerr(r.E_chain[f], out.E) < RTOL, f


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("single"))
def test_single_arm(name, oracle):
    """One long trajectory in MODE_SINGLE of the CTA kernel (more than one star, so not the one-star chain kernel).  The
    energy differences V - V0 and E - E0 are checked against the size of V itself (its pixel sum rounds at that scale);
    T - T0 has no such sum and is checked against its own largest value."""
    row = ROWS[name]
    counts, _, q, p, _, _ = _inputs(name)
    with _ctx(name, "single", False) as ctx:
        qc, pc, E, V, T = ctx.run_single(q, p, SINGLE_STEPS, 5e-2, f_pos=True, g_ff2=4.0, beta=1e-3)
    out = oracle("single", name)
    n = counts[0]
    S = _field_setup(name, 0, False)
    e_scale = abs(so.potential(S, q[0, : 3 * n], True, rad=row.rad))
    assert first_divergence(qc[0][:, : 3 * n], out.q, 1e-9) == -1
    assert first_divergence(pc[0][:, : 3 * n], out.p, 1e-8) == -1
    assert np.max(np.abs(V[0] - out.V)) < RTOL * e_scale
    assert np.max(np.abs(E[0] - out.E)) < RTOL * e_scale
    assert np.max(np.abs(T[0] - out.T)) < RTOL * np.max(np.abs(out.T))


# ------------------------------------------------------------------------------------------------ oracle restatements (CPU)
def test_oracle_patch_radius_matches_full_image():
    """rad > 0 routes V and dV/dq through patch_eval (plus prior and repulsion): on the 204-star field a 25x25 patch agrees
    with the full-image PSF to SURVEY 8d's 3e-13 (gradients and momenta relative to their per-coordinate scale) for the
    potential, the gradient and one leapfrog step; rad = 0 is the full-image path itself."""
    g = golden("field_eval_204")
    S = setup_from(g)
    q, p = g["q"], g["p"]
    assert relerr(so.potential(S, q, True, rad=12), so.potential(S, q, True)) < 3e-13
    g12, g0 = so.grad_potential(S, q, rad=12), so.grad_potential(S, q)
    assert _scale_err(g12, g0) < 3e-13
    c12, c0 = [], []
    q12, p12 = so.rhmc_step(S, q, p, counters=c12, rad=12)
    q0, p0 = so.rhmc_step(S, q, p, counters=c0)
    assert relerr(q12, q0) < 3e-13 and _scale_err(p12, p0) < 3e-13 and c12 == c0
    q0b, p0b = so.rhmc_step(S, q, p, rad=0)
    assert np.array_equal(q0b, q0) and np.array_equal(p0b, p0)
    assert np.array_equal(so.grad_potential(S, q, rad=0), g0) and so.potential(S, q, True, rad=0) == so.potential(S, q, True)


def test_oracle_per_star_stop_rule():
    """per_star=True stops each star's fixed-point loops on their own.  With one star that is the field-wide rule, bit for
    bit; with 204 stars the largest per-star count is the field-wide count and the states differ by less than the
    tolerance of the loops."""
    g = golden("kat1")
    S = setup_from(g)
    ca, cb = [], []
    qa, pa = so.rhmc_step(S, g["q"], g["p"], counters=ca, per_star=True)
    qb, pb = so.rhmc_step(S, g["q"], g["p"], counters=cb, per_star=False)
    assert np.array_equal(qa, qb) and np.array_equal(pa, pb) and ca == cb
    g = golden("field_eval_204")
    S = setup_from(g)
    ca, cb = [], []
    qa, pa = so.rhmc_step(S, g["q"], g["p"], counters=ca, per_star=True)
    qb, pb = so.rhmc_step(S, g["q"], g["p"], counters=cb)
    assert ca == cb
    assert np.max(np.abs(qa - qb)) < 1e-6 and not np.array_equal(qa, qb)


# ------------------------------------------------------------------------------------------------ coverage of the arms
@pytest.mark.gpu
def test_rows_cover_every_arm():
    """The union of the plans the tests above asserted (runs after them) covers every launch arm of the kernel."""
    assert PLANS, "run the whole module: the plans are recorded by the tests above"
    seen = lambda key: {pl[key] for pl in PLANS}
    assert seen("threads") >= {128, 256, 512}
    assert {(pl["tile_rows"], pl["tile_cols"]) for pl in PLANS} >= {(2, 4), (2, 2), (1, 2)}
    chunked = [pl for pl in PLANS if not pl["compact_tables"]]
    compact = [pl for pl in PLANS if pl["compact_tables"]]
    assert {-(-ROWS[pl["row"]].N // pl["chunk_stars"]) == 1 for pl in chunked} == {True, False}
    assert {pl["image_in_smem"] for pl in chunked} == {0, 1} and {pl["image_in_smem"] for pl in compact} == {0, 1}
    assert any(pl["rad"] > 0 for pl in chunked) and any(pl["rad"] == 0 for pl in chunked)
    assert seen("precision") == {32, 64}
    assert {pl["precision"] for pl in compact} == {32, 64} and {pl["precision"] for pl in chunked} == {32, 64}
    assert seen("mode") == {"eval", "step", "run", "single"}
    assert True in seen("shared_data") and seen("fixed_point_mode") == {0, 1}
