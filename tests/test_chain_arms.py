"""Every arm of the warp-resident one-star kernel (chain_kernel<4, DT, MODE, NCS, 255, PT>, chain_kernel.cuh) against the
float64 oracle.  The host sends a context to it for one star, at most 32 columns and 64 rows and a PSF that its column
tables can represent (chain_kernel_eligible, stellar_rhmc.cu); set_data then picks the image layout DT (float64, uint32 or
uint16 counts), precision 32 picks FP32 pixel arithmetic PT on uint16 counts, and the PSF width (or SRHMC_CHAIN_WINDOW=0)
picks the 24-column window or the full 32 columns (NCS).  Each row below chooses a shape, a precision and data that land on
one arm, first asserts that they did (RHMCContext.chain_plan), then compares V, dV/dq, H and H', leapfrog steps with their
fixed-point counts, chains with injected and with Philox draws, and long trajectories with the oracle.  Shapes other than
32 x 32 matter: the kernel's layout arithmetic, column mask, window clamp, reflections and support test all depend on R and
C separately.  The last GPU test checks that the rows together still cover every arm.

Rows "g" are FP32 shapes with an odd row count, whose row tables sat 8 bytes off the 16-byte alignment of their 128-bit
accesses; rows "k" are PSFs so narrow that a lane's column table started below the kernel's exponent cut-off, which now
take the CTA kernel (and "k-1.7" one that stays just inside the bound)."""
import functools
from dataclasses import dataclass, field

import numpy as np
import pytest

import stellar_oracle as so
from helpers import first_divergence, relerr

RTOL = 1e-10   # FP64: V, H, energies
QTOL = 1e-9    # FP64: q and p
F32_TOL = 1e-4
SMEM_MAX = 232448
F = 11         # chains per row: one full warp group of 8 and a partial group of 3
NITER, NSTEPS = 4, 5
NITER_PHILOX = 6
SINGLE_STEPS = 8

# every plan a test asserted, with what it ran: the last test checks that together they cover every arm
PLANS = []


@dataclass(frozen=True)
class Row:
    R: int
    C: int
    prec: int
    data: str                  # "u16": Poisson counts; "u32": one count above 65535; "f64": non-integer pixels
    expect: dict = field(hash=False)
    fwhm: float = 3.5
    env: tuple = ()
    prior: bool = True
    f_pos: bool = True
    schedule: bool = False     # g_ff2 schedule shorter than the chain
    stride: int = 1
    counter_max: int = 1000
    modes: str = "eval step run philox single"


def _plan(ck, win=24, nbytes=2, f32=0, **kw):
    return dict(chain_kernel=ck, window_cols=win, image_bytes=nbytes, pixel_f32=f32, **kw)


AWAY = dict(chain_kernel=0)
ROWS = {
    "a": Row(32, 32, 64, "u16", _plan(1)),
    "b": Row(32, 32, 64, "u32", _plan(1, nbytes=4), stride=2),
    "c": Row(40, 28, 64, "f64", _plan(1, nbytes=8), schedule=True),
    "d": Row(20, 17, 64, "u16", _plan(1), prior=False, counter_max=3),
    "e": Row(3, 5, 64, "u16", _plan(1), f_pos=False),
    "f-f64": Row(64, 32, 64, "f64", _plan(1, nbytes=8, blocks_per_sm=1, smem_bytes=140672),
                 env=(("SRHMC_CHAIN_CHUNKS", "3"),)),
    "f-u16": Row(64, 32, 64, "u16", _plan(1), env=(("SRHMC_CHAIN_CHUNKS", "3"),)),
    "g-45x32": Row(45, 32, 32, "u16", _plan(1, f32=1, tab_stride=1104)),
    "g-31x31": Row(31, 31, 32, "u16", _plan(1, f32=1, tab_stride=768), counter_max=3),
    "g-33x32": Row(33, 32, 32, "u16", _plan(1, f32=1, tab_stride=816), stride=3),
    "h": Row(64, 24, 32, "u16", _plan(1, f32=1, tab_stride=1552)),
    "i": Row(48, 24, 64, "u16", _plan(1, win=32), fwhm=1.8 * 2.354),
    "j": Row(32, 32, 32, "u16", _plan(1, win=32, f32=1, tab_stride=784), env=(("SRHMC_CHAIN_WINDOW", "0"),),
             schedule=True),
    "k-1.4": Row(32, 32, 64, "u16", AWAY, fwhm=1.4),
    "k-0.7": Row(40, 28, 64, "f64", AWAY, fwhm=0.7),
    "k-1.7": Row(32, 32, 64, "u16", _plan(1), fwhm=1.7),
    "l-65x32": Row(65, 32, 64, "u16", AWAY),
    "l-64x33": Row(64, 33, 64, "u16", AWAY),
    "m": Row(32, 32, 32, "f64", AWAY, modes="eval step"),
}


def _rows(mode):
    return [name for name, r in ROWS.items() if mode in r.modes.split()]


def _setup(row):
    return so.Setup(num_rows=row.R, num_cols=row.C, dt=0.2, g_xx=1.0, g_ff=1.0, g_ff2=1.0, use_prior=row.prior, alpha=2.0,
                    V_prior_const=0.7 if row.prior else None, PSF_FWHM_pix=row.fwhm)


def _schedule(row):
    return np.array([1.0, 2.0, 3.0]) if row.schedule else None


@functools.lru_cache(maxsize=None)
def _inputs(name):
    """Per chain: the data image, the start state and a momentum draw; plus the injected draws of the run.  The stars sit at
    the centre, on all four edges, just outside them and in two corners; their magnitudes span 15-22, so one warp mixes
    the table-logarithm and the series tiers of the potential."""
    row = ROWS[name]
    R, C = row.R, row.C
    rng = np.random.RandomState(sum(map(ord, name)))
    S = _setup(row)
    pos = [(R / 2, C / 2), (0.2, C / 2), (R - 1.2, C / 2), (R / 2, 0.3), (R / 2, C - 0.7), (-0.6, C / 3),
           (R + 0.4, 2 * C / 3), (R / 3, -0.5), (2 * R / 3, C + 0.5), (R - 0.8, C - 0.9), (0.5, 0.4)]
    q = np.array([[S.mag2flux_converter(m), x, y] for m, (x, y) in zip(np.linspace(15.0, 22.0, F), pos)])
    D = []
    for qi in q:
        truth = qi * np.array([0.95, 1.0, 1.0]) + np.array([0.0, *rng.uniform(-0.3, 0.3, 2)])
        D.append(rng.poisson(so.model_image(S, truth)).astype(float))
    D = np.stack(D)
    if row.data == "u32":
        D[0, 0, 0] = 70000.0   # far from chain 0's star at the centre
    elif row.data == "f64":
        D += 0.25
    p = np.stack([rng.randn(3) * np.sqrt(so.metric(S, qi)) for qi in q])
    normals = rng.randn(F, NITER + 1, 3)
    lnu = np.log(rng.random_sample((F, NITER + 1)))
    return D, q, p, normals, lnu


def _chain_setup(name, f):
    return _setup(ROWS[name]).clone(D=_inputs(name)[0][f])


def _pos_err(a, b):
    """Relative to max(|b|, 1): fluxes are relative, positions near an edge are compared to a pixel."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0))) if a.size else 0.0


def _scale_err(a, b, floor):
    """Per-coordinate scale over the chains (or rows) of a batch: element-wise with a floor at `floor` of the coordinate's
    largest value (test_gpu_parity.grad_relerr for floor = 1e-3; floor = 1 is relative to that largest value)."""
    a, b = np.asarray(a).reshape(-1, 3), np.asarray(b).reshape(-1, 3)
    scale = np.maximum(np.abs(b), floor * np.max(np.abs(b), axis=0, keepdims=True))
    return float(np.max(np.abs(a - b) / scale))


# ------------------------------------------------------------------------------------------------ oracle, once per module
@functools.lru_cache(maxsize=None)
def _oracle_eval(name):
    row = ROWS[name]
    _, q, _, _, _ = _inputs(name)
    out = []
    for f in range(F):
        S = _chain_setup(name, f)
        H, dH = so.metric(S, q[f], grad=True)
        out.append((so.potential(S, q[f], row.f_pos), so.grad_potential(S, q[f]), H, dH))
    return out


@functools.lru_cache(maxsize=None)
def _oracle_step(name):
    """States after 1 and 3 leapfrog steps, with the fixed-point counts of the last step of each."""
    row = ROWS[name]
    _, q, p, _, _ = _inputs(name)
    out = []
    for f in range(F):
        S, qq, pp, states = _chain_setup(name, f), q[f], p[f], []
        for s in range(3):
            cnt = []
            qq, pp = so.rhmc_step(S, qq, pp, 1e-6, row.counter_max, counters=cnt)
            if s in (0, 2):
                states.append((qq, pp, cnt[0]))
        out.append(states)
    return out


@functools.lru_cache(maxsize=None)
def _oracle_run(name):
    row = ROWS[name]
    _, q, _, normals, lnu = _inputs(name)
    return [so.run_rhmc(_chain_setup(name, f), q[f], normals[f], lnu[f], NITER, NSTEPS, 0.2, f_pos=row.f_pos,
                        counter_max=row.counter_max, schedule_g_ff2=_schedule(row)) for f in range(F)]


@functools.lru_cache(maxsize=None)
def _oracle_single(name):
    row = ROWS[name]
    _, q, p, _, _ = _inputs(name)
    return [so.run_single_rhmc(_chain_setup(name, f), q[f], p[f], SINGLE_STEPS, 0.2, f_pos=row.f_pos,
                               counter_max=row.counter_max) for f in range(F)]


# ------------------------------------------------------------------------------------------------ device side
def _env(monkeypatch, name, cta=False):
    for k, v in ROWS[name].env:
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("SRHMC_DISABLE_CHAIN_KERNEL", "1" if cta else "0")


def _ctx(name, mode):
    from hmc_stellar_toy_model_b200 import _capi
    from test_gpu_parity import make_ctx

    row = ROWS[name]
    ctx = make_ctx(_setup(row), n_fields=F, max_stars=1, precision=row.prec)
    ctx.set_data(_inputs(name)[0])
    plan = ctx.chain_plan()
    PLANS.append(dict(plan, row=name, mode=mode))
    for key, want in row.expect.items():
        assert plan[key] == want, (name, key, plan)
    if plan["chain_kernel"]:
        lay = _capi.chain_layout(row.R, plan["image_bytes"], plan["pixel_f32"])
        assert plan["smem_bytes"] == lay["smem_bytes"] <= SMEM_MAX and plan["tab_stride"] == lay["tab_stride"], plan
        assert plan["blocks_per_sm"] >= 1 and ctx.launch_plan()["chain_kernel"] == 1
    else:
        assert not any(v for k, v in plan.items() if k != "chain_kernel"), plan
    return ctx


def _f32_chain(name):
    """FP32 pixel arithmetic runs only in the gradient-only evaluations of the one-star kernel's steps."""
    return ROWS[name].prec == 32 and ROWS[name].expect["chain_kernel"] == 1


def _fp64_results(name):
    """Evaluations that return the potential stay FP64 in the FP32 build of the one-star kernel; the CTA kernel's FP32
    build renders every evaluation in float."""
    return ROWS[name].prec == 64 or _f32_chain(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("eval"))
def test_eval(name, monkeypatch):
    _env(monkeypatch, name)
    _, q, _, _, _ = _inputs(name)
    with _ctx(name, "eval") as ctx:
        V, grad, H, Hg = ctx.eval(q, f_pos=ROWS[name].f_pos, g_ff2=1.0)
    tol = RTOL if _fp64_results(name) else F32_TOL
    want = _oracle_eval(name)
    for f, (Vo, _, Ho, dHo) in enumerate(want):
        assert relerr(V[f], Vo) < tol, (f, V[f], Vo)
        assert relerr(H[f], Ho) < RTOL and np.allclose(Hg[f], dHo, rtol=RTOL, atol=0), f
    assert _scale_err(grad, np.stack([w[1] for w in want]), 1e-3 if tol == RTOL else 1.0) < tol


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("step"))
def test_steps(name, monkeypatch):
    row = ROWS[name]
    _env(monkeypatch, name)
    _, q, p, _, _ = _inputs(name)
    with _ctx(name, "step") as ctx:
        res = [ctx.step(q, p, k, 0.2, counter_max=row.counter_max, g_ff2=1.0, return_counts=True) for k in (1, 3)]
    want = _oracle_step(name)
    reached = False
    for k, (qk, pk, cnt) in enumerate(res):
        qo, po = np.stack([w[k][0] for w in want]), np.stack([w[k][1] for w in want])
        if row.prec == 64:
            assert _pos_err(qk, qo) < RTOL and _scale_err(pk, po, 1e-3) < QTOL, k
            assert [tuple(c) for c in cnt] == [w[k][2] for w in want], k
        else:
            assert _pos_err(qk, qo) < F32_TOL and _scale_err(pk, po, 1.0) < F32_TOL, k
        reached |= any(max(w[k][2]) == row.counter_max for w in want)
    assert reached == (row.counter_max < 1000), "the fixed-point cap should be reached exactly when it is small"


def _check_energies_at_own_states(name, r, stride):
    """E, V and T of every recorded row against the oracle at the chain's own (q, p): these evaluations are FP64 in every
    build, whatever path the trajectory took."""
    row = ROWS[name]
    for f in range(F):
        S = _chain_setup(name, f)
        for k in range(r.E_chain.shape[1]):
            S.g_ff2 = float(_schedule(row)[min(k * stride, 2)]) if row.schedule else 1.0
            qk, pk = r.q_chain[f, k], r.p_chain[f, k]
            H = so.metric(S, qk)
            V, T = so.potential(S, qk, row.f_pos), so.kinetic(pk, H)
            assert relerr(r.V_chain[f, k], V) < RTOL and relerr(r.E_chain[f, k], V + T) < RTOL, (f, k)
            assert abs(r.T_chain[f, k] - T) < RTOL * abs(V), (f, k)


def _check_run(name, r, outs, stride):
    if _f32_chain(name):
        _check_energies_at_own_states(name, r, stride)
        return
    for f, out in enumerate(outs):
        assert np.array_equal(r.A_chain[f].astype(bool), out.A[::stride]), f
        assert first_divergence(r.q_chain[f], out.q[::stride], QTOL) == -1, f
        assert first_divergence(r.p_chain[f], out.p[::stride], QTOL) == -1, f
        assert relerr(r.E_chain[f], out.E[::stride]) < RTOL and relerr(r.V_chain[f], out.V[::stride]) < RTOL, f
        assert np.max(np.abs(r.T_chain[f] - out.T[::stride])) < RTOL * np.max(np.abs(out.V)), f
        if stride == 1:
            assert abs(r.accept_rate[f] - out.A.mean()) < 1e-12, f


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("run"))
def test_run_injected_draws(name, monkeypatch):
    row = ROWS[name]
    _env(monkeypatch, name)
    _, q, _, normals, lnu = _inputs(name)
    with _ctx(name, "run") as ctx:
        r = ctx.run(q, NITER, NSTEPS, 0.2, normals=normals, lnu=lnu, g_ff2=1.0, f_pos=row.f_pos,
                    counter_max=row.counter_max, chain_stride=row.stride, schedule_g_ff2=_schedule(row))
    _check_run(name, r, _oracle_run(name), row.stride)


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("philox"))
def test_run_philox_replayed(name, monkeypatch):
    row = ROWS[name]
    _env(monkeypatch, name)
    _, q, _, _, _ = _inputs(name)
    with _ctx(name, "run") as ctx:
        normals, lnu = ctx.philox_draws(77, NITER_PHILOX)
        r = ctx.run(q, NITER_PHILOX, NSTEPS, 0.2, seed=77, g_ff2=1.0, f_pos=row.f_pos, counter_max=row.counter_max,
                    chain_stride=row.stride, schedule_g_ff2=_schedule(row))
    outs = [] if _f32_chain(name) else [
        so.run_rhmc(_chain_setup(name, f), q[f], normals[f], lnu[f], NITER_PHILOX, NSTEPS, 0.2, f_pos=row.f_pos,
                    counter_max=row.counter_max, schedule_g_ff2=_schedule(row)) for f in range(F)]
    _check_run(name, r, outs, row.stride)


def _energy_err(a, b):
    """Largest difference over the finite entries; inf where the two do not agree on which entries are infinite."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    fin = np.isfinite(b)
    if not np.array_equal(a[~fin], b[~fin]) or not np.all(np.isfinite(a[fin])):
        return np.inf
    return float(np.max(np.abs(a[fin] - b[fin]), initial=0.0))


@pytest.mark.gpu
@pytest.mark.parametrize("name", _rows("single"))
def test_run_single(name, monkeypatch):
    """MODE_SINGLE: every step also returns the potential, so every evaluation is FP64 in both builds.  V - V0 and E - E0
    are checked against the size of V; T - T0 against its own largest value.  A faint star whose flux passes below f_lim
    mid-trajectory has V = +inf at those steps (f_pos): the kernel must report +inf at exactly the same steps."""
    row = ROWS[name]
    _env(monkeypatch, name)
    _, q, p, _, _ = _inputs(name)
    with _ctx(name, "single") as ctx:
        qc, pc, E, V, T = ctx.run_single(q, p, SINGLE_STEPS, 0.2, counter_max=row.counter_max, f_pos=row.f_pos, g_ff2=1.0)
    for f, out in enumerate(_oracle_single(name)):
        e_scale = abs(so.potential(_chain_setup(name, f), q[f], row.f_pos))
        assert first_divergence(qc[f], out.q, QTOL) == -1, f
        assert _scale_err(pc[f], out.p, 1e-3) < QTOL, f
        assert _energy_err(V[f], out.V) < RTOL * e_scale and _energy_err(E[f], out.E) < RTOL * e_scale, f
        assert np.max(np.abs(T[f] - out.T)) < RTOL * max(np.max(np.abs(out.T)), 1.0), f


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n, r in ROWS.items() if r.prec == 64 and r.expect["chain_kernel"]])
def test_whole_batch_matches_cta_kernel(name, monkeypatch):
    """The one-star kernel and the CTA-per-field kernel on the whole batch, at the tolerances of
    test_gpu_parity.test_chain_kernel_matches_field_kernel_and_oracle."""
    from test_gpu_parity import grad_relerr

    row = ROWS[name]
    _, q, p, normals, lnu = _inputs(name)
    res = []
    for cta in (False, True):
        _env(monkeypatch, name, cta)
        with _ctx(name, "eval") if not cta else _cta_ctx(name) as ctx:
            ev = ctx.eval(q, f_pos=row.f_pos, g_ff2=1.0)
            st = ctx.step(q, p, 3, 0.2, counter_max=row.counter_max, g_ff2=1.0, return_counts=True)
            r = ctx.run(q, NITER, NSTEPS, 0.2, normals=normals, lnu=lnu, g_ff2=1.0, f_pos=row.f_pos,
                        counter_max=row.counter_max, chain_stride=row.stride, schedule_g_ff2=_schedule(row))
        res.append((ev, st, r))
    (ev, st, r), (ev2, st2, r2) = res
    assert relerr(ev[0], ev2[0]) < 1e-12 and grad_relerr(ev[1], ev2[1]) < 1e-10
    assert np.array_equal(ev[2], ev2[2]) and np.array_equal(ev[3], ev2[3])
    assert _pos_err(st[0], st2[0]) < 1e-10 and np.array_equal(st[2], st2[2])
    assert np.array_equal(r.A_chain, r2.A_chain)
    assert _pos_err(r.q_chain, r2.q_chain) < 1e-9 and relerr(r.E_chain, r2.E_chain) < 1e-11


def _cta_ctx(name):
    from test_gpu_parity import make_ctx

    row = ROWS[name]
    ctx = make_ctx(_setup(row), n_fields=F, max_stars=1, precision=row.prec)
    ctx.set_data(_inputs(name)[0])
    assert ctx.chain_plan()["chain_kernel"] == 0
    return ctx


@pytest.mark.gpu
def test_rows_cover_every_arm():
    """The union of the plans the tests above asserted (runs after them) covers every arm of the one-star kernel."""
    assert PLANS, "run the whole module: the plans are recorded by the tests above"
    on = [pl for pl in PLANS if pl["chain_kernel"]]
    assert {(pl["image_bytes"], pl["pixel_f32"]) for pl in on} == {(8, 0), (4, 0), (2, 0), (2, 1)}
    assert {pl["window_cols"] for pl in on} == {24, 32}
    assert {pl["window_cols"] for pl in on if pl["pixel_f32"]} == {24, 32}
    assert {pl["mode"] for pl in on} == {"eval", "step", "run", "single"}
    assert any(not pl["chain_kernel"] for pl in PLANS)
    odd_f32 = {ROWS[pl["row"]].R for pl in on if pl["pixel_f32"] and ROWS[pl["row"]].R % 2}
    assert len(odd_f32) >= 2, odd_f32


# ------------------------------------------------------------------------------------------------ host only (no device)
def test_chain_layout_is_aligned_for_every_row_count():
    """srhmc_chain_layout is the computation the kernel takes its shared-memory pointers from.  For every row count and
    image layout: each chain's image starts on its element size, each row table on 16 bytes (the kernel reads and writes
    it with 128-bit accesses), and the block fits the 227 KB a block may use.  R = 32 keeps the strides it always had."""
    from hmc_stellar_toy_model_b200 import _capi

    for nbytes, f32 in ((8, 0), (4, 0), (2, 0), (2, 1)):
        for R in range(1, 65):
            L = _capi.chain_layout(R, nbytes, f32)
            assert L["log_bytes"] == 64 * 16 and L["img_stride"] == (32 * R + 4) * nbytes, (R, nbytes, L)
            for g in range(8):
                assert (L["log_bytes"] + g * L["img_stride"]) % nbytes == 0, (R, nbytes, f32, g)
                assert (L["tab_base"] + g * L["tab_stride"]) % 16 == 0, (R, nbytes, f32, g, L)
            assert L["tab_base"] == L["log_bytes"] + 8 * L["img_stride"]
            assert L["tab_stride"] >= R * (16 + 8 * f32) + 16 and L["tab_stride"] - (R * (16 + 8 * f32) + 16) < 16
            assert L["smem_bytes"] == L["tab_base"] + 8 * L["tab_stride"] <= SMEM_MAX, (R, nbytes, f32, L)
    assert [_capi.chain_layout(32, b, f)["tab_stride"] for b, f in ((8, 0), (4, 0), (2, 0), (2, 1))] == [528] * 3 + [784]
    assert _capi.chain_layout(64, 8)["smem_bytes"] == 140672
    for bad in ((0, 2, 0), (65, 2, 0), (32, 1, 0), (32, 8, 1), (32, 4, 1)):
        with pytest.raises(_capi.SrhmcError):
            _capi.chain_layout(*bad)


def _column_exponent(C, fwhm, win, step=1.0 / 16):
    """NumPy restatement of chain_eval's first column of each lane (sub = 0..3) over star positions y in [-1, C + 1]: the
    window start jb, v0 = jb + 0.5 - y, the exponent v0^2 / 2s^2 of its weight and the argument -(8 v0 + 16) / 2s^2 of its
    first ratio."""
    inv2s2 = 1.0 / (2.0 * (fwhm / 2.354) ** 2)
    y = -1.0 + step * np.arange(int(round((C + 2) / step)) + 1)
    worst = 0.0
    for sub in range(4):
        jb = sub + (np.clip(np.ceil(y - (0.5 + 0.5 * win)), 0, max(C - win, 0)) if win < 32 else 0)
        v0 = jb + 0.5 - y
        worst = max(worst, float(np.max(np.maximum(v0 * v0, -(8.0 * v0 + 16.0)) * inv2s2)))
    return worst


def test_narrow_psf_eligibility_rule():
    """The host keeps a PSF on the one-star kernel only while every lane's column table starts at most 640 (50 below the
    kernel's cut-off at 690) over the support.  The library's bound equals the NumPy restatement, a 16 times finer scan of
    y finds no larger exponent, and the rows "k" land where the rule says."""
    from hmc_stellar_toy_model_b200 import _capi

    lib = _capi.load_library()
    for C in (1, 5, 17, 23, 24, 25, 28, 31, 32):
        for win in (24, 32):
            for fwhm in (0.5, 0.7, 1.0, 1.4, 1.6, 1.7, 2.0, 2.5, 3.5, 4.2):
                got = lib.srhmc_chain_column_exponent(C, fwhm, win)
                want = _column_exponent(C, fwhm, win)
                assert abs(got - want) <= 1e-12 * want, (C, win, fwhm, got, want)
                assert _column_exponent(C, fwhm, win, step=1.0 / 256) <= want * (1 + 1e-12), (C, win, fwhm)
    ok = lambda C, fwhm, win=24: lib.srhmc_chain_column_exponent(C, fwhm, win) <= 640.0
    assert ok(32, 3.5) and ok(32, 3.5, 32) and ok(32, 1.7) and not ok(32, 1.6) and not ok(32, 1.4) and not ok(28, 0.7)
    # the full width starts lane 0 at the first column wherever the star is: the bound there is FWHM ~2 px
    assert not ok(32, 2.1, 32) and ok(32, 2.2, 32)
    assert lib.srhmc_chain_column_exponent(33, 3.5, 24) == -1.0 and lib.srhmc_chain_column_exponent(32, 3.5, 16) == -1.0
    for name, row in ROWS.items():
        if row.R <= 64 and row.C <= 32 and not dict(row.env).get("SRHMC_CHAIN_WINDOW"):
            win = 32 if row.fwhm / 2.354 > 1.5 else 24
            assert ok(row.C, row.fwhm, win) == (name.startswith("k") is False or name == "k-1.7"), name
