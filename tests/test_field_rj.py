"""Reversible-jump chains on the device (field_kernel MODE_RUN_RJ, srhmc_run_rj, RHMCContext.run_rj) against the float64
restatement tests/rj_oracle.py, which tests/golden/rj_chain.npz (recorded from the unmodified reference) pins on the CPU.

Each GPU row first asserts the launch plan it runs, as test_field_arms.py does, then replays the device's own draw records
(philox_rj_draws, philox_draws) through rj_oracle.rj_run and compares moves, star counts, accept decisions, energies and
chains."""
import contextlib
import ctypes as C
import io
from dataclasses import dataclass, field

import numpy as np
import pytest
from scipy import stats

import rj_oracle as rj
import stellar_oracle as so
from helpers import first_divergence, golden, relerr, setup_from


# ------------------------------------------------------------------------------------------------ CPU
def _golden_preamble(g):
    """The test script of make_golden.rj_chain up to run_RHMC, on the drop-in's host-side set-up (no device needed):
    leaves np.random where the reference's run_RHMC started drawing."""
    from hmc_stellar_toy_model_b200.sampler_RHMC import gen_pow_law_sample, multi_gym

    nobj, nmodel = g["q_true"].shape[0], g["q_model"].shape[0]
    gym = multi_gym(dt=0.0, Nsteps=0, g_xx=0.05, g_ff=4.0, g_ff2=4.0)
    np.random.seed(int(g["seed"]))
    gym.num_rows = gym.num_cols = 32
    q_true = np.zeros((nobj, 3))
    fmin, fmax = gym.mag2flux_converter(20.0), gym.mag2flux_converter(15.0)
    mag = gym.flux2mag_converter(gen_pow_law_sample(2.0, fmin, fmax, nobj))
    for i in range(nobj):
        x = np.random.random() * (gym.num_rows - 2.0) + 1.0
        y = np.random.random() * (gym.num_cols - 2.0) + 1.0
        q_true[i] = np.array([mag[i], x, y])
    q_model = np.zeros((nmodel, 3))
    q_model[:, 0] = gym.flux2mag_converter(gen_pow_law_sample(2.0, fmin, fmax, nmodel))
    q_model[:, 1] = np.random.random(size=nmodel) * (gym.num_rows - 2.0) + 1.0
    q_model[:, 2] = np.random.random(size=nmodel) * (gym.num_cols - 2.0) + 1.0
    gym.gen_mock_data(q_true)
    assert np.array_equal(gym.D, g["D"]) and np.array_equal(q_model, g["q_model"])
    return fmin, fmax


def _golden_setup(g, fmin, fmax):
    return setup_from(g, fmin=fmin, fmax=fmax)


def test_oracle_replays_the_reference_rj_chain():
    """rj_run with the legacy np.random provider reproduces the reference's reversible-jump chain move for move."""
    g = golden("rj_chain")
    fmin, fmax = _golden_preamble(g)
    S = _golden_setup(g, fmin, fmax)
    q0 = so.format_q(S, g["q_model"])
    out = rj.rj_run(S, q0, int(g["niter"]), int(g["nsteps"]), float(g["dt"]), [0.4, 0.3, 0.3],
                    rj.LegacyDraws(S, [0.4, 0.3, 0.3]), n_max=30, K_split=1.0, beta_a=4.0, beta_b=4.0)
    assert np.array_equal(out["move_chain"], g["move_chain"])
    assert np.array_equal(out["N_chain"], g["N_chain"])
    assert np.array_equal(out["A_chain"], g["A_chain"])
    assert relerr(out["E_chain"], g["E_chain"]) < 1e-9
    assert first_divergence(out["q_chain"], g["q_chain"], 1e-7) == -1
    assert np.random.random(1)[0] == g["next_uniform"][0]  # the stream was consumed draw for draw


@pytest.mark.parametrize("a,b", [(2.0, 2.0), (4.0, 4.0), (0.5, 3.0)])
def test_beta_philox_is_beta_distributed(a, b):
    n = 100000
    share, nx, ny = rj.beta_philox(a, b, 12345, np.arange(n), 3)
    assert np.all((share > 0) & (share < 1)) and nx.max() < 64 and ny.max() < 64
    assert stats.kstest(share, stats.beta(a, b).cdf).pvalue > 1e-3


def test_proposals_restate_the_drop_in():
    """rj_birth / rj_death / rj_split / rj_merge against the drop-in's host proposals fed the same draws."""
    from hmc_stellar_toy_model_b200.sampler_RHMC import multi_gym

    g = golden("rj_chain")
    S = _golden_setup(g, 100.0, 4000.0)
    rng = np.random.RandomState(5)
    tq = np.stack([rng.uniform(200, 900, 4), rng.uniform(3, 29, 4), rng.uniform(3, 29, 4)], axis=1)
    tp = rng.randn(4, 3)
    gym = multi_gym(dt=0.0, Nsteps=0, g_xx=S.g_xx, g_ff=S.g_ff, g_ff2=S.g_ff2)
    gym.num_rows = gym.num_cols = 32
    gym.fmin, gym.fmax, gym.alpha, gym.V_prior_const = S.fmin, S.fmax, S.alpha, S.V_prior_const
    gym.K_split, gym.beta_a, gym.beta_b = 1.3, 2.0, 4.0
    gym._stars_metric = lambda *stars: [so.metric(S, np.asarray(s, float)) for s in stars]
    gym.T = lambda p, H: so.kinetic(np.asarray(p, float), np.asarray(H, float))
    for move, grow in ((1, True), (1, False), (2, True), (2, False)):
        gym.Nobjs, gym.d = 4, 12
        np.random.seed(9)
        fn = gym.birth_death_move if move == 1 else gym.split_merge_move
        q_h, p_h, lr_h = fn(tq.ravel().copy(), tp.ravel().copy(), grow)
        np.random.seed(9)
        d = rj.LegacyDraws(S, None)
        if move == 1 and grow:
            got = rj.rj_birth(S, tq, tp, *d.birth(0))
        elif move == 1:
            got = rj.rj_death(S, tq, tp, d.victim(0, 4))
        elif grow:
            got = rj.rj_split(S, tq, tp, *d.split(0, 4, 1.3, 2.0, 4.0), 1.3, 2.0, 4.0)
        else:
            pick, z = d.merge(0, rj.merge_weights(tq, 1.3, 2.0, 4.0))
            got = rj.rj_merge(S, tq, tp, pick // 4, pick % 4, z, 1.3, 2.0, 4.0)
        assert np.allclose(got[0].ravel(), q_h, rtol=1e-14, atol=0) and np.allclose(got[1].ravel(), p_h, rtol=1e-14, atol=0)
        assert abs(got[2] - lr_h) <= 1e-12 * max(1.0, abs(lr_h)), (move, grow)


def test_entry_points_refuse_without_a_context():
    from hmc_stellar_toy_model_b200 import _capi

    lib = _capi.load_library()
    want = -3 if lib.srhmc_device_count() == 0 else -1
    draws = np.zeros(14)
    assert lib.srhmc_run_rj(None, C.byref(_capi.RunArgs()), C.byref(_capi.RjArgs())) == want
    assert lib.srhmc_philox_rj_draws(None, 1, 0, 0, 1, 2.0, 2.0, _capi.dptr(draws)) == want


# ------------------------------------------------------------------------------------------------ GPU
P_MOVE = [0.2, 0.4, 0.4]


@dataclass(frozen=True)
class Row:
    R: int
    C: int
    N_max: int
    nstars: tuple
    expect: dict = field(hash=False)
    rad: int = 0
    shared: bool = False
    beta: tuple = (2.0, 4.0)
    niter: int = 11
    nsteps: int = 3
    inject: bool = False       # injected draws (_injected_draws) instead of the device's Philox


ROWS = {
    # the golden's 32x32 full-image set-up, beta_a != beta_b pins the merge weights' share convention
    "golden": Row(32, 32, 30, (5,), dict(compact=0, image_in_smem=1)),
    "compact": Row(64, 64, 150, (140,), dict(compact=1), rad=12, niter=5, nsteps=2),
    "global": Row(128, 128, 40, (30,), dict(compact=0, image_in_smem=0), niter=7, nsteps=2),
    "shared": Row(32, 32, 12, (6, 3, 9), dict(compact=0), shared=True),
    "ragged": Row(32, 32, 8, (0, 1, 2, 7), dict(compact=0), niter=15, inject=True),
}


def _setup(row):
    S = so.Setup(num_rows=row.R, num_cols=row.C, dt=5e-2, g_xx=0.05, g_ff=4.0, g_ff2=4.0, use_prior=True, alpha=2.0,
                 V_prior_const=0.7)
    S.fmin, S.fmax = S.mag2flux_converter(20.0), S.mag2flux_converter(15.0)
    return S


def _inputs(name):
    row = ROWS[name]
    rng = np.random.RandomState(sum(map(ord, name)))
    S = _setup(row)

    def stars(n):
        f = so.pow_law_sample(2.0, S.fmin, S.fmax, rng.random_sample(n))
        return np.stack([f, rng.uniform(1, row.R - 1, n), rng.uniform(1, row.C - 1, n)], axis=1)

    truth = stars(row.N_max)
    D = []
    q = np.zeros((len(row.nstars), 3 * row.N_max))
    shared_D = rng.poisson(so.model_image(S, truth.ravel())).astype(float)
    for f, n in enumerate(row.nstars):
        t = stars(n)
        D.append(shared_D if row.shared else rng.poisson(so.model_image(S, stars(row.N_max // 2).ravel())).astype(float))
        q[f, :3 * n] = t.ravel()
    return S, D, q


def _ctx(name):
    from test_gpu_parity import make_ctx

    row = ROWS[name]
    S, D, _ = _inputs(name)
    ctx = make_ctx(S, n_fields=len(row.nstars), max_stars=row.N_max, patch_radius=row.rad, shared_data=row.shared)
    ctx.set_data(D[0] if row.shared else np.stack(D))
    plan = ctx.launch_plan()
    got = dict(compact=plan["compact_tables"], image_in_smem=plan["image_in_smem"])
    for k, v in row.expect.items():
        assert got[k] == v, (name, k, plan)
    return ctx


def _rj_kw(row):
    S = _setup(row)
    return dict(P_move=P_MOVE, fmin=S.fmin, fmax=S.fmax, K_split=1.0, beta_a=row.beta[0], beta_b=row.beta[1])


def _injected_draws(row, seed):
    """Records (the oracle's restatement of the device records), normals and lnu of the ragged row, edited so that it reaches
    every refusal branch: field 0 (no star) draws a death and field 1 (one star) a merge at iteration 0; field 3 (N_max - 1
    stars) draws births at iterations 0 and 1, the first accepted whatever its ratio, so that the second needs N_max + 1."""
    F, L = len(row.nstars), row.niter + 1
    rec = rj.rj_records(seed, range(F), L, *row.beta)
    rng = np.random.RandomState(seed)
    normals = rng.randn(F, L, 3 * row.N_max)
    lnu = np.log(rng.random_sample((F, L)))
    # u_move in the birth/death band of P_MOVE (0.2 .. 0.6) or the split/merge band (0.6 .. 1); u_grow < 0.5 grows
    rec[0, 0, :2] = (0.3, 0.7)
    rec[1, 0, :2] = (0.8, 0.7)
    rec[3, :2, :2] = (0.3, 0.2)
    lnu[3, 0] = -1e4
    return rec, normals, lnu


def _ragged_checks(r):
    """The refusal branches, each a rejected jump with the state unchanged."""
    assert (r.move_chain[0, 0], r.N_chain[0, 0], r.A_chain[0, 0], r.N_chain[0, 1]) == (2, 0, 0, 0)  # death at N = 0
    assert (r.move_chain[1, 0], r.N_chain[1, 0], r.A_chain[1, 0], r.N_chain[1, 1]) == (4, 1, 0, 1)  # merge at N = 1
    assert (r.move_chain[3, 0], r.A_chain[3, 0], r.N_chain[3, 1]) == (1, 1, 8)                     # birth to N_max
    assert (r.move_chain[3, 1], r.A_chain[3, 1], r.N_chain[3, 2], r.overflow[3]) == (1, 0, 8, 1)    # overflow
    assert np.all(r.overflow[:3] == -1)


def test_ragged_draws_reach_every_refusal():
    """The oracle on the ragged row's injected draws (no device needed) takes the branches _ragged_checks asserts."""
    from types import SimpleNamespace

    row = ROWS["ragged"]
    S, D, q = _inputs("ragged")
    rec, normals, lnu = _injected_draws(row, 7)
    outs = [rj.rj_run(S.clone(D=D[f]), q[f, :3 * n], row.niter, row.nsteps, S.dt, P_MOVE,
                      rj.DeviceDraws(S, P_MOVE, rec[f], normals[f], lnu[f]), n_max=row.N_max, K_split=1.0,
                      beta_a=row.beta[0], beta_b=row.beta[1]) for f, n in enumerate(row.nstars)]
    _ragged_checks(SimpleNamespace(**{k: np.array([o[k] for o in outs]) for k in ("move_chain", "N_chain", "A_chain",
                                                                                     "overflow")}))


@pytest.mark.gpu
def test_philox_rj_draws_match_the_oracle_and_replay_bit_for_bit():
    row = ROWS["shared"]
    with _ctx("shared") as ctx:
        rec = ctx.philox_rj_draws(77, 40, beta_a=0.5, beta_b=3.0, field_id_base=3, field_id_stride=2)
        want = rj.rj_records(77, [3, 5, 7], 41, 0.5, 3.0)
        assert np.allclose(rec[..., :7], want[..., :7], rtol=1e-15, atol=1e-15)
        assert np.allclose(rec[..., 8:], want[..., 8:], rtol=1e-15, atol=1e-15)
        assert np.allclose(rec[..., 7], want[..., 7], rtol=1e-14, atol=0)
        _, q = _inputs("shared")[1:]
        kw = dict(nstars=list(row.nstars), f_pos=True, g_ff2=4.0, seed=77, field_id_base=3, field_id_stride=2)
        a = ctx.run_rj(q, 40, 2, 5e-2, **dict(_rj_kw(row), beta_a=0.5, beta_b=3.0), **kw)
        b = ctx.run_rj(q, 40, 2, 5e-2, draws=rec, **dict(_rj_kw(row), beta_a=0.5, beta_b=3.0), **kw)
    for k in ("q_chain", "E_chain", "A_chain", "N_chain", "move_chain", "n_final"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ROWS))
def test_device_run_matches_the_oracle(name):
    row = ROWS[name]
    S, D, q = _inputs(name)
    seed = 1000 + len(name)
    with _ctx(name) as ctx:
        if row.inject:
            rec, normals, lnu = _injected_draws(row, 7)
            injected = dict(draws=rec, normals=normals, lnu=lnu)
        else:
            injected = {}
        r = ctx.run_rj(q, row.niter, row.nsteps, S.dt, nstars=list(row.nstars), f_pos=True, g_ff2=4.0, seed=seed,
                       **_rj_kw(row), **injected)
        if not row.inject:
            rec = ctx.philox_rj_draws(seed, row.niter, beta_a=row.beta[0], beta_b=row.beta[1])
            normals, lnu = ctx.philox_draws(seed, row.niter)
    moves = set()
    for f, n in enumerate(row.nstars):
        Sf = S.clone(D=D[f])
        out = rj.rj_run(Sf, q[f, :3 * n], row.niter, row.nsteps, S.dt, P_MOVE,
                        rj.DeviceDraws(Sf, P_MOVE, rec[f], normals[f], lnu[f]), n_max=row.N_max, K_split=1.0,
                        beta_a=row.beta[0], beta_b=row.beta[1], rad=row.rad)
        assert np.array_equal(r.move_chain[f], out["move_chain"]), f
        assert np.array_equal(r.N_chain[f], out["N_chain"]), f
        assert np.array_equal(r.A_chain[f].astype(bool), out["A_chain"]), f
        assert relerr(r.E_chain[f], out["E_chain"]) < 1e-9, f
        assert first_divergence(r.q_chain[f], out["q_chain"], 1e-7) == -1, f
        assert r.n_final[f] == out["q_final"].size // 3 and r.overflow[f] == out["overflow"], f
        moves |= set(out["move_chain"][out["A_chain"]].tolist())
    assert moves & {1, 2, 3, 4}, "no jump was accepted: the row checks nothing trans-dimensional"
    if name == "ragged":
        _ragged_checks(r)


@pytest.mark.gpu
def test_within_model_only_reproduces_srhmc_run():
    row = ROWS["shared"]
    _, _, q = _inputs("shared")
    kw = dict(nstars=list(row.nstars), f_pos=True, g_ff2=4.0, seed=5)
    with _ctx("shared") as ctx:
        a = ctx.run(q, 9, 3, 5e-2, **kw)
        b = ctx.run_rj(q, 9, 3, 5e-2, **dict(_rj_kw(row), P_move=[1.0, 0.0, 0.0]), **kw)
        whole = ctx.run_rj(q, 9, 3, 5e-2, **_rj_kw(row), **kw)
    for k in ("q_chain", "E_chain", "A_chain", "q_final"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert np.all(b.move_chain == 0) and np.all(b.N_chain == np.array(row.nstars)[:, None])
    # the batch as two shards with explicit field ids
    from test_gpu_parity import make_ctx

    S, D, _ = _inputs("shared")
    parts = []
    for ids in ([0, 2], [1]):
        with make_ctx(S, n_fields=len(ids), max_stars=row.N_max, shared_data=True) as ctx:
            ctx.set_data(D[0])
            parts.append(ctx.run_rj(q[ids], 9, 3, 5e-2, field_ids=ids, **dict(kw, nstars=[row.nstars[i] for i in ids]),
                                    **_rj_kw(row)))
    for k in ("q_chain", "E_chain", "A_chain", "N_chain", "move_chain"):
        got = np.zeros_like(getattr(whole, k))
        got[[0, 2]], got[[1]] = getattr(parts[0], k), getattr(parts[1], k)
        assert np.array_equal(got, getattr(whole, k)), k


@pytest.mark.gpu
def test_refusals():
    from hmc_stellar_toy_model_b200._capi import SrhmcError
    from test_gpu_parity import make_ctx

    row = ROWS["golden"]
    _, _, q = _inputs("golden")
    good = _rj_kw(row)
    bad = [dict(P_move=[-0.1, 0.6, 0.5]), dict(P_move=[np.nan, 0.5, 0.5]), dict(P_move=[0, 0, 0]),
           dict(fmin=good["fmax"], fmax=good["fmin"]), dict(beta_a=0.0), dict(beta_b=-1.0), dict(K_split=0.0)]
    with _ctx("golden") as ctx:
        for change in bad:
            with pytest.raises(SrhmcError) as e:
                ctx.run_rj(q, 2, 1, 5e-2, nstars=[5], **dict(good, **change))
            assert e.value.code == -1, change
        with pytest.raises(SrhmcError):
            ctx.run_rj(q, 2, 1, 5e-2, nstars=[31], **good)
    S = _setup(row)
    for kw in (dict(precision=32), dict(use_prior=False)):
        S2 = S.clone(alpha=1.0) if "use_prior" in kw else S
        with make_ctx(S2, max_stars=30, **{k: v for k, v in kw.items() if k == "precision"}) as ctx:
            ctx.set_data(_inputs("golden")[1][0])
            with pytest.raises(SrhmcError) as e:
                ctx.run_rj(q, 2, 1, 5e-2, nstars=[5], **good)
            assert e.value.code == -1, kw


@pytest.mark.gpu
def test_drop_in_device_seed_runs_the_jumps_on_the_device():
    """multi_gym.run_RHMC with gym.device_seed set: the host path's attributes, shapes and dtypes, and the oracle's chain on
    the device draws; a too-small N_max raises the host path's ValueError."""
    g = golden("rj_chain")
    fmin, fmax = _golden_preamble(g)
    from hmc_stellar_toy_model_b200.sampler_RHMC import multi_gym

    def gym_run(n_max, seed=31):
        gym = multi_gym(dt=0.0, Nsteps=0, g_xx=0.05, g_ff=4.0, g_ff2=4.0)
        gym.num_rows = gym.num_cols = 32
        gym.fmin, gym.fmax = fmin, fmax
        gym.K_split, gym.beta_a, gym.beta_b = 1.0, 2.0, 4.0
        gym.use_prior, gym.alpha = True, 2.0
        gym.D = np.array(g["D"])
        gym.device_seed = seed
        state = np.random.get_state()
        with contextlib.redirect_stdout(io.StringIO()):
            gym.run_RHMC(np.copy(g["q_model"]), f_pos=True, delta=1e-6, Niter=30, Nsteps=5, dt=float(g["dt"]),
                         P_move=[0.4, 0.3, 0.3], N_max=n_max)
        assert all(np.array_equal(a, b) for a, b in zip(state[1:2], np.random.get_state()[1:2]))
        return gym

    gym = gym_run(30)
    L = 31
    for name, shape, dtype in (("q_chain", (L, 90), np.float64), ("p_chain", (L, 90), np.float64), ("E_chain", (L,), np.float64),
                               ("V_chain", (L,), np.float64), ("T_chain", (L,), np.float64), ("A_chain", (L,), np.bool_),
                               ("move_chain", (L,), np.int64), ("N_chain", (L,), np.int64)):
        a = getattr(gym, name)
        assert a.shape == shape and a.dtype == dtype, (name, a.shape, a.dtype)
    S = _golden_setup(g, fmin, fmax)
    ctx = gym._ctx
    rec = ctx.philox_rj_draws(31, 30, beta_a=2.0, beta_b=4.0)
    normals, lnu = ctx.philox_draws(31, 30)
    q0 = so.format_q(S, g["q_model"])
    out = rj.rj_run(S, q0, 30, 5, float(g["dt"]), [0.4, 0.3, 0.3], rj.DeviceDraws(S, [0.4, 0.3, 0.3], rec[0], normals[0], lnu[0]),
                    n_max=30, K_split=1.0, beta_a=2.0, beta_b=4.0)
    assert np.array_equal(gym.move_chain, out["move_chain"]) and np.array_equal(gym.N_chain, out["N_chain"])
    assert np.array_equal(gym.A_chain, out["A_chain"])
    assert relerr(gym.E_chain, out["E_chain"]) < 1e-9 and first_divergence(gym.q_chain, out["q_chain"], 1e-7) == -1
    assert gym.Nobjs == out["q_final"].size // 3
    with pytest.raises(ValueError):
        gym_run(5, seed=8)
