"""Reversible-jump chains of the large-field engine (BigFieldRHMC.run_rj, srhmc_big_rj_configure, csrc/big_rj.cuh) against
the float64 restatement tests/rj_oracle.py with the patch-limited PSF, against the CTA-per-field kernel's run_rj, and
against the engine's own within-model run.  Every oracle row runs on the three evaluation paths (fused tile kernel,
star-centric gradients on the tile lists, scatter / pixel / gather), eagerly and as one replayed graph."""
import numpy as np
import pytest

import rj_oracle as rj
import stellar_oracle as so
from helpers import first_divergence, relerr

RAD = 12
P_MOVE = [0.2, 0.4, 0.4]
BETA = (2.0, 3.0)
PATHS = ["tile", "star", "scatter"]


def _setup(R, C):
    S = so.Setup(num_rows=R, num_cols=C, dt=5e-2, g_xx=0.05, g_ff=4.0, g_ff2=4.0, use_prior=True, alpha=2.0,
                 V_prior_const=0.7)
    S.fmin, S.fmax = S.mag2flux_converter(20.0), S.mag2flux_converter(15.0)
    return S


def _stars(S, rng, n):
    f = so.pow_law_sample(2.0, S.fmin, S.fmax, rng.random_sample(n))
    return np.stack([f, rng.uniform(1, S.num_rows - 1, n), rng.uniform(1, S.num_cols - 1, n)], axis=1)


def _field(R, C, n_truth, n_start, seed):
    """Poisson data of n_truth stars and a start list of n_start others."""
    rng = np.random.RandomState(seed)
    S = _setup(R, C)
    truth = _stars(S, rng, n_truth)
    S.D = rng.poisson(so.model_image(S, truth.ravel())).astype(float)
    return S, _stars(S, rng, n_start)


def _draws(S, L, n_max, seed):
    """Device-record restatement, normals [L, 3 n_max] and lnu [L] for injection into both sides."""
    rec = rj.rj_records(seed, [0], L, *BETA)[0]
    rng = np.random.RandomState(seed)
    return rec, rng.randn(L, 3 * n_max), np.log(rng.random_sample(L))


def _oracle(S, q0, niter, nsteps, rec, normals, lnu, n_max, P_move=P_MOVE):
    return rj.rj_run(S, q0.ravel(), niter, nsteps, S.dt, P_move, rj.DeviceDraws(S, P_move, rec, normals, lnu), n_max=n_max,
                     K_split=1.0, beta_a=BETA[0], beta_b=BETA[1], rad=RAD)


# the oracle row: 64 x 64, 40 start stars, room for 60; these draws accept births, deaths, splits and merges
ORACLE_ROW = dict(R=64, C=64, n_truth=40, n_start=40, seed=5, n_max=60, niter=30, nsteps=2)


def test_oracle_row_accepts_every_jump():
    """The injected draws of the oracle row make the oracle accept all four jumps (no device needed)."""
    r = ORACLE_ROW
    S, q0 = _field(r["R"], r["C"], r["n_truth"], r["n_start"], r["seed"])
    out = _oracle(S, q0, r["niter"], r["nsteps"], *_draws(S, r["niter"] + 1, r["n_max"], r["seed"]), r["n_max"])
    assert set(out["move_chain"][out["A_chain"]].tolist()) >= {1, 2, 3, 4}


# ------------------------------------------------------------------------------------------------ GPU
def _consts(S):
    return dict(psf_fwhm_pix=S.PSF_FWHM_pix, B_count=S.B_count, f_lim=S.f_lim, f_low=S.mag2flux_converter(S.mB + 2),
                g0=S.g0, g1=S.g1, g2=S.g2, g_xx=S.g_xx, g_ff=S.g_ff, use_prior=S.use_prior, alpha=S.alpha,
                V_prior_const=S.V_prior_const)


_STREAM = None


def _engine(S, q0, n_max, path, monkeypatch, world=1):
    """One strip of the field (SRHMC_BIG_PATH / SRHMC_BIG_STAR pick the evaluation path when the strip is created)."""
    import torch

    from hmc_stellar_toy_model_b200 import bigfield as bf

    global _STREAM
    if _STREAM is None:
        _STREAM = torch.cuda.Stream()   # graph capture needs a non-default stream
    torch.cuda.set_stream(_STREAM)
    monkeypatch.setenv("SRHMC_BIG_PATH", "tile" if path == "star" else path)
    monkeypatch.setenv("SRHMC_BIG_STAR", "1" if path == "star" else "0")
    strips = []
    for r in range(world):
        s = bf.BigFieldStrip(rows=S.num_rows, cols=S.num_cols, rank=r, world=world, device=0, max_stars=n_max,
                             max_ghosts=n_max, patch_radius=RAD, halo=RAD, **_consts(S))
        s.set_stream(_STREAM.cuda_stream)
        s.set_data(S.D)
        s.set_stars(q0)
        strips.append(s)
    return bf.BigFieldRHMC(strips, bf.LocalComm() if world > 1 else bf.NoComm())


def _run_kw(S, **kw):
    return dict(dict(P_move=P_MOVE, fmin=S.fmin, fmax=S.fmax, K_split=1.0, beta_a=BETA[0], beta_b=BETA[1], g_ff2=4.0,
                     want=("q", "p")), **kw)


def _assert_matches_oracle(out, want, strip):
    assert np.array_equal(out["move_chain"], want["move_chain"])
    assert np.array_equal(out["N_chain"], want["N_chain"])
    assert np.array_equal(out["A_chain"].astype(bool), want["A_chain"])
    assert relerr(out["E_chain"], want["E_chain"]) < 1e-9
    assert first_divergence(out["q_chain"].reshape(len(want["q_chain"]), -1), want["q_chain"], 1e-7) == -1
    assert out["n_final"] == want["q_final"].size // 3 and out["overflow"] == want["overflow"]
    q, _, _ = strip.get_stars()
    assert strip.n == out["n_final"] and np.array_equal(strip.ids, np.arange(strip.n))
    assert relerr(q.ravel(), want["q_final"]) < 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("path", PATHS)
def test_run_rj_matches_the_oracle(path, graph, monkeypatch):
    r = ORACLE_ROW
    S, q0 = _field(r["R"], r["C"], r["n_truth"], r["n_start"], r["seed"])
    L = r["niter"] + 1
    rec, normals, lnu = _draws(S, L, r["n_max"], r["seed"])
    eng = _engine(S, q0, r["n_max"], path, monkeypatch)
    out = eng.run_rj(r["niter"], r["nsteps"], S.dt, draws=rec, normals=normals, lnu=lnu, use_graph=graph, **_run_kw(S))
    want = _oracle(S, q0, r["niter"], r["nsteps"], rec, normals, lnu, r["n_max"])
    _assert_matches_oracle(out, want, eng.strips[0])
    assert set(want["move_chain"][want["A_chain"]].tolist()) >= {1, 2, 3, 4}
    # recorded rows: table order, zero past N
    for l in range(L):
        assert not np.any(out["q_chain"][l, out["N_chain"][l]:]) and not np.any(out["p_chain"][l, out["N_chain"][l]:])
    # a later within-model run works from the final table
    after = eng.run(2, r["nsteps"], S.dt, g_ff2=4.0, seed=9)
    assert np.all(np.isfinite(after["E_chain"]))


@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
def test_run_rj_is_the_cta_kernels_chain(path, monkeypatch):
    """Same field and seed, no injection: the one-field CTA kernel (patch_radius = r) and the large-field engine draw the same
    records, normals and log-uniforms and take the same decisions."""
    from test_gpu_parity import make_ctx

    r = ORACLE_ROW
    S, q0 = _field(r["R"], r["C"], r["n_truth"], r["n_start"], r["seed"])
    seed, niter = 4242, 24
    kw = _run_kw(S)
    with make_ctx(S, n_fields=1, max_stars=r["n_max"], patch_radius=RAD) as ctx:
        ctx.set_data(S.D)
        q = np.zeros((1, 3 * r["n_max"]))
        q[0, :q0.size] = q0.ravel()
        want = ctx.run_rj(q, niter, r["nsteps"], S.dt, nstars=[len(q0)], f_pos=True, g_ff2=4.0, seed=seed,
                          **{k: kw[k] for k in ("P_move", "fmin", "fmax", "K_split", "beta_a", "beta_b")})
    eng = _engine(S, q0, r["n_max"], path, monkeypatch)
    out = eng.run_rj(niter, r["nsteps"], S.dt, seed=seed, **kw)
    assert np.array_equal(out["move_chain"], want.move_chain[0])
    assert np.array_equal(out["N_chain"], want.N_chain[0])
    assert np.array_equal(out["A_chain"], want.A_chain[0])
    assert relerr(out["E_chain"], want.E_chain[0]) < 1e-9
    assert out["n_final"] == want.n_final[0]
    assert np.any(out["move_chain"] != 0)


@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
def test_within_model_run_rj_is_run(path, monkeypatch):
    """P_move = [1, 0, 0] with injected normals and lnu takes run()'s decisions with run()'s energies; the stars are stored
    in another order, so the sums may differ in the last bits."""
    r = ORACLE_ROW
    S, q0 = _field(r["R"], r["C"], r["n_truth"], r["n_start"], r["seed"])
    niter, n = 12, len(q0)
    rng = np.random.RandomState(3)
    normals = rng.randn(niter + 1, n, 3)
    lnu = np.log(rng.random_sample(niter + 1))
    dt = 2e-2   # some iterations accept, some reject
    a = _engine(S, q0, n, path, monkeypatch).run(niter, r["nsteps"], dt, g_ff2=4.0, normals=normals, lnu=lnu)
    eng = _engine(S, q0, n, path, monkeypatch)
    before = eng.strips[0].launch_count
    b = eng.run_rj(niter, r["nsteps"], dt, normals=normals.reshape(niter + 1, -1), lnu=lnu,
                   **_run_kw(S, P_move=[1.0, 0.0, 0.0], want=()))
    assert np.array_equal(a["A_chain"], b["A_chain"]) and np.any(a["A_chain"]) and not np.all(a["A_chain"])
    assert relerr(b["E_chain"], a["E_chain"]) < 1e-12
    assert np.all(b["move_chain"] == 0) and np.all(b["N_chain"] == n) and b["n_final"] == n
    assert eng.strips[0].launch_count - before > 0 and eng.replayed_launches > 0


@pytest.mark.gpu
def test_merge_pick_across_cells(monkeypatch):
    """256 x 256 with 600 stars and K_split = 1: many pairs straddle the 38.6 px cut-off of the merge cells.  Records forced to
    merges with chosen u_a pick the oracle's dense-weight pair."""
    S, q0 = _field(256, 256, 500, 600, 11)
    niter, nsteps, n_max = 7, 1, 620
    L = niter + 1
    rec, normals, lnu = _draws(S, L, n_max, 11)
    rec[:, 0] = 0.9                     # the split / merge band of P_MOVE
    rec[:, 1] = 0.7                     # shrink: merge
    rec[:, 2] = [0.003, 0.21, 0.5, 0.77, 0.999, 0.35, 0.62, 0.08]
    lnu[:] = -1e4                       # accept (almost) every merge, so the table keeps changing
    eng = _engine(S, q0, n_max, "tile", monkeypatch)
    out = eng.run_rj(niter, nsteps, S.dt, draws=rec, normals=normals, lnu=lnu, use_graph=True, **_run_kw(S))
    want = _oracle(S, q0, niter, nsteps, rec, normals, lnu, n_max)
    _assert_matches_oracle(out, want, eng.strips[0])
    assert np.sum(want["A_chain"]) >= 4


def _refusal_draws(S, n_max):
    """Records that reach every refusal from an empty table of capacity 3 on 64 x 64: a death and a split at N = 0, a merge at
    N = 1, a merge of two stars 80 px apart (every weight zero), and a birth at N = 3 (overflow at iteration 7)."""
    L = 9
    rec, normals, lnu = _draws(S, L, n_max, 21)
    birth, death, split, merge = (0.3, 0.2), (0.3, 0.7), (0.8, 0.2), (0.8, 0.7)
    moves = [death, split, birth, merge, birth, merge, birth, birth, (0.1, 0.5)]
    for l, m in enumerate(moves):
        rec[l, :2] = m
    rec[2, 2:4] = (0.02, 0.02)          # first newborn near (2, 2)
    rec[4, 2:4] = (0.98, 0.98)          # second near (62, 62)
    rec[6, 2:4] = (0.02, 0.9)
    lnu[[2, 4, 6]] = -1e4
    return rec, normals, lnu


@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
def test_refusals_leave_the_state_unchanged(path, monkeypatch):
    S, _ = _field(64, 64, 30, 1, 21)
    n_max, niter = 3, 8
    rec, normals, lnu = _refusal_draws(S, n_max)
    q0 = np.zeros((0, 3))
    want = _oracle(S, q0, niter, 2, rec, normals, lnu, n_max)
    assert want["move_chain"].tolist()[:8] == [2, 3, 1, 4, 1, 4, 1, 1]
    assert want["N_chain"].tolist() == [0, 0, 0, 1, 1, 2, 2, 3, 3]
    assert want["A_chain"].tolist()[:8] == [False, False, True, False, True, False, True, False]
    assert want["overflow"] == 7
    eng = _engine(S, q0, n_max, path, monkeypatch)
    with pytest.raises(ValueError, match="iteration 7") as e:
        eng.run_rj(niter, 2, S.dt, draws=rec, normals=normals, lnu=lnu, **_run_kw(S))
    _assert_matches_oracle(e.value.result, want, eng.strips[0])


@pytest.mark.gpu
def test_entry_point_refusals(monkeypatch):
    from hmc_stellar_toy_model_b200 import _capi

    S, q0 = _field(64, 64, 30, 20, 3)
    eng = _engine(S, q0, 40, "scatter", monkeypatch)
    with pytest.raises(_capi.SrhmcError) as e:
        eng.run_rj(3, 1, S.dt, **_run_kw(S, beta_a=0.5))
    assert e.value.code == -1
    eng.fixed_point_mode = 1
    with pytest.raises(ValueError):
        eng.run_rj(3, 1, S.dt, **_run_kw(S))
    # the C entry points refuse a strip of a tiled field, precision 32 and a per-star stop rule phase
    rjargs = _capi.RjArgs(P_move=(_capi.C.c_double * 3)(0.5, 0.25, 0.25), fmin=S.fmin, fmax=S.fmax, K_split=1.0, beta_a=2.0,
                          beta_b=2.0)
    tiled = _engine(S, q0, 40, "scatter", monkeypatch, world=2)
    with pytest.raises(ValueError):
        tiled.run_rj(3, 1, S.dt, **_run_kw(S))
    with pytest.raises(_capi.SrhmcError) as e:
        tiled.strips[0].rj_configure(rjargs, 4)
    assert e.value.code == -1
    S32, q32 = _field(1152, 1152, 10, 10, 4)
    big = _engine(S32, q32, 40, "tile", monkeypatch)
    big.strips[0].set_precision(32)
    with pytest.raises(_capi.SrhmcError) as e:
        big.strips[0].rj_configure(rjargs, 4)
    assert e.value.code == -1
    s = eng.strips[0]
    s.rj_configure(rjargs, 4)
    st = _capi.BigStep(dt=S.dt, delta=1e-6, g_ff2=4.0, counter_max=1000, f_pos=1, iteration=0, fixed_point_mode=1, seed=0)
    with pytest.raises(_capi.SrhmcError) as e:
        s.phase("PS_ADVANCE", st)
    assert e.value.code == -1
    s.rj_finish(4)


def _c5_catalogue_strip(max_stars):
    """bench.py's large field (8192^2, 1e5 mock stars) on one strip holding its find_peaks catalogue."""
    import importlib.util
    import os

    from hmc_stellar_toy_model_b200 import bigfield as bf

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_for_rj_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    t = bench.c5_truth(8192, 8192, 100000, 77)
    ftc = bench.exp_constants()["flux_to_count"]
    strip = bf.BigFieldStrip(rows=8192, cols=8192, rank=0, world=1, device=0, max_stars=max_stars, max_ghosts=1, patch_radius=RAD,
                             halo=RAD, **t["consts"])
    strip.gen_mock_data(t["q_true"], seed=77)
    np.random.seed(78)
    cat = strip.find_peaks(ftc, 22.0)
    strip.set_stars(cat)
    fmin, fmax = 10 ** (0.4 * (22.5 - 20)) * ftc, 10 ** (0.4 * (22.5 - 15)) * ftc
    return strip, cat, t, fmin, fmax


@pytest.mark.gpu
def test_full_size_field_from_its_catalogue():
    """8192^2 with 1e5 mock stars from its find_peaks catalogue, a few replayed iterations: no error flag, N moves as the
    accepted moves say, finite energies, rows zero past N."""
    import torch

    from hmc_stellar_toy_model_b200 import bigfield as bf

    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    strip, cat, t, fmin, fmax = _c5_catalogue_strip(200000)
    strip.set_stream(stream.cuda_stream)
    out = bf.BigFieldRHMC([strip]).run_rj(5, 3, t["run"]["dt"], P_move=[0.4, 0.3, 0.3], fmin=fmin, fmax=fmax, seed=7,
                                          g_ff2=4.0, use_graph=True)
    N, mv, A = out["N_chain"].astype(int), out["move_chain"], out["A_chain"].astype(bool)
    step = {0: 0, 1: 1, 2: -1, 3: 1, 4: -1}
    expect = N[:-1] + np.array([step[m] if a else 0 for m, a in zip(mv[:-1], A[:-1])])
    assert np.array_equal(N[1:], expect)
    assert N[0] == len(cat)
    assert np.all(np.isfinite(out["E_chain"]))
    for l in range(len(N)):
        assert not np.any(out["q_chain"][l, N[l]:])
    strip.close()
