"""K chains of one field in one large-field context (srhmc_big_set_chains): chain c is the one-chain engine's chain drawn from
Philox field c, bit for bit, whatever K and the other chains' states; one launch sequence covers every chain; R-hat over the
context's own chains on the device."""
import numpy as np
import pytest

import stellar_oracle as so
from helpers import relerr
from hmc_stellar_toy_model_b200 import bigfield as bf

RUN = dict(nsteps=5, dt=2e-2, f_pos=True, g_ff2=4.0, seed=11)


# ------------------------------------------------------------------ host logic
def test_chain_starts_sorts_each_chain_by_its_own_tiles():
    rng = np.random.RandomState(0)
    n, K, cols = 300, 4, 200
    q = np.stack([rng.uniform(1, 9, n), rng.uniform(0, 250, n), rng.uniform(0, cols, n)], axis=1)
    qk = np.stack([q + np.array([0.0, 1.0, -1.0]) * 30 * rng.normal(size=(n, 1)) for _ in range(K)])
    for start in (q, qk):
        q_store, ids, slots = bf.chain_starts(start, K, cols)
        assert q_store.shape == (K, n, 3) and ids.shape == (K, n) and slots.shape == (K, n)
        per = np.broadcast_to(start, (K, n, 3))
        for c in range(K):
            assert np.array_equal(ids[c], bf.tile_order(per[c], cols))
            assert np.array_equal(q_store[c], per[c][ids[c]])
            # the slot of a stored star is its column in a recorded row: ascending id, the same for every chain
            row = np.empty(n, dtype=np.int64)
            row[slots[c]] = ids[c]
            assert np.array_equal(row, bf.slot_ids(ids[c]))
    _, ids, _ = bf.chain_starts(qk, K, cols)
    assert not all(np.array_equal(ids[0], ids[c]) for c in range(1, K))   # the starts sort differently
    with pytest.raises(ValueError):
        bf.chain_starts(qk[:3], K, cols)


# ------------------------------------------------------------------ GPU
def _field(name):
    if name == "philox":
        from test_bigfield_samples import _philox_field

        return _philox_field()
    from test_bigfield import _synthetic_field

    return _synthetic_field(256, 256, 3277, 31)   # the C3 shape: 256^2, 0.05 stars per pixel


def _one(S, D, q0, fpm=0, start=None):
    from test_bigfield import _engine

    eng = _engine(S, q0.ravel(), D=D, halo=20, fixed_point_mode=fpm)
    if start is not None:
        eng.strips[0].set_stars(start)
    return eng


def _chains(S, D, q0, K, fpm=0, start=None):
    eng = _one(S, D, q0, fpm)
    eng.strips[0].set_chains(K)
    eng.strips[0].set_stars(q0 if start is None else start)
    return eng


def _philox_draws(S, n, niter, c, seed=RUN["seed"]):
    from hmc_stellar_toy_model_b200 import RHMCContext
    from test_bigfield import _consts

    with RHMCContext(n_fields=1, num_rows=16, num_cols=16, max_stars=n, **_consts(S)) as ctx:
        normals, lnu = ctx.philox_draws(seed, niter, field_id_base=c)
    return normals[0].reshape(niter + 1, n, 3), lnu[0]


def _assert_chain(outk, engk, c, out1, eng1, n):
    for k in ("E_chain", "V_chain", "T_chain", "A_chain"):
        assert np.array_equal(outk[k][c], out1[k]), (c, k)
    assert outk["n_accepted"][c] == out1["n_accepted"] and outk["accept_rate"][c] == out1["accept_rate"]
    for w in ("q_chain", "p_chain"):
        if w in out1:
            assert np.array_equal(outk[w][c], out1[w]), (c, w)
    for a, b in zip(engk.stars(n), eng1.stars(n)):
        assert np.array_equal(a[c], b), c


@pytest.mark.gpu
@pytest.mark.parametrize("field", ["philox", "c3"])
@pytest.mark.parametrize("K", [2, 5])
@pytest.mark.parametrize("fpm", [0, 1])
@pytest.mark.parametrize("mode", ["graph", "eager"])
def test_chain_zero_is_the_one_chain_engine(field, K, fpm, mode, monkeypatch):
    """Chain 0 of K chains: E / V / T / A rows, final q / p / grad and recorded q / p rows equal a one-chain tile-path run
    from the same start with the same seed, bit for bit (graph replay, and eager with a g_ff2 schedule)."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    S, D, q0 = _field(field)
    n, niter = len(q0), 6
    kw = dict(RUN, want=("q", "p"))
    if mode == "eager":
        kw.update(use_graph=False, schedule_g_ff2=[4.0, 3.5, 3.0, 4.0])
    engk = _chains(S, D, q0, K, fpm)
    outk = engk.run(niter, **kw)
    assert (engk.replayed_launches > 0) == (mode == "graph")
    assert outk["E_chain"].shape == (K, niter + 1) and outk["q_chain"].shape == (K, niter + 1, n, 3)
    eng1 = _one(S, D, q0, fpm)
    out1 = eng1.run(niter, **kw)
    assert 0 < out1["A_chain"].sum()
    _assert_chain(outk, engk, 0, out1, eng1, n)


@pytest.mark.gpu
@pytest.mark.parametrize("fpm", [0, 1])
def test_chain_c_is_philox_field_c(fpm, monkeypatch):
    """Chain c of K = 4 equals a one-chain run with the normals / log u of RHMCContext.philox_draws(field_id_base=c)."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    S, D, q0 = _field("philox")
    n, niter, K = len(q0), 7, 4
    engk = _chains(S, D, q0, K, fpm)
    outk = engk.run(niter, **RUN, want=("q", "p"))
    for c in range(1, K):
        normals, lnu = _philox_draws(S, n, niter, c)
        eng1 = _one(S, D, q0, fpm)
        out1 = eng1.run(niter, **RUN, want=("q", "p"), normals=normals, lnu=lnu)
        _assert_chain(outk, engk, c, out1, eng1, n)
    assert not np.array_equal(outk["E_chain"][0], outk["E_chain"][1])


def _perturbed_starts(q0, K, seed=5):
    rng = np.random.RandomState(seed)
    return np.stack([q0 * np.array([1.0 + 0.02 * rng.normal(), 1.0, 1.0]) + np.concatenate(
        [np.zeros((len(q0), 1)), rng.uniform(-8, 8, (len(q0), 2)) * (rng.uniform(size=(len(q0), 1)) < 0.1)], axis=1)
        for _ in range(K)])


@pytest.mark.gpu
def test_chains_from_different_starts(monkeypatch):
    """K = 3 chains from perturbed catalogues whose tile orders differ: each equals its own one-chain replay (Philox field c),
    and the recorded rows are in global-id order."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    S, D, q0 = _field("philox")
    n, niter, K = len(q0), 7, 3
    starts = np.clip(_perturbed_starts(q0, K), [0, 1, 1], [np.inf, 254, 94])
    engk = _chains(S, D, q0, K, start=starts)
    ids = engk.strips[0].ids
    assert ids.shape == (K, n) and not np.array_equal(ids[0], ids[1])
    outk = engk.run(niter, **RUN, want=("q",))
    for c in range(K):
        assert np.array_equal(outk["q_chain"][c, 0], starts[c])   # row 0: the start, in global-id order
        normals, lnu = _philox_draws(S, n, niter, c)
        eng1 = _one(S, D, q0, start=starts[c])
        out1 = eng1.run(niter, **RUN, want=("q",), normals=normals, lnu=lnu)
        _assert_chain(outk, engk, c, out1, eng1, n)


@pytest.mark.gpu
def test_chain_results_do_not_depend_on_k(monkeypatch):
    """Chain c of K = 3 equals chain c of K = 7 bit for bit (different starts per chain)."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    S, D, q0 = _field("philox")
    n, niter = len(q0), 7
    starts = np.clip(_perturbed_starts(q0, 7, seed=8), [0, 1, 1], [np.inf, 254, 94])
    e3 = _chains(S, D, q0, 3, start=starts[:3])
    o3 = e3.run(niter, **RUN, want=("q", "p"))
    e7 = _chains(S, D, q0, 7, start=starts)
    o7 = e7.run(niter, **RUN, want=("q", "p"))
    s3, s7 = e3.stars(n), e7.stars(n)
    for k in ("E_chain", "V_chain", "T_chain", "A_chain", "q_chain", "p_chain"):
        assert np.array_equal(o7[k][:3], o3[k]), k
    for a, b in zip(s7, s3):
        assert np.array_equal(a[:3], b)


@pytest.mark.gpu
@pytest.mark.parametrize("fpm", [0, 1])
def test_k_chains_enqueue_one_launch_sequence(fpm, monkeypatch):
    """A K = 4 iteration enqueues exactly the kernels of a one-chain tile-path iteration: graph nodes and launch_count."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    S, D, q0 = _field("philox")
    counts = {}
    for K in (1, 4):
        eng = _chains(S, D, q0, K, fpm) if K > 1 else _one(S, D, q0, fpm)
        eng.run(4, **RUN, want=("q",))
        s = eng.strips[0]
        l0 = s.launch_count
        eng.run(4, **RUN, want=("q",), use_graph=False)
        counts[K] = (eng._graph_nodes, s.launch_count - l0)
    assert counts[4] == counts[1] and counts[1][0] > 0


@pytest.mark.gpu
def test_chain_convergence_stats_on_the_device(monkeypatch):
    """One K = 4 engine with recorded q: bf.convergence_stats(engine) equals bf.convergence_stats of the four one-chain
    replays bit for bit, and oracle.convergence_stats of the downloaded rows (R to 1e-12, n_eff to 1e-9)."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    S, D, q0 = _field("philox")
    n, niter, K = len(q0), 59, 4
    starts = np.clip(_perturbed_starts(q0, K, seed=2), [0, 1, 1], [np.inf, 254, 94])
    engk = _chains(S, D, q0, K, start=starts)
    outk = engk.run(niter, **RUN, want=("q",))
    singles = []
    for c in range(K):
        normals, lnu = _philox_draws(S, n, niter, c)
        e = _one(S, D, q0, start=starts[c])
        e.run(niter, **RUN, want=("q",), normals=normals, lnu=lnu)
        singles.append(e)
    chains = outk["q_chain"].reshape(K, niter + 1, -1)
    for thin, warm in ((1, 0), (2, 10), (5, 3)):
        R, n_eff = bf.convergence_stats(engk, thin_rate=thin, warm_up_num=warm)
        R1, n1 = bf.convergence_stats(singles, thin_rate=thin, warm_up_num=warm)
        assert np.array_equal(R, R1) and np.array_equal(n_eff, n1), (thin, warm)
        Ro, no = so.convergence_stats(chains, thin_rate=thin, warm_up_num=warm)
        assert R.shape == (n, 3) and np.all(np.isfinite(R))
        assert relerr(R.ravel(), Ro) < 1e-12 and relerr(n_eff.ravel(), no) < 1e-9, (thin, warm)
    assert np.array_equal(bf.convergence_stats([engk])[0], bf.convergence_stats(engk)[0])


@pytest.mark.gpu
def test_chain_refusals_and_reset(monkeypatch):
    """What K > 1 does not cover raises with its message; set_chains(3) then set_chains(1) on a field below 2 tiles per SM
    returns the engine to the scatter path: its launch sequence and accept decisions equal an untouched engine's exactly, its
    E / V / T rows to 1e-12 and q rows and final stars to 1e-9 (the scatter path adds the model image with FP64 atomics, so
    two untouched engines also differ in the last bits)."""
    from hmc_stellar_toy_model_b200._capi import SrhmcError
    from test_bigfield import _engine

    monkeypatch.delenv("SRHMC_BIG_PATH", raising=False)
    monkeypatch.delenv("SRHMC_BIG_STAR", raising=False)
    S, D, q0 = _field("philox")   # 4 x 2 tiles: the scatter path at creation
    n = len(q0)
    ref = _engine(S, q0.ravel(), D=D, halo=20)
    l0 = ref.strips[0].launch_count
    r = ref.run(5, **RUN, want=("q",), use_graph=False)
    ref_launches = ref.strips[0].launch_count - l0
    eng = _engine(S, q0.ravel(), D=D, halo=20)
    s = eng.strips[0]
    for k in (0, 65):
        with pytest.raises(SrhmcError, match="a context holds 1..64"):
            s.set_chains(k)
    s.set_chains(3)
    s.set_stars(q0)
    with pytest.raises(ValueError, match="injected normals / lnu"):
        eng.run(3, **RUN, lnu=np.zeros(4))
    for call, name in ((lambda: eng.run_rj(3, 5, 2e-2, P_move=[1, 0, 0], fmin=1.0, fmax=2.0), "run_rj"),
                       (lambda: eng.steps(2, 2e-2), "steps"), (lambda: eng.evaluate(), "evaluate"),
                       (lambda: eng.energies(), "energies")):
        with pytest.raises(ValueError, match=name):
            call()
    lib, h = s._lib, s._h
    for rc_call, msg in ((lambda: lib.srhmc_big_set_precision(h, 32), "precision 32 needs one chain"),
                         (lambda: lib.srhmc_big_set_momenta(h, bf._capi.dptr(np.zeros((n, 3)))), "holds 3 chains"),
                         (lambda: lib.srhmc_big_read_samples(h, 0, 0, None, None), "srhmc_big_read_chain_samples"),
                         (lambda: lib.srhmc_big_read_chains(h, 1, None, None, None, None, None, None), "srhmc_big_read_chain_rows"),
                         (lambda: lib.srhmc_big_set_draws(h, None, None, 1), "Philox")):
        with pytest.raises(SrhmcError, match=msg):
            bf.check(rc_call())
    with pytest.raises(SrhmcError, match="srhmc_big_set_chain_stars"):
        bf.BigFieldStrip.set_table(s, q0)
    # mismatched id sets: chain 1 without its last star
    ids = np.arange(n - 1, dtype=np.int64)
    bf.check(lib.srhmc_big_set_chain_stars(h, 1, bf._capi.dptr(np.ascontiguousarray(q0[:-1])),
                                           ids.ctypes.data_as(bf.C.POINTER(bf.C.c_int64)), n - 1))
    with pytest.raises(SrhmcError, match="chain 1 holds other star ids"):
        eng.run(3, **RUN)
    # out of scope at creation: a strip of a tiled field
    with pytest.raises(SrhmcError, match="strip of 2"):
        _engine(S, q0.ravel(), world=2, D=D, halo=20).strips[0].set_chains(2)
    # reset
    s.set_chains(1)
    s.set_stars(q0)
    l0 = s.launch_count
    o = eng.run(5, **RUN, want=("q",), use_graph=False)
    assert s.launch_count - l0 == ref_launches   # the scatter path's launch sequence
    assert np.array_equal(o["A_chain"], r["A_chain"])
    for k in ("E_chain", "V_chain", "T_chain"):
        assert relerr(o[k], r[k]) < 1e-12, k
    assert relerr(o["q_chain"], r["q_chain"]) < 1e-9
    for a, b in zip(eng.stars(n), ref.stars(n)):
        assert relerr(a, b) < 1e-9
