"""Sample rows of the large-field engine (srhmc_big_set_recording / srhmc_big_read_samples, BigFieldRHMC.run(want=...)) and
the convergence statistics over the resident rows of several engines (srhmc_big_convergence_stats, bf.convergence_stats):
host helpers on CPU; on the GPU the reference's own recorded chains, exact consistency of the rows with the engine's state,
tiling, and the statistics against the oracle."""
import ctypes as C

import numpy as np
import pytest

import stellar_oracle as so
from helpers import first_divergence, golden, relerr, setup_from
from hmc_stellar_toy_model_b200 import bigfield as bf


# ------------------------------------------------------------------ CPU: host helpers
def test_record_want_and_rows():
    assert bf.record_want(()) == () and bf.record_want("q") == ("q",)
    assert bf.record_want(["p", "q"]) == ("q", "p") and bf.record_want(("p",)) == ("p",)
    with pytest.raises(ValueError):
        bf.record_want(("q", "grad"))
    assert [bf.record_rows(L, 1) for L in (1, 7)] == [1, 7]
    assert [bf.record_rows(L, 3) for L in (1, 3, 4, 6, 7)] == [1, 1, 2, 2, 3]
    # row r is iteration r * stride: the rows of stride k are range(L)[::k]
    for L in range(1, 12):
        for k in range(1, 5):
            assert bf.record_rows(L, k) == len(range(L)[::k])
    with pytest.raises(ValueError):
        bf.record_rows(5, 0)


def test_slot_order_is_ascending_id():
    """Rows are stored in ascending global-id order whatever the storage (tile) order of the strip: two strips that own the
    same ids in different storage orders share one column layout."""
    rng = np.random.RandomState(4)
    ids = rng.permutation(40)[:25].astype(np.int64)
    other = rng.permutation(ids)
    assert np.array_equal(bf.slot_ids(ids), np.sort(ids)) and np.array_equal(bf.slot_ids(ids), bf.slot_ids(other))
    # the slot the device assigns a stored star is the rank of its id among the strip's ids: column slot[k] of a row holds
    # stored star k, whose global id is slot_ids(ids)[slot[k]]
    slot = np.argsort(np.argsort(ids, kind="stable"), kind="stable")
    assert np.array_equal(bf.slot_ids(ids)[slot], ids)


# ------------------------------------------------------------------ GPU
def _philox_field():
    """The 700-star field of test_bigfield.py::test_bigfield_philox_chain_tiled_equals_untiled."""
    S = so.Setup(num_rows=256, num_cols=96, g_xx=0.05, g_ff=4.0, g_ff2=4.0, use_prior=True, alpha=2.0, V_prior_const=1.0)
    rng = np.random.RandomState(3)
    n = 700
    fl = S.mag2flux_converter(rng.uniform(15.5, 20.0, n))
    q = np.stack([fl, rng.uniform(1, 255, n), rng.uniform(1, 95, n)], axis=1)
    lam = S.B_count * np.ones((256, 96))
    sig = S.PSF_FWHM_pix / 2.354
    ci, cj = np.arange(0.5, 256), np.arange(0.5, 96)
    ex = np.exp(-((ci[None] - q[:, 1:2]) ** 2) / (2 * sig ** 2))
    ey = np.exp(-((cj[None] - q[:, 2:3]) ** 2) / (2 * sig ** 2)) / (2 * np.pi * sig ** 2)
    lam += np.einsum("k,ki,kj->ij", q[:, 0], ex, ey)
    D = rng.poisson(lam).astype(float)
    q0 = q * np.array([1.03, 1.0, 1.0]) + np.array([0.0, 0.05, -0.05])
    return S, D, q0


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["scatter", "tile", "star"])
def test_bigfield_samples_match_reference_chain(path, monkeypatch):
    """chain_multi100 (100 stars, prior, g_ff2 schedule: eager path) with the reference's draws injected: the recorded q / p
    rows against the reference's own q_chain / p_chain at the tolerances the CTA kernel meets (test_gpu_parity.py::
    test_run_rhmc_crowded_chain): 1e-6 over the chain, 1e-10 up to the first accepted iteration; row 0 is the start state."""
    from test_bigfield import _engine, _set_path

    _set_path(monkeypatch, path)
    g = golden("chain_multi100")
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    niter, nsteps, dt = int(g["niter"]), int(g["nsteps"]), float(g["dt"])
    eng = _engine(S, q0, halo=13)
    out = eng.run(niter, nsteps, dt, f_pos=True, g_ff2=S.g_ff2, normals=g["normals"].reshape(niter + 1, -1, 3),
                  lnu=g["lnu"], schedule_g_ff2=g["schedule_g_ff2"], want=("q", "p"))
    L = niter + 1
    assert out["q_chain"].shape == (L, 100, 3) and out["p_chain"].shape == (L, 100, 3)
    assert np.array_equal(out["A_chain"].astype(bool), g["A_chain"])
    assert np.array_equal(out["q_chain"][0].ravel(), q0)
    q, p = out["q_chain"].reshape(L, -1), out["p_chain"].reshape(L, -1)
    assert first_divergence(q, g["q_chain"], 1e-6) == -1
    assert first_divergence(p, g["p_chain"], 1e-6) == -1
    first_accept = int(np.argmax(g["A_chain"])) + 1
    assert first_divergence(q[: first_accept + 1], g["q_chain"][: first_accept + 1], 1e-10) == -1
    assert first_divergence(p[: first_accept + 1], g["p_chain"][: first_accept + 1], 1e-10) == -1


def _philox_run(niter, lnu, start=None, **kw):
    from test_bigfield import _engine

    S, D, q0 = _philox_field()
    eng = _engine(S, (q0 if start is None else start).ravel(), world=kw.pop("world", 1), D=D, halo=20)
    out = eng.run(niter, 5, 2e-2, f_pos=True, g_ff2=4.0, seed=11, lnu=None if lnu is None else lnu[: niter + 1], **kw)
    return eng, out


@pytest.mark.gpu
def test_bigfield_samples_are_the_engine_state(monkeypatch):
    """Tile path, 700-star Philox field, bit for bit: a rejected iteration's next row repeats its row; after a rejected last
    iteration stars() is the last row; stride-k rows are the stride-1 rows [::k]; a graph replay records what the eager run
    records; recording leaves E / V / T / A and the final stars unchanged.  The chain starts where 200 iterations from the
    field's start ended (from the start itself every trajectory still lowers the energy); odd iterations draw log u = +inf
    (accepted only when dE < 0), even ones -inf (always accepted), so the chain holds both outcomes."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    burn, _ = _philox_run(199, None)
    start = burn.stars(700)[0]
    niter = 31
    lnu = np.where(np.arange(niter + 1) % 2 == 1, np.inf, -np.inf)
    run = lambda it, **kw: _philox_run(it, lnu, start=start, **kw)   # noqa: E731
    eng, a = run(niter, want=("q", "p"))
    assert eng.replayed_launches > 0   # the captured-graph path
    A = a["A_chain"].astype(bool)
    rejected = np.nonzero(~A[:-1])[0]
    assert A.any() and len(rejected) > 0
    for l in rejected:
        assert np.array_equal(a["q_chain"][l + 1], a["q_chain"][l]), l
    for l in np.nonzero(A[:-1])[0]:
        assert not np.array_equal(a["q_chain"][l + 1], a["q_chain"][l]), l
    # the run that ends with the first rejected iteration: its final stars are its last row
    l_rej = int(rejected[0])
    eng_t, t = run(l_rej, want=("q",))
    assert not t["A_chain"][-1]
    assert np.array_equal(eng_t.stars(700)[0], t["q_chain"][-1])
    assert np.array_equal(t["q_chain"], a["q_chain"][: l_rej + 1])
    # stride 3
    _, s3 = run(niter, want=("q", "p"), chain_stride=3)
    assert s3["q_chain"].shape[0] == bf.record_rows(niter + 1, 3)
    assert np.array_equal(s3["q_chain"], a["q_chain"][::3]) and np.array_equal(s3["p_chain"], a["p_chain"][::3])
    # eager enqueueing against the graph replay
    eng_e, e = run(niter, want=("q", "p"), use_graph=False)
    assert eng_e.replayed_launches == 0
    for k in ("q_chain", "p_chain", "E_chain", "V_chain", "T_chain", "A_chain"):
        assert np.array_equal(e[k], a[k]), k
    # recording off
    eng_o, o = run(niter)
    assert "q_chain" not in o and "p_chain" not in o
    for k in ("E_chain", "V_chain", "T_chain", "A_chain"):
        assert np.array_equal(o[k], a[k]), k
    assert np.array_equal(eng_o.stars(700)[0], eng.stars(700)[0])


@pytest.mark.gpu
def test_bigfield_graph_cache_follows_the_recording_setup(monkeypatch):
    """One engine, successive runs: a graph captured with recording is not replayed without it and the reverse, and after an
    eager run that freed or re-allocated the rows, a graph run with the earlier set-up records into the current rows."""
    from test_bigfield import _engine, _set_path

    _set_path(monkeypatch, "tile")
    S, D, q0 = _philox_field()
    ref = _engine(S, q0.ravel(), D=D, halo=20)
    r = ref.run(7, 5, 2e-2, f_pos=True, g_ff2=4.0, seed=11, want=("q",))
    r_stars = ref.stars(700)[0]
    eng = _engine(S, q0.ravel(), D=D, halo=20)
    for mode, want in (("graph", ("q",)), ("eager", ()), ("graph", ("q",)), ("eager", ("q", "p")), ("graph", ()),
                       ("graph", ("q",)), ("eager", ("p",)), ("graph", ("q",))):
        for s in eng.strips:
            s.set_stars(q0)
        if mode == "eager":
            eng.run(3, 5, 2e-2, f_pos=True, g_ff2=4.0, seed=5, use_graph=False, want=want)
            continue
        out = eng.run(7, 5, 2e-2, f_pos=True, g_ff2=4.0, seed=11, want=want)
        assert eng.replayed_launches > 0
        for k in ("A_chain", "E_chain", "V_chain", "T_chain"):
            assert np.array_equal(out[k], r[k]), (want, k)
        assert np.array_equal(eng.stars(700)[0], r_stars)
        assert ("q_chain" in out) == ("q" in want)
        if "q" in want:
            assert np.array_equal(out["q_chain"], r["q_chain"])


@pytest.mark.gpu
def test_bigfield_samples_tiled_equal_untiled(monkeypatch):
    """4 strips through LocalComm record the untiled chain: q rows to 1e-9, accept decisions exact, every star covered."""
    from test_bigfield import _set_path

    _set_path(monkeypatch, "tile")
    _, a = _philox_run(8, None, want=("q",))
    _, b = _philox_run(8, None, want=("q",), world=4)
    assert np.array_equal(a["A_chain"], b["A_chain"]) and 0 < a["A_chain"].sum()
    assert not np.any(np.isnan(b["q_chain"]))
    assert relerr(b["q_chain"], a["q_chain"]) < 1e-9


def _stats_engines(world, seeds, starts, niter, S, D):
    from test_bigfield import _engine

    engs = []
    for seed, q0 in zip(seeds, starts):
        eng = _engine(S, q0.ravel(), world=world, D=D, halo=20)
        eng.run(niter, 4, 2e-2, f_pos=True, g_ff2=4.0, seed=seed, want=("q",))
        engs.append(eng)
    return engs


@pytest.mark.gpu
def test_bigfield_convergence_stats_match_oracle(monkeypatch):
    """K = 3 untiled chains (different seeds and starts, 240 rows) and K = 2 chains tiled in 2 strips (same start, different
    seeds): bf.convergence_stats on the resident rows equals oracle.convergence_stats of the downloaded chains, R to 1e-12 and
    n_eff to 1e-9, for several (thin, warm-up) pairs."""
    monkeypatch.setenv("SRHMC_BIG_PATH", "scatter")
    from test_bigfield import _synthetic_field

    S, D, q0 = _synthetic_field(256, 96, 150, 23)
    rng = np.random.RandomState(9)
    starts3 = [q0 * np.array([1.0 + 0.02 * rng.normal(), 1.0, 1.0]) + np.array([0.0, 0.1, -0.1]) * rng.normal(size=3)
               for _ in range(3)]
    cases = [(1, _stats_engines(1, (1, 2, 3), starts3, 239, S, D)),
             (2, _stats_engines(2, (4, 5), (q0, q0), 239, S, D))]
    for world, engs in cases:
        rows = 240
        for e in engs:
            assert len(e.strips) == world and e.strips[0].n_global == 150
        chains = np.stack([e._samples("q", rows).reshape(rows, -1) for e in engs])
        assert not np.any(np.isnan(chains))
        for thin, warm in ((1, 0), (2, 10), (5, 3)):
            R, n_eff = bf.convergence_stats(engs, thin_rate=thin, warm_up_num=warm)
            Ro, no = so.convergence_stats(chains, thin_rate=thin, warm_up_num=warm)
            assert R.shape == (150, 3) and np.all(np.isfinite(R)) and np.all(np.isfinite(n_eff))
            assert relerr(R.ravel(), Ro) < 1e-12, (world, thin, warm)
            assert relerr(n_eff.ravel(), no) < 1e-9, (world, thin, warm)


@pytest.mark.gpu
def test_bigfield_convergence_stats_rejections(monkeypatch):
    """srhmc_big_convergence_stats refuses one chain, chains that own different stars, hold different row counts or strides,
    or recorded no q (the device check needs a second GPU and is not exercised here)."""
    monkeypatch.setenv("SRHMC_BIG_PATH", "scatter")
    from hmc_stellar_toy_model_b200._capi import SrhmcError
    from test_bigfield import _engine, _synthetic_field

    S, D, q0 = _synthetic_field(256, 96, 150, 23)

    def eng_of(q, niter, want=("q",), stride=1):
        e = _engine(S, q.ravel(), D=D, halo=20)
        e.run(niter, 2, 2e-2, f_pos=True, g_ff2=4.0, seed=niter, want=want, chain_stride=stride)
        return e

    base = eng_of(q0, 19)
    lib = bf._capi.load_library()

    def stats(engs):
        h = (C.c_void_p * len(engs))(*[e.strips[0]._h.value for e in engs])
        r, ne = np.empty(450), np.empty(450)
        bf.check(lib.srhmc_big_convergence_stats(h, len(engs), 1, 0, bf._capi.dptr(r), bf._capi.dptr(ne)))
        return r

    assert np.all(np.isfinite(stats([base, eng_of(q0, 19)])))
    for others, msg in (([], "at least two chains"),
                        ([eng_of(q0[:120], 19)], "same stars"),
                        ([eng_of(q0, 29)], "rows at stride"),
                        ([eng_of(q0, 39, stride=2)], "rows at stride"),
                        ([eng_of(q0, 19, want=("p",))], "no recorded q")):
        with pytest.raises(SrhmcError, match=msg):
            stats([base] + others)
    with pytest.raises(SrhmcError, match="fewer than two samples"):
        bf.convergence_stats([base, eng_of(q0, 19)], thin_rate=10, warm_up_num=0)
    with pytest.raises(ValueError):
        bf.convergence_stats([base])
