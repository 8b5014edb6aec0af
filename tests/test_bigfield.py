"""Large-field engine (csrc/big_field.cu, bigfield.py): host geometry on CPU (incl. a 2-rank gloo exchange of the
boundary lists), and on the GPU the untiled engine against the CTA-resident kernel / the oracle, and a tiling run on
one device through LocalComm against the untiled engine."""
import os
import socket
import sys

import numpy as np
import pytest

import stellar_oracle as so
from helpers import golden, relerr, setup_from
from hmc_stellar_toy_model_b200 import bigfield as bf


# ------------------------------------------------------------------ CPU: geometry and host logic
def test_strip_geometry():
    for rows, world in ((64, 1), (64, 2), (8192, 8), (1000, 3)):
        b = bf.strip_bounds(rows, world)
        assert b[0][0] == 0 and b[-1][1] == rows and all(b[i][1] == b[i + 1][0] for i in range(world - 1))
        x = np.random.RandomState(0).uniform(-2, rows + 2, 500)
        own = bf.owner_of(x, rows, world)
        for r, (lo, hi) in enumerate(b):
            inside = (x >= lo) & (x < hi)
            assert np.all(own[inside] == r)
        assert np.all(own[x < 0] == 0) and np.all(own[x >= rows] == world - 1)
    assert bf.data_window(100, 33, 66, 20) == (13, 73)
    assert bf.data_window(100, 0, 33, 20) == (0, 53)
    with pytest.raises(ValueError):
        bf.strip_bounds(3, 8)


def test_tile_order_is_a_stable_row_major_tile_sort():
    """set_stars stores a strip's stars in 64x64-tile order (locality for the tile lists and footprint sums)."""
    rng = np.random.RandomState(1)
    q = np.stack([rng.uniform(1, 2, 500), rng.uniform(-3, 400, 500), rng.uniform(-2, 700, 500)], axis=1)
    order = bf.tile_order(q, 700)
    assert sorted(order.tolist()) == list(range(500))
    key = (np.floor(q[order, 1]) // 64) * (700 // 64 + 1) + np.floor(q[order, 2]) // 64
    assert np.all(np.diff(key) >= 0)
    same = np.diff(key) == 0
    assert np.all(np.diff(order)[same] > 0)          # stable inside a tile
    assert bf.tile_order(q[:1], 700).tolist() == [0] and len(bf.tile_order(q[:0], 700)) == 0


def test_ghost_lists_cover_every_star_that_can_touch_a_neighbour():
    rows, world, rad, halo = 256, 4, 12, 24
    rng = np.random.RandomState(1)
    x = rng.uniform(0, rows, 4000)
    own = bf.owner_of(x, rows, world)
    bounds = bf.strip_bounds(rows, world)
    reach = halo + rad + 1
    for r, (lo, hi) in enumerate(bounds):
        row0, nrows = bf.data_window(rows, lo, hi, halo)
        # every foreign star whose patch touches my data rows must be in a neighbour's list for me
        touches = (np.floor(x) + rad >= row0) & (np.floor(x) - rad <= row0 + nrows - 1) & (own != r)
        got = np.zeros_like(touches)
        for nb in (r - 1, r + 1):
            if 0 <= nb < world:
                nlo, nhi = bounds[nb]
                to_lo, to_hi = bf.ghost_mask(x, nlo, nhi, reach, nb, world)
                sel = (own == nb) & (to_hi if nb < r else to_lo)
                got |= sel
        assert np.all(got[touches]), r


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rows, rad, halo, cap = 128, 12, 24, 160
        rng = np.random.RandomState(7)
        stars = np.stack([rng.uniform(100, 1000, 300), rng.uniform(0, rows, 300), rng.uniform(0, 64, 300)], axis=1)
        mine = stars[bf.owner_of(stars[:, 1], rows, world) == rank]
        lo, hi = bf.strip_bounds(rows, world)[rank]
        to_lo, to_hi = bf.ghost_mask(mine[:, 1], lo, hi, halo + rad + 1, rank, world)
        # the device PACK layout: [2][1 + 3 cap], count first
        send = np.zeros((2, 1 + 3 * cap))
        for i, m in enumerate((to_lo, to_hi)):
            sel = mine[m][:cap]
            send[i, 0] = len(sel)
            send[i, 1:1 + 3 * len(sel)] = sel.ravel()
        recv = torch.zeros(world * send.size, dtype=torch.float64)
        dist.all_gather_into_tensor(recv, torch.from_numpy(send.ravel().copy()))
        recv = recv.numpy().reshape(world, 2, 1 + 3 * cap)
        # what the EVAL phase reads: list 1 of rank-1 and list 0 of rank+1
        ghosts = []
        if rank > 0:
            n = int(recv[rank - 1, 1, 0])
            ghosts.append(recv[rank - 1, 1, 1:1 + 3 * n].reshape(n, 3))
        if rank < world - 1:
            n = int(recv[rank + 1, 0, 0])
            ghosts.append(recv[rank + 1, 0, 1:1 + 3 * n].reshape(n, 3))
        ghosts = np.concatenate(ghosts) if ghosts else np.zeros((0, 3))
        row0, nrows = bf.data_window(rows, lo, hi, halo)
        foreign = stars[bf.owner_of(stars[:, 1], rows, world) != rank]
        need = foreign[(np.floor(foreign[:, 1]) + rad >= row0) & (np.floor(foreign[:, 1]) - rad <= row0 + nrows - 1)]
        have = {tuple(g) for g in ghosts}
        ok = all(tuple(s) in have for s in need)
        # sum-reduce of the energy partials and max-reduce of the counters
        sc = torch.tensor([1.0 + rank, 2.0, 0.0, 0.5 * rank], dtype=torch.float64)
        dist.all_reduce(sc)
        cnt = torch.tensor([3 + rank, 7 - rank], dtype=torch.int32)
        dist.all_reduce(cnt, op=dist.ReduceOp.MAX)
        q.put((rank, ok, len(need), sc.tolist(), cnt.tolist()))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_boundary_exchange():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, ok, n_need, sc, cnt in res:
        assert ok and n_need > 0
        assert sc == [3.0, 4.0, 0.0, 0.5] and cnt == [4, 7]


# ------------------------------------------------------------------ GPU
def _consts(S):
    return dict(psf_fwhm_pix=S.PSF_FWHM_pix, B_count=S.B_count, f_lim=S.f_lim, f_low=S.mag2flux_converter(S.mB + 2),
                g0=S.g0, g1=S.g1, g2=S.g2, g_xx=S.g_xx, g_ff=S.g_ff, use_prior=S.use_prior, alpha=S.alpha,
                V_prior_const=S.V_prior_const if S.V_prior_const is not None else 0.0)


def _engine(S, q, world=1, rad=12, halo=20, D=None, fixed_point_mode=0):
    import torch

    # one explicit side stream for the engine AND the LocalComm tensor ops (CUDA-graph capture needs a non-default one)
    global _STREAM
    if _STREAM is None:
        _STREAM = torch.cuda.Stream()
    torch.cuda.set_stream(_STREAM)
    stream = _STREAM.cuda_stream
    strips = []
    for r in range(world):
        s = bf.BigFieldStrip(rows=S.num_rows, cols=S.num_cols, rank=r, world=world, device=0, max_stars=q.size // 3,
                             max_ghosts=q.size // 3, patch_radius=rad, halo=halo, **_consts(S))
        s.set_stream(stream)
        s.set_data(S.D if D is None else D)
        s.set_stars(q.reshape(-1, 3))
        strips.append(s)
    return bf.BigFieldRHMC(strips, bf.LocalComm() if world > 1 else bf.NoComm(), fixed_point_mode=fixed_point_mode)


_STREAM = None


def _grad_close(a, b, tol):
    a, b = np.asarray(a).reshape(-1, 3), np.asarray(b).reshape(-1, 3)
    scale = np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b), axis=0, keepdims=True))
    return float(np.max(np.abs(a - b) / scale)) < tol


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("path", ["scatter", "tile"])
def test_bigfield_eval_matches_reference_values(world, path, monkeypatch):
    """204 stars on 64x64 (golden from the reference): V and dV/dq through the scatter / pixel / gather kernels,
    untiled and tiled into 2 strips on one device."""
    _set_path(monkeypatch, path)  # EVAL through the star-parallel kernels, the fused tile kernel or the star-centric kernel
    g = golden("field_eval_204")
    S = setup_from(g)
    eng = _engine(S, g["q"], world=world, halo=14)
    eng.evaluate(want_V=True, g_ff2=S.g_ff2)
    V, _ = eng.energies()
    _, _, grad = eng.stars(204)
    # reference dVdq includes the prior term alpha/f (sampler_RHMC.py:408-409); the engine keeps the pixel part
    gref = g["dVdq"].reshape(-1, 3).copy()
    gref[:, 0] -= S.alpha / g["q"].reshape(-1, 3)[:, 0]
    assert relerr(V, g["V"]) < 1e-10
    assert _grad_close(grad, gref, 1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("path", ["scatter", "tile", "star"])
def test_bigfield_steps_match_cta_kernel(world, path, monkeypatch):
    """Three leapfrog steps of the 204-star field: same q, p as the CTA-resident kernel (which is parity-checked
    against the reference), including the field-wide stop rule of the fixed-point loops via the two-phase scheme."""
    _set_path(monkeypatch, path)  # EVAL through the star-parallel kernels, the fused tile kernel or the star-centric kernel
    from test_gpu_parity import make_ctx

    g = golden("field_eval_204")
    S = setup_from(g)
    with make_ctx(S, max_stars=204, patch_radius=12) as ctx:
        ctx.set_data(S.D)
        q_ref, p_ref = ctx.step(g["q"][None], g["p"][None], 3, float(g["dt"]), g_ff2=S.g_ff2)
    eng = _engine(S, g["q"], world=world, halo=14)
    for s in eng.strips:
        s.set_momenta(g["p"].reshape(-1, 3)[s.ids])
    eng.steps(3, float(g["dt"]), g_ff2=S.g_ff2)
    q, p, _ = eng.stars(204)
    assert relerr(q.ravel(), q_ref[0]) < 1e-10
    assert _grad_close(p, p_ref[0], 1e-8)
    # and the first step against the reference's own recorded step
    eng2 = _engine(S, g["q"], world=world, halo=14)
    for s in eng2.strips:
        s.set_momenta(g["p"].reshape(-1, 3)[s.ids])
    eng2.steps(1, float(g["dt"]), g_ff2=S.g_ff2)
    q1, p1, _ = eng2.stars(204)
    assert relerr(q1.ravel(), g["q1"]) < 1e-10 and _grad_close(p1, g["p1"], 1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1])
@pytest.mark.parametrize("path", ["scatter", "tile", "star"])
def test_bigfield_chain_matches_reference_chain(world, path, monkeypatch):
    """RHMC-big-sim3-like chain (100 stars, prior, g_ff2 schedule) recorded from the reference: accept decisions and
    energies from the large-field engine with the reference's draws injected."""
    _set_path(monkeypatch, path)  # EVAL through the star-parallel kernels, the fused tile kernel or the star-centric kernel
    g = golden("chain_multi100")
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    niter, nsteps, dt = int(g["niter"]), int(g["nsteps"]), float(g["dt"])
    eng = _engine(S, q0, world=world, halo=13)  # a 32-row image is too small to tile at r = 12; tiling: next test
    out = eng.run(niter, nsteps, dt, f_pos=True, g_ff2=S.g_ff2, normals=g["normals"].reshape(niter + 1, -1, 3),
                  lnu=g["lnu"], schedule_g_ff2=g["schedule_g_ff2"])
    assert np.array_equal(out["A_chain"].astype(bool), g["A_chain"])
    assert relerr(out["E_chain"], g["E_chain"]) < 1e-9
    assert relerr(out["V_chain"], g["V_chain"]) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["scatter", "tile", "star"])
def test_bigfield_philox_chain_tiled_equals_untiled(path, monkeypatch):
    """Device-RNG chain on a 256x96 field with 700 stars: a 4-strip tiling reproduces the untiled run (same accept
    decisions, energies to 1e-10) because the draws are keyed by global star id."""
    _set_path(monkeypatch, path)  # EVAL through the star-parallel kernels, the fused tile kernel or the star-centric kernel
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
    outs = []
    for world in (1, 4):
        eng = _engine(S, q0.ravel(), world=world, D=D, halo=20)
        outs.append((eng.run(6, 5, 2e-2, f_pos=True, g_ff2=4.0, seed=11), eng.stars(n)[0]))
    a, b = outs
    assert np.array_equal(a[0]["A_chain"], b[0]["A_chain"]) and 0 < a[0]["A_chain"].sum()
    assert relerr(b[0]["E_chain"], a[0]["E_chain"]) < 1e-10
    assert relerr(b[1], a[1]) < 1e-9


def _synthetic_field(rows, cols, n, seed):
    S = so.Setup(num_rows=rows, num_cols=cols, g_xx=0.05, g_ff=4.0, g_ff2=4.0, use_prior=True, alpha=2.0, V_prior_const=1.0)
    rng = np.random.RandomState(seed)
    fl = S.mag2flux_converter(rng.uniform(15.5, 20.0, n))
    q = np.stack([fl, rng.uniform(1, rows - 1, n), rng.uniform(1, cols - 1, n)], axis=1)
    # a few stars hugging the edges and corners: clipped patches, edge tiles
    q[:4, 1:] = [[0.2, 0.3], [rows - 0.4, cols - 0.2], [0.7, cols - 0.6], [rows - 0.3, 0.9]]
    sig = S.PSF_FWHM_pix / 2.354
    ci, cj = np.arange(0.5, rows), np.arange(0.5, cols)
    ex = np.exp(-((ci[None] - q[:, 1:2]) ** 2) / (2 * sig ** 2))
    ey = np.exp(-((cj[None] - q[:, 2:3]) ** 2) / (2 * sig ** 2)) / (2 * np.pi * sig ** 2)
    lam = S.B_count + np.einsum("k,ki,kj->ij", q[:, 0], ex, ey)
    D = rng.poisson(lam).astype(float)
    q0 = q * np.array([1.03, 1.0, 1.0]) + np.array([0.0, 0.05, -0.05])
    return S, D, q0


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,world", [(200, 330, 1), (333, 321, 1), (333, 321, 3)])
def test_bigfield_tile_kernel_equals_star_parallel_kernels(rows, cols, world, monkeypatch):
    """The fused tile evaluation (one CTA per 64x64 tile, D read once) against the scatter / pixel / gather kernels on
    fields whose edges cut tiles (odd column count: unaligned row starts), untiled and as 3 strips: V and dV/dq to
    1e-12, and the tile path bit-identical run to run (no floating-point atomics)."""
    S, D, q0 = _synthetic_field(rows, cols, 900, 5)
    res = {}
    for run, path in (("scatter", "scatter"), ("tile", "tile"), ("tile_rerun", "tile")):
        monkeypatch.setenv("SRHMC_BIG_PATH", path)
        eng = _engine(S, q0.ravel(), world=world, D=D, halo=20)
        eng.evaluate(want_V=True, g_ff2=4.0)
        res[run] = (eng.energies()[0], eng.stars(900)[2])
    assert relerr(res["tile"][0], res["scatter"][0]) < 1e-13
    assert _grad_close(res["tile"][1], res["scatter"][1], 1e-11)
    assert res["tile"][0] == res["tile_rerun"][0] and np.array_equal(res["tile"][1], res["tile_rerun"][1])



def _set_path(monkeypatch, path):
    """"scatter" | "tile" | "star": the star-centric gradient kernel rides on the tile path's lists (SRHMC_BIG_STAR forces it
    on for fields the automatic rule would hand to the tile kernel, e.g. 204 stars in one tile -> the long-list code path)."""
    monkeypatch.setenv("SRHMC_BIG_PATH", "tile" if path == "star" else path)
    monkeypatch.setenv("SRHMC_BIG_STAR", "1" if path == "star" else "0")


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,n,world", [(200, 330, 900, 1), (333, 321, 900, 1), (333, 321, 900, 3), (640, 700, 700, 1),
                                               (640, 700, 700, 2)])
def test_bigfield_star_kernel_equals_tile_kernel(rows, cols, n, world, monkeypatch):
    """Gradient-only evaluation by the star-centric kernel (one warp per star, neighbours from the tile lists) against the
    fused tile kernel: clipped patches at edges and corners, odd column counts, long lists (900 stars on 200x330: ~70 records
    per tile -> the re-scanning path) and short ones (700 stars on 640x700: the register-cached path), untiled and tiled with
    ghosts from the neighbouring strips.  dV/dq to 1e-12 of the per-coordinate scale, and bit-identical run to run."""
    S, D, q0 = _synthetic_field(rows, cols, n, 5)
    res = {}
    for path in ("tile", "star", "star2"):
        _set_path(monkeypatch, path[:4])
        eng = _engine(S, q0.ravel(), world=world, D=D, halo=20)
        eng.evaluate(want_V=False, g_ff2=4.0)
        res[path] = eng.stars(n)[2]
        if path == "star":
            assert all(s.launch_count > 0 for s in eng.strips)
    assert np.all(np.isfinite(res["star"]))
    a, b = res["star"].reshape(-1, 3), res["tile"].reshape(-1, 3)
    err = float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b), axis=0, keepdims=True))))
    assert err < 1e-11, err   # different summation order (whole patch at once vs per-tile partial sums): rounding only
    assert np.array_equal(res["star"], res["star2"])


@pytest.mark.gpu
def test_bigfield_star_kernel_wide_patch(monkeypatch):
    """Patch radius 14 (29 x 29 patches: the 31-row instantiation of the star-centric kernel) against the tile kernel and the
    patch oracle, untiled and as two strips."""
    S, D, q0 = _synthetic_field(640, 700, 500, 8)
    _, gref = so.patch_eval(S, D, q0, 14)
    for world in (1, 2):
        res = {}
        for path in ("tile", "star"):
            _set_path(monkeypatch, path)
            eng = _engine(S, q0.ravel(), world=world, D=D, rad=14, halo=24)
            eng.evaluate(want_V=False, g_ff2=4.0)
            res[path] = eng.stars(500)[2]
        assert _grad_close(res["star"], res["tile"], 1e-11)
        assert _grad_close(res["star"], gref, 1e-10)


@pytest.mark.gpu
def test_bigfield_star_kernel_spot_check_against_patch_oracle(monkeypatch):
    """The star-centric kernel chosen by the automatic rule (very sparse 1600x1600 field: 400 stars on 625 tiles) against the
    NumPy patch oracle, and the same field with 3000 stars (tile kernel by the rule, star kernel forced)."""
    monkeypatch.delenv("SRHMC_BIG_PATH", raising=False)
    for n, force in ((400, None), (3000, "1")):
        if force:
            monkeypatch.setenv("SRHMC_BIG_STAR", force)
        else:
            monkeypatch.delenv("SRHMC_BIG_STAR", raising=False)
        S, D, q0 = _synthetic_field(1600, 1600, n, 21)
        eng = _engine(S, q0.ravel(), D=D, halo=20)
        eng.evaluate(want_V=False, g_ff2=4.0)
        grad = eng.stars(n)[2]
        _, gref = so.patch_eval(S, D, q0, 12)
        assert _grad_close(grad, gref, 1e-10)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("path", ["scatter", "tile"])
def test_bigfield_per_star_stop_rule_matches_cta_kernel(world, path, monkeypatch):
    """fixed_point_mode = 1 (every star's implicit loops stop at its own convergence; one merged per-star kernel between two
    evaluations, no max all-reduce): three leapfrog steps of the 204-star field against the CTA-resident kernel in the same
    mode, untiled and as two strips -- and within the fixed-point tolerance of the reference's stop rule."""
    _set_path(monkeypatch, path)
    from test_gpu_parity import make_ctx

    g = golden("field_eval_204")
    S = setup_from(g)
    ref = {}
    for mode in (0, 1):
        with make_ctx(S, max_stars=204, patch_radius=12, fixed_point_mode=mode) as ctx:
            ctx.set_data(S.D)
            ref[mode] = ctx.step(g["q"][None], g["p"][None], 3, float(g["dt"]), g_ff2=S.g_ff2)
    eng = _engine(S, g["q"], world=world, halo=14, fixed_point_mode=1)
    for s in eng.strips:
        s.set_momenta(g["p"].reshape(-1, 3)[s.ids])
    eng.steps(3, float(g["dt"]), g_ff2=S.g_ff2)
    q, p, _ = eng.stars(204)
    assert relerr(q.ravel(), ref[1][0][0]) < 1e-10
    assert _grad_close(p, ref[1][1][0], 1e-8)
    # the two stop rules differ by what the extra iterations of an already converged star change: far below delta = 1e-6
    assert 0 < relerr(ref[1][0][0], ref[0][0][0]) < 1e-6


@pytest.mark.gpu
def test_bigfield_per_star_chain_tiled_equals_untiled(monkeypatch):
    """Device-RNG chain in the per-star mode: a 4-strip tiling reproduces the untiled run (decisions, energies to 1e-10)."""
    _set_path(monkeypatch, "tile")
    S, D, q0 = _synthetic_field(256, 96, 700, 3)
    outs = []
    for world in (1, 4):
        eng = _engine(S, q0.ravel(), world=world, D=D, halo=20, fixed_point_mode=1)
        outs.append((eng.run(6, 5, 2e-2, f_pos=True, g_ff2=4.0, seed=11), eng.stars(700)[0]))
    a, b = outs
    assert np.array_equal(a[0]["A_chain"], b[0]["A_chain"]) and 0 < a[0]["A_chain"].sum()
    assert relerr(b[0]["E_chain"], a[0]["E_chain"]) < 1e-10
    assert relerr(b[1], a[1]) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_bigfield_sparse_chain_star_kernel_tiled_equals_untiled(mode, monkeypatch):
    """A sparse field (150 stars on 640x700: the automatic rule hands the gradient-only evaluations to the star-centric
    kernel, the potential to the tile kernel) through whole Metropolis iterations, untiled and as three strips with ghosts, in
    both stop-rule modes: same decisions, energies to 1e-10 -- and the same chain as with the tile kernel alone."""
    monkeypatch.setenv("SRHMC_BIG_PATH", "tile")
    S, D, q0 = _synthetic_field(640, 700, 150, 17)
    outs = {}
    for star, world in (("auto", 1), ("auto", 3), ("0", 1)):
        if star == "auto":
            monkeypatch.delenv("SRHMC_BIG_STAR", raising=False)
        else:
            monkeypatch.setenv("SRHMC_BIG_STAR", star)
        eng = _engine(S, q0.ravel(), world=world, D=D, halo=20, fixed_point_mode=mode)
        outs[(star, world)] = (eng.run(6, 5, 2e-2, f_pos=True, g_ff2=4.0, seed=11), eng.stars(150)[0])
    a, b, c = outs[("auto", 1)], outs[("auto", 3)], outs[("0", 1)]
    assert 0 < a[0]["A_chain"].sum()
    for other in (b, c):
        assert np.array_equal(a[0]["A_chain"], other[0]["A_chain"])
        assert relerr(other[0]["E_chain"], a[0]["E_chain"]) < 1e-10
        assert relerr(other[1], a[1]) < 1e-9

@pytest.mark.gpu
def test_bigfield_tile_kernel_dense_list_chunks_and_auto_path(monkeypatch):
    """1600x1600 field (625 tiles > 2 x SM count: the tile path is chosen automatically) and a clump of 300 stars in
    one tile (38 table chunks): V and dV/dq against the NumPy oracle restatement with the same patch truncation."""
    monkeypatch.delenv("SRHMC_BIG_PATH", raising=False)
    S, D, q0 = _synthetic_field(1600, 1600, 2000, 9)
    rng = np.random.RandomState(2)
    q0[100:400, 1] = rng.uniform(700, 760, 300)
    q0[100:400, 2] = rng.uniform(900, 960, 300)
    eng = _engine(S, q0.ravel(), world=1, D=D, halo=20)
    eng.evaluate(want_V=True, g_ff2=4.0)
    V = eng.energies()[0]
    grad = eng.stars(2000)[2]
    Vo, go = so.patch_eval(S, D, q0, rad=12)
    assert relerr(V, Vo) < 1e-12
    assert _grad_close(grad, go, 1e-10)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["scatter", "tile"])
def test_bigfield_peer_exchange_equals_untiled(path, monkeypatch):
    """The library's own collectives (exchange kernels over peer-mapped memory, here between three strips of one process
    on their own streams): a Philox chain of the tiled field reproduces the untiled run -- same accept decisions, energies
    to 1e-10 -- with no collective issued by the caller; and three leapfrog steps agree star by star."""
    monkeypatch.setenv("SRHMC_BIG_PATH", path)
    S, D, q = _synthetic_field(230, 128, 400, 8)
    q = q.ravel()
    n = q.size // 3
    ref = _engine(S, q, world=1, D=D, halo=20)
    a = ref.run(5, 4, 2e-2, f_pos=True, g_ff2=4.0, seed=5)
    qa = ref.stars(n)[0]
    strips = []
    for r in range(3):
        s = bf.BigFieldStrip(rows=S.num_rows, cols=S.num_cols, rank=r, world=3, device=0, max_stars=n, max_ghosts=n,
                             patch_radius=12, halo=20, **_consts(S))
        s.set_data(D)
        s.set_stars(q.reshape(-1, 3))
        strips.append(s)
    eng = bf.BigFieldRHMC(strips, bf.PeerComm(strips))
    b = eng.run(5, 4, 2e-2, f_pos=True, g_ff2=4.0, seed=5)
    assert np.array_equal(a["A_chain"], b["A_chain"]) and 0 < a["A_chain"].sum()
    assert relerr(b["E_chain"], a["E_chain"]) < 1e-10
    assert relerr(eng.stars(n)[0], qa) < 1e-9
    for s in strips:
        s.close()


class _FakeStrip:
    """Stands in for BigFieldStrip in the host-side plumbing test of PeerComm (no device)."""

    def __init__(self, rank, world):
        self.rank, self.world = rank, world
        self.imported = None

    def comm_export(self):
        return bytes([self.rank]) * 64, 0x1000 * (self.rank + 1)

    def comm_import(self, handles=None, raw_ptrs=None):
        self.imported = handles if handles is not None else list(raw_ptrs)


def _peer_handles_worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        s = _FakeStrip(rank, world)
        comm = bf.PeerComm([s], dist)
        q.put((rank, s.imported, comm.in_process))
    finally:
        dist.destroy_process_group()


def test_peer_comm_distributes_handles_in_rank_order():
    """One strip per process: every rank ends up with the world's 64-byte mailbox handles concatenated in rank order (the
    layout srhmc_big_comm_import expects); strips of one process exchange raw pointers in rank order instead."""
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_peer_handles_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    want = bytes([0]) * 64 + bytes([1]) * 64
    for rank, imported, in_process in res:
        assert imported == want and not in_process
    strips = [_FakeStrip(r, 3) for r in (2, 0, 1)]
    comm = bf.PeerComm(strips)
    assert comm.in_process and all(s.imported == [0x1000, 0x2000, 0x3000] for s in strips)


@pytest.mark.gpu
def test_bigfield_full_size_spot_check_against_patch_oracle():
    """BASELINE configs[4] at full size (8192 x 8192, 1e5 stars, device mock data): the pixel gradients of 200 random stars
    against the NumPy patch-limited restatement evaluated on an 81 x 81 crop around each star (every star whose patch can
    overlap the star's patch has its centre inside the crop); stars next to the image edges are always among them."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_for_bigfield", os.path.join(os.path.dirname(os.path.dirname(
        os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(bench)
    finally:
        sys.argv = argv
    rows = cols = 8192
    n = 100000
    t = bench.c5_truth(rows, cols, n, 77)
    c = t["consts"]
    S = so.Setup(num_rows=rows, num_cols=cols, g_xx=c["g_xx"], g_ff=c["g_ff"], g_ff2=4.0, use_prior=True, alpha=c["alpha"],
                 V_prior_const=c["V_prior_const"])
    strip = bf.BigFieldStrip(rows=rows, cols=cols, rank=0, world=1, device=0, max_stars=n, max_ghosts=1, patch_radius=12,
                             halo=24, **c)
    D = strip.gen_mock_data(t["q_true"], seed=77, return_data=True)
    q0 = t["q0"]
    strip.set_stars(q0)
    eng = bf.BigFieldRHMC([strip])
    eng.evaluate(want_V=True, g_ff2=4.0)
    grad = eng.stars(n)[2]
    rng = np.random.RandomState(1)
    near_edge = np.nonzero((q0[:, 1] < 14) | (q0[:, 1] > rows - 14) | (q0[:, 2] < 14) | (q0[:, 2] > cols - 14))[0][:20]
    picks = np.unique(np.concatenate([rng.choice(n, 180, replace=False), near_edge]))
    worst = 0.0
    scale = np.max(np.abs(grad), axis=0)
    for k in picks:
        x, y = q0[k, 1], q0[k, 2]
        i0, i1 = max(0, int(np.floor(x)) - 40), min(rows, int(np.floor(x)) + 41)
        j0, j1 = max(0, int(np.floor(y)) - 40), min(cols, int(np.floor(y)) + 41)
        sel = np.nonzero((np.abs(q0[:, 1] - x) <= 26) & (np.abs(q0[:, 2] - y) <= 26))[0]
        qs = q0[sel] - np.array([0.0, i0, j0])
        Sc = S.clone(num_rows=i1 - i0, num_cols=j1 - j0)
        _, go = so.patch_eval(Sc, D[i0:i1, j0:j1], qs, rad=12)
        mine = go[np.nonzero(sel == k)[0][0]]
        err = np.abs(grad[k] - mine) / np.maximum(np.abs(mine), 1e-6 * scale)
        worst = max(worst, float(err.max()))
    assert worst < 1e-9, worst
    strip.close()
