"""GPU parity tests proper: the CUDA path, called through the C ABI, against the reference's recorded outputs
(tests/golden) and the NumPy oracle on seeded inputs.  FP64 tolerance from BASELINE.json's north_star:
V, gradients and metric <= 1e-10 relative; chains reproduce trajectories and accept decisions step for step."""
import numpy as np
import pytest

import stellar_oracle as so
from helpers import first_divergence, golden, relerr, setup_from

pytestmark = pytest.mark.gpu

RTOL = 1e-10  # north_star FP64 tolerance


def make_ctx(S, n_fields=1, max_stars=1, **kw):
    from hmc_stellar_toy_model_b200 import RHMCContext
    f_low = S.mag2flux_converter(S.mB + 2)
    return RHMCContext(n_fields=n_fields, num_rows=S.num_rows, num_cols=S.num_cols, max_stars=max_stars,
                       psf_fwhm_pix=S.PSF_FWHM_pix, B_count=S.B_count, f_lim=S.f_lim, f_low=f_low, g0=S.g0, g1=S.g1,
                       g2=S.g2, g_xx=S.g_xx, g_ff=S.g_ff, use_prior=S.use_prior, alpha=S.alpha,
                       V_prior_const=S.V_prior_const if S.V_prior_const is not None else 0.0, use_Vc=S.use_Vc,
                       Vc_r_pow=S.Vc_r_pow, **kw)


def grad_relerr(a, b):
    """Element-wise relative error with a floor at 1e-12 of the per-coordinate-type scale (components that vanish
    by cancellation carry absolute, not relative, rounding error)."""
    a = np.asarray(a).reshape(-1, 3)
    b = np.asarray(b).reshape(-1, 3)
    scale = np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b), axis=0, keepdims=True))
    return float(np.max(np.abs(a - b) / scale))


@pytest.mark.parametrize("name,nstar", [("kat1", 1), ("kat2", 2), ("field_eval_204", 204)])
def test_eval_matches_reference(name, nstar):
    g = golden(name)
    S = setup_from(g)
    with make_ctx(S, max_stars=nstar) as ctx:
        ctx.set_data(S.D)
        V, grad, H, Hg = ctx.eval(g["q"], f_pos=True, g_ff2=S.g_ff2, beta=S.beta)
    assert relerr(V[0], g["V"]) < RTOL
    assert grad_relerr(grad[0], g["dVdq"]) < RTOL
    assert relerr(H[0], g["H"]) < RTOL
    assert np.allclose(Hg[0], g["dH"], rtol=RTOL, atol=0)


@pytest.mark.parametrize("name,nstar", [("kat1", 1), ("kat2", 2)])
def test_step_trajectory_matches_reference(name, nstar):
    g = golden(name)
    S = setup_from(g)
    with make_ctx(S, max_stars=nstar) as ctx:
        ctx.set_data(S.D)
        q, p = g["q"][None], g["p"][None]
        for i in range(1, len(g["q_traj"])):
            q, p = ctx.step(q, p, 1, float(g["dt"]), g_ff2=S.g_ff2, beta=S.beta)
            assert relerr(q[0], g["q_traj"][i]) < RTOL, i
            assert relerr(p[0], g["p_traj"][i]) < 1e-9, i
        # the same trajectory in one resident launch
        q2, p2 = ctx.step(g["q"][None], g["p"][None], len(g["q_traj"]) - 1, float(g["dt"]), g_ff2=S.g_ff2, beta=S.beta)
        assert relerr(q2[0], g["q_traj"][-1]) < RTOL


def test_step_204_stars_and_counts():
    g = golden("field_eval_204")
    S = setup_from(g)
    counters = []
    so.rhmc_step(S, g["q"], g["p"], 1e-6, 1000, counters=counters)
    with make_ctx(S, max_stars=204) as ctx:
        ctx.set_data(S.D)
        q, p, counts = ctx.step(g["q"][None], g["p"][None], 1, float(g["dt"]), g_ff2=S.g_ff2, beta=S.beta,
                                return_counts=True)
    assert relerr(q[0], g["q1"]) < RTOL
    assert grad_relerr(p[0], g["p1"]) < 1e-9
    assert tuple(counts[0]) == counters[0]


@pytest.mark.parametrize("name", ["chain_one_star_m19", "chain_one_star_m21", "chain_one_star_m15",
                                  "chain_one_star_m20_sep1"])
def test_run_rhmc_one_star_chain(name):
    g = golden(name)
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    niter = int(g["niter"])
    with make_ctx(S, max_stars=1) as ctx:
        ctx.set_data(S.D)
        r = ctx.run(q0[None], niter, int(g["nsteps"]), float(g["dt"]), normals=g["normals"][None], lnu=g["lnu"][None],
                    g_ff2=S.g_ff2, beta=S.beta, f_pos=True)
    assert np.array_equal(r.A_chain[0].astype(bool), g["A_chain"]), "accept decisions differ"
    assert first_divergence(r.q_chain[0], g["q_chain"], 1e-9) == -1
    assert first_divergence(r.p_chain[0], g["p_chain"], 1e-8) == -1
    assert relerr(r.E_chain[0], g["E_chain"]) < RTOL
    assert relerr(r.V_chain[0], g["V_chain"]) < RTOL
    assert relerr(r.T_chain[0], g["T_chain"]) < 1e-8
    assert abs(r.accept_rate[0] - g["A_chain"].mean()) < 1e-12


@pytest.mark.parametrize("name", ["chain_multi30_vc", "chain_multi100"])
def test_run_rhmc_crowded_chain(name):
    """Crowded field with prior, repulsion and both schedules (RHMC-big-sim2/3.py).

    The 30-star repulsive system is chaotic: a ONE-ulp perturbation of two inputs of the NumPy oracle grows by
    ~1e3 per accepted trajectory (2e-16 -> 2e-13 -> 5e-10 over this fixture; scripts/dbg_chain.py).  So the
    whole-chain comparison checks the accept decisions exactly and the energies to 1e-9, bounds the state error
    loosely, and the 1e-10-class check is done per trajectory, restarting every iteration from the reference's
    own recorded (q, p)."""
    g = golden(name)
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    n = q0.size // 3
    niter, nsteps, dt = int(g["niter"]), int(g["nsteps"]), float(g["dt"])
    with make_ctx(S, max_stars=n) as ctx:
        ctx.set_data(S.D)
        r = ctx.run(q0[None], niter, nsteps, dt, normals=g["normals"][None], lnu=g["lnu"][None],
                    g_ff2=S.g_ff2, beta=S.beta, f_pos=True, schedule_g_ff2=g["schedule_g_ff2"],
                    schedule_beta=g["schedule_beta"])
        assert np.array_equal(r.A_chain[0].astype(bool), g["A_chain"])
        assert first_divergence(r.q_chain[0], g["q_chain"][:, : 3 * n], 1e-6) == -1
        first_accept = int(np.argmax(g["A_chain"])) + 1
        assert first_divergence(r.q_chain[0][: first_accept + 1], g["q_chain"][: first_accept + 1, : 3 * n], RTOL) == -1
        assert relerr(r.E_chain[0], g["E_chain"]) < 1e-9
        assert relerr(r.V_chain[0], g["V_chain"]) < 1e-9
        # restart parity from the reference's recorded states: one step at the 1e-10 class, a whole
        # trajectory within the chaos-limited bound
        for l in range(0, niter + 1, 3):
            Sl = S.clone(dt=dt, g_ff2=float(g["schedule_g_ff2"][l]), beta=float(g["schedule_beta"][l]))
            q, p = g["q_chain"][l, : 3 * n].copy(), g["p_chain"][l, : 3 * n].copy()
            q1, p1 = ctx.step(q[None], p[None], 1, dt, g_ff2=Sl.g_ff2, beta=Sl.beta)
            qg, pg = ctx.step(q[None], p[None], nsteps, dt, g_ff2=Sl.g_ff2, beta=Sl.beta)
            for s in range(nsteps):
                q, p = so.rhmc_step(Sl, q, p)
                if s == 0:
                    assert relerr(q1[0], q) < RTOL, l
                    assert grad_relerr(p1[0], p) < RTOL, l
            assert relerr(qg[0], q) < 1e-6, l


def test_run_single_rhmc():
    g = golden("single_traj")
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    with make_ctx(S, max_stars=1) as ctx:
        ctx.set_data(S.D)
        qc, pc, E, V, T = ctx.run_single(q0[None], g["p0"][None], int(g["nsteps"]), float(g["dt"]), f_pos=True,
                                         g_ff2=S.g_ff2, beta=S.beta)
    assert first_divergence(qc[0], g["q_chain"], 1e-9) == -1
    assert first_divergence(pc[0], g["p_chain"], 1e-8) == -1
    assert np.allclose(V[0], g["V_chain"], rtol=0, atol=1e-6)
    assert np.allclose(T[0], g["T_chain"], rtol=0, atol=1e-6)
    assert np.allclose(E[0], g["E_chain"], rtol=0, atol=1e-6)


def test_batch_of_ragged_fields_against_oracle():
    """Several fields in one launch with different star counts (incl. an empty field)."""
    rng = np.random.RandomState(7)
    base = so.Setup(num_rows=24, num_cols=24, dt=0.02, g_xx=0.05, g_ff=4.0, g_ff2=3.0, use_prior=True, alpha=1.7,
                    V_prior_const=0.3, use_Vc=True, beta=1e-3, Vc_r_pow=3.0)
    counts = [0, 1, 7, 12, 3]
    F, N = len(counts), 12
    q = np.zeros((F, 3 * N))
    p = np.zeros((F, 3 * N))
    D = np.zeros((F, 24, 24))
    setups = []
    for f, n in enumerate(counts):
        qq = np.zeros(3 * n)
        qq[0::3] = base.mag2flux_converter(rng.uniform(15, 22, n))
        qq[1::3] = rng.uniform(1, 23, n)
        qq[2::3] = rng.uniform(1, 23, n)
        S = base.clone()
        S.D = rng.poisson(so.model_image(S, qq)).astype(float)
        setups.append(S)
        D[f] = S.D
        q[f, : 3 * n] = qq
        p[f, : 3 * n] = rng.randn(3 * n) * np.sqrt(so.metric(S, qq)) if n else 0.0
    with make_ctx(base, n_fields=F, max_stars=N) as ctx:
        ctx.set_data(D)
        V, grad, H, Hg = ctx.eval(q, nstars=counts, f_pos=True, g_ff2=3.0, beta=1e-3)
        q1, p1 = ctx.step(q, p, 3, 0.02, g_ff2=3.0, beta=1e-3, nstars=counts)
    for f, n in enumerate(counts):
        S = setups[f]
        qq, pp = q[f, : 3 * n], p[f, : 3 * n]
        assert relerr(V[f], so.potential(S, qq, True)) < RTOL
        if n:
            assert grad_relerr(grad[f, : 3 * n], so.grad_potential(S, qq)) < RTOL
            for _ in range(3):
                qq, pp = so.rhmc_step(S, qq, pp)
            assert relerr(q1[f, : 3 * n], qq) < 1e-9
        assert np.all(grad[f, 3 * n:] == 0)


def test_potential_infinite_outside_support():
    g = golden("kat1")
    S = setup_from(g)
    with make_ctx(S, n_fields=3, max_stars=1) as ctx:
        ctx.set_data(np.repeat(S.D[None], 3, axis=0))
        q = np.array([[S.f_lim * 0.5, 16.0, 16.0], [500.0, -1.5, 16.0], [500.0, 16.0, 33.5]])
        V, _, _, _ = ctx.eval(q, f_pos=True)
        assert np.all(np.isinf(V))
        V2, _, _, _ = ctx.eval(q, f_pos=False)
        assert np.isfinite(V2[0]) and np.isinf(V2[1]) and np.isinf(V2[2])


def test_patch_truncation_radius12_within_tolerance():
    """SURVEY 8d: a 25x25 patch (radius 12) reproduces the full-image gradient to ~1e-13."""
    g = golden("field_eval_204")
    S = setup_from(g)
    with make_ctx(S, max_stars=204, patch_radius=12) as ctx:
        ctx.set_data(S.D)
        V, grad, _, _ = ctx.eval(g["q"], f_pos=True, g_ff2=S.g_ff2)
    assert relerr(V[0], g["V"]) < RTOL
    assert grad_relerr(grad[0], g["dVdq"]) < RTOL


def test_philox_chain_replays_through_oracle():
    """Device-RNG chain: dump the Philox draws, replay them through the NumPy oracle, expect the same chain."""
    g = golden("chain_one_star_m19")
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    niter, nsteps, dt = 25, 10, 0.2
    with make_ctx(S, n_fields=2, max_stars=1) as ctx:
        ctx.set_data(np.repeat(S.D[None], 2, axis=0))
        normals, lnu = ctx.philox_draws(1234, niter)
        r = ctx.run(np.repeat(q0[None], 2, axis=0), niter, nsteps, dt, seed=1234, g_ff2=S.g_ff2, f_pos=True)
    assert abs(normals.mean()) < 0.3 and 0.7 < normals.std() < 1.3
    assert not np.allclose(normals[0], normals[1])
    for f in range(2):
        out = so.run_rhmc(S, q0, normals[f], lnu[f], niter, nsteps, dt)
        assert np.array_equal(r.A_chain[f].astype(bool), out.A)
        assert first_divergence(r.q_chain[f], out.q, 1e-9) == -1
        assert relerr(r.E_chain[f], out.E) < RTOL


def test_fp32_build_within_1e4():
    """FP32 pixel arithmetic: <= 1e-4 relative (scale-relative for gradient components, SURVEY hard part 4)."""
    g = golden("field_eval_204")
    S = setup_from(g)
    with make_ctx(S, max_stars=204, precision=32) as ctx:
        ctx.set_data(S.D)
        V, grad, H, _ = ctx.eval(g["q"], f_pos=True, g_ff2=S.g_ff2)
    assert relerr(V[0], g["V"]) < 1e-4
    a, b = grad[0].reshape(-1, 3), g["dVdq"].reshape(-1, 3)
    assert np.max(np.abs(a - b) / np.max(np.abs(b), axis=0, keepdims=True)) < 1e-4
    assert relerr(H[0], g["H"]) < 1e-12


def test_chain_kernel_matches_field_kernel_and_oracle(monkeypatch):
    """The warp-resident one-star kernel and the generic CTA-per-field kernel are two implementations of the same
    path: run an odd-sized batch of one-star chains through both (and two of them through the oracle)."""
    import bench
    wl = bench.workload_c2(3, seed=5)  # 33 chains, 11 magnitudes
    F = wl["D"].shape[0] - 2           # 31: leaves one half-warp idle
    D, q0 = wl["D"][:F], wl["q0"][:F]
    q0 = q0 + np.random.RandomState(1).uniform(-0.4, 0.4, q0.shape) * np.array([0.0, 1.0, 1.0])
    cfg = dict(wl["cfg"], n_fields=F)
    niter, nsteps, dt = 30, 10, 0.2
    from hmc_stellar_toy_model_b200 import RHMCContext
    res = {}
    for name, off in (("chain", "0"), ("field", "1")):
        monkeypatch.setenv("SRHMC_DISABLE_CHAIN_KERNEL", off)
        with RHMCContext(**cfg) as ctx:
            ctx.set_data(D)
            normals, lnu = ctx.philox_draws(99, niter)
            r = ctx.run(q0, niter, nsteps, dt, seed=99, g_ff2=1.0, f_pos=True)
            V, grad, H, Hg = ctx.eval(q0, f_pos=True, g_ff2=1.0)
            q1, p1, cnt = ctx.step(q0, normals[:, 0] * np.sqrt(H), 3, dt, g_ff2=1.0, return_counts=True)
            res[name] = (r, V, grad, H, Hg, q1, p1, cnt, normals, lnu)
    a, b = res["chain"], res["field"]
    assert np.array_equal(a[0].A_chain, b[0].A_chain)
    assert relerr(a[0].q_chain, b[0].q_chain) < 1e-9
    assert relerr(a[0].E_chain, b[0].E_chain) < 1e-11
    assert relerr(a[1], b[1]) < 1e-12 and grad_relerr(a[2], b[2]) < 1e-10
    assert np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4])
    assert relerr(a[5], b[5]) < 1e-10 and np.array_equal(a[7], b[7])
    assert np.array_equal(a[8], b[8]) and np.array_equal(a[9], b[9])
    k = exp = None
    for f in (0, F - 1):
        S = so.Setup(num_rows=32, num_cols=32, g_xx=1.0, g_ff=1.0, g_ff2=1.0, V_prior_const=0.0, D=D[f])
        out = so.run_rhmc(S, q0[f], a[8][f], a[9][f], niter, nsteps, dt)
        assert np.array_equal(a[0].A_chain[f].astype(bool), out.A)
        assert first_divergence(a[0].q_chain[f], out.q, 1e-9) == -1
        assert relerr(a[0].E_chain[f], out.E) < RTOL


def test_device_math_accuracy():
    """The kernels' own exp / log / reciprocal against libm."""
    g = golden("kat1")
    S = setup_from(g)
    rng = np.random.RandomState(3)
    with make_ctx(S, max_stars=1) as ctx:
        x = -rng.uniform(0, 250, 20000) ** rng.choice([1.0, 0.5, 2.0], 20000) % 650.0
        x[:4] = [0.0, -1e-300, -700.0, -1e-9]
        y = ctx.device_math(0, x)
        assert np.max(np.abs(y - np.exp(x)) / np.exp(x)) < 5e-16
        v = np.concatenate([rng.uniform(1e-3, 1e6, 20000), 10 ** rng.uniform(-300, 300, 2000), [1.0, 2.0, 0.5, 24.98]])
        w = ctx.device_math(1, v)
        assert np.max(np.abs(w - np.log(v)) / np.maximum(np.abs(np.log(v)), 1.0)) < 5e-16
        r = ctx.device_math(2, v)
        assert np.max(np.abs(r * v - 1.0)) < 5e-16


def test_u32_image_path_is_lossless(monkeypatch):
    """Integer-valued data take a compact integer shared-memory layout; results are bit-identical to the float64
    layout (SRHMC_DISABLE_U32_IMAGES=1), and non-integer data silently use float64.  The golden image (largest count 46)
    takes the uint16 layout.  The same image with one corner pixel raised to 70 000 takes the uint32 layout: that pixel
    sets bit 1 of the flags of to_counts_kernel, and the context then keeps the uint32 copy.  The pixel lies 16 rows and
    16 columns from the star, where the PSF weight is below 2^-80, so the chain still follows the star."""
    g = golden("chain_one_star_m21")
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    assert S.D.max() <= 65535 and min(q0[1], q0[2]) > 12
    D32 = S.D.copy()
    D32[0, 0] = 70000.0
    for D in (S.D, D32):
        outs = []
        for off in ("0", "1"):
            monkeypatch.setenv("SRHMC_DISABLE_U32_IMAGES", off)
            with make_ctx(S, max_stars=1) as ctx:
                ctx.set_data(D)
                r = ctx.run(q0[None], 20, 10, 0.2, normals=g["normals"][None, :21], lnu=g["lnu"][None, :21], g_ff2=S.g_ff2)
                outs.append(r)
        assert np.array_equal(outs[0].q_chain, outs[1].q_chain) and np.array_equal(outs[0].E_chain, outs[1].E_chain)
        assert np.array_equal(outs[0].A_chain, outs[1].A_chain)


def test_chunked_scheduler_is_bit_identical(monkeypatch):
    """The chain kernel may split a chain's iterations into chunks that migrate between warps (work scheduler for
    batches that do not fill the resident warps evenly).  Chunking must not change a single bit of any output."""
    g = golden("chain_one_star_m19")
    S = setup_from(g)
    q0 = so.format_q(S, g["q_model"])
    F, niter = 37, 45
    rng = np.random.RandomState(5)
    D = rng.poisson(np.repeat(so.model_image(S, q0)[None], F, axis=0)).astype(float)
    q = np.repeat(q0[None], F, axis=0)
    outs = []
    for chunks in ("1", "7", "46"):
        monkeypatch.setenv("SRHMC_CHAIN_CHUNKS", chunks)
        with make_ctx(S, n_fields=F, max_stars=1) as ctx:
            ctx.set_data(D)
            outs.append(ctx.run(q, niter, 10, 0.2, seed=99, g_ff2=S.g_ff2, f_pos=True))
    for o in outs[1:]:
        for name in ("q_chain", "p_chain", "E_chain", "V_chain", "T_chain", "A_chain", "q_final", "accept_rate"):
            assert np.array_equal(getattr(outs[0], name), getattr(o, name)), name
    assert 0.3 < outs[0].accept_rate.mean() <= 1.0
