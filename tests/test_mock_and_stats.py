"""SURVEY.md 8f rows 3-4: device-side mock data (model render + counter-based Poisson) and chain statistics.

CPU part: the oracle's restatements are pinned -- convergence_stats against the reference itself (through the py2->py3
shim, with its Python-2 integer division restored) and against a committed golden; the Philox Poisson sampler against
the Poisson distribution.  GPU part: the CUDA kernels against the oracle, value for value."""
import os

import numpy as np
import pytest

import ref_shim
import stellar_oracle as so
from helpers import GOLDEN_DIR, relerr


def _ar1_chains(seed, nchain, niter, d, phi):
    rng = np.random.RandomState(seed)
    x = np.zeros((nchain, niter, d))
    eps = rng.randn(nchain, niter, d)
    for t in range(1, niter):
        x[:, t] = phi * x[:, t - 1] + eps[:, t]
    return x + rng.randn(nchain, 1, d) * 0.05 + np.arange(d) * 3.0


def test_convergence_stats_golden():
    """Fixture recorded from the reference (tests/golden/make_golden.py: utils.convergence_stats run under Python-2
    division semantics)."""
    with np.load(os.path.join(GOLDEN_DIR, "conv_stats.npz")) as z:
        for tag in ("a", "b"):
            R, neff = so.convergence_stats(z["chain_" + tag], int(z["thin_" + tag]), int(z["warm_" + tag]))
            assert relerr(R, z["R_" + tag]) < 1e-12
            assert relerr(neff, z["neff_" + tag]) < 1e-10


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.available(), reason="reference checkout not present")
def test_convergence_stats_matches_live_reference():
    utils = ref_shim.load()[0]
    x = _ar1_chains(5, 6, 400, 3, 0.6)
    for thin, warm in ((5, 0), (1, 37), (3, 100)):
        R0, n0 = utils.convergence_stats(x, thin_rate=thin, warm_up_num=warm)
        R1, n1 = so.convergence_stats(x, thin, warm)
        assert relerr(R1, R0) < 1e-12 and relerr(n1, n0) < 1e-10


def test_philox_poisson_distribution():
    """Mean, variance and a chi-square against the Poisson pmf for the three regimes of the sampler (multiplication
    method, PTRS near the background level, PTRS for a bright pixel); independent streams for different seeds / offsets."""
    from scipy import stats

    for lam, n in ((3.3, 200000), (24.98145266935892, 200000), (2850.0, 100000)):
        d = so.poisson_philox(np.full(n, lam), seed=11)
        assert np.all(d == np.floor(d)) and d.min() >= 0
        assert abs(d.mean() - lam) < 5 * np.sqrt(lam / n)
        assert abs(d.var() / lam - 1.0) < 5 * np.sqrt(2.0 / n)
        lo, hi = int(stats.poisson.ppf(1e-4, lam)), int(stats.poisson.ppf(1 - 1e-4, lam))
        edges = np.arange(lo, hi + 2) - 0.5
        obs, _ = np.histogram(d, bins=edges)
        exp = n * stats.poisson.pmf(np.arange(lo, hi + 1), lam)
        keep = exp > 20
        chi2 = np.sum((obs[keep] - exp[keep]) ** 2 / exp[keep])
        assert chi2 < stats.chi2.ppf(1 - 1e-6, keep.sum() - 1), (lam, chi2, keep.sum())
    a = so.poisson_philox(np.full(1000, 25.0), seed=1)
    assert not np.array_equal(a, so.poisson_philox(np.full(1000, 25.0), seed=2))
    b = so.poisson_philox(np.full(1500, 25.0), seed=1, index_base=500)
    assert np.array_equal(a[500:], b[:500])  # the draw of a pixel depends on its global index only
    big = so.poisson_philox(np.full(10, 25.0), seed=1, index_base=2**33 + 5)
    assert not np.array_equal(big, a[5:15])  # the high counter word is used


def test_philox_matches_published_vectors():
    """Known-answer test of Philox4x32-10 (Random123 kat_vectors): zero key/counter and the all-ones vector."""
    r = so.philox4x32_10(0, 0, 0, 0, 0)
    assert [int(v) for v in r] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    r = so.philox4x32_10(0xFFFFFFFFFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF)
    assert [int(v) for v in r] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]


# ------------------------------------------------------------------------------------------------------- GPU
def _ctx(F, R, C, N, **kw):
    from hmc_stellar_toy_model_b200.context import RHMCContext

    S = so.Setup()
    base = dict(n_fields=F, num_rows=R, num_cols=C, max_stars=N, psf_fwhm_pix=S.PSF_FWHM_pix, B_count=S.B_count, f_lim=S.f_lim,
                f_low=S.mag2flux_converter(S.mB + 2), g0=S.g0, g1=S.g1, g2=S.g2, g_xx=1.0, g_ff=1.0)
    base.update(kw)
    return RHMCContext(**base), S


def _random_fields(seed, F, R, C, N):
    rng = np.random.RandomState(seed)
    S = so.Setup()
    q = np.zeros((F, N, 3))
    q[:, :, 0] = S.mag2flux_converter(rng.uniform(15, 21, size=(F, N)))
    q[:, :, 1] = rng.uniform(-0.5, R + 0.5, size=(F, N))
    q[:, :, 2] = rng.uniform(-0.5, C + 0.5, size=(F, N))
    return q.reshape(F, 3 * N)


@pytest.mark.gpu
@pytest.mark.parametrize("R,C,N", [(32, 32, 1), (48, 40, 7), (64, 64, 70), (20, 150, 3)])
def test_gen_model_matches_oracle(R, C, N):
    F = 5
    ctx, S = _ctx(F, R, C, N)
    S.num_rows, S.num_cols = R, C
    q = _random_fields(3, F, R, C, N)
    nstars = np.array([N, max(0, N - 1), N, 0, N], dtype=np.int32)
    got = ctx.gen_model(q, nstars)
    for f in range(F):
        want = so.model_image(S, q[f, :3 * nstars[f]])
        assert relerr(got[f], want) < 1e-13  # separable product vs exp of the sum: a few ulp per star


@pytest.mark.gpu
def test_gen_mock_data_value_for_value_and_sharding():
    """Device Poisson data equal the oracle's restatement driven by the same Philox counters, pixel for pixel; a shard of
    the batch with its global field offset reproduces the same images; the data are installed in the context."""
    F, R, C, N = 24, 32, 32, 2
    ctx, S = _ctx(F, R, C, N)
    S.num_rows, S.num_cols = R, C
    q = _random_fields(9, F, R, C, N)
    q[0, 0] = S.mag2flux_converter(13.0)  # a very bright star: lambda of several 1e4 in the core
    D = ctx.gen_mock_data(q, seed=1234)
    lam = np.stack([so.model_image(S, q[f]) for f in range(F)])
    want = so.poisson_philox(ctx.gen_model(q), seed=1234)
    assert np.array_equal(D, want)
    assert abs(np.mean((D - lam) / np.sqrt(lam))) < 5 / np.sqrt(D.size)
    assert abs(np.var((D - lam) / np.sqrt(lam)) - 1.0) < 0.05
    sub, _ = _ctx(8, R, C, N)
    Dsub = sub.gen_mock_data(q[8:16], seed=1234, field_id_base=8)
    assert np.array_equal(Dsub, D[8:16])
    assert not np.array_equal(ctx.gen_mock_data(q, seed=1235), D)
    # the generated images are the context's data: V equals the oracle's on them
    D = ctx.gen_mock_data(q, seed=1234, return_data=True)
    V = ctx.eval(q, f_pos=False)[0]
    for f in (0, 5, 23):
        S.D = D[f]
        assert abs(V[f] - so.potential(S, q[f])) <= 1e-10 * abs(V[f])


@pytest.mark.gpu
def test_low_background_uses_multiplication_method():
    F, R, C = 4, 32, 32
    ctx, S = _ctx(F, R, C, 1, B_count=2.5, f_lim=1.0)
    q = _random_fields(2, F, R, C, 1)
    D = ctx.gen_mock_data(q, seed=5)
    assert np.array_equal(D, so.poisson_philox(ctx.gen_model(q), seed=5))
    assert (D == 0).sum() > 50  # exp(-2.5) = 8 % of the background pixels


@pytest.mark.gpu
def test_gym_device_mock_data():
    from hmc_stellar_toy_model_b200 import sampler_RHMC as gyms

    gym = gyms.multi_gym(Nsteps=5, dt=0.1, g_xx=1., g_ff=1., g_ff2=1.)
    gym.num_rows = gym.num_cols = 32
    q_true = np.array([[18.0, 12.3, 14.1], [20.0, 20.5, 9.9]])
    state = np.random.get_state()[1].copy()
    gym.gen_mock_data(q_true, device_seed=77)
    assert np.array_equal(np.random.get_state()[1], state)  # the global legacy stream is untouched
    lam = gym.gen_model(q_true)
    z = (gym.D - lam) / np.sqrt(lam)
    assert gym.D.shape == (32, 32) and abs(z.mean()) < 0.2 and abs(z.std() - 1) < 0.15
    assert np.isfinite(gym.V(gym.format_q(q_true.copy()), f_pos=True))


@pytest.mark.gpu
def test_bigfield_mock_data_tiled_equals_untiled():
    """A 3-strip tiling and the untiled engine generate the same counts on every shared row (global pixel counters, fixed
    summation order of the model), and the untiled image equals the oracle's Poisson draw of the patch-limited model."""
    from hmc_stellar_toy_model_b200 import bigfield as bf

    rows, cols, n = 300, 210, 120
    S = so.Setup()
    rng = np.random.RandomState(4)
    qt = np.stack([S.mag2flux_converter(rng.uniform(15, 20, n)), rng.uniform(1, rows - 1, n), rng.uniform(1, cols - 1, n)], axis=1)
    kw = dict(rows=rows, cols=cols, device=0, max_stars=n, max_ghosts=n, patch_radius=12, halo=24, psf_fwhm_pix=S.PSF_FWHM_pix,
              B_count=S.B_count, f_lim=S.f_lim, f_low=S.mag2flux_converter(S.mB + 2), g0=S.g0, g1=S.g1, g2=S.g2, g_xx=1.0, g_ff=1.0)
    whole = bf.BigFieldStrip(rank=0, world=1, **kw)
    D = whole.gen_mock_data(qt, seed=99, return_data=True)
    assert np.all(D == np.floor(D)) and D.min() >= 0
    for r in range(3):
        s = bf.BigFieldStrip(rank=r, world=3, **kw)
        Dr = s.gen_mock_data(qt, seed=99, return_data=True)
        assert np.array_equal(Dr, D[s.row0:s.row0 + s.nrows])
        s.close()
    # patch-limited model of the oracle: same counters -> same counts except where a 1-ulp difference of lambda flips a
    # rejection test (none expected at this size)
    lam = np.full((rows, cols), S.B_count)
    sig2 = (S.PSF_FWHM_pix / 2.354) ** 2
    for f, x, y in qt:
        mi, mj = int(np.floor(x)), int(np.floor(y))
        i0, i1, j0, j1 = max(0, mi - 12), min(rows - 1, mi + 12), max(0, mj - 12), min(cols - 1, mj + 12)
        ex = np.exp(-((np.arange(i0, i1 + 1) + 0.5 - x) ** 2) / (2 * sig2))
        ey = np.exp(-((np.arange(j0, j1 + 1) + 0.5 - y) ** 2) / (2 * sig2)) / (2 * np.pi * sig2)
        lam[i0:i1 + 1, j0:j1 + 1] += f * ex[:, None] * ey[None, :]
    want = so.poisson_philox(lam, seed=99)
    assert np.mean(want != D) < 1e-4
    z = (D - lam) / np.sqrt(lam)
    assert abs(z.mean()) < 5 / np.sqrt(D.size) and abs(z.var() - 1) < 0.05
    # the engine runs on the generated data
    whole.set_stars(qt)
    eng = bf.BigFieldRHMC([whole])
    eng.evaluate(want_V=True)
    V, _ = eng.energies()
    assert np.isfinite(V)
    whole.close()


@pytest.mark.gpu
# rows 1700 (n = 850 samples per split chain) takes the single-CTA kernel, the others the chain-parallel pair
@pytest.mark.parametrize("thin,warm,rows", [(5, 0, 500), (1, 37, 500), (3, 100, 500), (1, 0, 1700)],
                         ids=["5-0", "1-37", "3-100", "1-0-1700"])
def test_convergence_stats_device_matches_oracle(thin, warm, rows):
    from hmc_stellar_toy_model_b200 import utils

    x = _ar1_chains(7, 12, rows, 3, 0.7)
    R0, n0 = so.convergence_stats(x, thin, warm)
    R1, n1 = utils.convergence_stats(x, thin_rate=thin, warm_up_num=warm)
    assert relerr(R1, R0) < 1e-12 and relerr(n1, n0) < 1e-9
    a = (np.random.RandomState(1).rand(12, 500, 1) < 0.7).astype(float)
    assert np.array_equal(utils.acceptance_rate(a), so.acceptance_rate(a))
    assert np.array_equal(utils.acceptance_rate(a, 10, 200), so.acceptance_rate(a, 10, 200))


@pytest.mark.gpu
def test_run_stats_on_resident_chains():
    """2 magnitudes x 64 one-star chains: R and n_eff per magnitude group straight from the device-resident q_chain equal
    the oracle's statistics of the downloaded chains."""
    F, R_, C_ = 128, 32, 32
    ctx, S = _ctx(F, R_, C_, 1)
    S.num_rows, S.num_cols = R_, C_
    q = np.zeros((F, 3))
    q[:64, 0], q[64:, 0] = S.mag2flux_converter(17.0), S.mag2flux_converter(20.0)
    q[:, 1:] = 16.0
    ctx.gen_mock_data(q, seed=3, return_data=False)
    a, keep = ctx.make_run_args(q, 200, 5, 0.2, seed=42, want=("q",))
    ctx.run_upload(a)
    ctx.run_launch(a)
    Rg, ng = ctx.run_stats(n_groups=2, thin_rate=2, warm_up_num=20)   # before (and without needing) the download
    ctx.run_download(a)
    chains = keep["q_chain"].reshape(F, 201, 3)
    for g in range(2):
        R0, n0 = so.convergence_stats(chains[64 * g:64 * (g + 1)], 2, 20)
        assert relerr(Rg[g], R0) < 1e-11 and relerr(ng[g], n0) < 1e-8
    # positions mix (R ~ 1); the flux means differ between chains because every chain has its own data realisation
    assert np.all(np.isfinite(Rg)) and np.all(Rg[:, 1:] < 1.2) and np.all(ng > 0)


# ------------------------------------------------------------------------------------------------------- find_peaks
def _peaks_setup():
    from helpers import golden

    g = golden("find_peaks")
    L = so.LightSetup(num_rows=32, num_cols=32)
    L.D = g["D"]
    return g, L


def test_find_peaks_oracle_matches_golden():
    """Fixture recorded from lightsource_gym.find_peaks (samplers.py:129-254) with its own jitter draws."""
    g, L = _peaks_setup()
    assert np.array_equal(so.ls_find_peaks(L, g["jitter"], linear_pix_density=0.25, no_perturb=True), g["q_seed0"])
    got = so.ls_find_peaks(L, g["jitter"], linear_pix_density=0.25, Nstep=400)
    assert got.shape == g["q_seed"].shape and relerr(got, g["q_seed"]) < 1e-12


@pytest.mark.gpu
def test_find_peaks_gym_replays_reference_script():
    """The drop-in gym with the reference's seed: same jitter draws consumed from the global stream, same surviving and
    merged peaks, positions and fluxes to 1e-6 (the |dV/V| < 1e-9 stop test may fire one step apart)."""
    from hmc_stellar_toy_model_b200 import samplers as m

    g, L = _peaks_setup()
    np.random.seed(int(g["seed"]))
    gym = m.lightsource_gym()
    gym.num_rows = gym.num_cols = 32
    gym.gen_mock_data(q_true=g["q_true"])
    assert np.array_equal(gym.D, g["D"])
    state = np.random.get_state()
    gym.find_peaks(linear_pix_density=0.25, Nstep=400, dt_f_coeff=1e-1, dt_xy_coeff=1e-1)
    assert gym.q_seed.shape == g["q_seed"].shape
    assert relerr(gym.q_seed, g["q_seed"]) < 1e-6
    np.random.set_state(state)
    gym.find_peaks(linear_pix_density=0.25, no_perturb=True)
    assert np.array_equal(gym.q_seed, g["q_seed0"])
    assert np.random.random(1)[0] == g["next_uniform"][0]  # the global stream is where the reference left it


@pytest.mark.gpu
def test_find_peaks_descent_matches_oracle_per_seed():
    g, L = _peaks_setup()
    ctx, _ = _ctx(1, 32, 32, 1, B_count=L.B_count, f_lim=0.0, f_low=1.0, g0=1.0, g1=1.0, g2=1.0, enable_hessian=True)
    ctx.set_data(L.D)
    f_lim = so.mag2flux(L.mB - 1.0) * L.flux_to_count
    _, want, alive0, steps0 = so.ls_find_peaks(L, g["jitter"], linear_pix_density=0.25, Nstep=400, return_all=True)
    q, alive, steps = ctx.find_peaks_descend(g["q_seed0"], 400, 1e-1, 1e-1, f_lim)
    assert np.array_equal(alive, alive0)
    assert np.mean(steps == steps0) > 0.9 and np.max(np.abs(steps - steps0)) <= 1
    same = steps == steps0
    assert relerr(q[same & alive], want[same & alive]) < 1e-9
    assert relerr(q[alive], want[alive]) < 1e-6


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.available(), reason="reference checkout not present")
def test_find_peaks_oracle_matches_live_reference():
    """A second configuration (24x40 image, two stars, coarser grid, larger steps) straight against the reference."""
    utils, _, smp = ref_shim.load()
    np.random.seed(123)
    gym = smp.lightsource_gym()
    gym.num_rows = gym.num_cols = 36
    fl = lambda m: utils.mag2flux(m) * gym.flux_to_count  # noqa: E731
    q_true = np.array([[fl(17.5), 12.2, 25.1], [fl(20.0), 27.7, 9.4]])
    gym.gen_mock_data(q_true=q_true)
    state = np.random.get_state()
    n_side = int(0.2 * 36) - 1
    jitter = np.random.randn(n_side * n_side, 2)
    np.random.set_state(state)
    with ref_shim.quiet():
        gym.find_peaks(linear_pix_density=0.2, Nstep=150, dt_f_coeff=0.2, dt_xy_coeff=0.05, dr_tol=1.5, dmag_tol=0.7)
    L = so.LightSetup(num_rows=36, num_cols=36)
    L.D = gym.D
    got = so.ls_find_peaks(L, jitter, linear_pix_density=0.2, Nstep=150, dt_f_coeff=0.2, dt_xy_coeff=0.05, dr_tol=1.5,
                           dmag_tol=0.7)
    assert got.shape == gym.q_seed.shape and relerr(got, gym.q_seed) < 1e-12


@pytest.mark.gpu
def test_device_noise_profile_matches_the_host_profile():
    """gen_noise_profile (sampler_RHMC.py:118-145) with device_seed: 300 Poisson realisations drawn in one launch; the
    residual histogram agrees with the np.random one within sampling noise, is reproducible, and leaves the global
    np.random stream untouched."""
    from hmc_stellar_toy_model_b200.sampler_RHMC import multi_gym

    gym = multi_gym(dt=0.2, Nsteps=10, g_xx=1.0, g_ff=1.0, g_ff2=1.0)
    gym.num_rows = gym.num_cols = 32
    q_true = np.array([[18.0, 16.0, 16.0], [20.5, 8.3, 22.1]])
    np.random.seed(3)
    gym.gen_noise_profile(np.copy(q_true), N_trial=300)
    host = gym.hist_noise.copy()
    state = np.random.get_state()[1].copy()
    gym.gen_noise_profile(np.copy(q_true), N_trial=300, device_seed=11)
    dev = gym.hist_noise.copy()
    assert np.array_equal(np.random.get_state()[1], state)
    gym.gen_noise_profile(np.copy(q_true), N_trial=300, device_seed=11)
    assert np.array_equal(dev, gym.hist_noise)
    assert abs(dev.sum() - host.sum()) < 1e-3 * host.sum()
    width = gym.centers_noise[1] - gym.centers_noise[0]
    assert np.sum(np.abs(dev - host)) * width < 0.02   # total-variation distance of two 3e5-sample histograms
