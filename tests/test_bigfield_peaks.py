"""Peak finding on a large image (srhmc_big_find_peaks, BigFieldStrip.find_peaks): the seed grid and the windowed
descent of the NumPy checker on the CPU, and on the GPU the device descent and merge against the checkers
(window_peaks_oracle.window_find_peaks, stellar_oracle.merge_peaks and stellar_oracle.ls_find_peaks)."""
import os
import re

import numpy as np
import pytest

import stellar_oracle as so
import window_peaks_oracle as wo
from helpers import golden, relerr
from hmc_stellar_toy_model_b200 import _capi
from hmc_stellar_toy_model_b200 import bigfield as bf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FTC = 1.0 / (0.00546689 * 4.62)
RAD = 12

# Recall thresholds, set from the oracle run on the 128^2 field below (window_find_peaks + merge_peaks found all 7
# isolated bright stars within 1 px, with 34 catalogue entries for 24 stars): every truth star brighter than mag 19 with
# no other truth star within 6 px must have a catalogue entry within 1 px (at least 90 % of them on the GPU's larger
# fields), and the catalogue may hold at most twice as many entries as there are truth stars.
ISO_MAG, ISO_SEP, HIT_PX, MAX_CAT_PER_STAR = 19.0, 6.0, 1.0, 2.0


def _truth(rows, cols, seed):
    """Star list at the large-field density of the benchmark (1.49e-3 stars/px, power law alpha = 2 in mag [15, 20])."""
    rng = np.random.RandomState(seed)
    n = int(round(1.49e-3 * rows * cols))
    alpha = 2.0
    fmin, fmax = so.mag2flux(20.0) * FTC, so.mag2flux(15.0) * FTC
    u = rng.random_sample(n)
    fl = np.exp(np.log(fmin ** (1 - alpha) + u * (fmax ** (1 - alpha) - fmin ** (1 - alpha))) / (1 - alpha))
    x = rng.random_sample(n) * (rows - 2.0) + 1.0
    y = rng.random_sample(n) * (cols - 2.0) + 1.0
    return np.stack([fl, x, y], axis=1)


def _recall(q_true, cat):
    """(found, isolated bright stars) and the catalogue size."""
    mag = so.flux2mag(q_true[:, 0] / FTC)
    from scipy.spatial import cKDTree

    tt = cKDTree(q_true[:, 1:])
    near = tt.query(q_true[:, 1:], k=2)[0][:, 1]
    iso = (mag < ISO_MAG) & (near > ISO_SEP)
    if len(cat) == 0:
        return 0, int(iso.sum())
    d = cKDTree(cat[:, 1:]).query(q_true[iso, 1:])[0]
    return int(np.sum(d < HIT_PX)), int(iso.sum())


def _light(D):
    L = so.LightSetup(num_rows=D.shape[0], num_cols=D.shape[1])
    L.D = np.asarray(D, dtype=float)
    return L


def _limits(L):
    return so.mag2flux(L.mB - 1.0) * L.flux_to_count, so.mag2flux(L.mB - 1.5) * L.flux_to_count


def _field128():
    L = _light(np.zeros((128, 128)))
    q_true = _truth(128, 128, 5)
    lam = so.model_image(so.Setup(num_rows=128, num_cols=128, B_count=L.B_count), q_true.ravel())
    L.D = so.poisson_philox(lam, seed=9)
    return L, q_true


def _small_field():
    """16 x 16 image with two stars: with r = 15 every window is the whole image."""
    L = _light(np.zeros((16, 16)))
    rng = np.random.RandomState(3)
    q_true = np.array([[so.mag2flux(18.5) * FTC, 5.3, 9.7], [so.mag2flux(20.0) * FTC, 11.6, 4.2]])
    lam = so.model_image(so.Setup(num_rows=16, num_cols=16, B_count=L.B_count), q_true.ravel())
    L.D = rng.poisson(lam).astype(float)
    jitter = rng.randn(7 * 7, 2)
    return L, jitter


# ------------------------------------------------------------------ CPU
def test_peak_seeds_match_the_reference_grid():
    g = golden("find_peaks")
    L = _light(g["D"])
    f_seed = _limits(L)[1]
    assert np.array_equal(bf.peak_seeds(32, 32, 0.25, g["jitter"], f_seed), g["q_seed0"])
    L40 = _light(np.zeros((40, 40)))
    jitter = np.random.RandomState(2).randn(7 * 7, 2)
    want = so.ls_find_peaks(L40, jitter, linear_pix_density=0.2, no_perturb=True)
    assert np.array_equal(bf.peak_seeds(40, 40, 0.2, jitter, f_seed), want)


def test_peak_seeds_index_non_square_grids_by_column_count():
    jitter = np.random.RandomState(4).randn(3 * 5, 2)
    q = bf.peak_seeds(20, 30, 0.2, jitter, 7.0)
    assert q.shape == (15, 3) and np.all(q[:, 0] == 7.0)
    i, j = 2, 3
    t = i * 5 + j
    assert q[t, 1] == 5.0 * (i + 0.5 + 0.1 * jitter[t, 0]) and q[t, 2] == 5.0 * (j + 0.5 + 0.1 * jitter[t, 1])


def test_window_descent_is_the_reference_descent_when_the_window_covers_the_image():
    L, jitter = _small_field()
    f_lim, f_seed = _limits(L)
    _, want, alive0, steps0 = so.ls_find_peaks(L, jitter, linear_pix_density=0.5, Nstep=400, return_all=True)
    q, alive, steps = wo.window_find_peaks(L, bf.peak_seeds(16, 16, 0.5, jitter, f_seed), 15, f_lim, Nstep=400)
    assert np.array_equal(alive, alive0) and np.array_equal(steps, steps0)
    assert relerr(q, want) < 1e-12


def test_window_descent_recovers_isolated_bright_stars():
    L, q_true = _field128()
    f_lim, f_seed = _limits(L)
    seeds = bf.peak_seeds(128, 128, 0.2, np.random.RandomState(6).randn(24 * 24, 2), f_seed)
    q, alive, _ = wo.window_find_peaks(L, seeds, RAD, f_lim)
    cat = so.merge_peaks(L, q[alive])
    found, iso = _recall(q_true, cat)
    assert iso >= 5 and found == iso, (found, iso)
    assert len(cat) <= MAX_CAT_PER_STAR * len(q_true), (len(cat), len(q_true))


def test_whole_image_stop_rule_reports_every_empty_sky_seed():
    """The reference's stop test divides by V of the whole image.  The 128^2 field in the corner of a 4096^2 image
    (1e-9 |V| ~ 0.9 there, above the first-step change of an empty-sky seed): every seed away from a star stops after one
    step, still alive, and nearly every grid point becomes a peak.  The window rule on the same image keeps the
    catalogue near the star count."""
    L, q_true = _field128()
    f_lim, f_seed = _limits(L)
    big = np.random.RandomState(8).poisson(L.B_count, size=(4096, 4096)).astype(float)
    big[:128, :128] = L.D
    Lb = _light(big)
    seeds = bf.peak_seeds(128, 128, 0.2, np.random.RandomState(6).randn(24 * 24, 2), f_seed)
    q, alive, steps = wo.window_find_peaks(Lb, seeds, RAD, f_lim, whole_image_stop=True)
    cat = so.merge_peaks(Lb, q[alive])
    assert np.mean(alive) > 0.9 and np.mean(steps == 1) > 0.8, (np.mean(alive), np.mean(steps == 1))
    assert len(cat) > 0.9 * len(seeds), (len(cat), len(seeds))
    qw, aw, _ = wo.window_find_peaks(Lb, seeds, RAD, f_lim)
    assert len(so.merge_peaks(Lb, qw[aw])) <= MAX_CAT_PER_STAR * len(q_true)


def test_peaks_args_layout_matches_the_header():
    text = open(os.path.join(ROOT, "include", "stellar_rhmc.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    body = re.search(r"typedef struct srhmc_big_peaks_args \{(.*?)\} srhmc_big_peaks_args;", text, flags=re.S).group(1)
    names = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        rest = decl.split(None, 2)[2] if decl.startswith("const") else decl.split(None, 1)[1]
        names += [n.replace("*", "").strip() for n in rest.split(",")]
    assert names == [f[0] for f in _capi.BigPeaksArgs._fields_]
    assert "srhmc_big_find_peaks" in _capi.SIGNATURES


# ------------------------------------------------------------------ GPU
def _strip(rows, cols, rad=RAD, world=1, max_stars=1):
    """A strip with the benchmark's large-field constants (prior on, alpha = 2, fluxes in mag [15, 20])."""
    B = so.mag2flux(23.0) * FTC
    fmin, fmax = so.mag2flux(20.0) * FTC, so.mag2flux(15.0) * FTC
    vpc = float(np.log(float(rows) * cols) - np.log(-1.0 / (1.0 / fmax - 1.0 / fmin)))
    return bf.BigFieldStrip(rows=rows, cols=cols, rank=0, world=world, device=0, max_stars=max_stars, max_ghosts=1024,
                            patch_radius=rad, halo=rad, psf_fwhm_pix=3.5, B_count=B, f_lim=B,
                            f_low=so.mag2flux(25.0) * FTC, g0=0.035997054345069765, g1=0.4523523265306124,
                            g2=0.008141675878296745, g_xx=0.05, g_ff=4.0, use_prior=True, alpha=2.0, V_prior_const=vpc)


def _mock(rows, seed, max_stars=1):
    s = _strip(rows, rows, max_stars=max_stars)
    q_true = _truth(rows, rows, seed)
    D = s.gen_mock_data(q_true, seed=seed, return_data=True)
    return s, q_true, D


def _compare_descent(q, alive, steps, want, alive0, steps0):
    assert np.array_equal(alive, alive0)
    same = steps == steps0
    assert np.mean(same) > 0.9 and np.max(np.abs(steps - steps0)) <= 1, (np.mean(same), np.max(np.abs(steps - steps0)))
    assert relerr(q[same], want[same]) < 1e-9


@pytest.mark.gpu
def test_find_peaks_matches_the_reference_on_a_whole_image_window():
    L, jitter = _small_field()
    merged, want, alive0, steps0 = so.ls_find_peaks(L, jitter, linear_pix_density=0.5, Nstep=400, return_all=True)
    s = _strip(16, 16, rad=15)
    s.set_data(L.D)
    cat, q, alive, steps = s.find_peaks(FTC, L.mB - 1.0, linear_pix_density=0.5, Nstep=400, jitter=jitter, return_all=True)
    _compare_descent(q, alive, steps, want, alive0, steps0)
    assert cat.shape == merged.shape and relerr(cat, merged) < 1e-6
    # jitter=None takes the reference's draws from the global stream
    np.random.seed(17)
    a = s.find_peaks(FTC, L.mB - 1.0, linear_pix_density=0.5, Nstep=400)
    np.random.seed(17)
    draws = np.array([[np.random.randn(), np.random.randn()] for _ in range(49)])
    after = np.random.random()
    np.random.seed(17)
    s.find_peaks(FTC, L.mB - 1.0, linear_pix_density=0.5, Nstep=400)
    assert np.random.random() == after
    assert np.array_equal(a, s.find_peaks(FTC, L.mB - 1.0, linear_pix_density=0.5, Nstep=400, jitter=draws))
    s.close()


@pytest.mark.gpu
def test_windowed_descent_matches_the_oracle_on_every_seed_of_1024():
    s, _, D = _mock(1024, 21)
    L = _light(D)
    f_lim, f_seed = _limits(L)
    n = 203 * 203
    seeds = bf.peak_seeds(1024, 1024, 0.2, np.random.RandomState(22).randn(n, 2), f_seed)
    out = s.descend_seeds(seeds, 1000, 0.1, 0.1, f_lim)
    want, alive0, steps0 = wo.window_find_peaks(L, seeds, RAD, f_lim)
    _compare_descent(out["q"], out["alive"], out["steps"], want, alive0, steps0)
    s.close()


@pytest.mark.gpu
def test_device_merge_and_descent_on_2048():
    s, q_true, D = _mock(2048, 31)
    L = _light(D)
    f_lim, f_seed = _limits(L)
    n = 408 * 408
    seeds = bf.peak_seeds(2048, 2048, 0.2, np.random.RandomState(32).randn(n, 2), f_seed)
    out = s.descend_seeds(seeds, 1000, 0.1, 0.1, f_lim, merge=(1.0, 0.5, FTC))
    sub = np.sort(np.random.RandomState(33).choice(n, 300, replace=False))
    want, alive0, steps0 = wo.window_find_peaks(L, seeds[sub], RAD, f_lim)
    _compare_descent(out["q"][sub], out["alive"][sub], out["steps"][sub], want, alive0, steps0)
    # the device merge of the device's own descended seeds is merge_peaks of them
    qa = out["q"][out["alive"]]
    _assert_no_pair_at_a_tolerance(qa, 1.0, 0.5)
    assert np.array_equal(out["q"][out["kept"]], so.merge_peaks(L, qa, 1.0, 0.5))
    assert out["n_kept"] == out["kept"].sum() and out["rounds"] >= 2
    s.close()


def _assert_no_pair_at_a_tolerance(q, dr_tol, dmag_tol):
    """No pair within 1e-9 of either tolerance: the rounding of log10 or of the squared distance decides no case."""
    from scipy.spatial import cKDTree

    pairs = cKDTree(q[:, 1:]).query_pairs(abs(dr_tol) + 1e-6, output_type="ndarray")
    if len(pairs) == 0:
        return
    i, j = pairs[:, 0], pairs[:, 1]
    d2 = (q[i, 1] - q[j, 1]) ** 2 + (q[i, 2] - q[j, 2]) ** 2
    dm = np.abs(so.flux2mag(q[i, 0] / FTC) - so.flux2mag(q[j, 0] / FTC))
    assert np.all(np.abs(d2 - dr_tol ** 2) > 1e-9) and np.all(np.abs(dm - dmag_tol) > 1e-9)


def _merge_cases(rng):
    m2f = lambda m: so.mag2flux(np.asarray(m, dtype=float)) * FTC  # noqa: E731
    parts = []
    k = np.arange(40)
    parts.append(np.stack([m2f(np.full(40, 19.0)), 10.0 + 0.9 * k, np.full(40, 20.3)], 1))    # a line 0.9 px apart
    parts.append(np.stack([m2f(rng.uniform(17.0, 20.0, 1000)), 40.1 + 0.8 * rng.random_sample(1000),
                           50.1 + 0.8 * rng.random_sample(1000)], 1))                               # 1000 seeds in one cell
    for x, y in ((29.95, 5.5), (30.05, 5.7), (5.5, 29.9), (5.8, 30.2), (44.9, 44.9), (45.1, 45.2), (44.95, 45.3)):
        parts.append(np.array([[m2f(18.2), x, y]]))                                                 # across cell borders
    parts.append(np.stack([m2f([18.0, 18.3, 18.7, 19.0, 19.6, 18.1]), np.full(6, 60.5), np.full(6, 3.5)], 1))  # magnitude only
    parts.append(np.array([[m2f(18.5), -3.2, 10.0], [m2f(18.6), -3.9, 10.4], [m2f(18.4), 70.5, 70.2],
                           [m2f(18.5), 70.9, 69.8], [m2f(18.5), -1000.0, -1000.3], [m2f(18.5), -1000.5, -1000.0],
                           [m2f(18.5), 10.0, -2.5], [m2f(19.5), 10.1, -2.9]]))                      # outside the 64^2 image
    rest = np.concatenate(parts[1:])
    return np.concatenate([parts[0], rest[rng.permutation(len(rest))]])


@pytest.mark.gpu
@pytest.mark.parametrize("dr_tol", [0.3, 1.0, 2.5])
def test_device_merge_equals_merge_peaks(dr_tol):
    s = _strip(64, 64)
    s.gen_mock_data(np.zeros((0, 3)), seed=1)
    L = _light(np.zeros((64, 64)))
    q = _merge_cases(np.random.RandomState(40))
    _assert_no_pair_at_a_tolerance(q, dr_tol, 0.5)
    out = s.descend_seeds(q, 0, 0.1, 0.1, 1.0, merge=(dr_tol, 0.5, FTC))
    assert np.array_equal(out["q"], q) and out["alive"].all() and not out["steps"].any()
    want = so.merge_peaks(L, q, dr_tol, 0.5)
    assert np.array_equal(q[out["kept"]], want), (out["n_kept"], len(want))
    assert out["n_kept"] == len(want)
    if dr_tol == 1.0:   # the line (seeds 0..39): keep, remove, keep, ... one more round per seed of the chain
        assert np.array_equal(out["kept"][:40], np.arange(40) % 2 == 0) and out["rounds"] >= 40
    s.close()


@pytest.mark.gpu
def test_found_catalogue_runs_rhmc_on_2048():
    strip, q_true, _ = _mock(2048, 51, max_stars=408 * 408)
    cat = strip.find_peaks(FTC, 22.0)
    found, iso = _recall(q_true, cat)
    assert iso > 100 and found >= 0.9 * iso, (found, iso)
    assert 0.5 * len(q_true) <= len(cat) <= MAX_CAT_PER_STAR * len(q_true), (len(cat), len(q_true))
    strip.set_stars(cat)
    out = bf.BigFieldRHMC([strip]).run(2, nsteps=10, dt=5e-2, g_ff2=4.0, seed=3)   # raises on an error flag
    assert np.all(np.isfinite(out["E_chain"]))
    strip.close()


@pytest.mark.gpu
def test_find_peaks_refusals():
    s2 = _strip(64, 64, world=2)
    with pytest.raises(_capi.SrhmcError) as e:
        s2.find_peaks(FTC, 22.0)
    assert e.value.code == -5
    s2.close()
    s = _strip(64, 64)
    with pytest.raises(_capi.SrhmcError) as e:
        s.find_peaks(FTC, 22.0)
    assert e.value.code == -5
    s.gen_mock_data(np.zeros((0, 3)), seed=1)
    bad = np.array([[100.0, 3.0, 4.0], [100.0, np.nan, 4.0]])
    with pytest.raises(_capi.SrhmcError) as e:
        s.descend_seeds(bad, 10, 0.1, 0.1, 1.0, merge=(1.0, 0.5, FTC))
    assert e.value.code == -1
    with pytest.raises(_capi.SrhmcError) as e:
        s.descend_seeds(bad[:1], 10, 0.1, 0.1, 1.0, merge=(np.inf, 0.5, FTC))
    assert e.value.code == -1
    s.close()
