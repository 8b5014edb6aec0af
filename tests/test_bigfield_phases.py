"""Fused phases of the large-field engine (csrc/big_field.cu) against the phases they fuse.

A fused phase runs the per-star code of the phases it replaces in one kernel, with the same arithmetic in the same order,
so its results must be bit for bit those of the unfused sequence:

    EVAL_KICK2_KICK1   =  EVAL, KICK2, KICK1            (field-wide stop rule, inside a trajectory)
    EVAL_V_KICK2       =  EVAL_V, KICK2                 (last step of a trajectory, with the potential)
    EVAL_PS_ADVANCE    =  EVAL_KICK2, PS_ADVANCE        (per-star stop rule, inside a trajectory)
    EVAL_KICK2         =  EVAL, KICK2                   (per-star stop rule, last step)

Each case runs a few leapfrog steps of the same start state both ways, on every evaluation path (scatter / pixel / gather,
the FP64 tile kernel, the star-centric kernel, the FP32 tile kernel) and untiled or as two strips, and compares q, p,
dV/dq and the energies with exact equality.

The scatter kernel adds the stars' PSFs into the model image with FP64 atomics, so its gradient is the same run to run only
where no two patches overlap: that path runs on a field of 36 stars whose patches are disjoint (a grid with stars on the
corners, one outside the image, and a row on the edge between the two strips)."""
import numpy as np
import pytest

from helpers import golden, setup_from

NSTEPS = 3


def _engines(field, world, path, mode, monkeypatch):
    """Two engines with the same start state (q, p, data) and the step parameters to run them with."""
    from test_bigfield import _engine, _set_path, _synthetic_field

    _set_path(monkeypatch, "tile" if path == "fp32" else path)
    if field == "sparse256x96":
        S, D, q = _sparse_field(_synthetic_field)
        p, halo, dt, g_ff2 = None, 20, 2e-2, 4.0
    elif field == "golden204":
        g = golden("field_eval_204")
        S = setup_from(g)
        q, D, p, halo, dt, g_ff2 = g["q"], None, g["p"].reshape(-1, 3), 14, float(g["dt"]), S.g_ff2
    else:   # 256 x 96 with stars on the edges and corners: reflections, clipped patches, stars near the strip edges
        S, D, q = _synthetic_field(256, 96, 700, 3)
        p, halo, dt, g_ff2 = None, 20, 2e-2, 4.0
    engines = []
    for _ in range(2):
        eng = _engine(S, np.asarray(q).ravel(), world=world, D=D, halo=halo, fixed_point_mode=mode)
        for s in eng.strips:
            if path == "fp32":
                s.set_precision(32)
            if p is not None:
                s.set_momenta(p[s.ids])
        engines.append(eng)
    st = engines[0]._step_struct(dt, 1e-6, g_ff2, 1000, True, 0, 11)
    if p is None:
        for eng in engines:
            eng._all("MOMENTUM", st)   # device Philox keyed by the global star id: the same momenta in both engines
    return engines, st, np.asarray(q, dtype=np.float64).reshape(-1, 3)


def _sparse_field(synthetic_field):
    """_synthetic_field's constants on a 9 x 4 grid of stars 30 or more pixels apart in both directions (patches of
    25 x 25 pixels that stay disjoint while the stars move)."""
    S, _, q = synthetic_field(256, 96, 36, 4)
    x, y = np.meshgrid(np.linspace(0.2, 255.6, 9), np.linspace(0.3, 95.8, 4), indexing="ij")
    q[:, 1], q[:, 2] = x.ravel(), y.ravel()
    q[0, 1] = -0.1   # starts outside the image: its position momentum is reflected
    sig = S.PSF_FWHM_pix / 2.354
    ci, cj = np.arange(0.5, 256), np.arange(0.5, 96)
    ex = np.exp(-((ci[None] - q[:, 1:2]) ** 2) / (2 * sig ** 2))
    ey = np.exp(-((cj[None] - q[:, 2:3]) ** 2) / (2 * sig ** 2)) / (2 * np.pi * sig ** 2)
    D = np.random.RandomState(4).poisson(S.B_count + np.einsum("k,ki,kj->ij", q[:, 0], ex, ey)).astype(float)
    return S, D, q


def _run(eng, st, fused):
    """NSTEPS leapfrog steps from an evaluation at the start state, through the fused phases or the phases they fuse;
    the step of the field-wide stop rule ends with the potential (EVAL_V_KICK2), the per-star one without (EVAL_KICK2)."""
    def phases(fused_name, *parts):
        for name in ((fused_name,) if fused else parts):
            eng._all(name, st)

    eng._ghosts(st)
    eng._all("EVAL", st)
    if st.fixed_point_mode == 0:
        eng._all("KICK1", st)
        for t in range(NSTEPS):
            eng._advance(st)
            if t < NSTEPS - 1:
                phases("EVAL_KICK2_KICK1", "EVAL", "KICK2", "KICK1")
            else:
                phases("EVAL_V_KICK2", "EVAL_V", "KICK2")
    else:
        eng._all("PS_ADVANCE", st)
        eng._ghosts(st)
        for t in range(NSTEPS):
            if t < NSTEPS - 1:
                phases("EVAL_PS_ADVANCE", "EVAL_KICK2", "PS_ADVANCE")
                eng._ghosts(st)
            else:
                phases("EVAL_KICK2", "EVAL", "KICK2")
    eng._all("ENERGY", st)
    if eng.multi:
        eng.comm.sum_scalars(eng.strips)


CASES = [(field, path) for field in ("golden204", "synthetic256x96") for path in ("tile", "star", "fp32")]
CASES.append(("sparse256x96", "scatter"))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("field,path", CASES)
def test_fused_phases_equal_the_phases_they_fuse(field, path, world, mode, monkeypatch):
    (fused, unfused), st, q0 = _engines(field, world, path, mode, monkeypatch)
    _run(fused, st, True)
    _run(unfused, st, False)
    a, b = fused.stars(len(q0)), unfused.stars(len(q0))
    for name, x, y in zip(("q", "p", "dV/dq"), a, b):
        assert np.all(np.isfinite(x)), name
        assert np.array_equal(x, y), name
    assert np.all(np.any(a[0] != q0, axis=1))   # every star moved
    Va, Ta = fused.energies()
    Vb, Tb = unfused.energies()
    assert np.isfinite(Va) and Va == Vb and Ta == Tb
