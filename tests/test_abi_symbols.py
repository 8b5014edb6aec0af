"""The C-ABI library builds, loads without a GPU, exports every symbol include/stellar_rhmc.h declares, the ctypes
binding covers all of them, and every compute entry point refuses loudly when there is no device (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "stellar_rhmc.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(srhmc_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_and_bound():
    from hmc_stellar_toy_model_b200 import _capi

    lib = _capi.load_library()
    names = _declared_symbols()
    assert len(names) >= 40 and "srhmc_run" in names and "srhmc_big_phase" in names
    for n in names:
        assert hasattr(lib, n), "library does not export %s" % n
        assert n in _capi.SIGNATURES, "ctypes binding lacks %s" % n
    assert set(_capi.SIGNATURES) <= set(names), sorted(set(_capi.SIGNATURES) - set(names))
    assert lib.srhmc_abi_version() == _capi.ABI_VERSION == 3


def test_struct_layouts_match_the_header():
    """Field order of the ctypes structures against the header's struct bodies."""
    from hmc_stellar_toy_model_b200 import _capi

    text = open(os.path.join(ROOT, "include", "stellar_rhmc.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)

    def fields(struct):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
        out = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            names = decl.split(None, 1)[1] if not decl.startswith("const") else decl.split(None, 2)[2]
            for n in names.split(","):
                out.append(n.replace("*", "").strip())
        return out

    for struct, cls in (("srhmc_config", _capi.Config), ("srhmc_run_args", _capi.RunArgs), ("srhmc_ls_args", _capi.LsArgs),
                        ("srhmc_big_config", _capi.BigConfig), ("srhmc_big_step", _capi.BigStep),
                        ("srhmc_big_buffers_t", _capi.BigBuffers), ("srhmc_launch_plan", _capi.LaunchPlan),
                        ("srhmc_chain_plan", _capi.ChainPlan), ("srhmc_chain_layout_t", _capi.ChainLayout)):
        assert fields(struct) == [f[0] for f in cls._fields_], struct


def test_no_cpu_fallback_without_a_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from hmc_stellar_toy_model_b200 import RHMCContext, _capi
    from hmc_stellar_toy_model_b200 import bigfield as bf

    kw = dict(psf_fwhm_pix=3.5, B_count=25.0, f_lim=25.0, f_low=4.0, g0=0.036, g1=0.45, g2=0.008, g_xx=1.0, g_ff=1.0)
    with pytest.raises(_capi.SrhmcError) as e:
        RHMCContext(n_fields=1, num_rows=32, num_cols=32, max_stars=1, **kw)
    assert e.value.code == -3 and "no CPU path" in str(e.value)
    with pytest.raises(_capi.SrhmcError) as e:
        bf.BigFieldStrip(rows=64, cols=64, rank=0, world=1, device=0, max_stars=4, max_ghosts=1, patch_radius=12, halo=12,
                         **kw)
    assert e.value.code == -3
    tf = C.c_double()
    assert _capi.load_library().srhmc_measure_fma_peak(0, 64, C.byref(tf), None) == -3
    assert _capi.load_library().srhmc_device_count() == 0


def test_scheduler_never_plans_an_empty_chunk(monkeypatch):
    """Host logic of the one-star kernel's work scheduler (no device needed): the run is cut into n chunks of
    ceil(L/n) iterations and every chunk must hold at least one iteration -- an empty last chunk would wait for a
    predecessor that never publishes (L = 385 in 24 chunks and L = 1001 in 40 were such cases)."""
    from hmc_stellar_toy_model_b200 import _capi

    lib = _capi.load_library()

    def ok(n, L):
        return n >= 1 and (n - 1) * -(-L // n) < L

    for L in list(range(1, 700)) + [1000, 1001, 1024, 4097, 10001]:
        for parts in (0, 2, 4, 8):
            n = lib.srhmc_plan_chunks(1375, 1184, L, parts)
            if parts == 0:
                assert ok(n, L), (L, parts, n)
            elif n:
                assert n % parts == 0 and ok(n, L), (L, parts, n)
            else:
                assert not ok(parts, L), (L, parts)
    assert lib.srhmc_plan_chunks(1375, 1184, 1001, 8) == 48 and lib.srhmc_plan_chunks(1375, 1184, 1001, 0) == 16
    assert lib.srhmc_plan_chunks(100, 1184, 1001, 0) == 1  # everything resident at once: no chunking
    for c in (1, 5, 24, 40, 500, 5000):
        monkeypatch.setenv("SRHMC_CHAIN_CHUNKS", str(c))
        for L in (1, 7, 385, 1001):
            assert ok(lib.srhmc_plan_chunks(1375, 1184, L, 0), L), (c, L)
