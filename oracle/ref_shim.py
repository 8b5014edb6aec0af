"""Import-time Python-3 shim for the UNMODIFIED reference, a checkout named by $SRHMC_REFERENCE_DIR.

TEST INFRASTRUCTURE ONLY.  Nothing in the product package imports this file.

The reference (jaekor91/HMC-stellar-toy-model) is Python 2 + matplotlib; neither
exists in this image.  This module loads `utils.py`, `sampler_RHMC.py` and
`samplers.py` straight from the read-only checkout (no source is copied into
this repository) after three mechanical, semantics-preserving rewrites:

  * `print "x"`  ->  `print("x")`          (14 statements in sampler_RHMC.py, ...)
  * `xrange`     ->  `range`
  * `np.infty`, `np.product` aliases for NumPy >= 2

and with stub `matplotlib*` modules registered so the import-time rcParams
writes in utils.py:2-16,22 succeed.  The reference is not part of this
repository, so callers must gate on `available()`.

Used by: tests/golden/make_golden.py (fixture generator) and the CPU tests that
pin oracle/stellar_oracle.py against the live reference.
"""
from __future__ import annotations

import os
import re
import sys
import types

import numpy as np

REFERENCE_DIR = os.environ.get("SRHMC_REFERENCE_DIR", "")

_PRINT_RE = re.compile(r"^(\s*)print\s+(?!\()(.*?)\s*$", re.M)
_loaded: dict[str, types.ModuleType] = {}


def available() -> bool:
    return bool(REFERENCE_DIR) and os.path.isfile(os.path.join(REFERENCE_DIR, "sampler_RHMC.py"))


class _Anything(types.ModuleType):
    """A module whose every attribute is a do-nothing callable / namespace."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        if name == "rcParams":
            value = {}
        else:
            value = _Anything(self.__name__ + "." + name)
        setattr(self, name, value)
        return value

    def __call__(self, *a, **k):
        return _Anything(self.__name__ + "()")

    def __iter__(self):  # `fig, ax = plt.subplots(...)`
        return iter((_Anything("fig"), _Anything("ax")))


def _install_stubs() -> None:
    for name in (
        "matplotlib",
        "matplotlib.pyplot",
        "matplotlib.ticker",
        "matplotlib.patches",
        "matplotlib.colors",
        "mpl_toolkits",
        "mpl_toolkits.axes_grid1",
    ):
        if name not in sys.modules:
            sys.modules[name] = _Anything(name)
    if not hasattr(np, "infty"):
        np.infty = np.inf
    if not hasattr(np, "product"):
        np.product = np.prod


def _py3(src: str) -> str:
    src = src.replace("xrange", "range")
    # the one Python-2 integer division on a path we pin (utils.convergence_stats, utils.py:111: both operands are ints)
    src = src.replace("n = L_chain/2 ", "n = L_chain//2 ")
    return _PRINT_RE.sub(lambda m: "%sprint(%s)" % (m.group(1), m.group(2)), src)


def _load(name: str) -> types.ModuleType:
    if name in _loaded:
        return _loaded[name]
    path = os.path.join(REFERENCE_DIR, name + ".py")
    with open(path, "r") as fh:
        src = _py3(fh.read())
    mod = types.ModuleType(name)
    mod.__file__ = path
    # the reference modules `from utils import *`
    saved = sys.modules.get(name)
    sys.modules[name] = mod
    try:
        exec(compile(src, path, "exec"), mod.__dict__)
    except Exception:
        if saved is None:
            sys.modules.pop(name, None)
        else:
            sys.modules[name] = saved
        raise
    _loaded[name] = mod
    return mod


def load():
    """Return (utils, sampler_RHMC, samplers) modules of the live reference."""
    if not available():
        raise RuntimeError("reference checkout not present: set SRHMC_REFERENCE_DIR to a checkout of the reference "
                           "(now %r)" % REFERENCE_DIR)
    _install_stubs()
    utils = _load("utils")
    sampler_rhmc = _load("sampler_RHMC")
    samplers = _load("samplers")
    return utils, sampler_rhmc, samplers


class quiet:
    """Context manager silencing the reference's progress prints."""

    def __enter__(self):
        self._out = sys.stdout
        sys.stdout = open(os.devnull, "w")

    def __exit__(self, *exc):
        sys.stdout.close()
        sys.stdout = self._out
        return False
