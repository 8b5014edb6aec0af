"""Large crowded fields: one field too big for a single CTA, on one GPU or tiled in row strips over the GPUs of a node
(BASELINE configs[2] scaled up, configs[4]; SURVEY.md 8e).

The numerics run in csrc/big_field.cu behind the `srhmc_big_*` C ABI (include/stellar_rhmc.h): per leapfrog step a fixed
sequence of phases is enqueued on one CUDA stream, with no host synchronisation inside a chain.  When the field is
tiled, three tiny collectives per step ride on the same stream between the phases:

    all-gather   boundary stars (f, x, y) within  halo + r  rows of a strip edge  -> the neighbours' ghost lists
    all-reduce   max of the two fixed-point iteration counts (the reference's field-wide stop rule)
    all-reduce   sum of [V_pixels, T, #out-of-support, V_prior] at the two ends of a trajectory -> dE, so every rank
                 takes the same Metropolis decision (shared Philox log-uniform)

PyTorch appears here only as the owner of the NCCL communicator and as a zero-copy view of the library's device buffers
(`__cuda_array_interface__`); `torch.distributed` can be replaced by `LocalComm`, which runs all ranks of a tiling on
ONE GPU in lock-step (used by the tests to check the tiled numerics against the untiled engine).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi
from ._capi import check_big as check
from .utils import mag2flux

PHASE = dict(PACK=0, EVAL=1, EVAL_V=2, KICK1=3, PFIX_QFIX=4, QFIX_KICK=5, KICK2=6, MOMENTUM=7, ENERGY=8, RECORD_E0=9,
             ACCEPT=10, RESET_ITER=11, EVAL_KICK2=12, EVAL_V_KICK2=13, EVAL_KICK2_KICK1=14, PS_ADVANCE=15, EVAL_PS_ADVANCE=16,
             RJ_BEGIN=17, RJ_JUMP=18, RJ_ACCEPT=19)


# ----------------------------------------------------------------------------------------------- host-side geometry
def tile_order(q, cols, tile=64):
    """Permutation that sorts stars [n,3] (f, x, y) by the 64x64 tile holding them (row-major over the tiles, original order
    inside a tile)."""
    q = np.asarray(q, dtype=np.float64).reshape(-1, 3)
    if len(q) < 2:
        return np.arange(len(q), dtype=np.int64)
    ti = np.floor(q[:, 1] * (1.0 / tile)).astype(np.int64)      # floor(x / tile) = floor(x) // tile
    tj = np.floor(q[:, 2] * (1.0 / tile)).astype(np.int64)
    key = ti * (int(cols) // tile + 1) + tj
    key -= key.min()
    if key.max() < 65536:
        key = key.astype(np.uint16)   # NumPy's stable sort of 16-bit keys is a radix sort: ~4x faster on 1e5 stars
    return np.argsort(key, kind="stable").astype(np.int64)


def chain_starts(q, chains, cols):
    """Storage of K chains of one whole field: q [N,3] (every chain starts there) or [K,N,3] (chain c starts at q[c]) ->
    (q_store [K,N,3], ids [K,N], slots [K,N]).  Chain c is stored in the 64x64-tile order of its own start (tile_order): chains
    started from different catalogues sort differently, and the tile kernel sums each tile's stars in id order, so this keeps
    chain c equal to a one-chain engine started from q[c].  ids[c] is the global id of each stored star; slots[c] the column
    of each stored star in a recorded row (the rank of its id), the same ascending-id columns for every chain."""
    q = np.asarray(q, dtype=np.float64)
    if q.ndim == 3:
        if q.shape[0] != chains or q.shape[2] != 3:
            raise ValueError("per-chain starts must be [K=%d, N, 3], got %s" % (chains, q.shape))
    else:
        q = q.reshape(-1, 3)
        q = np.broadcast_to(q, (chains,) + q.shape)
    ids = np.stack([tile_order(q[c], cols) for c in range(chains)]).reshape(chains, q.shape[1])
    q_store = np.ascontiguousarray(np.take_along_axis(q, ids[:, :, None], axis=1))
    slots = np.argsort(np.argsort(ids, axis=1, kind="stable"), axis=1, kind="stable")
    return q_store, ids, slots


def strip_bounds(rows: int, world: int):
    """Owned row ranges [lo, hi) of `world` equal-height strips (the last one takes the remainder)."""
    base = rows // world
    if base < 1:
        raise ValueError("more ranks than image rows")
    bounds = [(r * base, (r + 1) * base) for r in range(world)]
    bounds[-1] = (bounds[-1][0], rows)
    return bounds


def data_window(rows: int, lo: int, hi: int, halo: int):
    """Local data rows [row0, row0 + nrows) of a strip: the strip plus `halo` rows on each interior side."""
    row0 = max(0, lo - halo)
    row1 = min(rows, hi + halo)
    return row0, row1 - row0


def owner_of(x, rows: int, world: int):
    """Rank owning a star whose row coordinate is x (stars outside the image belong to the edge strips)."""
    base = rows // world
    r = np.floor(np.asarray(x, dtype=float) / base).astype(np.int64)
    return np.clip(r, 0, world - 1)


def ghost_mask(x, lo: int, hi: int, reach: int, rank: int, world: int):
    """Which of a rank's stars go to the lower / upper neighbour: the device PACK phase, restated for the tests."""
    x = np.asarray(x, dtype=float)
    to_lo = (x < lo + reach) if rank > 0 else np.zeros(x.shape, bool)
    to_hi = (x >= hi - reach) if rank < world - 1 else np.zeros(x.shape, bool)
    return to_lo, to_hi


def peak_seeds(rows, cols, linear_pix_density, jitter, f_seed):
    """Seed grid of lightsource_gym.find_peaks (samplers.py:163-176): int(density * rows) - 1 rows by
    int(density * cols) - 1 columns at spacing 1 / density; seed t = i * n_col + j sits at
    (spacing * (i + 0.5 + 0.1 jitter[t, 0]), spacing * (j + 0.5 + 0.1 jitter[t, 1])) with flux f_seed.  jitter
    [n_row * n_col, 2] holds the draws in the reference's order.  The reference's flat index i * n_row + j overwrites
    seeds on a non-square grid; on a square one the two are the same."""
    n_row = max(0, int(linear_pix_density * rows) - 1)
    n_col = max(0, int(linear_pix_density * cols) - 1)
    spacing = 1 / float(linear_pix_density)
    jitter = np.asarray(jitter, dtype=np.float64).reshape(n_row * n_col, 2)
    i = np.repeat(np.arange(n_row), n_col)
    j = np.tile(np.arange(n_col), n_row)
    q = np.empty((n_row * n_col, 3))
    q[:, 0] = f_seed
    q[:, 1] = spacing * (i + 0.5 + 0.1 * jitter[:, 0])
    q[:, 2] = spacing * (j + 0.5 + 0.1 * jitter[:, 1])
    return q


# ----------------------------------------------------------------------------------------------- sample rows
def record_want(want):
    """The chains a run records: a subset of ("q", "p") -> the canonical tuple (empty: recording off)."""
    want = (want,) if isinstance(want, str) else tuple(want)
    bad = set(want) - {"q", "p"}
    if bad:
        raise ValueError("want must be a subset of ('q', 'p'), got %r" % (sorted(bad),))
    return tuple(w for w in ("q", "p") if w in want)


def record_rows(n_iters: int, stride: int):
    """Rows kept of n_iters iterations at chain_stride `stride`: ceil(n_iters / stride) (row r = iteration r * stride)."""
    if stride < 1:
        raise ValueError("chain_stride must be >= 1")
    return -(-int(n_iters) // int(stride))


def slot_ids(ids):
    """Global ids of a strip's stars in slot order: the column order of its recorded rows and statistics (ascending id,
    independent of the tile order the stars are stored in)."""
    return np.sort(np.asarray(ids, dtype=np.int64))


class _DevView:
    """Zero-copy torch view of a device buffer owned by the library."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def _as_tensor(ptr, n, typestr, device):
    import torch

    return torch.as_tensor(_DevView(ptr, n, typestr), device=torch.device("cuda", device))


class BigFieldStrip:
    """One rank's strip: thin wrapper over the srhmc_big_* entry points."""

    def __init__(self, *, rows, cols, rank, world, device, max_stars, max_ghosts, patch_radius, halo, psf_fwhm_pix,
                 B_count, f_lim, f_low, g0, g1, g2, g_xx, g_ff, use_prior=False, alpha=2.0, V_prior_const=0.0, chains=1):
        """chains: K chains of the same field in this context (srhmc_big_set_chains: world = 1, FP64, device draws; every
        evaluation on the tile kernel).  With K > 1 set_stars takes [N,3] or [K,N,3], ids is [K,N] and the per-star arrays
        gain a leading chain axis."""
        self._lib = _capi.load_library()
        lo, hi = strip_bounds(rows, world)[rank]
        row0, nrows = data_window(rows, lo, hi, halo)
        if halo < patch_radius:
            raise ValueError("halo (%d rows) must be at least the patch radius (%d)" % (halo, patch_radius))
        if world > 1 and (hi - lo) < halo + patch_radius + 1:
            # otherwise stars two strips away could touch the local rows and the neighbour exchange is not enough
            raise ValueError("strips of %d rows are too thin for halo %d / patch radius %d" % (hi - lo, halo, patch_radius))
        self.rows, self.cols, self.rank, self.world, self.device = rows, cols, rank, world, device
        self.max_stars = max(1, max_stars)
        self.lo, self.hi, self.row0, self.nrows, self.halo, self.rad = lo, hi, row0, nrows, halo, patch_radius
        cfg = _capi.BigConfig(abi_version=_capi.ABI_VERSION, device=device, rows_global=rows, cols=cols, own_lo=lo,
                              own_hi=hi, row0=row0, nrows=nrows, nrows_halo=halo, max_stars=max(1, max_stars),
                              max_ghosts=max(1, max_ghosts), patch_radius=patch_radius, use_prior=int(bool(use_prior)),
                              world_size=world, rank=rank, psf_fwhm_pix=psf_fwhm_pix, B_count=B_count, f_lim=f_lim,
                              f_low=f_low, g0=g0, g1=g1, g2=g2, g_xx=g_xx, g_ff=g_ff, alpha=alpha,
                              V_prior_const=V_prior_const)
        self._h = C.c_void_p()
        check(self._lib.srhmc_big_create(C.byref(cfg), C.byref(self._h)))
        self.n = 0
        self.n_global = 0
        self.ids = np.zeros(0, dtype=np.int64)
        self._views = None
        self.chains = 1
        self.layout = 0
        if chains != 1:
            self.set_chains(chains)

    def set_chains(self, k):
        """K chains of this field (srhmc_big_set_chains); every chain's stars are cleared.  k = 1 returns to the one-chain
        engine on the evaluation path chosen at creation."""
        check(self._lib.srhmc_big_set_chains(self._h, int(k)))
        self.chains = int(k)
        self.layout += 1   # the per-chain buffers moved: no graph captured before may be replayed
        self.n = self.n_global = 0
        self.ids = np.zeros((0,) if k == 1 else (k, 0), dtype=np.int64)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.srhmc_big_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, ptr):
        check(self._lib.srhmc_big_set_stream(self._h, C.c_void_p(ptr)))

    def adopt_stream(self, ptr):
        check(self._lib.srhmc_big_adopt_stream(self._h, C.c_void_p(ptr)))

    def synchronize(self):
        check(self._lib.srhmc_big_synchronize(self._h))

    @property
    def launch_count(self):
        return int(self._lib.srhmc_big_launch_count(self._h))

    def set_data_window(self, D_local):
        D_local = np.ascontiguousarray(D_local, dtype=np.float64)
        assert D_local.shape == (self.nrows, self.cols), (D_local.shape, self.nrows, self.cols)
        check(self._lib.srhmc_big_set_data(self._h, _capi.dptr(D_local)))

    def set_data(self, D_global):
        self.set_data_window(np.asarray(D_global)[self.row0:self.row0 + self.nrows])

    def set_precision(self, precision):
        """32: gradient-only evaluations through the FP32 tile kernel (float copy of the data); 64: everything FP64."""
        check(self._lib.srhmc_big_set_precision(self._h, int(precision)))

    def gen_mock_data(self, q_true, seed=0, return_data=False):
        """Device-side gen_mock_data (sampler_RHMC.py:77-99) for this strip's data window.  q_true [N,3] (f, x, y) is the
        truth list of the WHOLE field, the same on every rank; the Philox counter of a pixel is its global index, so the
        halo rows of neighbouring strips (and an untiled run) get identical counts."""
        q = np.ascontiguousarray(np.asarray(q_true, dtype=np.float64).reshape(-1, 3))
        out = np.empty((self.nrows, self.cols)) if return_data else None
        check(self._lib.srhmc_big_mock_data(self._h, _capi.dptr(q), len(q), int(seed), _capi.dptr(out)))
        return out

    def set_stars(self, q_global):
        """Take the stars of the global list [N,3] (f, x, y) whose row coordinate falls in this strip.  K > 1 chains (whole
        field): [N,3] starts every chain there, [K,N,3] chain c at q_global[c] (chain_starts)."""
        if self.chains > 1:
            q, ids, _ = chain_starts(q_global, self.chains, self.cols)
            for c in range(self.chains):
                idc = np.ascontiguousarray(ids[c])
                check(self._lib.srhmc_big_set_chain_stars(self._h, c, _capi.dptr(q[c]), idc.ctypes.data_as(C.POINTER(C.c_int64)),
                                                          idc.size))
            self.n, self.ids, self.n_global = ids.shape[1], ids, ids.shape[1]
            return
        q_global = np.asarray(q_global, dtype=np.float64).reshape(-1, 3)
        mine = np.nonzero(owner_of(q_global[:, 1], self.rows, self.world) == self.rank)[0].astype(np.int64)
        # stars are stored in 64x64-tile order (row-major over the tiles, stable inside a tile): consecutive warps of the
        # star-centric gradient kernel then read neighbouring patches (DRAM pages and L2 lines are shared instead of being
        # opened once per 200-byte row segment).  `ids` carries the permutation: every per-star array of the API is in this order.
        q = q_global if len(mine) == len(q_global) else q_global[mine]
        order = tile_order(q, self.cols)
        mine, q = mine[order], np.ascontiguousarray(q[order])
        check(self._lib.srhmc_big_set_stars(self._h, _capi.dptr(q), mine.ctypes.data_as(C.POINTER(C.c_int64)), len(mine)))
        self.n, self.ids, self.n_global = len(mine), mine, len(q_global)

    def set_table(self, q):
        """Store the stars [n,3] as a table in the given order (storage index = table index, ids 0..n-1): the layout of
        reversible-jump runs."""
        q = np.ascontiguousarray(np.asarray(q, dtype=np.float64).reshape(-1, 3))
        ids = np.arange(len(q), dtype=np.int64)
        check(self._lib.srhmc_big_set_stars(self._h, _capi.dptr(q), ids.ctypes.data_as(C.POINTER(C.c_int64)), len(q)))
        self.n, self.ids, self.n_global = len(q), ids, len(q)

    def get_stars(self):
        """(q, p, grad) in storage order: [n,3] each, [K,n,3] with K > 1 chains."""
        if self.chains > 1:
            q, p, g = (np.zeros((self.chains, self.n, 3)) for _ in range(3))
            for c in range(self.chains):
                check(self._lib.srhmc_big_get_chain_stars(self._h, c, _capi.dptr(q[c]), _capi.dptr(p[c]), _capi.dptr(g[c])))
            return q, p, g
        q, p, g = (np.zeros((self.n, 3)) for _ in range(3))
        check(self._lib.srhmc_big_get_stars(self._h, _capi.dptr(q), _capi.dptr(p), _capi.dptr(g)))
        return q, p, g

    def set_momenta(self, p):
        p = np.ascontiguousarray(p, dtype=np.float64).reshape(self.n, 3)
        check(self._lib.srhmc_big_set_momenta(self._h, _capi.dptr(p)))

    def set_draws(self, normals, lnu, n_iters, rows=None):
        rows = self.n if rows is None else rows
        z = None if normals is None else np.ascontiguousarray(normals, dtype=np.float64).reshape(n_iters, rows, 3)
        u = None if lnu is None else np.ascontiguousarray(lnu, dtype=np.float64).reshape(n_iters)
        check(self._lib.srhmc_big_set_draws(self._h, _capi.dptr(z), _capi.dptr(u), n_iters))

    def rj_configure(self, rj, n_iters):
        """Enter reversible-jump mode for the coming n_iters iterations (srhmc_big_rj_configure)."""
        check(self._lib.srhmc_big_rj_configure(self._h, C.byref(rj), int(n_iters)))

    def rj_finish(self, n_iters):
        """Leave reversible-jump mode: (N_chain, move_chain, n_final, overflow); the strip then holds the n_final stars."""
        N = np.zeros(n_iters, dtype=np.int32)
        mv = np.zeros(n_iters, dtype=np.uint8)
        nf, ov = C.c_int32(), C.c_int32()
        out = _capi.RjArgs(N_chain=_capi.iptr(N), move_chain=_capi.bptr(mv), n_final=C.pointer(nf), overflow=C.pointer(ov))
        check(self._lib.srhmc_big_rj_finish(self._h, int(n_iters), C.byref(out)))
        self.n = self.n_global = int(nf.value)
        self.ids = np.arange(self.n, dtype=np.int64)
        return N, mv, int(nf.value), int(ov.value)

    def read_table_samples(self, nrows, want):
        """{name: [nrows, max_stars, 3]} of the rows a reversible-jump run recorded (table order, zero past N)."""
        out = {w: np.empty((int(nrows), self.max_stars, 3)) for w in want}
        check(self._lib.srhmc_big_read_samples(self._h, 0, int(nrows), _capi.dptr(out.get("q")), _capi.dptr(out.get("p"))))
        return out

    def alloc_chains(self, n_iters):
        check(self._lib.srhmc_big_alloc_chains(self._h, n_iters))

    def read_chains(self, n_iters):
        """E / V / T / A_chain [n_iters] and n_accepted; with K > 1 chains [K, n_iters] and [K]."""
        err = C.c_int32()
        if self.chains > 1:
            E, V, T = (np.zeros((self.chains, n_iters)) for _ in range(3))
            A = np.zeros((self.chains, n_iters), dtype=np.uint8)
            nacc = np.zeros(self.chains)
            check(self._lib.srhmc_big_read_chain_rows(self._h, n_iters, _capi.dptr(E), _capi.dptr(V), _capi.dptr(T),
                                                      _capi.bptr(A), _capi.dptr(nacc), C.byref(err)))
        else:
            E, V, T = (np.zeros(n_iters) for _ in range(3))
            A = np.zeros(n_iters, dtype=np.uint8)
            acc = C.c_double()
            check(self._lib.srhmc_big_read_chains(self._h, n_iters, _capi.dptr(E), _capi.dptr(V), _capi.dptr(T),
                                                  _capi.bptr(A), C.byref(acc), C.byref(err)))
            nacc = float(acc.value)
        if err.value == 1:
            raise RuntimeError("an owned star drifted out of the local data window (halo %d rows): re-partition "
                               "more often or enlarge the halo" % self.halo)
        if err.value == 2:
            raise RuntimeError("boundary star list overflow: raise max_ghosts")
        if err.value == 3:
            raise RuntimeError("more than 1024 stars touch one 64x64 tile: the fused tile evaluation cannot hold the list")
        if err.value == 4:
            raise RuntimeError("peer exchange timed out: a rank of the tiling never delivered its contribution")
        return dict(E_chain=E, V_chain=V, T_chain=T, A_chain=A, n_accepted=nacc)

    def set_recording(self, n_iters, stride=1, want=()):
        """Record the sample rows of the coming run (see srhmc_big_set_recording); want=() turns recording off."""
        want = record_want(want)
        check(self._lib.srhmc_big_set_recording(self._h, int(n_iters), int(stride), int("q" in want), int("p" in want)))

    def read_samples(self, row0, nrows, want=("q",), chain=None):
        """{name: [nrows, n, 3]} of recorded rows [row0, row0 + nrows), stars in slot order (`slot_ids(self.ids)`); with
        K > 1 chains those of chain `chain`."""
        want = record_want(want)
        out = {w: np.empty((int(nrows), self.n, 3)) for w in want}
        if self.chains > 1:
            check(self._lib.srhmc_big_read_chain_samples(self._h, int(chain), int(row0), int(nrows), _capi.dptr(out.get("q")),
                                                         _capi.dptr(out.get("p"))))
            return out
        check(self._lib.srhmc_big_read_samples(self._h, int(row0), int(nrows), _capi.dptr(out.get("q")),
                                               _capi.dptr(out.get("p"))))
        return out

    def find_peaks(self, flux_to_count, mag_lim, linear_pix_density=0.2, dr_tol=1., dmag_tol=0.5, Nstep=1000,
                   dt_f_coeff=0.1, dt_xy_coeff=0.1, jitter=None, return_all=False):
        """lightsource_gym.find_peaks (samplers.py:129-254) on this strip's image, which must be the whole field
        (world_size = 1): seeds on the jittered grid (`peak_seeds`, flux mag_lim - 0.5), descent of every seed on a
        pure-background model with potential and gradient over its (2 patch_radius + 1)^2 window, and the greedy merge.
        jitter=None draws np.random.randn in the reference's order from the global stream.  Returns the catalogue [k,3]
        (f in counts, x, y) in seed order, ready for set_stars; with return_all also the descended seeds (q [n,3],
        alive [n], steps [n])."""
        f_lim = mag2flux(mag_lim) * flux_to_count
        f_seed = mag2flux(mag_lim - 0.5) * flux_to_count
        n = max(0, int(linear_pix_density * self.rows) - 1) * max(0, int(linear_pix_density * self.cols) - 1)
        if jitter is None:
            jitter = np.random.randn(n, 2)
        seeds = peak_seeds(self.rows, self.cols, linear_pix_density, jitter, f_seed)
        out = self.descend_seeds(seeds, Nstep, dt_f_coeff, dt_xy_coeff, f_lim, merge=(dr_tol, dmag_tol, flux_to_count))
        catalogue = out["q"][out["kept"]]
        return (catalogue, out["q"], out["alive"], out["steps"]) if return_all else catalogue

    def descend_seeds(self, seeds, Nstep, dt_f_coeff, dt_xy_coeff, f_lim, merge=None):
        """srhmc_big_find_peaks on seeds [n,3]: dict of the descended q, alive and steps; with merge = (dr_tol, dmag_tol,
        flux_to_count) also the kept mask, n_kept and the number of merge rounds.  Nstep = 0 leaves the seeds alive where
        they are, so the merge alone runs on a given list."""
        seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.float64).reshape(-1, 3))
        n = len(seeds)
        q = np.empty((n, 3))
        alive = np.empty(n, dtype=np.uint8)
        steps = np.empty(n, dtype=np.int32)
        kept = np.empty(n, dtype=np.uint8) if merge is not None else None
        n_kept, rounds = C.c_int32(), C.c_int32()
        dr_tol, dmag_tol, flux_to_count = merge if merge is not None else (1.0, 0.5, 1.0)
        args = _capi.BigPeaksArgs(seeds=_capi.dptr(seeds), n=n, nstep=int(Nstep), dt_f_coeff=float(dt_f_coeff),
                                  dt_xy_coeff=float(dt_xy_coeff), f_lim=float(f_lim), dr_tol=float(dr_tol),
                                  dmag_tol=float(dmag_tol), flux_to_count=float(flux_to_count), q=_capi.dptr(q),
                                  alive=_capi.bptr(alive), steps=_capi.iptr(steps), kept=_capi.bptr(kept),
                                  n_kept=C.pointer(n_kept) if merge is not None else None, merge_rounds=C.pointer(rounds))
        check(self._lib.srhmc_big_find_peaks(self._h, C.byref(args)))
        out = dict(q=q, alive=alive.astype(bool), steps=steps)
        if merge is not None:
            out.update(kept=kept.astype(bool), n_kept=int(n_kept.value), rounds=int(rounds.value))
        return out

    def read_scalars(self):
        s = np.zeros(8)
        check(self._lib.srhmc_big_read_scalars(self._h, _capi.dptr(s)))
        return s

    def phase(self, name, step):
        check(self._lib.srhmc_big_phase(self._h, PHASE[name], C.byref(step)))

    def comm_export(self):
        """(64-byte CUDA IPC handle, raw device pointer) of this strip's peer-exchange mailbox."""
        handle = C.create_string_buffer(64)
        raw = C.c_void_p()
        check(self._lib.srhmc_big_comm_export(self._h, handle, C.byref(raw)))
        return handle.raw, raw.value

    def comm_import(self, handles=None, raw_ptrs=None):
        """Map the mailboxes of all ranks: `handles` = world x 64 bytes (other processes) or `raw_ptrs` = world device
        pointers (strips of this process)."""
        hb = None if handles is None else C.create_string_buffer(bytes(handles), 64 * self.world)
        rp = None if raw_ptrs is None else (C.c_void_p * self.world)(*[int(p) for p in raw_ptrs])
        check(self._lib.srhmc_big_comm_import(self._h, hb, rp))

    def views(self):
        """torch views of the communication buffers (needs torch + CUDA)."""
        if self._views is None:
            b = _capi.BigBuffers()
            check(self._lib.srhmc_big_buffers(self._h, C.byref(b)))
            self._views = dict(
                send=_as_tensor(b.ghost_send, b.ghost_send_doubles, "<f8", self.device),
                recv=_as_tensor(b.ghost_recv, b.ghost_recv_doubles, "<f8", self.device),
                scalars=_as_tensor(b.scalars, b.n_scalars, "<f8", self.device),
                gscalars=_as_tensor(b.global_scalars, b.n_scalars, "<f8", self.device),
                counters=_as_tensor(b.counters, b.n_counters, "<i4", self.device))
        return self._views


# ----------------------------------------------------------------------------------------------- collectives
class NoComm:
    """world_size = 1."""

    def max_counters(self, strips):
        pass

    def gather_ghosts(self, strips):
        pass

    def sum_scalars(self, strips):
        pass  # the ACCEPT / RECORD_E0 phases copy the local scalars themselves


class TorchDistComm:
    """One strip per process, NCCL through torch.distributed on the current CUDA stream."""

    def __init__(self, dist=None):
        if dist is None:
            import torch.distributed as dist  # noqa: PLC0415
        self.dist = dist

    def max_counters(self, strips):
        (s,) = strips
        self.dist.all_reduce(s.views()["counters"], op=self.dist.ReduceOp.MAX)

    def gather_ghosts(self, strips):
        (s,) = strips
        v = s.views()
        self.dist.all_gather_into_tensor(v["recv"], v["send"])

    def sum_scalars(self, strips):
        (s,) = strips
        v = s.views()
        v["gscalars"].copy_(v["scalars"])
        self.dist.all_reduce(v["gscalars"], op=self.dist.ReduceOp.SUM)


class PeerComm:
    """The library's own collectives: exchange kernels over peer-mapped memory (NVLink P2P / CUDA IPC) enqueued by the
    phases themselves (KICK1, PFIX_QFIX, EVAL_KICK2_KICK1: max of the fixed-point counts they produce; PACK: boundary lists
    into the neighbours' buffers; RECORD_E0 / ACCEPT: sum of the energy partials) -- no NCCL call on the path, and one
    strip per process can replay a captured CUDA graph of an iteration.

    PeerComm(strips)            all strips of the tiling live in this process (each on its OWN stream: the exchange kernels
                                wait for each other), mailboxes shared by raw device pointers;
    PeerComm([strip], dist)     one strip per process: the 64-byte IPC handles travel once through
                                torch.distributed.all_gather_object at set-up."""

    def __init__(self, strips, dist=None):
        strips = list(strips)
        self.in_process = dist is None
        if dist is None:
            assert len(strips) == strips[0].world, "in-process peer exchange needs every strip of the tiling"
            ptrs = [s.comm_export()[1] for s in sorted(strips, key=lambda s: s.rank)]
            for s in strips:
                s.comm_import(raw_ptrs=ptrs)
        else:
            (s,) = strips
            handle, _ = s.comm_export()
            handles = [None] * s.world
            dist.all_gather_object(handles, handle)
            s.comm_import(handles=b"".join(handles))
            dist.barrier()

    def max_counters(self, strips):
        pass

    def gather_ghosts(self, strips):
        pass

    def sum_scalars(self, strips):
        pass


class LocalComm:
    """All strips of a tiling hosted by this process on ONE device and stream: the collectives become tensor ops.
    Summation order is rank order, like a deterministic all-reduce."""

    def max_counters(self, strips):
        import torch

        m = torch.stack([s.views()["counters"] for s in strips]).max(dim=0).values
        for s in strips:
            s.views()["counters"].copy_(m)

    def gather_ghosts(self, strips):
        import torch

        allsend = torch.cat([s.views()["send"] for s in strips])
        for s in strips:
            s.views()["recv"].copy_(allsend)

    def sum_scalars(self, strips):
        import torch

        tot = torch.stack([s.views()["scalars"] for s in strips]).sum(dim=0)
        for s in strips:
            s.views()["gscalars"].copy_(tot)


# ----------------------------------------------------------------------------------------------- orchestration
class BigFieldRHMC:
    """RHMC on one large field.  `strips` is the list of strips hosted by THIS process: one for a normal run (with
    NoComm or TorchDistComm), all of them for the single-GPU emulation of a tiling (LocalComm)."""

    def __init__(self, strips, comm=None, fixed_point_mode=0):
        """fixed_point_mode: 0 = the reference's stop rule for the two implicit loops of RHMC_single_step (iterate until the
        slowest star of the whole field has converged, sampler_RHMC.py:531-545: parity with the reference, two max
        all-reduces per leapfrog step when tiled); 1 = every star stops at its own convergence (what
        srhmc_config.fixed_point_mode = 1 is for the CTA kernels): per-step results within `delta` of mode 0, three kernels
        and one exchange per leapfrog step."""
        self.strips = list(strips)
        self.comm = comm if comm is not None else NoComm()
        self.multi = self.strips[0].world > 1
        self.fixed_point_mode = int(fixed_point_mode)

    @property
    def chains(self):
        """K: the chains of the field each strip holds (BigFieldStrip(chains=K))."""
        return self.strips[0].chains

    def _one_chain(self, what):
        if self.chains > 1:
            raise ValueError("%s runs one chain: this engine holds %d (K chains run through run())" % (what, self.chains))

    def _step_struct(self, dt, delta, g_ff2, counter_max, f_pos, iteration, seed):
        return _capi.BigStep(dt=float(dt), delta=float(delta), g_ff2=float(g_ff2), counter_max=int(counter_max),
                             f_pos=int(bool(f_pos)), iteration=int(iteration),
                             fixed_point_mode=self.fixed_point_mode, seed=int(seed))

    def _all(self, name, st):
        for s in self.strips:
            s.phase(name, st)

    def evaluate(self, want_V=True, **kw):
        """One gradient (and potential) evaluation at the current star state."""
        self._one_chain("evaluate")
        st = self._step_struct(kw.get("dt", 0.0), 1e-6, kw.get("g_ff2", 1.0), 1000, kw.get("f_pos", True), 0, 0)
        self._ghosts(st)
        self._all("EVAL_V" if want_V else "EVAL", st)
        self._all("ENERGY", st)
        if self.multi:
            self.comm.sum_scalars(self.strips)

    def _advance(self, st):
        """Steps (2)-(4) of RHMC_single_step after the first half kick, up to the point where the gradient at the new
        position is needed (ghost exchange included)."""
        if self.multi:
            self.comm.max_counters(self.strips)
        self._all("PFIX_QFIX", st)
        if self.multi:
            self.comm.max_counters(self.strips)
        self._all("QFIX_KICK", st)
        self._ghosts(st)

    def _ghosts(self, st):
        if self.multi:
            self._all("PACK", st)
            self.comm.gather_ghosts(self.strips)

    def leapfrog(self, st, want_V):
        """One RHMC_single_step (sampler_RHMC.py:522-566); needs the gradient at the current q."""
        if st.fixed_point_mode:
            self._all("PS_ADVANCE", st)
            self._ghosts(st)
        else:
            self._all("KICK1", st)
            self._advance(st)
        self._all("EVAL_V_KICK2" if want_V else "EVAL_KICK2", st)

    def trajectory(self, st, nsteps, want_V_last):
        """nsteps leapfrog steps.  The last half kick of a step and the first half kick of the next one use the same
        gradient, so inside the trajectory they ride in one fused phase behind the evaluation (EVAL_KICK2_KICK1):
        four kernels per step on one GPU."""
        if nsteps <= 0:
            return
        if st.fixed_point_mode:
            # per-star stop rule (fixed_point_mode = 1): no iteration count couples the stars, so everything between two
            # evaluations is one kernel -- three kernels and ONE exchange (the ghost lists) per leapfrog step on N ranks
            self._all("PS_ADVANCE", st)
            self._ghosts(st)
            for t in range(nsteps):
                if t < nsteps - 1:
                    self._all("EVAL_PS_ADVANCE", st)
                    self._ghosts(st)
                else:
                    self._all("EVAL_V_KICK2" if want_V_last else "EVAL_KICK2", st)
            return
        self._all("KICK1", st)
        for t in range(nsteps):
            self._advance(st)
            if t < nsteps - 1:
                self._all("EVAL_KICK2_KICK1", st)
            else:
                self._all("EVAL_V_KICK2" if want_V_last else "EVAL_KICK2", st)

    def steps(self, nsteps, dt, delta=1e-6, counter_max=1000, g_ff2=1.0):
        """nsteps leapfrog steps from the current (q, p) (srhmc_step semantics)."""
        self._one_chain("steps")
        st = self._step_struct(dt, delta, g_ff2, counter_max, True, 0, 0)
        self._ghosts(st)
        self._all("EVAL", st)
        self.trajectory(st, nsteps, False)

    def _iteration(self, st, nsteps):
        self._all("MOMENTUM", st)
        self._all("ENERGY", st)
        if self.multi:
            self.comm.sum_scalars(self.strips)
        self._all("RECORD_E0", st)
        self.trajectory(st, nsteps, True)
        self._all("ENERGY", st)
        if self.multi:
            self.comm.sum_scalars(self.strips)
        self._all("ACCEPT", st)

    def run(self, niter, nsteps, dt, delta=1e-6, counter_max=1000, f_pos=True, g_ff2=1.0, seed=0, normals=None, lnu=None,
            schedule_g_ff2=None, use_graph=None, want=(), chain_stride=1):
        """Move-0 leg of multi_gym.run_RHMC (sampler_RHMC.py:1009-1083) for iterations 0..niter, all enqueued on
        the stream; `normals` [niter+1, N_global, 3] / `lnu` [niter+1] inject the reference's draws (parity mode),
        otherwise device Philox keyed by global star id.

        want: a subset of ("q", "p"): the samples recorded on the device and returned as out["q_chain"] / out["p_chain"],
        [ceil((niter+1) / chain_stride), N_global, 3] in global-id order, NaN for stars hosted elsewhere.  Row r is the state
        at the start of iteration r * chain_stride (q before the trajectory, p as drawn), as in multi_gym.run_RHMC.  The
        rows stay on the device for `convergence_stats` until the next run.

        use_graph: capture ONE Metropolis iteration (all its phases and, when tiled, its NCCL collectives) into a CUDA
        graph and replay it niter+1 times -- the chain row and RNG counter then come from a device-side iteration
        counter.  Default: on for an untiled field without a g_ff2 schedule.

        K > 1 chains (BigFieldStrip(chains=K)): chain c draws from Philox field c (chain 0 is the one-chain run), every
        launch covers the K chains; E / V / T / A_chain are [K, L], n_accepted and accept_rate [K], q_chain / p_chain
        [K, Ls, N_global, 3].  Injected normals / lnu need one chain."""
        if self.chains > 1 and (normals is not None or lnu is not None):
            raise ValueError("injected normals / lnu need one chain: K = %d chains draw from Philox fields 0..K-1" % self.chains)
        L = niter + 1
        want = record_want(want)
        Ls = record_rows(L, chain_stride)
        self._rj_graph_key = None   # set_recording below may move the buffers run_rj's captured graph writes
        # a change of the recording set-up may move its buffers: no graph captured before it may be replayed after it
        rec = (want, int(chain_stride), L, tuple((s.n, s.layout) for s in self.strips))
        if rec != getattr(self, "_rec", None):
            self._graph_key = None
        for s in self.strips:
            if s.chains == 1:
                s.set_draws(None if normals is None else np.asarray(normals)[:, s.ids, :], lnu, L)
            s.alloc_chains(L)
            s.set_recording(L, chain_stride, want)
        self._rec = rec
        st0 = self._step_struct(dt, delta, g_ff2, counter_max, f_pos, 0, seed)
        self._ghosts(st0)
        self._all("EVAL_V", st0)
        has_sched = schedule_g_ff2 is not None and len(schedule_g_ff2) > 0
        dist_comm = isinstance(self.comm, TorchDistComm)
        peer_in_process = isinstance(self.comm, PeerComm) and self.comm.in_process and len(self.strips) > 1
        if use_graph is None:
            use_graph = not has_sched and L >= 3 and not dist_comm and not peer_in_process
        if use_graph and peer_in_process:
            raise ValueError("strips that exchange through PeerComm inside one process run on separate streams: no graph")
        if use_graph and dist_comm:
            # measured on 2 x B200 (torch 2.11, NCCL 2.28.9): replaying a graph that contains the captured
            # collectives dead-locked; the tiled path therefore enqueues its phases eagerly
            raise ValueError("CUDA-graph replay is not available with torch.distributed collectives")
        if use_graph and has_sched:
            raise ValueError("a g_ff2 schedule changes a launch parameter every iteration: run with use_graph=False")
        self.replayed_launches = 0
        if use_graph:
            import torch

            self._all("RESET_ITER", st0)
            # one captured iteration serves every later run with the same launch parameters (the chain row and the RNG
            # counter come from the device-side iteration counter; the buffers are owned by the strips and never move)
            key = (int(nsteps), float(dt), float(delta), float(g_ff2), int(counter_max), bool(f_pos), int(seed), L,
                   tuple(s.n for s in self.strips), self.fixed_point_mode, want, int(chain_stride))
            if normals is not None or lnu is not None:
                key = None  # injected draws live in buffers that are re-allocated per run: always capture afresh
            if key is None or getattr(self, "_graph_key", None) != key:
                stg = self._step_struct(dt, delta, g_ff2, counter_max, f_pos, -1, seed)
                run_stream = torch.cuda.current_stream()
                graph = torch.cuda.CUDAGraph()
                before = [s.launch_count for s in self.strips]
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    cap = torch.cuda.current_stream().cuda_stream
                    for s in self.strips:
                        s.adopt_stream(cap)
                    self._iteration(stg, nsteps)
                for s in self.strips:
                    s.adopt_stream(run_stream.cuda_stream)
                self._graph, self._graph_key = graph, key
                self._graph_nodes = sum(s.launch_count - b for s, b in zip(self.strips, before))
                self.replayed_launches = -self._graph_nodes  # the capture itself executed nothing
            for _ in range(L):
                self._graph.replay()
            self.replayed_launches += self._graph_nodes * L  # kernels executed by the replays (not seen by launch_count)
        else:
            for l in range(L):
                g = g_ff2
                if has_sched:
                    g = float(schedule_g_ff2[min(l, len(schedule_g_ff2) - 1)])
                self._iteration(self._step_struct(dt, delta, g, counter_max, f_pos, l, seed), nsteps)
        out = self.strips[0].read_chains(L)
        for s in self.strips[1:]:
            s.read_chains(L)  # synchronises and surfaces per-strip errors
        out["accept_rate"] = out["n_accepted"] / float(L)
        for w in want:
            out[w + "_chain"] = self._samples(w, Ls)
        return out

    def run_rj(self, niter, nsteps, dt, *, P_move, fmin, fmax, K_split=1., beta_a=2., beta_b=2., seed=0, draws=None, normals=None,
               lnu=None, delta=1e-6, counter_max=1000, f_pos=True, g_ff2=1.0, want=("q",), chain_stride=1, use_graph=None):
        """multi_gym.run_RHMC with birth/death and split/merge moves (P_move[1:] != 0) on an untiled field: the semantics of
        RHMCContext(patch_radius=r).run_rj for one field (tests/rj_oracle.rj_run with rad = r), the star count on the device.
        The strip's stars are first re-stored as a table in the order of the list given to set_stars (ids 0..n-1); the
        momentum of star k is keyed by its table index, the jump record of iteration l by (seed, field 0, l).  draws
        [niter+1, 14], normals [niter+1, 3 max_stars] and lnu [niter+1] replace the device's draws.  alpha and V_prior_const
        are the strip's.

        Returns run()'s dict plus N_chain, move_chain (0 within, 1 birth, 2 death, 3 split, 4 merge), n_final, overflow and
        q_chain / p_chain [ceil((niter+1) / chain_stride), max_stars, 3] in table order, zero past N.  Afterwards the strip
        holds the n_final stars (get_stars, ids), and a later run() starts from them.  An iteration whose proposal needed more
        than max_stars stars is rejected; the run then raises ValueError, as the drop-in does, with the result dict as its
        `result` attribute.  use_graph: one captured
        iteration replayed niter+1 times (default: on for niter >= 2)."""
        self._one_chain("run_rj")
        if self.multi or len(self.strips) != 1:
            raise ValueError("reversible-jump runs need the whole field on one device (world_size = 1)")
        if self.fixed_point_mode != 0:
            raise ValueError("reversible-jump runs use the reference stop rule (fixed_point_mode = 0)")
        (s,) = self.strips
        L = niter + 1
        want = record_want(want)
        Ls = record_rows(L, chain_stride)
        q_list = np.empty((s.n, 3))
        q_list[s.ids] = s.get_stars()[0]
        s.set_table(q_list)
        rj = _capi.RjArgs(P_move=(C.c_double * 3)(*[float(x) for x in P_move]), fmin=float(fmin), fmax=float(fmax),
                          K_split=float(K_split), beta_a=float(beta_a), beta_b=float(beta_b),
                          draws=_capi.dptr(None if draws is None else np.ascontiguousarray(draws, dtype=np.float64).reshape(L, 14)))
        s.rj_configure(rj, L)
        try:
            s.set_draws(normals, lnu, L, rows=s.max_stars)
            s.alloc_chains(L)
            s.set_recording(L, chain_stride, want)
            self._graph_key = self._rec = None   # run()'s captured graph and recording set-up are not this run's
            st0 = self._step_struct(dt, delta, g_ff2, counter_max, f_pos, 0, seed)
            s.phase("EVAL_V", st0)
            if use_graph is None:
                use_graph = L >= 3
            self.replayed_launches = 0
            if use_graph:
                import torch

                s.phase("RESET_ITER", st0)
                # one captured iteration serves every later run_rj with the same launch parameters and buffers
                key = (int(nsteps), float(dt), float(delta), float(g_ff2), int(counter_max), bool(f_pos), int(seed), L,
                       tuple(float(x) for x in P_move), float(fmin), float(fmax), float(K_split), float(beta_a),
                       float(beta_b), want, int(chain_stride))
                if draws is not None or normals is not None or lnu is not None:
                    key = None   # injected draws live in buffers that are re-allocated per run: always capture afresh
                if key is None or getattr(self, "_rj_graph_key", None) != key:
                    stg = self._step_struct(dt, delta, g_ff2, counter_max, f_pos, -1, seed)
                    run_stream = torch.cuda.current_stream()
                    graph = torch.cuda.CUDAGraph()
                    before = s.launch_count
                    with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                        s.adopt_stream(torch.cuda.current_stream().cuda_stream)
                        self._rj_iteration(stg, nsteps)
                    s.adopt_stream(run_stream.cuda_stream)
                    self._rj_graph, self._rj_graph_key = graph, key
                    self._rj_graph_nodes = s.launch_count - before
                for _ in range(L):
                    self._rj_graph.replay()
                self.replayed_launches = self._rj_graph_nodes * L
            else:
                for l in range(L):
                    self._rj_iteration(self._step_struct(dt, delta, g_ff2, counter_max, f_pos, l, seed), nsteps)
            out = s.read_chains(L)
            if want:
                for w, v in s.read_table_samples(Ls, want).items():
                    out[w + "_chain"] = v
        finally:
            N, mv, n_final, overflow = s.rj_finish(L)
        out.update(N_chain=N, move_chain=mv, n_final=n_final, overflow=overflow, accept_rate=out["n_accepted"] / float(L))
        if overflow >= 0:
            err = ValueError("the proposal of iteration %d needs %d stars but max_stars = %d" % (overflow, s.max_stars + 1,
                                                                                              s.max_stars))
            err.result = out   # the chains of the run, overflowing iterations rejected
            raise err
        return out

    def _rj_iteration(self, st, nsteps):
        """One reversible-jump iteration: leg 1, the jump, the gradient at the edited table and leg 2 are enqueued every time;
        the device skips what the iteration's move does not run."""
        self._all("MOMENTUM", st)
        self._all("ENERGY", st)
        self._all("RECORD_E0", st)
        self._all("RJ_BEGIN", st)
        self.trajectory(st, nsteps, True)
        self._all("RJ_JUMP", st)
        self._all("EVAL_V", st)
        self.trajectory(st, nsteps, True)
        self._all("ENERGY", st)
        self._all("RJ_ACCEPT", st)

    def _samples(self, name, rows, chunk_bytes=256 << 20):
        """Recorded rows of every strip hosted here in global-id order, downloaded in pieces of about `chunk_bytes`
        ([K, rows, N_global, 3] with K > 1 chains)."""
        n_global = self.strips[0].n_global
        if self.chains > 1:
            (s,) = self.strips
            out = np.full((self.chains, rows, n_global, 3), np.nan)
            step = max(1, chunk_bytes // max(1, 24 * s.n))
            for c in range(self.chains):
                cols = slot_ids(s.ids[c])
                for r0 in range(0, rows, step):
                    nr = min(step, rows - r0)
                    out[c][r0:r0 + nr, cols, :] = s.read_samples(r0, nr, (name,), chain=c)[name]
            return out
        out = np.full((rows, n_global, 3), np.nan)
        for s in self.strips:
            cols = slot_ids(s.ids)
            step = max(1, chunk_bytes // max(1, 24 * s.n))
            for r0 in range(0, rows, step):
                nr = min(step, rows - r0)
                out[r0:r0 + nr, cols, :] = s.read_samples(r0, nr, (name,))[name]
        return out

    def energies(self):
        """(V, T) at the last EVAL_V + ENERGY of the strips hosted here (all of them, or world_size = 1)."""
        self._one_chain("energies")
        sc = sum(s.read_scalars() for s in self.strips)
        V = np.inf if sc[2] > 0 else sc[0] + sc[3]
        return float(V), float(sc[1])

    def stars(self, n_global):
        """(q, p, grad) of the stars hosted by this process scattered into global-id order (NaN elsewhere); [K, N, 3] each
        with K > 1 chains."""
        if self.chains > 1:
            (s,) = self.strips
            q, p, g = (np.full((self.chains, n_global, 3), np.nan) for _ in range(3))
            a, b, c = s.get_stars()
            for k in range(self.chains):
                q[k, s.ids[k]], p[k, s.ids[k]], g[k, s.ids[k]] = a[k], b[k], c[k]
            return q, p, g
        q = np.full((n_global, 3), np.nan)
        p = np.full((n_global, 3), np.nan)
        g = np.full((n_global, 3), np.nan)
        for s in self.strips:
            a, b, c = s.get_stars()
            q[s.ids], p[s.ids], g[s.ids] = a, b, c
        return q, p, g


def convergence_stats(engines, thin_rate=5, warm_up_num=0):
    """utils.convergence_stats (split-chain R-hat and n_eff, the reference's quirks kept) over the q rows that K >= 2 runs of
    the same field recorded on the device (`run(..., want=("q",))`): each engine is one chain, all hosted on one device with
    the same tiling and row count (different seeds or starts).  One variable-parallel kernel per strip; returns (R, n_eff),
    each [N_global, 3] in global-id order, NaN for stars hosted by other processes.  `engines` may also be ONE engine of
    K >= 2 chains (BigFieldStrip(chains=K)): the statistics then cover its own chains."""
    if isinstance(engines, BigFieldRHMC):
        engines = [engines]
    engines = list(engines)
    if len(engines) == 1 and engines[0].chains > 1:
        (s,) = engines[0].strips
        r, ne = np.empty(3 * s.n), np.empty(3 * s.n)
        check(s._lib.srhmc_big_chain_convergence_stats(s._h, int(thin_rate), int(warm_up_num), _capi.dptr(r), _capi.dptr(ne)))
        R = np.full((s.n_global, 3), np.nan)
        n_eff = np.full((s.n_global, 3), np.nan)
        cols = slot_ids(s.ids[0])
        R[cols], n_eff[cols] = r.reshape(-1, 3), ne.reshape(-1, 3)
        return R, n_eff
    if len(engines) < 2:
        raise ValueError("convergence statistics need at least two chains (utils.py:94)")
    nstrips = len(engines[0].strips)
    if any(len(e.strips) != nstrips for e in engines):
        raise ValueError("every chain must host the same strips")
    n_global = engines[0].strips[0].n_global
    R = np.full((n_global, 3), np.nan)
    n_eff = np.full((n_global, 3), np.nan)
    lib = _capi.load_library()
    for i in range(nstrips):
        strips = [e.strips[i] for e in engines]
        s0 = strips[0]
        handles = (C.c_void_p * len(strips))(*[s._h.value for s in strips])
        r, ne = np.empty(3 * s0.n), np.empty(3 * s0.n)
        check(lib.srhmc_big_convergence_stats(handles, len(strips), int(thin_rate), int(warm_up_num), _capi.dptr(r),
                                              _capi.dptr(ne)))
        cols = slot_ids(s0.ids)
        R[cols], n_eff[cols] = r.reshape(-1, 3), ne.reshape(-1, 3)
    return R, n_eff
