// Fused tile evaluation of the large-field engine (BASELINE configs[4]; north_star: "one CTA per image tile, the
// residual image staged in shared memory").  One gradient evaluation of the whole field (reference:
// base_class.dVdq / base_class.V, sampler_RHMC.py:365-425 / 294-351, PSF truncated to the (2r+1)^2 patch) reads
// the data image from HBM exactly ONCE and never materialises Lambda or rho in global memory:
//
//   bin        one thread per star (own stars: inside the scalar kernel that finishes the position update; ghosts: a
//              small kernel after the exchange): append a pair record (star id, box patch x tile, footprint slot) to
//              the fixed-capacity list of each of the <= 2x2 tiles its patch touches (one atomic per pair)
//   tile       one CTA per 64x64 tile: sort the tile's list by star id (fixed summation order), render
//              Lambda = B + sum f PSF for the tile in registers (4x4 pixels per thread; per-star row/column
//              Gaussian tables in shared memory), read D, rho = D/Lambda - 1 into the shared tile, V partial of
//              the owned rows, then one warp per owned star of the list: the three residual-weighted PSF
//              reductions over patch x tile  -> gpart[star][slot of this tile in the star's 2x2 footprint]
//              (EVAL_V: the last tile to finish sums the per-tile potential partials in tile order); the CTA
//              re-zeroes its list counter for the next evaluation
//   gsum       per owned star: sum of its footprint slots in fixed order, scale -> g[3n]; fused into the scalar kernel
//              that consumes the gradient (big_kick_kernel, big_perstar_kernel) or run on its own (big_gsum_kernel)
//
// No floating-point atomics anywhere: results are bit-reproducible run to run.
#pragma once

namespace {

constexpr int kTile = 64;        // tile edge in pixels (>= 2 kMaxRad + 1, so a patch touches at most 2x2 tiles)
constexpr int kTileThreads = 256;
constexpr int kTileChunk = 16;   // pairs per table build (each warp builds the tables of two pairs)
constexpr int kTileMaxList = 1024;  // stars per tile list (0.13 stars/px over tile + halo)

struct TileSrc {
    const double* q;
    const double* ga;
    const double* gb;
    int n_own, cap;
};

// star record of source id `sid`: own stars [0, n_own), then the two ghost lists (capacity `cap` each)
__device__ __forceinline__ const double* tile_source(const TileSrc& S, int sid) {
    if (sid < S.n_own) return S.q + 3 * (size_t)sid;
    sid -= S.n_own;
    if (sid < S.cap) return (S.ga && sid < (int)S.ga[0]) ? S.ga + 1 + 3 * (size_t)sid : nullptr;
    sid -= S.cap;
    return (S.gb && sid < S.cap && sid < (int)S.gb[0]) ? S.gb + 1 + 3 * (size_t)sid : nullptr;
}

struct TileSpan {
    int ti0, ti1, tj0, tj1;
};

__device__ __forceinline__ TileSpan tile_span(const BigParams& P, int i0, int i1, int j0, int j1) {
    TileSpan t;
    t.ti0 = (i0 - P.row0) / kTile;
    t.ti1 = (i1 - P.row0) / kTile;
    t.tj0 = j0 / kTile;
    t.tj1 = j1 / kTile;
    return t;
}

// (star, tile) pair record: star id, the box patch x tile in tile coordinates (6 bits each) + the index of the tile in the
// star's 2x2 footprint, and the star itself -- so the tile kernel needs ONE trip to global memory for its list instead of
// three dependent ones (count -> records -> star data)
struct __align__(16) PairRec {   // 32 bytes
    int sid, box;
    double f, x, y;
};
constexpr int kTileRecs = 64;    // records of a tile list kept whole in shared memory (later ones are re-read from L2)

__device__ __forceinline__ PairRec ld_rec(const PairRec* p) {   // two 16-byte L2 loads
    const int4 a = __ldcg(reinterpret_cast<const int4*>(p));
    const double2 b = __ldcg(reinterpret_cast<const double2*>(p) + 1);
    PairRec r;
    r.sid = a.x; r.box = a.y;
    r.f = __hiloint2double(a.w, a.z);
    r.x = b.x; r.y = b.y;
    return r;
}

__device__ __forceinline__ int pack_box(int ia, int ib, int ja, int jb, int slot) {
    return ia | (ib << 6) | (ja << 12) | (jb << 18) | (slot << 24);
}

// Append the pair records of one source star to the lists of the tiles its patch touches.  `owned`: the star belongs
// to this rank, so leaving the local data window is an error (flag 1).  List overflow raises flag 3.
__device__ __forceinline__ void bin_star(const BigParams& P, int ntx, int sid, double f, double x, double y, bool owned, int* cnt,
                                         PairRec* list, int* err) {
    int i0, i1, j0, j1, mi, mj;
    bool clipped;
    if (!patch_of(P, x, y, i0, i1, j0, j1, mi, mj, clipped)) {
        if (owned) atomicExch(err, 1);  // an owned star left the local data window
        return;
    }
    if (owned && clipped) atomicExch(err, 1);
    const TileSpan t = tile_span(P, i0, i1, j0, j1);
    for (int ti = t.ti0; ti <= t.ti1; ++ti)
        for (int tj = t.tj0; tj <= t.tj1; ++tj) {
            const int tile = ti * ntx + tj;
            const int pos = atomicAdd(&cnt[tile], 1);
            if (pos >= kTileMaxList) {
                atomicExch(err, 3);  // list capacity exceeded (density above 0.13 stars/px)
                continue;
            }
            const int r0 = P.row0 + ti * kTile, c0 = tj * kTile;
            PairRec rec;
            rec.sid = sid;
            rec.box = pack_box(max(i0, r0) - r0, min(i1, r0 + kTile - 1) - r0, max(j0, c0) - c0, min(j1, c0 + kTile - 1) - c0,
                               (ti - t.ti0) * 2 + (tj - t.tj0));
            rec.f = f; rec.x = x; rec.y = y;
            list[(size_t)tile * kTileMaxList + pos] = rec;
        }
}

// sources [sid0, sid1): own stars are [0, n_own), the ghost lists follow (tile_source)
template <bool LIVE>
__global__ void big_bin_kernel(const BigParams P, const TileSrc S, int ntx, int sid0, int sid1, int* cnt, PairRec* list, int* err,
                               const int* nd /* live owned stars: sid1 */) {
    if (LIVE) sid1 = *nd;
    TileSrc Sc = S;   // chain blockIdx.y: its stars into its own lists
    Sc.q = chain_slice(S.q, 3 * P.X.M);
    cnt += blockIdx.y * P.X.tiles;
    list += blockIdx.y * P.X.tiles * kTileMaxList;
    for (int sid = sid0 + blockIdx.x * blockDim.x + threadIdx.x; sid < sid1; sid += gridDim.x * blockDim.x) {
        const double* src = tile_source(Sc, sid);
        if (!src) continue;
        bin_star(P, ntx, sid, src[0], src[1], src[2], sid < S.n_own, cnt, list, err);
    }
}

constexpr int kTabPad = 4;                 // zero guard entries on each side of a 32-entry factor table
constexpr int kTabLen = 32 + 2 * kTabPad;  // a thread reads 4 consecutive entries starting anywhere in [-3, 31]

// Factor tables of one (star, tile) pair, built by one warp with two warp-wide exponentials (exp_neg: the kernels'
// own branch-free FP64 exponential, fastmath.cuh) and used by BOTH the render and the gather phase:
//   rowf[kTabPad + k] = ex        of row (ia & ~1) + k,     ex = exp(-(i+.5-x)^2/2s^2)
//   colf[kTabPad + k] = f ey      of column (ja & ~1) + k,  ey = norm exp(-(j+.5-y)^2/2s^2)
// (even origins: see build_pair_tab) zero outside the box and in the guards; (dx0, dy0) = offsets of the box's first row / column from the star, from which
// the gather phase forms ex dx and ey dy.
struct PairTab {
    double rowf[kTabLen];
    double colf[kTabLen];
    double dx0, dy0;
};

struct TileSmem {
    double rho[kTile][kTile];          // 32 KB
    PairTab tab[kTileChunk];           // 656 B each
    PairRec rec[kTileRecs];            // the first records of the list, in arrival order
    union {
        int sid[kTileMaxList];         // star id of every record (ranking key): dead once the list is ranked ...
        double rowd[kTileChunk][32];   // ... then ex_k dx_k of row ia + k per table slot (gather phase; no guards needed)
    };
    unsigned short order[kTileMaxList];  // order[r] = arrival index of the record with the r-th smallest star id
    int box[kTileChunk][4];
    double red[32];
    double2 ltab[kLogTableSize];       // table of log_pos (fastmath.cuh), built per CTA when the potential is wanted
    unsigned long long mbar;           // completion barrier of the TMA tile load
    bool is_last;
};

__device__ __forceinline__ void build_pair_tab(const BigParams& P, const PairRec& rec, int r0, int c0, int lane,
                                               PairTab& T, int* box, double* rowd) {
    const double f = rec.f, x = rec.x, y = rec.y;
    const int ia = rec.box & 63, ib = (rec.box >> 6) & 63, ja = (rec.box >> 12) & 63, jb = (rec.box >> 18) & 63;
    const double dx = ((double)(r0 + ia + lane) + 0.5) - x, dy = ((double)(c0 + ja + lane) + 0.5) - y;
    const double ex = (ia + lane <= ib) ? exp_neg(-(dx * dx) * P.inv2s2) : 0.0;
    // entry kTabPad + k belongs to row (ia & ~1) + k / column (ja & ~1) + k: a thread's four consecutive entries then start
    // at an even index and load as two 16-byte words (half the shared-memory wavefronts of four 8-byte loads)
    const int io = ia & 1, jo = ja & 1;
    T.rowf[kTabPad + io + lane] = ex;
    rowd[lane] = ex * dx;
    T.colf[kTabPad + jo + lane] = (ja + lane <= jb) ? exp_neg(-(dy * dy) * P.inv2s2) * (P.norm * f) : 0.0;
    if (lane == 0) {
        T.rowf[kTabPad + (io ? 0 : 32)] = 0.0;   // the 33rd body entry this pair's parity leaves unwritten
        T.colf[kTabPad + (jo ? 0 : 32)] = 0.0;
        T.dx0 = dx;
        T.dy0 = dy;
        if (box) {
            box[0] = ia; box[1] = ib; box[2] = ja; box[3] = jb;
        }
    }
}

// reciprocals of four pixels from one MUFU.RCP64H (product tree: the same number of FP64 instructions as four Newton
// reciprocals, a quarter of the MUFU / move instructions; <= 4 roundings per result)
__device__ __forceinline__ void rcp4(const double (&a)[4], double (&r)[4]) {
    const double p01 = a[0] * a[1], p23 = a[2] * a[3];
    const double ip = rcp_fast(p01 * p23);
    const double r01 = p23 * ip, r23 = p01 * ip;
    r[0] = a[1] * r01;
    r[1] = a[0] * r01;
    r[2] = a[3] * r23;
    r[3] = a[2] * r23;
}

// ---- TMA / mbarrier primitives (sm_90+ PTX; SASS: UTMALDG, SYNCS)
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 2-D tile global -> shared through the tensor map (coordinates: x = column, y = local row), completion on `bar`
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, int x, int y, unsigned long long* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 16-byte asynchronous copy global -> shared (LDGSTS): no registers held while the data are in flight
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
// 8-byte asynchronous copy global -> shared
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// blockIdx.y read where it is used: the chain tile kernel applies its chain offsets at each use, so that no offset pointer
// is held in a register across the kernel (asm volatile: the read is neither hoisted nor merged)
__device__ __forceinline__ unsigned chain_at_use() {
    unsigned y;
    asm volatile("mov.u32 %0, %%ctaid.y;" : "=r"(y));
    return y;
}

// MODE 0: gradient; 1: gradient + pixel potential; 2: mock data -- the rendered model of the tile is Poisson-sampled
// (poisson.cuh, counter = global pixel index) into Dout and nothing else happens.
// CHAINS: the launch covers the context's chains, chain c = blockIdx.y with its own lists, partials, ticket and fixed-point
// counters (counter j of chain c at fp_counters[j K + c]); the shared data tile is the same for every chain.  A template flag
// so that the one-chain instantiations keep their code.
template <int MODE, bool CHAINS = false>
__global__ void __launch_bounds__(kTileThreads, 4) big_tile_kernel(const BigParams P, const TileSrc S, int ntx,
                                                                const double* __restrict__ D,
                                                                int* __restrict__ cnt,
                                                                const PairRec* __restrict__ list, double* __restrict__ gpart,
                                                                double* vpart, unsigned int* ticket, double* scalars,
                                                                int* fp_counters, double* __restrict__ Dout,
                                                                unsigned long long mock_seed,
                                                                const __grid_constant__ CUtensorMap tmapD, int use_tma) {
    constexpr bool WANT_V = MODE == 1;
    // chain offsets are applied where each buffer is used (offset pointers held across the kernel cost registers)
    const int tile = CHAINS ? (int)(chain_at_use() * P.X.tiles) + blockIdx.x : blockIdx.x;   // this chain's list of this tile
    extern __shared__ __align__(128) unsigned char tile_smem_raw[];
    TileSmem& sm = *reinterpret_cast<TileSmem*>(tile_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = kTileThreads / 32;
    const int ti = blockIdx.x / ntx, tj = blockIdx.x % ntx;
    const int r0 = P.row0 + ti * kTile, c0 = tj * kTile;  // global pixel of the tile origin
    const int vr = min(kTile, P.row0 + P.nrows - r0), vc = min(kTile, P.C - c0);  // valid rows / columns

    const int ty = tid >> 4, tx = tid & 15;
    const int pr = 4 * ty, pc = 4 * tx;  // thread owns the 4x4 pixel block at (pr, pc)
    // The tile's data pixels first: every thread copies its own 4x4 block asynchronously straight into the rho buffer, so
    // the HBM latency is covered by the list sort, the table build and the render; the residual later overwrites the
    // block in place (a thread only ever touches its own block before the barrier that precedes the gather).
    if (MODE != 2 && use_tma) {
        // the whole 64x64 tile in one TMA transfer (tiles cut by the image edge are zero-filled by the copy engine);
        // nothing has touched the rho buffer yet, so no proxy fence is needed before the asynchronous write
        if (tid == 0) {
            mbar_init(&sm.mbar, 1);
            mbar_expect_tx(&sm.mbar, kTile * kTile * 8);
            tma_load_2d(&sm.rho[0][0], &tmapD, c0, r0 - P.row0, &sm.mbar);
        }
    } else if (MODE != 2) {
        const bool vec = ((P.C & 1) == 0) && (pc + 3 < vc);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int li = pr + a;
            if (li < vr) {
                const double* row = D + (size_t)(r0 + li - P.row0) * P.C + c0 + pc;
                if (vec) {
                    cp_async16(&sm.rho[li][pc], row);
                    cp_async16(&sm.rho[li][pc + 2], row + 2);
                } else {
#pragma unroll
                    for (int b = 0; b < 4; ++b) sm.rho[li][pc + b] = (pc + b < vc) ? __ldg(row + b) : 0.0;
                }
            } else {
#pragma unroll
                for (int b = 0; b < 4; ++b) sm.rho[li][pc + b] = 0.0;
            }
        }
        cp_async_commit();
    }

    // ---- the tile's pair list, ranked by star id so that every sum below has a fixed order.  The first kTileRecs records
    //      are fetched speculatively together with the count (one trip to L2 instead of two dependent ones); they carry
    //      the star's (f, x, y), so no third trip follows.
    list += (size_t)tile * kTileMaxList;
    PairRec spec;
    spec.sid = 0; spec.box = 0; spec.f = spec.x = spec.y = 0.0;
    if (tid < kTileRecs) spec = ld_rec(&list[tid]);
    const int nl = min(cnt[tile], kTileMaxList);  // an overflow was flagged when the list was filled
    // the fixed-point iteration counters of the leapfrog step are free between its last reader and the next step
    if (fp_counters && blockIdx.x == 0 && tid < 2) fp_counters[CHAINS ? tid * gridDim.y + blockIdx.y : tid] = 0;
    // guard entries of the factor tables stay zero for the whole launch; the 32 body entries are rewritten per pair
    for (int k = tid; k < kTileChunk * 4 * kTabPad; k += kTileThreads) {
        const int pair = k / (4 * kTabPad), e = k % (4 * kTabPad), side = e / kTabPad, g = e % kTabPad;
        double* t = (side & 1) ? sm.tab[pair].colf : sm.tab[pair].rowf;
        t[(side & 2) ? kTabPad + 32 + g : g] = 0.0;
    }
    if (WANT_V && tid < kLogTableSize) {
        // (rc_k, -ln rc_k) with rc_k ~ 1/(bin centre): ln x = e ln2 - ln rc_k + log1p(m rc_k - 1) is an identity for the
        // ROUNDED rc_k, so the table only needs -ln rc_k to double accuracy
        const double rc = 1.0 / (1.0 + ((double)tid + 0.5) / (double)kLogTableSize);
        sm.ltab[tid] = make_double2(rc, -log(rc));
    }
    if (tid < min(nl, kTileRecs)) {
        sm.rec[tid] = spec;
        sm.sid[tid] = spec.sid;
    }
    for (int k = kTileRecs + tid; k < nl; k += kTileThreads) sm.sid[k] = __ldcg(&list[k].sid);   // dense tiles only
    __syncthreads();
    for (int k = tid; k < nl; k += kTileThreads) {
        const int mine = sm.sid[k];
        int r = 0;
        for (int m = 0; m < nl; ++m) r += sm.sid[m] < mine;
        sm.order[r] = (unsigned short)k;
    }
    __syncthreads();
    if (tid == 0) cnt[CHAINS ? (int)(chain_at_use() * P.X.tiles) + blockIdx.x : blockIdx.x] = 0;  // every thread has read the count: ready for the next evaluation's binning
    // record with the s-th smallest star id
    auto rec_at = [&](int s) -> PairRec {
        const int k = sm.order[s];
        return k < kTileRecs ? sm.rec[k] : ld_rec(&list[k]);
    };

    // ---- render Lambda = B + sum f PSF over the list, in list order
    double lam[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) lam[a][b] = P.F.B;
    for (int base = 0; base < nl; base += kTileChunk) {
        const int nc = min(kTileChunk, nl - base);
        for (int s = warp; s < nc; s += kWarps)
            build_pair_tab(P, rec_at(base + s), r0, c0, lane, sm.tab[s], sm.box[s], sm.rowd[s]);
        __syncthreads();
        // pairs whose box meets the 8 image rows of this warp (lane s tests pair s), visited in list order
        const int4 mybox = *reinterpret_cast<const int4*>(sm.box[lane & (kTileChunk - 1)]);
        unsigned hits = __ballot_sync(0xffffffffu, lane < nc && 8 * warp <= mybox.y && 8 * warp + 7 >= mybox.x);
        while (hits) {
            const int s = __ffs(hits) - 1;
            hits &= hits - 1;
            const int4 bx = *reinterpret_cast<const int4*>(sm.box[s]);   // (ia, ib, ja, jb)
            if (pr + 3 < bx.x || pr > bx.y || pc + 3 < bx.z || pc > bx.w) continue;
            // pr - (ia & ~1) in [-2, 32], even: inside the padded table, 16-byte aligned
            const double2* te = reinterpret_cast<const double2*>(&sm.tab[s].rowf[kTabPad + pr - (bx.x & ~1)]);
            const double2* tf = reinterpret_cast<const double2*>(&sm.tab[s].colf[kTabPad + pc - (bx.z & ~1)]);
            const double2 e01 = te[0], e23 = te[1], f01 = tf[0], f23 = tf[1];
            const double ex[4] = {e01.x, e01.y, e23.x, e23.y}, fy[4] = {f01.x, f01.y, f23.x, f23.y};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) lam[a][b] = fma(ex[a], fy[b], lam[a][b]);
        }
        if (base + kTileChunk < nl) __syncthreads();  // the tables are rewritten by the next chunk
    }

    if (MODE == 2) {
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int li = pr + a, lj = pc + b;
                if (li < vr && lj < vc)
                    Dout[(size_t)(r0 + li - P.row0) * P.C + c0 + lj] =
                        poisson_draw(lam[a][b], mock_seed, (unsigned long long)(r0 + li) * (unsigned long long)P.C + (unsigned long long)(c0 + lj));
            }
        return;
    }

    // ---- residual into the shared tile; pixel potential of the owned rows
    if (use_tma) mbar_wait(&sm.mbar, 0u);   // initialised by thread 0 before the barrier that follows the list sort
    else cp_async_wait_all();               // this thread's own copies (it reads nothing else here)
    double v = 0.0;
    if (!WANT_V && vr == kTile && vc == kTile) {
        // tile inside the image, gradient only: no per-pixel edge selects (a third of this phase's instructions)
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int li = pr + a;
            const double2 d0 = *reinterpret_cast<const double2*>(&sm.rho[li][pc]);
            const double2 d1 = *reinterpret_cast<const double2*>(&sm.rho[li][pc + 2]);
            double il[4];
            rcp4(lam[a], il);
            *reinterpret_cast<double2*>(&sm.rho[li][pc]) = make_double2(fma(d0.x, il[0], -1.0), fma(d0.y, il[1], -1.0));
            *reinterpret_cast<double2*>(&sm.rho[li][pc + 2]) = make_double2(fma(d1.x, il[2], -1.0), fma(d1.y, il[3], -1.0));
        }
    } else {
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int li = pr + a, gi = r0 + li;
            const bool own = WANT_V && li < vr && gi >= P.own_lo && gi < P.own_hi;
            const double2 d0 = *reinterpret_cast<const double2*>(&sm.rho[li][pc]);
            const double2 d1 = *reinterpret_cast<const double2*>(&sm.rho[li][pc + 2]);
            const double d[4] = {d0.x, d0.y, d1.x, d1.y};
            double rho[4], il[4];
            rcp4(lam[a], il);
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const bool in = li < vr && pc + b < vc;
                rho[b] = in ? fma(d[b], il[b], -1.0) : 0.0;
                if (WANT_V && own && pc + b < vc) v += lam[a][b] - d[b] * (lam[a][b] >= 2.3e-308 ? log_pos(lam[a][b], sm.ltab) : CUDART_NAN);  // ln of a non-positive model is NaN, as in NumPy
            }
            *reinterpret_cast<double2*>(&sm.rho[li][pc]) = make_double2(rho[0], rho[1]);
            *reinterpret_cast<double2*>(&sm.rho[li][pc + 2]) = make_double2(rho[2], rho[3]);
        }
    }
    if (WANT_V) {
        double a1[1] = {v};
        block_sum<1>(a1, sm.red);
        if (tid == 0) vpart[CHAINS ? chain_at_use() * P.X.vpart + blockIdx.x : blockIdx.x] = a1[0];
    }
    __syncthreads();

    // ---- gather: one warp per owned star of the list (sampler_RHMC.py:404-406 restricted to patch x tile);
    //      lanes own the columns of the box.  A single-chunk list still has its tables in shared memory; otherwise
    //      the warp rebuilds the pair's tables in its own slot.
    const bool keep = nl <= kTileChunk;
    for (int s = warp; s < nl; s += kWarps) {
        const PairRec rec = rec_at(s);
        if (rec.sid >= S.n_own) continue;  // ghosts are rendered only
        PairTab& T = sm.tab[keep ? s : warp];
        if (!keep) {
            __syncwarp();
            build_pair_tab(P, rec, r0, c0, lane, T, nullptr, sm.rowd[warp]);
            __syncwarp();
        }
        const int ia = rec.box & 63, ib = (rec.box >> 6) & 63, ja = (rec.box >> 12) & 63, jb = (rec.box >> 18) & 63;
        const double fy = T.colf[kTabPad + (ja & 1) + lane];     // f ey of this lane's column, 0 past the box
        const double dyl = T.dy0 + (double)lane;
        const double* col = &sm.rho[ia][min(ja + lane, kTile - 1)];
        const double* rf = &T.rowf[kTabPad + (ia & 1)];
        const double* rd = sm.rowd[keep ? s : warp];
        double a0 = 0.0, a1 = 0.0;
        const int nr = ib - ia + 1;
#pragma unroll 5
        for (int k = 0; k < nr; ++k) {   // two broadcast loads, one residual load, two DFMAs per row
            const double rho = col[k * kTile];
            a0 = fma(rho, rf[k], a0);
            a1 = fma(rho, rd[k], a1);
        }
        // three warp sums with six shuffles: fold the values onto lane groups first
        if (ja + lane > jb) a0 = a1 = 0.0;  // lanes past the box read a clamped column
        double sf = fy * a0, sx = fy * a1, sy = (fy * dyl) * a0, sz = 0.0;
        {
            const bool hi = lane & 16;
            const double k0 = hi ? sy : sf, k1 = hi ? sz : sx, t0 = hi ? sf : sy, t1 = hi ? sx : sz;
            const double x0 = k0 + __shfl_xor_sync(0xffffffffu, t0, 16), x1 = k1 + __shfl_xor_sync(0xffffffffu, t1, 16);
            const bool h8 = lane & 8;
            double yv = (h8 ? x1 : x0) + __shfl_xor_sync(0xffffffffu, h8 ? x0 : x1, 8);
            yv += __shfl_xor_sync(0xffffffffu, yv, 4);
            yv += __shfl_xor_sync(0xffffffffu, yv, 2);
            yv += __shfl_xor_sync(0xffffffffu, yv, 1);
            // lane 0: sum sf, lane 8: sum sx, lane 16: sum sy
            if ((lane & 7) == 0 && lane < 24)
                gpart[((size_t)(CHAINS ? rec.sid + chain_at_use() * P.X.M : rec.sid) * 4 + (rec.box >> 24)) * 3 + (lane >> 3)] = yv;
        }
    }
    // ---- pixel potential: the last tile to finish sums the per-tile partials in tile order -> scalars[0]
    if (WANT_V) {
        if (CHAINS) {
            const unsigned c = chain_at_use();
            ticket += c * 2;
            vpart += c * P.X.vpart;
            scalars += c * kScalars;
        }
        if (last_block_ticket(ticket, &sm.is_last)) {
            double w[1] = {0.0};
            for (int b = tid; b < (int)gridDim.x; b += kTileThreads) w[0] += __ldcg(vpart + b);
            block_sum<1>(w, sm.red);
            if (tid == 0) {
                scalars[0] = w[0];
                *ticket = 0u;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ FP32 gradient tile kernel
// The FP32 build of the tile evaluation (north_star: "<= 1e-4 in the FP32 build"): gradient-only evaluations (every
// leapfrog step but the last of a trajectory) read a float copy of the data window -- half the HBM bytes -- and do the
// render, the residual (MUFU.RCP) and the residual-weighted sums in float; star state, the tables' exponentials, the
// footprint sums and every evaluation that also returns the potential stay FP64, so the energies of the Metropolis test
// are exact for the state reached.  Same structure as big_tile_kernel<0> (one CTA per 64x64 tile, TMA tile load).
struct PairTabF {
    float rowf[kTabLen];
    float colf[kTabLen];
    float dx0, dy0;
};

struct TileSmemF {
    float rho[kTile][kTile];           // 16 KB, TMA destination
    PairTabF tab[kTileChunk];
    PairRec rec[kTileRecs];
    int sid[kTileMaxList];
    unsigned short order[kTileMaxList];
    int box[kTileChunk][4];
    unsigned long long mbar;
};

__device__ __forceinline__ void build_pair_tab_f(const BigParams& P, const PairRec& rec, int r0, int c0, int lane,
                                                 PairTabF& T, int* box) {
    const double f = rec.f, x = rec.x, y = rec.y;
    const int ia = rec.box & 63, ib = (rec.box >> 6) & 63, ja = (rec.box >> 12) & 63, jb = (rec.box >> 18) & 63;
    const double dx = ((double)(r0 + ia + lane) + 0.5) - x, dy = ((double)(c0 + ja + lane) + 0.5) - y;
    T.rowf[kTabPad + lane] = (ia + lane <= ib) ? (float)exp_neg(-(dx * dx) * P.inv2s2) : 0.0f;
    T.colf[kTabPad + lane] = (ja + lane <= jb) ? (float)(exp_neg(-(dy * dy) * P.inv2s2) * (P.norm * f)) : 0.0f;
    if (lane == 0) {
        T.dx0 = (float)dx;
        T.dy0 = (float)dy;
        if (box) {
            box[0] = ia; box[1] = ib; box[2] = ja; box[3] = jb;
        }
    }
}

__global__ void __launch_bounds__(kTileThreads, 5)
big_tile32_kernel(const BigParams P, const TileSrc S, int ntx, int* __restrict__ cnt, const PairRec* __restrict__ list,
                  double* __restrict__ gpart, int* fp_counters, const __grid_constant__ CUtensorMap tmapD32) {
    extern __shared__ __align__(128) unsigned char tile32_smem_raw[];
    TileSmemF& sm = *reinterpret_cast<TileSmemF*>(tile32_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = kTileThreads / 32;
    const int ti = blockIdx.x / ntx, tj = blockIdx.x % ntx;
    const int r0 = P.row0 + ti * kTile, c0 = tj * kTile;
    const int vr = min(kTile, P.row0 + P.nrows - r0), vc = min(kTile, P.C - c0);
    const int ty = tid >> 4, tx = tid & 15;
    const int pr = 4 * ty, pc = 4 * tx;
    if (tid == 0) {
        mbar_init(&sm.mbar, 1);
        mbar_expect_tx(&sm.mbar, kTile * kTile * 4);
        tma_load_2d(&sm.rho[0][0], &tmapD32, c0, r0 - P.row0, &sm.mbar);
    }
    list += (size_t)blockIdx.x * kTileMaxList;
    PairRec spec;
    spec.sid = 0; spec.box = 0; spec.f = spec.x = spec.y = 0.0;
    if (tid < kTileRecs) spec = ld_rec(&list[tid]);   // speculative: in flight together with the count
    const int nl = min(cnt[blockIdx.x], kTileMaxList);
    if (fp_counters && blockIdx.x == 0 && tid < 2) fp_counters[tid] = 0;
    for (int k = tid; k < kTileChunk * 4 * kTabPad; k += kTileThreads) {
        const int pair = k / (4 * kTabPad), e = k % (4 * kTabPad), side = e / kTabPad, g = e % kTabPad;
        float* t = (side & 1) ? sm.tab[pair].colf : sm.tab[pair].rowf;
        t[(side & 2) ? kTabPad + 32 + g : g] = 0.0f;
    }
    if (tid < min(nl, kTileRecs)) {
        sm.rec[tid] = spec;
        sm.sid[tid] = spec.sid;
    }
    for (int k = kTileRecs + tid; k < nl; k += kTileThreads) sm.sid[k] = __ldcg(&list[k].sid);
    __syncthreads();
    for (int k = tid; k < nl; k += kTileThreads) {
        const int mine = sm.sid[k];
        int r = 0;
        for (int m = 0; m < nl; ++m) r += sm.sid[m] < mine;
        sm.order[r] = (unsigned short)k;
    }
    __syncthreads();
    if (tid == 0) cnt[blockIdx.x] = 0;
    auto rec_at = [&](int s) -> PairRec {
        const int k = sm.order[s];
        return k < kTileRecs ? sm.rec[k] : ld_rec(&list[k]);
    };

    float lam[4][4];
    const float Bf = (float)P.F.B;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) lam[a][b] = Bf;
    for (int base = 0; base < nl; base += kTileChunk) {
        const int nc = min(kTileChunk, nl - base);
        for (int s = warp; s < nc; s += kWarps) build_pair_tab_f(P, rec_at(base + s), r0, c0, lane, sm.tab[s], sm.box[s]);
        __syncthreads();
        for (int s = 0; s < nc; ++s) {
            const int ia = sm.box[s][0], ja = sm.box[s][2];
            if (pr + 3 < ia || pr > sm.box[s][1] || pc + 3 < ja || pc > sm.box[s][3]) continue;
            const float* te = &sm.tab[s].rowf[kTabPad + pr - ia];
            const float* tf = &sm.tab[s].colf[kTabPad + pc - ja];
            const float ex[4] = {te[0], te[1], te[2], te[3]}, fy[4] = {tf[0], tf[1], tf[2], tf[3]};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) lam[a][b] = fmaf(ex[a], fy[b], lam[a][b]);
        }
        if (base + kTileChunk < nl) __syncthreads();
    }
    mbar_wait(&sm.mbar, 0u);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int li = pr + a;
        const float4 d4 = *reinterpret_cast<const float4*>(&sm.rho[li][pc]);
        const float d[4] = {d4.x, d4.y, d4.z, d4.w};
        float rho[4];
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            float rc;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(lam[a][b]));
            rho[b] = (li < vr && pc + b < vc) ? fmaf(d[b], rc, -1.0f) : 0.0f;
        }
        *reinterpret_cast<float4*>(&sm.rho[li][pc]) = make_float4(rho[0], rho[1], rho[2], rho[3]);
    }
    __syncthreads();
    const bool keep = nl <= kTileChunk;
    for (int s = warp; s < nl; s += kWarps) {
        const PairRec rec = rec_at(s);
        if (rec.sid >= S.n_own) continue;
        PairTabF& T = sm.tab[keep ? s : warp];
        if (!keep) {
            __syncwarp();
            build_pair_tab_f(P, rec, r0, c0, lane, T, nullptr);
            __syncwarp();
        }
        const int ia = rec.box & 63, ib = (rec.box >> 6) & 63, ja = rec.box >> 12 & 63, jb = (rec.box >> 18) & 63;
        const float fy = T.colf[kTabPad + lane];
        const float dyl = T.dy0 + (float)lane;
        const float* col = &sm.rho[ia][min(ja + lane, kTile - 1)];
        const float* rf = &T.rowf[kTabPad];
        float a0 = 0.0f, a1 = 0.0f, dxk = T.dx0;
        const int nr = ib - ia + 1;
#pragma unroll 4
        for (int k = 0; k < nr; ++k) {
            const float e = rf[k];
            const float rho = col[k * kTile];
            a0 = fmaf(rho, e, a0);
            a1 = fmaf(rho * e, dxk, a1);
            dxk += 1.0f;
        }
        if (ja + lane > jb) a0 = a1 = 0.0f;
        double sf = (double)fy * (double)a0, sx = (double)fy * (double)a1, sy = ((double)fy * (double)dyl) * (double)a0, sz = 0.0;
        {
            const bool hi = lane & 16;
            const double k0 = hi ? sy : sf, k1 = hi ? sz : sx, t0 = hi ? sf : sy, t1 = hi ? sx : sz;
            const double x0 = k0 + __shfl_xor_sync(0xffffffffu, t0, 16), x1 = k1 + __shfl_xor_sync(0xffffffffu, t1, 16);
            const bool h8 = lane & 8;
            double yv = (h8 ? x1 : x0) + __shfl_xor_sync(0xffffffffu, h8 ? x0 : x1, 8);
            yv += __shfl_xor_sync(0xffffffffu, yv, 4);
            yv += __shfl_xor_sync(0xffffffffu, yv, 2);
            yv += __shfl_xor_sync(0xffffffffu, yv, 1);
            if ((lane & 7) == 0 && lane < 24) gpart[((size_t)rec.sid * 4 + (rec.box >> 24)) * 3 + (lane >> 3)] = yv;
        }
    }
}

__global__ void big_to_float_kernel(const double* __restrict__ src, float* __restrict__ dst, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = (float)src[i];
}

// g = scaled sum of the footprint slots of star k, in slot order (sampler_RHMC.py:404-406)
__device__ __forceinline__ void gsum_star(const BigParams& P, int k, double f, double x, double y, const double* gpart,
                                          double& gf, double& gx, double& gy) {
    int i0, i1, j0, j1, mi, mj;
    bool clipped;
    double sf = 0.0, sx = 0.0, sy = 0.0;
    if (patch_of(P, x, y, i0, i1, j0, j1, mi, mj, clipped)) {
        const TileSpan t = tile_span(P, i0, i1, j0, j1);
        for (int ti = t.ti0; ti <= t.ti1; ++ti)
            for (int tj = t.tj0; tj <= t.tj1; ++tj) {
                const double* o = gpart + ((size_t)k * 4 + (ti - t.ti0) * 2 + (tj - t.tj0)) * 3;
                sf += __ldcg(o); sx += __ldcg(o + 1); sy += __ldcg(o + 2);
            }
    }
    // the tile kernel's sums carry the factor f (its column table is f ey)
    gf = -sf / f;
    gx = -sx * P.inv_s2;
    gy = -sy * P.inv_s2;
}

template <bool LIVE>
__global__ void big_gsum_kernel(const BigParams P, const double* q, int n_own, const double* gpart, double* g, const int* nd) {
    if (LIVE) n_own = *nd;
    q += blockIdx.y * 3 * P.X.M; g += blockIdx.y * 3 * P.X.M;
    gpart += blockIdx.y * 12 * P.X.M;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_own; k += gridDim.x * blockDim.x)
        gsum_star(P, k, q[3 * k], q[3 * k + 1], q[3 * k + 2], gpart, g[3 * k], g[3 * k + 1], g[3 * k + 2]);
}

}  // namespace
