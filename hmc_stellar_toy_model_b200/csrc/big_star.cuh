// Star-centric gradient evaluation of the large-field engine for SPARSE fields (BASELINE configs[4]: 1.5e-3 stars per pixel,
// ~12 (star, tile) pairs per 64x64 tile).  Reference: base_class.dVdq, sampler_RHMC.py:365-425, PSF truncated to the
// (2r+1)^2 patch -- the same patch-limited model as big_tile_kernel, which stays the evaluation that also returns the
// potential (one in `nsteps` evaluations), the dense-field path, the FP32 path and the mock-data generator.
//
// One WARP per owned star, no block barrier, no shared tile:
//   * lane c owns column j0 + c of the star's patch: its column of Lambda lives in registers (NR rows), its column of the data
//     goes global -> shared by 8-byte cp.async issued first (no registers held while the loads are in flight under everything
//     else: 16 warps per SM instead of 8 with the data in registers, which measured 1.4x slower than this);
//   * Lambda = B + own PSF + the PSF of every NEIGHBOUR whose patch meets this patch.  Neighbours come from the tile lists the
//     position update has just filled (pair records carry (f, x, y); ghosts of the neighbouring ranks are in the lists too): the
//     warp reads the first 32 records of the <= 2x2 tiles its patch touches -- one trip to L2, in flight together with the data
//     -- and a neighbour is taken from the ONE tile that holds the upper-left pixel of the two patches' intersection (a star
//     sits in the list of every tile it touches).  Neighbours are added in star-id order (repeated warp minimum), so the sum
//     does not depend on the order the atomics filled the lists: results stay bit-reproducible run to run;
//   * rho = D / Lambda - 1 (product-tree reciprocal) and the three residual-weighted sums of the star's own PSF over its own
//     patch, folded over the lanes with shuffles: the complete pixel gradient of the star, written to footprint slot 0 of
//     `gpart` (the other slots are zeroed), so big_kick_kernel / big_gsum_kernel consume it unchanged.
// Measured on 8192^2 / 1e5 stars (BASELINE configs[4], 3.6 neighbours per star): 331 us per gradient against 242 us for the
// tile kernel (ncu: 1850 warp-instructions per star -- 210 per neighbour pass, 220 for the copies' address arithmetic -- at
// IPC 2.1 with 16 warps per SM), i.e. C5 275 vs 352 M star-steps/s: every neighbour costs two warp-wide exponentials per
// STAR here and per TILE there.  The kernel therefore serves the fields the tile kernel is worst at -- few stars on a large
// image, where one CTA per tile still streams every pixel: the host picks it when the mean tile list holds fewer than ~1.5
// records (no neighbours to speak of, and only the patches are read from HBM), or when SRHMC_BIG_STAR=1.  Tiles with more
// than 32 records are handled by re-scanning the list in every pass (correct for any density, slow when lists are long).
#pragma once

namespace {

constexpr int kStarWarps = 4;

__device__ __forceinline__ double shfl_f64(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// pair record through the read-only path (the lists are not written while this kernel runs): the second read of a record
// -- the (f, x, y) of a neighbour once its turn has come -- then hits L1
__device__ __forceinline__ PairRec ldg_rec(const PairRec* p) {
    const int4 a = __ldg(reinterpret_cast<const int4*>(p));
    const double2 b = __ldg(reinterpret_cast<const double2*>(p) + 1);
    PairRec r;
    r.sid = a.x; r.box = a.y;
    r.f = __hiloint2double(a.w, a.z);
    r.x = b.x; r.y = b.y;
    return r;
}

template <int NR, bool LIVE>   // rows / columns of the largest patch: 2 rad + 1 <= NR <= 31; LIVE: the star count is *nd
__global__ void __launch_bounds__(32 * kStarWarps, 4)
big_star_kernel(const BigParams P, int n_own, const double* __restrict__ q, const double* __restrict__ D, int ntx,
                const int* __restrict__ cnt, const PairRec* __restrict__ list, double* __restrict__ gpart, int* fp_counters,
                const int* nd /* live stars (reversible-jump mode), or nullptr: n_own */) {
    __shared__ double s_d[kStarWarps][NR][32];  // data patch: lane c copies and reads column j0 + c only
    __shared__ double2 s_row[kStarWarps][32];   // own star: {ex, ex dx} of row i0 + r
    __shared__ double s_nex[kStarWarps][32];    // current neighbour: ex of row i0 + r (0 outside its patch)
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // the fixed-point iteration counters of the leapfrog step are free between its last reader and the next step
    if (fp_counters && blockIdx.x == 0 && threadIdx.x < 2) fp_counters[threadIdx.x] = 0;
    if (LIVE) n_own = *nd;
    for (int k = blockIdx.x * kStarWarps + warp; k < n_own; k += gridDim.x * kStarWarps) {
        const double f = q[3 * k], x = q[3 * k + 1], y = q[3 * k + 2];
        double* out = gpart + (size_t)k * 12;
        int i0, i1, j0, j1, mi, mj;
        bool clipped;
        if (!patch_of(P, x, y, i0, i1, j0, j1, mi, mj, clipped)) {   // flagged when the star was binned
            if (lane < 12) out[lane] = 0.0;
            continue;
        }
        const int nr = i1 - i0 + 1, nc = j1 - j0 + 1;
        const bool okc = lane < nc;
        // ---- this lane's column of the data: up to NR asynchronous 8-byte copies in flight (lanes past the patch copy its
        //      last column: finite values that meet a zero weight)
        const double* dp = D + (size_t)(i0 - P.row0) * P.C + j0 + min(lane, nc - 1);
        for (int r = 0; r < nr; ++r) cp_async8(&s_d[warp][r][lane], dp + (size_t)r * P.C);
        cp_async_commit();
        // ---- the first 32 records of the tiles this patch touches (speculative: in flight together with the counts)
        const TileSpan t = tile_span(P, i0, i1, j0, j1);
        const int ntj = t.tj1 - t.tj0 + 1, ntl = (t.ti1 - t.ti0 + 1) * ntj;   // 1, 2 or 4 tiles
        PairRec c[4];   // only the star ids stay live across the passes below
        int nT[4];
        const PairRec* lst[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const bool on = u < ntl;
            const int tile = on ? (t.ti0 + (ntj == 2 ? (u >> 1) : u)) * ntx + t.tj0 + (ntj == 2 ? (u & 1) : 0) : 0;
            lst[u] = list + (size_t)tile * kTileMaxList;
            nT[u] = on ? min(__ldg(cnt + tile), kTileMaxList) : 0;
            if (on) {
                c[u] = ldg_rec(lst[u] + lane);
            } else {
                c[u].sid = 0; c[u].box = 0; c[u].f = c[u].x = c[u].y = 0.0;
            }
        }
        // ---- own tables (same expressions as build_pair_tab) and Lambda = B + own PSF
        const double dx = ((double)(i0 + lane) + 0.5) - x, dy = ((double)(j0 + lane) + 0.5) - y;
        const double exl = (lane < nr) ? exp_neg(-(dx * dx) * P.inv2s2) : 0.0;
        const double fy = okc ? exp_neg(-(dy * dy) * P.inv2s2) * (P.norm * f) : 0.0;
        __syncwarp();   // the previous star's readers of the warp's tables are done
        s_row[warp][lane] = make_double2(exl, exl * dx);
        __syncwarp();
        double lam[NR];
#pragma unroll
        for (int r = 0; r < NR; ++r) lam[r] = fma(s_row[warp][r].x, fy, P.F.B);

        // ---- neighbours.  A record of tile u qualifies when it is another star whose patch meets this patch and the
        //      upper-left pixel of the intersection lies in tile u.
        auto qualifies = [&](const PairRec& rc, int u) -> bool {
            if (rc.sid == k) return false;
            int a0, a1, b0, b1, m0, m1;
            bool cl;
            if (!patch_of(P, rc.x, rc.y, a0, a1, b0, b1, m0, m1, cl)) return false;
            const int it = max(i0, a0), jt = max(j0, b0);
            if (it > min(i1, a1) || jt > min(j1, b1)) return false;
            const int ti = t.ti0 + (ntj == 2 ? (u >> 1) : u), tj = t.tj0 + (ntj == 2 ? (u & 1) : 0);
            return (it - P.row0) / kTile == ti && jt / kTile == tj;
        };
        int sid[4];     // star id of this lane's cached record of tile u, or "none" when it does not qualify
        bool dense = false;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            sid[u] = (lane < nT[u] && qualifies(c[u], u)) ? c[u].sid : 0x7fffffff;
            dense |= nT[u] > 32;
        }
        int last = -1;
        while (true) {
            // smallest qualifying star id above `last`: cached records first, then (long lists only) the rest of the lists
            int best = 0x7fffffff;
            const PairRec* bp = nullptr;
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (sid[u] > last && sid[u] < best) {
                    best = sid[u];
                    bp = lst[u] + lane;
                }
            if (dense) {
                for (int u = 0; u < ntl; ++u)
                    for (int base = 32; base < nT[u]; base += 32) {
                        if (base + lane >= nT[u]) continue;
                        const PairRec rc = ldg_rec(lst[u] + base + lane);
                        if (rc.sid > last && rc.sid < best && qualifies(rc, u)) {
                            best = rc.sid;
                            bp = lst[u] + base + lane;
                        }
                    }
            }
            const int m = __reduce_min_sync(FULL, best);
            if (m == 0x7fffffff) break;
            last = m;
            const int src = __ffs(__ballot_sync(FULL, best == m)) - 1;
            const unsigned long long pa = __shfl_sync(FULL, (unsigned long long)bp, src);
            const PairRec nb = ldg_rec(reinterpret_cast<const PairRec*>(pa));   // same address in every lane: one L1 hit
            const double nf = nb.f, nx = nb.x, ny = nb.y;
            int a0, a1, b0, b1, m0, m1;
            bool cl;
            patch_of(P, nx, ny, a0, a1, b0, b1, m0, m1, cl);
            const int gi = i0 + lane, gj = j0 + lane;
            const double ndx = ((double)gi + 0.5) - nx, ndy = ((double)gj + 0.5) - ny;
            const double nex = (lane < nr && gi >= a0 && gi <= a1) ? exp_neg(-(ndx * ndx) * P.inv2s2) : 0.0;
            const double nfy = (okc && gj >= b0 && gj <= b1) ? exp_neg(-(ndy * ndy) * P.inv2s2) * (P.norm * nf) : 0.0;
            __syncwarp();
            s_nex[warp][lane] = nex;
            __syncwarp();
#pragma unroll
            for (int r = 0; r < NR; ++r) lam[r] = fma(s_nex[warp][r], nfy, lam[r]);   // rows outside either patch add 0
        }

        // ---- residual and the three weighted sums of this star's PSF over its patch
        cp_async_wait_all();   // this lane reads only what it copied itself
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int r = 0; r + 3 < NR; r += 4) {
            if (r >= nr) break;
            const double a[4] = {lam[r], lam[r + 1], lam[r + 2], lam[r + 3]};
            double il[4];
            rcp4(a, il);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const double dv = (r + e < nr) ? s_d[warp][r + e][lane] : 0.0;   // rows past the patch were not copied
                const double rho = fma(dv, il[e], -1.0);
                const double2 w = s_row[warp][r + e];   // ... and carry zero weights
                s0 = fma(rho, w.x, s0);
                s1 = fma(rho, w.y, s1);
            }
        }
#pragma unroll
        for (int r = NR & ~3; r < NR; ++r) {
            if (r >= nr) break;
            const double rho = fma(s_d[warp][r][lane], rcp_fast(lam[r]), -1.0);
            const double2 w = s_row[warp][r];
            s0 = fma(rho, w.x, s0);
            s1 = fma(rho, w.y, s1);
        }
        // the sums carry the factor f of the column table, as the tile kernel's do (gsum_star divides it out)
        const double sf = warp_sum(fy * s0), sx = warp_sum(fy * s1), sy = warp_sum((fy * dy) * s0);
        if (lane < 12) out[lane] = lane == 0 ? sf : (lane == 1 ? sx : (lane == 2 ? sy : 0.0));
    }
}

}  // namespace
