// Peak finding on a large image (srhmc_big_find_peaks): lightsource_gym.find_peaks (samplers.py:129-254) with every
// potential and gradient of a seed taken over its (2r+1)^2 window (DESIGN.md §4.5).  Included by big_field.cu.
//
// Descent: one warp per seed, seeds in row-major grid order (neighbouring warps read neighbouring windows).  The warp
// keeps its window of the data image in shared memory, one column per lane, and re-stages it only when the seed moves to
// another pixel.  One pass per position yields V and the three gradient components through the separable tables, as
// peaks_kernel does on a whole small image:
//   Lambda_ij = B + f n ex_i ey_j,  rho = D/Lambda - 1,  c0_j = sum_i rho_ij ex_i,  c1_j = sum_i rho_ij ex_i dx_i,
//   g_f = -n sum_j ey_j c0_j,  g_x = -(f/s^2) n sum_j ey_j c1_j,  g_y = -(f/s^2) n sum_j ey_j dy_j c0_j,
//   V = -sum(D ln Lambda - Lambda).
// The reference's stop test |dV/V| < 1e-9 compares both potentials on the window of the NEW position: when a step changes
// the seed's pixel, V at the old position is evaluated once more on the new window.
//
// Merge: the greedy reduction (samplers.py:234-252) keeps alive seed i iff no earlier kept seed j conflicts with it,
// conflict = NOT(dist^2 > dr_tol^2 OR |mag_i - mag_j| > dmag_tol) (a NaN comparison is false, as in NumPy).  Alive seeds
// are binned into cells of side max(|dr_tol|, 1) px (cell indices clamped to the grid), so every conflicting pair lies
// in a 3x3 neighbourhood; seeds with a non-finite coordinate go to one extra list that every seed checks.  Rounds then
// decide seeds: removed if an earlier conflicting neighbour is kept, kept if every earlier conflicting neighbour is
// removed.  By induction on the seed index a decision equals the sequential one, and the earliest undecided seed is
// decided in every round.

constexpr int kSeedWarps = 8;

enum : unsigned char { kMergeOpen = 0, kMergeKept = 1, kMergeRemoved = 2, kMergeDead = 3 };

__global__ void __launch_bounds__(32 * kSeedWarps) big_seed_descent_kernel(const BigParams P, const double* __restrict__ D, int n,
                                                                           int nstep, double dt_f_coeff, double dt_xy_coeff,
                                                                           double f_lim, double* __restrict__ q,
                                                                           unsigned char* __restrict__ alive, int* __restrict__ steps) {
    extern __shared__ __align__(16) double seed_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wrows = 2 * P.rad + 1;
    double* win = seed_smem + (size_t)warp * (wrows * 32 + 64);  // [wrows][32]: lane j holds window column j
    double* tex = win + wrows * 32;                              // ex[32], ex*dx[32] of the window rows
    const int seed = blockIdx.x * kSeedWarps + warp;
    if (seed >= n) return;
    double f = q[3 * seed], x = q[3 * seed + 1], y = q[3 * seed + 2];
    int i0, i1, j0, j1, mi, mj;
    bool clipped;
    auto stage = [&]() {
        patch_of(P, x, y, i0, i1, j0, j1, mi, mj, clipped);   // world 1: local rows are global rows
        const int j = j0 + lane;
        if (j <= j1)
            for (int r = 0; r <= i1 - i0; ++r) win[r * 32 + lane] = D[(size_t)(i0 + r) * P.C + j];
    };
    // V and gradient of (pf, px, py) over the staged window; every lane gets the sums
    auto pass = [&](double pf, double px, double py, double& V, double& gf, double& gx, double& gy) {
        const int nrow = i1 - i0 + 1;
        __syncwarp();
        if (lane < nrow) {
            const double dx = ((double)(i0 + lane) + 0.5) - px;
            const double e = exp(-(dx * dx) * P.inv2s2);
            tex[lane] = e;
            tex[32 + lane] = e * dx;
        }
        __syncwarp();
        double sv = 0.0, sf = 0.0, sx = 0.0, sy = 0.0;
        const int j = j0 + lane;
        if (j <= j1) {
            const double dy = ((double)j + 0.5) - py;
            const double ey = exp(-(dy * dy) * P.inv2s2) * P.norm, fey = pf * ey;
            double c0 = 0.0, c1 = 0.0;
            for (int r = 0; r < nrow; ++r) {
                const double lam = fma(tex[r], fey, P.F.B);
                const double d = win[r * 32 + lane];
                const double rho = d / lam - 1.0;
                c0 = fma(rho, tex[r], c0);
                c1 = fma(rho, tex[32 + r], c1);
                sv += d * log(lam) - lam;
            }
            sf = ey * c0;
            sx = ey * c1;
            sy = ey * dy * c0;
        }
        V = -warp_sum(sv);
        gf = -warp_sum(sf);
        gx = -warp_sum(sx) * pf * P.inv_s2;
        gy = -warp_sum(sy) * pf * P.inv_s2;
    };

    stage();
    double V, gf, gx, gy;
    pass(f, x, y, V, gf, gx, gy);
    double V_prev = V;
    bool live = true;
    int it = 0;
    for (int i = 0; i < nstep; ++i) {
        const double dt_f = f * dt_f_coeff, dt_xy = dt_xy_coeff / f;  // samplers.py:207-208
        const double fo = f, xo = x, yo = y;
        f -= gf * dt_f;
        x -= gx * dt_xy;
        y -= gy * dt_xy;
        it = i + 1;
        if (f < f_lim) {  // faint: the seed disappears (samplers.py:215-217)
            live = false;
            break;
        }
        const int pmi = mi, pmj = mj;
        int ni0, ni1, nj0, nj1, nmi, nmj;
        patch_of(P, x, y, ni0, ni1, nj0, nj1, nmi, nmj, clipped);
        if (nmi != pmi || nmj != pmj) {
            stage();
            double g0, g1, g2;
            pass(fo, xo, yo, V_prev, g0, g1, g2);
        }
        pass(f, x, y, V, gf, gx, gy);
        if (fabs((V - V_prev) / V_prev) < 1e-9) break;
        V_prev = V;
    }
    if (lane == 0) {
        q[3 * seed] = f; q[3 * seed + 1] = x; q[3 * seed + 2] = y;
        alive[seed] = live ? 1 : 0;
        steps[seed] = it;
    }
}

__device__ __forceinline__ bool merge_wild(double x, double y) { return !isfinite(x) || !isfinite(y); }

// cell of a seed with finite coordinates, clamped to the grid
__device__ __forceinline__ int merge_cell_1d(double v, double inv_cell, int nc) {
    const double c = floor(v * inv_cell);
    return c > 0.0 ? (c > (double)(nc - 1) ? nc - 1 : (int)c) : 0;
}

// samplers.py:248-250 in NumPy's operation order (no contraction: the rounding is the host's)
__device__ __forceinline__ bool merge_conflict(const double* q, const double* mag, int i, int j, double dr2, double dmag_tol) {
    const double dx = __dsub_rn(q[3 * j + 1], q[3 * i + 1]), dy = __dsub_rn(q[3 * j + 2], q[3 * i + 2]);
    const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    return !(d2 > dr2 || fabs(__dsub_rn(mag[i], mag[j])) > dmag_tol);
}

// puts item i at (x, y) at the head of its cell's list (linked through `next`; head[ncx * ncy] is the non-finite list)
__device__ __forceinline__ void merge_cell_insert(int i, double x, double y, double inv_cell, int ncx, int ncy, int* head, int* next) {
    const int c = merge_wild(x, y) ? ncx * ncy : merge_cell_1d(x, inv_cell, ncx) * ncy + merge_cell_1d(y, inv_cell, ncy);
    next[i] = atomicExch(&head[c], i);
}

// magnitude, state and cell list of every seed
__global__ void big_merge_bin_kernel(int n, const double* q, const unsigned char* alive, double flux_to_count, double inv_cell,
                                     int ncx, int ncy, double* mag, int* head, int* next, unsigned char* state, int* n_open) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!alive[i]) {
        state[i] = kMergeDead;
        return;
    }
    // flux2mag (utils.py:27-28) of f / flux_to_count
    mag[i] = __dsub_rn(22.5, __dmul_rn(2.5, log10(q[3 * i] / flux_to_count)));
    merge_cell_insert(i, q[3 * i + 1], q[3 * i + 2], inv_cell, ncx, ncy, head, next);
    state[i] = kMergeOpen;
    atomicAdd(n_open, 1);
}

// one round: decisions from the previous round's states only (st_in -> st_out), so the round count is deterministic
__global__ void big_merge_round_kernel(int n, const double* q, const double* mag, const int* head, const int* next, double inv_cell,
                                       int ncx, int ncy, double dr2, double dmag_tol, const unsigned char* st_in,
                                       unsigned char* st_out, int* n_decided) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned char s = st_in[i];
    if (s != kMergeOpen) {
        st_out[i] = s;
        return;
    }
    bool any_kept = false, all_removed = true;
    auto visit = [&](int j) {
        if (j < i && merge_conflict(q, mag, i, j, dr2, dmag_tol)) {
            const unsigned char sj = st_in[j];
            any_kept |= sj == kMergeKept;
            all_removed &= sj == kMergeRemoved;
        }
    };
    const double x = q[3 * i + 1], y = q[3 * i + 2];
    if (merge_wild(x, y)) {
        for (int j = 0; j < i && !any_kept; ++j)
            if (st_in[j] != kMergeDead) visit(j);
    } else {
        const int cx = merge_cell_1d(x, inv_cell, ncx), cy = merge_cell_1d(y, inv_cell, ncy);
        for (int a = max(0, cx - 1); a <= min(ncx - 1, cx + 1) && !any_kept; ++a)
            for (int b = max(0, cy - 1); b <= min(ncy - 1, cy + 1) && !any_kept; ++b)
                for (int j = head[a * ncy + b]; j >= 0 && !any_kept; j = next[j]) visit(j);
        for (int j = head[ncx * ncy]; j >= 0 && !any_kept; j = next[j]) visit(j);
    }
    const unsigned char out = any_kept ? kMergeRemoved : (all_removed ? kMergeKept : kMergeOpen);
    st_out[i] = out;
    if (out != kMergeOpen) atomicAdd(n_decided, 1);
}

__global__ void big_merge_kept_kernel(int n, const unsigned char* state, unsigned char* kept, int* n_kept) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool k = state[i] == kMergeKept;
    kept[i] = k ? 1 : 0;
    if (k) atomicAdd(n_kept, 1);
}
