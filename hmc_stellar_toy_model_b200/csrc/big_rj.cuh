// Reversible-jump chains of the large-field engine (srhmc_big_rj_configure; phases SRHMC_BIG_RJ_BEGIN, RJ_JUMP, RJ_ACCEPT):
// multi_gym.run_RHMC with birth/death and split/merge moves on one field of any size, the star count on the device.
//
// The stars are stored in table order (storage index = table index), so the table edits follow np.delete / np.vstack and
// the Philox momentum of star k is keyed by k, as in field_rj.cuh.  The live count N sits in BigRj::N; every per-star kernel
// of an iteration reads its count from BigRj (N, or n1 / n2 for the step phases of leg 1 / leg 2) and is launched for
// max_stars, so one captured graph serves every N.  A leg the device skips (leg 2 of a within-model iteration, both legs of
// a refused jump) sees the count 0: its per-star kernels do nothing and its evaluations render an empty star list.  The
// pixel potential those evaluations leave is replaced at the accept phase by the one of the leg that ran.
#pragma once
#include <climits>

#include "rj_moves.cuh"

namespace {

struct BigRj {
    int N;               // live stars
    int n1, n2;          // the stars the step phases of leg 1 / leg 2 see: N, or 0 when the device skips the leg
    int N0;              // N at the iteration's start
    int code, status;    // move code (rj_move_code) and RjStatus of the iteration
    int jumped;          // the table was edited: leg 2 runs and p is negated after it
    int d0, d1, par;     // removed rows (-1: none) and split parent
    int n_new;           // N after the edit
    int overflow;        // first iteration whose proposal needed more than max_stars stars, -1 if none
    double lr;           // log ratio of the proposal
    double V1;           // pixel potential after leg 1
    double Vend;         // pixel potential at the end of the iteration's trajectory
    double rowA[6];      // proposed row (q, p): the split's child one
    double rowB[6];      // proposed row: the newborn, the split's child two or the merged star
    double rec[kRjDraws];
};

constexpr int kRjThreads = 1024;   // the one-block proposal kernel
constexpr int kRjNb = 48;          // nonzero-weight merge partners of a row sorted in registers; more take the selection pass

// Merge cells: exp(-s^2 / (2 K^2)) is exactly 0.0 in double once s^2 / (2 K^2) exceeds ~745.13, so every pair of nonzero
// weight lies closer than K sqrt(2 * 746) and within the 3 x 3 cells around either star (cells of that side, widened by one
// part in 1e12 against the rounding of the cell index).
inline double rj_merge_cell(double K) { return K * std::sqrt(2.0 * 746.0) * (1.0 + 1e-12); }

// Calls f(j, w) for every star j with a nonzero merge weight w = w(i, j), in ascending j, until f returns false.
template <typename F>
__device__ void merge_row_visit(const RjParams& R, const double* q, int i, double inv_cell, int ncx, int ncy, const int* head,
                                const int* next, F f) {
    const double xi = q[3 * i + 1], yi = q[3 * i + 2];
    const int cx = merge_cell_1d(xi, inv_cell, ncx), cy = merge_cell_1d(yi, inv_cell, ncy);
    auto w_of = [&](int j) { return merge_weight_of(R, q + 3 * i, q + 3 * j); };
    int js[kRjNb];
    int m = 0;
    bool full = false;
    for (int a = max(0, cx - 1); a <= min(ncx - 1, cx + 1); ++a)
        for (int b = max(0, cy - 1); b <= min(ncy - 1, cy + 1); ++b)
            for (int j = head[a * ncy + b]; j >= 0; j = next[j])
                if (w_of(j) != 0.0) {
                    if (m < kRjNb) js[m++] = j;
                    else full = true;
                }
    if (!full) {
        for (int t = 1; t < m; ++t) {
            const int v = js[t];
            int u = t;
            for (; u > 0 && js[u - 1] > v; --u) js[u] = js[u - 1];
            js[u] = v;
        }
        for (int t = 0; t < m; ++t)
            if (!f(js[t], w_of(js[t]))) return;
        return;
    }
    for (int last = -1;;) {   // a row with more partners than the register list: select them in ascending order
        int best = INT_MAX;
        for (int a = max(0, cx - 1); a <= min(ncx - 1, cx + 1); ++a)
            for (int b = max(0, cy - 1); b <= min(ncy - 1, cy + 1); ++b)
                for (int j = head[a * ncy + b]; j >= 0; j = next[j])
                    if (j > last && j < best && w_of(j) != 0.0) best = j;
        if (best == INT_MAX || !f(best, w_of(best))) return;
        last = best;
    }
}

// The iteration's draw record, move and refusals that depend on N alone; N_chain / move_chain rows
__global__ void big_rj_begin_kernel(const RjParams R, BigRj* st, int max_stars, unsigned long long seed, int iter_host,
                                    const int* iter_dev, int* N_chain, unsigned char* move_chain) {
    if (threadIdx.x || blockIdx.x) return;
    const int iter = iter_dev ? *iter_dev : iter_host;
    double* rec = st->rec;
    if (R.draws) {
        for (int i = 0; i < kRjDraws; ++i) rec[i] = R.draws[(size_t)iter * kRjDraws + i];
    } else {
        rj_record(seed, 0u, (uint32_t)iter, R.beta_a, R.beta_b, rec);
    }
    const int code = rj_move_code(R, rec), n = st->N;
    int status = RJ_OK;
    if ((code == 1 || code == 3) && n + 1 > max_stars) status = RJ_OVERFLOW;
    if ((code == 2 || code == 3) && n == 0) status = RJ_REFUSED;
    if (code == 4 && n < 2) status = RJ_REFUSED;
    if (status == RJ_OVERFLOW && st->overflow < 0) st->overflow = iter;
    st->code = code;
    st->status = status;
    st->N0 = n;
    st->jumped = 0;
    st->n1 = status == RJ_OK ? n : 0;
    st->n2 = 0;
    if (N_chain) N_chain[iter] = n;
    if (move_chain) move_chain[iter] = (unsigned char)code;
}

// merge: the cell lists of the table (head reset to -1 by the host)
__global__ void big_rj_merge_bin_kernel(const BigRj* st, const double* q, double inv_cell, int ncx, int ncy, int* head, int* next) {
    if (st->status != RJ_OK || st->code != 4) return;
    const int n = st->N;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        merge_cell_insert(i, q[3 * i + 1], q[3 * i + 2], inv_cell, ncx, ncy, head, next);
}

// merge: rowsum[i] = sum over j ascending of w(i, j) -- the dense row's sum, its zero terms being exact no-ops.  A star with a
// non-finite position makes every row NaN, as it makes the dense weights NaN.
__global__ void big_rj_merge_rows_kernel(const RjParams R, const BigRj* st, const double* q, double inv_cell, int ncx, int ncy,
                                         const int* head, const int* next, double* rowsum) {
    if (st->status != RJ_OK || st->code != 4) return;
    const int n = st->N;
    const bool wild = head[ncx * ncy] >= 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        double s = 0.0;
        if (wild) {
            s = CUDART_NAN;
        } else {
            merge_row_visit(R, q, i, inv_cell, ncx, ncy, head, next, [&](int, double w) {
                s += w;
                return true;
            });
        }
        rowsum[i] = s;
    }
}

// One block: keeps the pixel potential of leg 1, and on a jump picks the merge pair (fixed-order scan of the row sums: thread t
// sums rows [t m, (t + 1) m), thread 0 the thread sums in order, then the first flat index i n + j whose cumulative weight
// exceeds u W) and computes the proposal: its rows, log ratio, removed rows and new count.
__global__ void __launch_bounds__(kRjThreads) big_rj_propose_kernel(const BigParams P, const RjParams R, double g_ff2, BigRj* st,
                                                                    const double* q, const double* p, const double* rowsum,
                                                                    const double* scalars, double inv_cell, int ncx, int ncy,
                                                                    const int* head, const int* next) {
    __shared__ double part[kRjThreads];
    const int tid = threadIdx.x;
    if (tid == 0) st->V1 = scalars[0];
    const int code = st->code;
    if (st->status != RJ_OK || code == 0) return;
    const int n = st->N;
    const double* rec = st->rec;
    int d0 = -1, d1 = -1;
    if (code == 4) {
        const int m = (n + kRjThreads - 1) / kRjThreads;
        double s = 0.0;
        for (int i = tid * m; i < min(n, (tid + 1) * m); ++i) s += rowsum[i];
        part[tid] = s;
        __syncthreads();
        if (tid) return;
        double W = 0.0;
        for (int t = 0; t < kRjThreads; ++t) W += part[t];
        if (W > 0.0 && isfinite(W)) {
            const double target = rec[2] * W;
            double cum = 0.0;
            int row = -1;
            for (int t = 0; t < kRjThreads && row < 0; ++t) {
                if (!(cum + part[t] > target) && t < kRjThreads - 1) {
                    cum += part[t];
                    continue;
                }
                for (int i = t * m; i < min(n, (t + 1) * m); ++i) {
                    if (cum + rowsum[i] > target) {
                        row = i;
                        break;
                    }
                    cum += rowsum[i];
                }
            }
            // the running sum fell short of u W by rounding: the last row of nonzero weight, and in it the last pair
            const double target_row = row >= 0 ? target : CUDART_INF;
            if (row < 0)
                for (row = n - 1; row >= 0 && !(rowsum[row] > 0.0); --row) {}
            if (row >= 0) {
                int pick = -1, last = -1;
                merge_row_visit(R, q, row, inv_cell, ncx, ncy, head, next, [&](int j, double w) {
                    last = j;
                    cum += w;
                    if (cum > target_row) {
                        pick = j;
                        return false;
                    }
                    return true;
                });
                d0 = row;
                d1 = pick >= 0 ? pick : last;
            }
        }
        if (d1 < 0) {   // all weights zero, or not finite
            st->status = RJ_REFUSED;
            return;
        }
    } else if (tid) {
        return;
    }
    // thread 0: the proposal (rj_moves.cuh), as rj_propose of field_rj.cuh
    double* rowA = st->rowA;
    double* rowB = st->rowB;
    const double K = R.K_split, k2 = K * K, kernel_norm = log(2.0 * CUDART_PI * k2);
    double lr = 0.0;
    int par = -1;
    if (code == 1) {
        rj_newborn(R, P.Rg, P.C, P.F.alpha, rec, rowB);
        draw_momentum(P.F, g_ff2, rowB, rec + 8, rowB + 3);
        lr = rj_lr_birth(P.F, rowB[0], star_T(P.F, g_ff2, rowB, rowB + 3));
    } else if (code == 2) {
        d0 = rj_index(rec, n);
        lr = rj_lr_death(P.F, q[3 * d0], star_T(P.F, g_ff2, q + 3 * d0, p + 3 * d0));
    } else if (code == 3) {
        par = rj_index(rec, n);
        const double off_r = rec[5] * K, off_c = rec[6] * K, share = rec[7];
        rj_children(q[3 * par], q[3 * par + 1], q[3 * par + 2], off_r, off_c, share, rowA, rowB);
        draw_momentum(P.F, g_ff2, rowA, rec + 8, rowA + 3);
        draw_momentum(P.F, g_ff2, rowB, rec + 11, rowB + 3);
        lr = rj_lr_split(R, kernel_norm, q[3 * par], share, off_r, off_c, pair_T(P.F, g_ff2, rowA, rowA + 3, rowB, rowB + 3),
                         star_T(P.F, g_ff2, q + 3 * par, p + 3 * par));
    } else {
        const double* a = q + 3 * d0;
        const double* b = q + 3 * d1;
        const double share = a[0] / (a[0] + b[0]);
        const double gap2 = (a[1] - b[1]) * (a[1] - b[1]) + (a[2] - b[2]) * (a[2] - b[2]);
        rj_merged(a, b, share, rowB);
        const double T_pair = pair_T(P.F, g_ff2, a, p + 3 * d0, b, p + 3 * d1);
        draw_momentum(P.F, g_ff2, rowB, rec + 8, rowB + 3);
        lr = rj_lr_merge(R, kernel_norm, rowB[0], share, gap2, T_pair, star_T(P.F, g_ff2, rowB, rowB + 3));
    }
    const int n_new = (code == 1 || code == 3) ? n + 1 : n - 1;   // a merge removes two rows and appends one
    st->lr = lr;
    st->d0 = d0;
    st->d1 = d1;
    st->par = par;
    st->n_new = n_new;
    st->n2 = n_new;
    st->jumped = 1;
}

// The edited table into (qn, pn): the kept rows in order (np.delete) with p negated, the split parent replaced by child one,
// the appended row last (np.vstack)
__global__ void big_rj_edit_kernel(const BigRj* st, const double* q, const double* p, double* qn, double* pn) {
    if (!st->jumped) return;
    const int code = st->code, n = st->N, n_new = st->n_new, par = st->par;
    const int lo = st->d1 < 0 ? st->d0 : min(st->d0, st->d1), hi = st->d1 < 0 ? -1 : max(st->d0, st->d1);
    const int n_kept = code == 2 ? n - 1 : (code == 4 ? n - 2 : n);
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_new; k += gridDim.x * blockDim.x) {
        if (k >= n_kept || (code == 3 && k == par)) {
            const double* r = k >= n_kept ? st->rowB : st->rowA;
            for (int c = 0; c < 3; ++c) {
                qn[3 * k + c] = r[c];
                pn[3 * k + c] = r[3 + c];
            }
            continue;
        }
        int src = k;
        if (lo >= 0 && src >= lo) ++src;
        if (hi >= 0 && src >= hi) ++src;
        for (int c = 0; c < 3; ++c) {
            qn[3 * k + c] = q[3 * src + c];
            pn[3 * k + c] = -p[3 * src + c];
        }
    }
}

__global__ void big_rj_commit_kernel(BigRj* st, const double* qn, const double* pn, double* q, double* p) {
    if (!st->jumped) return;
    const int n_new = st->n_new;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * n_new; i += gridDim.x * blockDim.x) {
        q[i] = qn[i];
        p[i] = pn[i];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) st->N = n_new;
}

// Metropolis test: ln u < -dE for a within-model iteration (big_accept_kernel's), ln u < -dE + log_ratio for a jump; a refused
// jump is rejected.  Rejection restores q and g of the iteration's start (its N0 rows); an accepted jump negates p again.
__global__ void big_rj_accept_kernel(BigRj* st, const double* scalars, double* state, unsigned long long seed, int iter_host,
                                     const int* iter_dev, const double* lnu_in, double* q, double* p, double* g, const double* q0,
                                     const double* g0, unsigned char* A_chain) {
    const int iter = iter_dev ? *iter_dev : iter_host;
    const int code = st->code, jumped = st->jumped;
    const double Vpix = jumped ? scalars[0] : st->V1;
    const double V = (scalars[2] > 0.0) ? CUDART_INF : Vpix + scalars[3];
    const double dE = (V + scalars[1]) - state[0];
    const double lnu = lnu_in ? lnu_in[iter] : philox_lnu(seed, 0u, (uint32_t)iter);
    bool accept = false;
    if (st->status == RJ_OK) {
        if (code == 0) {
            accept = (dE < 0.0) || (lnu < -dE);
        } else {
            const double ln_alpha = -dE + st->lr;
            accept = (ln_alpha > 0.0) || (lnu < ln_alpha);
        }
    }
    if (!accept) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * st->N0; i += gridDim.x * blockDim.x) {
            q[i] = q0[i];
            g[i] = g0[i];
        }
    } else if (jumped) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * st->n_new; i += gridDim.x * blockDim.x) p[i] = -p[i];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (A_chain) A_chain[iter] = accept ? 1 : 0;
        state[2] = accept ? 1.0 : 0.0;
        state[3] += accept ? 1.0 : 0.0;
        st->Vend = Vpix;
    }
}

// after every block of big_rj_accept_kernel: the pixel potential and N of the state the chain continues from
__global__ void big_rj_finish_kernel(BigRj* st, double* scalars, const double* state, int* iter_dev) {
    if (state[2] != 0.0) {
        scalars[0] = st->Vend;
    } else {
        scalars[0] = state[1];
        st->N = st->N0;
    }
    if (iter_dev) *iter_dev += 1;
}

}  // namespace
