// Reversible-jump chains of the CTA-per-field kernel (field_kernel MODE_RUN_RJ): multi_gym.run_RHMC with
// P_move[1:] != 0 (drop-in sampler_RHMC.py _run_RHMC_rj, birth_death_move, split_merge_move; reference
// sampler_RHMC.py:1009-1198, 1200-1445), every iteration of F fields inside one launch.
//
// Iteration l: schedules, momentum refresh and E0 exactly as MODE_RUN; the move comes from u_move (np.random.choice's
// rule).  Move 0 is a MODE_RUN iteration.  A jump runs leg 1 (nsteps leapfrog steps), p = -p, edits the star table,
// re-evaluates the pixel gradient at the edited q, runs leg 2, p = -p, and accepts when ln u < -dE + log_ratio; a rejection
// restores q, the pixel gradient, V and N of the iteration's start.  Table order follows np.delete / np.vstack: a death or
// a merge removes rows keeping the order of the others, a newborn, a second child or a merged star is appended last.
//
// The one deliberate difference from the reference: where it raises (a death or a split with no star, a merge with fewer
// than two stars or all pair weights zero, a proposal needing more than Nmax stars) the jump is rejected with the state
// unchanged; the first iteration whose proposal needed more than Nmax stars is reported in RjParams.overflow.
#pragma once
#include "rj_moves.cuh"

namespace srhmc {

// c.red slots above the ones block_sum (<= 5 values: red[0, 160)) and fp_count_slots (red[224]) use
constexpr int kRjRec = 192;               // the iteration's draw record, kRjDraws doubles
constexpr int kRjBc = kRjRec + kRjDraws;  // proposal broadcast: [0] merge pick, [1] log ratio, [2..7] row A, [8..13] row B
constexpr int kRjStart = kRjBc + 14;      // E0, V and N of the iteration's start (3 doubles, red[220, 223))
static_assert(kRjStart + 3 <= 224, "the reversible-jump slots must stay below fp_count_slots");

// Merge weight of the ordered pair (i, j) of the table (merge_weight_of, rj_moves.cuh)
template <typename T>
__device__ __forceinline__ double merge_weight(const Ctx<T>& c, const RjParams& R, int i, int j) {
    return merge_weight_of(R, c.q + 3 * i, c.q + 3 * j);
}

// Removes rows d0 and d1 (-1: none) of q and p keeping the order of the others (np.delete).  Rows only move down, so a
// pass over nt rows reads before any of its writes and writes below every row a later pass reads.
template <typename T>
__device__ void remove_rows(const Ctx<T>& c, int n, int d0, int d1) {
    for (int base = 0; base < n; base += blockDim.x) {
        const int k = base + threadIdx.x;
        int dst = -1;
        double qv[3], pv[3];
        if (k < n && k != d0 && k != d1) {
            dst = k - (d0 >= 0 && k > d0) - (d1 >= 0 && k > d1);
            for (int i = 0; i < 3; ++i) {
                qv[i] = c.q[3 * k + i];
                pv[i] = c.p[3 * k + i];
            }
        }
        __syncthreads();
        if (dst >= 0 && dst != k)
            for (int i = 0; i < 3; ++i) {
                c.q[3 * dst + i] = qv[i];
                c.p[3 * dst + i] = pv[i];
            }
        __syncthreads();
    }
}

// The proposal of jump `code` (1 birth, 2 death, 3 split, 4 merge) on the table q, p of n stars after leg 1 (p already
// negated).  Returns the new star count, with the table holding the proposed stars and red[kRjBc + 1] the proposal's log
// ratio, or -RJ_REFUSED with the table untouched.  All threads of the CTA call it.  Out of line, and given plain pointers
// rather than the kernel's Ctx: it runs once per jump, and either inlining it or taking the Ctx's address would push the
// leapfrog loop around it into local memory.
static __device__ __noinline__ int rj_propose(const FieldParams& P, double* q, double* p, double* red, int n, double g_ff2,
                                       const RjParams& R, int code, const double* rec, double* part) {
    Ctx<double> c;  // the fields the helpers below read
    c.P = &P;
    c.q = q;
    c.p = p;
    c.red = red;
    c.N = n;
    c.g_ff2 = g_ff2;
    const int tid = threadIdx.x, nt = blockDim.x;
    double* bc = c.red + kRjBc;
    int d0 = -1, d1 = -1;
    if (code == 2) d0 = rj_index(rec, n);
    if (code == 4) {
        // weights of all n^2 ordered pairs: thread t sums the flat indices [t m, (t + 1) m) in order, thread 0 adds the
        // partial sums in thread order and picks the first flat index i n + j whose cumulative weight exceeds u W
        const int np = n * n, m = (np + nt - 1) / nt;
        double s = 0.0;
        for (int f = tid * m; f < min(np, (tid + 1) * m); ++f) s += merge_weight(c, R, f / n, f % n);
        part[tid] = s;
        __syncthreads();
        if (tid == 0) {
            double W = 0.0;
            for (int t = 0; t < nt; ++t) W += part[t];
            int pick = -1;
            if (W > 0.0 && isfinite(W)) {
                const double target = rec[2] * W;
                double cum = 0.0;
                int last = -1;
                for (int t = 0; t < nt && pick < 0; ++t) {
                    if (!(cum + part[t] > target) && t < nt - 1) {
                        cum += part[t];
                        continue;
                    }
                    for (int f = t * m; f < min(np, (t + 1) * m); ++f) {
                        const double w = merge_weight(c, R, f / n, f % n);
                        if (w > 0.0) last = f;
                        cum += w;
                        if (cum > target) {
                            pick = f;
                            break;
                        }
                    }
                }
                if (pick < 0) pick = last;  // the running sum fell short of u W by rounding: the last pair of nonzero weight
            }
            bc[0] = (double)pick;
        }
        __syncthreads();
        const int pick = (int)bc[0];
        if (pick < 0) return -RJ_REFUSED;
        d0 = pick / n;
        d1 = pick % n;
    }
    const double K = R.K_split, k2 = K * K, kernel_norm = log(2.0 * CUDART_PI * k2);
    double* rowA = bc + 2;
    double* rowB = bc + 8;
    if (tid == 0) {
        double lr = 0.0;
        if (code == 1) {
            // newborn: row, column and flux from the prior, momentum from H of the newborn
            rj_newborn(R, P.R, P.C, P.alpha, rec, rowB);
            draw_momentum(P, g_ff2, rowB, rec + 8, rowB + 3);
            lr = rj_lr_birth(P, rowB[0], star_T(P, g_ff2, rowB, rowB + 3));
        } else if (code == 2) {
            lr = rj_lr_death(P, c.q[3 * d0], star_T(P, g_ff2, c.q + 3 * d0, c.p + 3 * d0));
        } else if (code == 3) {
            // the parent becomes child one in place, child two is appended
            const int par = rj_index(rec, n);
            const double fp = c.q[3 * par], rp = c.q[3 * par + 1], cp = c.q[3 * par + 2];
            const double off_r = rec[5] * K, off_c = rec[6] * K, share = rec[7];
            rj_children(fp, rp, cp, off_r, off_c, share, rowA, rowB);
            draw_momentum(P, g_ff2, rowA, rec + 8, rowA + 3);
            draw_momentum(P, g_ff2, rowB, rec + 11, rowB + 3);
            lr = rj_lr_split(R, kernel_norm, fp, share, off_r, off_c, pair_T(P, g_ff2, rowA, rowA + 3, rowB, rowB + 3),
                             star_T(P, g_ff2, c.q + 3 * par, c.p + 3 * par));
            bc[0] = (double)par;
        } else {
            // merge of the ordered pair (one, two): the merged star uses the share f_one / (f_one + f_two)
            const double* a = c.q + 3 * d0;
            const double* b = c.q + 3 * d1;
            const double share = a[0] / (a[0] + b[0]);
            const double gap2 = (a[1] - b[1]) * (a[1] - b[1]) + (a[2] - b[2]) * (a[2] - b[2]);
            rj_merged(a, b, share, rowB);
            const double T_pair = pair_T(P, g_ff2, a, c.p + 3 * d0, b, c.p + 3 * d1);
            draw_momentum(P, g_ff2, rowB, rec + 8, rowB + 3);
            lr = rj_lr_merge(R, kernel_norm, rowB[0], share, gap2, T_pair, star_T(P, g_ff2, rowB, rowB + 3));
        }
        bc[1] = lr;
    }
    __syncthreads();
    if (d0 >= 0) remove_rows(c, n, d0, d1);
    const int n_new = (code == 1 || code == 3) ? n + 1 : n - 1;
    if (tid == 0) {
        if (code == 3) {
            const int par = (int)bc[0];
            for (int i = 0; i < 3; ++i) {
                c.q[3 * par + i] = rowA[i];
                c.p[3 * par + i] = rowA[3 + i];
            }
        }
        if (code != 2)
            for (int i = 0; i < 3; ++i) {
                c.q[3 * (n_new - 1) + i] = rowB[i];
                c.p[3 * (n_new - 1) + i] = rowB[3 + i];
            }
    }
    __syncthreads();
    return n_new;
}

template <typename T, int MR, int MC, int KV3>
__device__ void run_rj_field(Ctx<T>& c, const LaunchArgs& A, double* scratch, int field) {
    const FieldParams& P = *c.P;
    const RjParams& R = *reinterpret_cast<const RjParams*>(scratch);
    const int tid = threadIdx.x, nt = blockDim.x, S = 3 * P.Nmax;
    double* qs = scratch + kRjHeaderDoubles + (size_t)field * R.field_stride;  // q, pixel gradient at the iteration's start
    double* gs = qs + S;
    double* part = gs + S;  // merge weights: one partial sum per thread
    double* rec = c.red + kRjRec;
    // E0, V and N at the iteration's start: kept in shared memory over the legs, out of the registers the leapfrog needs
    double* st = c.red + kRjStart;
    const size_t rows = (size_t)A.n_rows;
    const int L = A.niter + 1;
    const uint32_t fid = A.philox_field(field);
    double Vpix = eval_pixels<T, MR, MC, KV3>(c, true);
    int n_acc = 0, overflow = -1;
    for (int l = 0; l < L; ++l) {
        if (A.gff2_sched && l < A.n_gff2) c.g_ff2 = A.gff2_sched[l];
        if (A.beta_sched && l < A.n_beta) c.beta = A.beta_sched[l];
        for (int k = tid; k < c.N; k += nt) {
            const Metric m = metric_of(P, c.q[3 * k], c.g_ff2);
            double z[3];
            if (A.normals) {
                const double* zp = A.normals + ((size_t)field * L + l) * S + 3 * k;
                z[0] = zp[0]; z[1] = zp[1]; z[2] = zp[2];
            } else {
                philox_normals3(A.seed, fid, (uint32_t)l, (uint32_t)k, z);
            }
            c.p[3 * k] = z[0] * sqrt(m.Hff);
            c.p[3 * k + 1] = z[1] * sqrt(m.Hxx);
            c.p[3 * k + 2] = z[2] * sqrt(m.Hxx);
            qs[3 * k] = c.q[3 * k]; qs[3 * k + 1] = c.q[3 * k + 1]; qs[3 * k + 2] = c.q[3 * k + 2];
            gs[3 * k] = c.g[3 * k]; gs[3 * k + 1] = c.g[3 * k + 1]; gs[3 * k + 2] = c.g[3 * k + 2];
        }
        if (tid == 0) {
            if (R.draws) {
                const double* dp = R.draws + ((size_t)field * L + l) * kRjDraws;
                for (int i = 0; i < kRjDraws; ++i) rec[i] = dp[i];
            } else {
                rj_record(A.seed, fid, (uint32_t)l, R.beta_a, R.beta_b, rec);
            }
        }
        __syncthreads();
        const Energies e0 = energies(c, Vpix, A.f_pos, true);
        const bool keep = (l % A.chain_stride) == 0;
        const int code = rj_move_code(R, rec);
        if (tid == 0) {
            st[0] = e0.V + e0.T;
            st[1] = Vpix;
            st[2] = (double)c.N;
        }
        if (keep) {
            const size_t row = (size_t)field * rows + (size_t)(l / A.chain_stride);
            if (A.q_chain)
                for (int i = tid; i < 3 * c.N; i += nt) A.q_chain[row * S + i] = c.q[i];
            if (A.p_chain)
                for (int i = tid; i < 3 * c.N; i += nt) A.p_chain[row * S + i] = c.p[i];
            if (tid == 0) {
                if (A.E_chain) A.E_chain[row] = e0.V + e0.T;
                if (A.V_chain) A.V_chain[row] = e0.V;
                if (A.T_chain) A.T_chain[row] = e0.T;
                if (R.N_chain) R.N_chain[row] = c.N;
                if (R.move_chain) R.move_chain[row] = (unsigned char)code;
            }
        }
        __syncthreads();
        // refusals that depend on the star count alone are known before leg 1
        int status = RJ_OK;
        if ((code == 1 || code == 3) && c.N + 1 > P.Nmax) status = RJ_OVERFLOW;
        if ((code == 2 || code == 3) && c.N == 0) status = RJ_REFUSED;
        if (code == 4 && c.N < 2) status = RJ_REFUSED;
        // one leg for move 0, two around the proposal for a jump; the leapfrog loop has this one call site
        const int legs = status != RJ_OK ? 0 : (code == 0 ? 1 : 2);
        for (int leg = 0; leg < legs; ++leg) {
            if (leg == 1) {
                for (int i = tid; i < 3 * c.N; i += nt) c.p[i] = -c.p[i];
                __syncthreads();
                const int n_new = rj_propose(P, c.q, c.p, c.red, c.N, c.g_ff2, R, code, rec, part);
                if (n_new < 0) {
                    status = -n_new;
                    break;
                }
                c.N = n_new;
                // the cached pixel gradient belongs to the table before the edit (V: for nsteps = 0)
                Vpix = eval_pixels<T, MR, MC, KV3>(c, true);
            }
            for (int s = 0; s < A.nsteps; ++s)
                rhmc_step<T, MR, MC, KV3>(c, A.delta, A.counter_max, leg == legs - 1 && s == A.nsteps - 1, Vpix, nullptr);
        }
        bool accept = false;
        if (status == RJ_OK) {
            if (code != 0) {
                for (int i = tid; i < 3 * c.N; i += nt) c.p[i] = -c.p[i];
                __syncthreads();
            }
            const Energies e1 = energies(c, Vpix, A.f_pos, true);
            const double dE = (e1.V + e1.T) - st[0];
            const double lnu = A.lnu ? A.lnu[(size_t)field * L + l] : philox_lnu(A.seed, fid, (uint32_t)l);
            if (code == 0) {
                accept = (dE < 0.0) || (lnu < -dE);
            } else {
                const double ln_alpha = -dE + c.red[kRjBc + 1];
                accept = (ln_alpha > 0.0) || (lnu < ln_alpha);
            }
        } else if (status == RJ_OVERFLOW && overflow < 0) {
            overflow = l;
        }
        if (keep && tid == 0 && A.A_chain) A.A_chain[(size_t)field * rows + (size_t)(l / A.chain_stride)] = accept ? 1 : 0;
        if (accept) {
            ++n_acc;
        } else {
            __syncthreads();
            c.N = (int)st[2];
            for (int i = tid; i < 3 * c.N; i += nt) {
                c.q[i] = qs[i];
                c.g[i] = gs[i];
            }
            Vpix = st[1];
        }
        __syncthreads();
    }
    if (A.q_out)
        for (int i = tid; i < 3 * c.N; i += nt) A.q_out[(size_t)field * S + i] = c.q[i];
    if (tid == 0) {
        if (A.accept_rate) A.accept_rate[field] = (double)n_acc / (double)L;
        if (R.n_final) R.n_final[field] = c.N;
        if (R.overflow) R.overflow[field] = overflow;
    }
}

}  // namespace srhmc
