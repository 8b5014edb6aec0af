// The per-star algebra of the reversible-jump moves (drop-in sampler_RHMC.py birth_death_move, split_merge_move; reference
// sampler_RHMC.py:1200-1445), on plain values, shared by the CTA-per-field kernel (field_rj.cuh) and the large-field engine
// (big_field.cu): the move code and index mapping of a draw record (rj_draws.cuh), the Beta density, the merge weight, a
// star's kinetic energy, the momentum of a proposed star and the four log ratios.
#pragma once
#include <math_constants.h>

#include "rj_draws.cuh"

namespace srhmc {

// a jump that runs, one refused with the state unchanged, one that would need more than the star capacity
enum RjStatus : int { RJ_OK = 0, RJ_REFUSED = 1, RJ_OVERFLOW = 2 };

// ln of the Beta(a, b) density (scipy.stats.beta.logpdf)
__device__ __forceinline__ double beta_logpdf(const RjParams& R, double x) {
    return (R.beta_a - 1.0) * log(x) + (R.beta_b - 1.0) * log1p(-x) - R.ln_beta;
}

// Merge weight of the ordered pair (a, b) of rows (f, x, y) (drop-in _merge_weights): Beta density of the share
// f_b / (f_a + f_b), zero within 1e-6 of one half, times the Gaussian split kernel at the pair's separation
__device__ __forceinline__ double merge_weight_of(const RjParams& R, const double* a, const double* b) {
    const double fi = a[0], fj = b[0];
    const double share = fj / (fi + fj);
    // outside (0, 1) (a flux at or below 0, possible with f_pos = 0) the Beta density is 0, as scipy's BETA.pdf gives it
    if (!(share > 0.0 && share < 1.0) || fabs(share - 0.5) < 1e-6) return 0.0;
    const double dr = a[1] - b[1], dc = a[2] - b[2];
    const double k2 = R.K_split * R.K_split;
    return exp(beta_logpdf(R, share)) * (exp(-(dr * dr + dc * dc) / (2.0 * k2)) / (2.0 * CUDART_PI * k2));
}

// 0 within, 1 birth, 2 death, 3 split, 4 merge (gym.move_types) from u_move (np.random.choice's rule) and u_grow
__device__ __forceinline__ int rj_move_code(const RjParams& R, const double* rec) {
    const int move = rec[0] < R.cdf0 ? 0 : (rec[0] < R.cdf1 ? 1 : 2);
    const bool grow = rec[1] < 0.5;
    return move == 0 ? 0 : (move == 1 ? (grow ? 1 : 2) : (grow ? 3 : 4));
}

// np.random.randint(0, n) from the record's u_a: the death victim or the split parent
__device__ __forceinline__ int rj_index(const double* rec, int n) { return min((int)floor(rec[2] * n), n - 1); }

// the newborn (flux, row, col) of a birth: position uniform inside the one-pixel border, flux from the power-law prior
__device__ __forceinline__ void rj_newborn(const RjParams& R, int rows, int cols, double alpha, const double* rec, double* q3) {
    q3[1] = rec[2] * (rows - 2.0) + 1.0;
    q3[2] = rec[3] * (cols - 2.0) + 1.0;
    q3[0] = exp(log(R.pl_lo + rec[4] * R.pl_span) / (1.0 - alpha));
}

// T(p, H(q)) of one star
__device__ __forceinline__ double star_T(const FieldParams& P, double g_ff2, const double* q3, const double* p3) {
    double quad = 0.0, logdet = 0.0;
    kinetic_terms(metric_of(P, q3[0], g_ff2), p3[0], p3[1], p3[2], quad, logdet);
    return (quad + logdet) / 2.0;
}

// T of two stars together (the split's children, the merge's pair): one sum of quad and one of logdet, as the reference
// evaluates the kinetic energy of the concatenated pair
__device__ __forceinline__ double pair_T(const FieldParams& P, double g_ff2, const double* qa, const double* pa, const double* qb,
                                         const double* pb) {
    double quad = 0.0, logdet = 0.0;
    kinetic_terms(metric_of(P, qa[0], g_ff2), pa[0], pa[1], pa[2], quad, logdet);
    kinetic_terms(metric_of(P, qb[0], g_ff2), pb[0], pb[1], pb[2], quad, logdet);
    return (quad + logdet) / 2.0;
}

// p3 = z sqrt(H(q3)): the momentum of a proposed star
__device__ __forceinline__ void draw_momentum(const FieldParams& P, double g_ff2, const double* q3, const double* z, double* p3) {
    const Metric m = metric_of(P, q3[0], g_ff2);
    p3[0] = z[0] * sqrt(m.Hff);
    p3[1] = z[1] * sqrt(m.Hxx);
    p3[2] = z[2] * sqrt(m.Hxx);
}

// the two children of a split of (fp, rp, cp) with offsets (off_r, off_c) and flux share `share`
__device__ __forceinline__ void rj_children(double fp, double rp, double cp, double off_r, double off_c, double share, double* a,
                                            double* b) {
    a[0] = share * fp;
    a[1] = rp + (1.0 - share) * off_r;
    a[2] = cp + (1.0 - share) * off_c;
    b[0] = (1.0 - share) * fp;
    b[1] = rp - share * off_r;
    b[2] = cp - share * off_c;
}

// the merged star of the ordered pair (a, b): flux sum, position weighted by share = f_a / (f_a + f_b)
__device__ __forceinline__ void rj_merged(const double* a, const double* b, double share, double* m) {
    m[0] = a[0] + b[0];
    m[1] = share * a[1] + (1.0 - share) * b[1];
    m[2] = share * a[2] + (1.0 - share) * b[2];
}

// ---- the log ratios of the four proposals (T_*: kinetic energies of the stars that appear or disappear; kernel_norm =
// ln(2 pi K^2) of the split kernel)
__device__ __forceinline__ double rj_lr_birth(const FieldParams& P, double f_new, double T_new) {
    return P.alpha * log(f_new) - 3.0 / 2.0 + T_new + P.Vpc;
}
__device__ __forceinline__ double rj_lr_death(const FieldParams& P, double f_old, double T_old) {
    return -P.alpha * log(f_old) + 3.0 / 2.0 - T_old - P.Vpc;
}
__device__ __forceinline__ double rj_lr_split(const RjParams& R, double kernel_norm, double fp, double share, double off_r,
                                              double off_c, double T_children, double T_parent) {
    const double k2 = R.K_split * R.K_split;
    return (-3.0 / 2.0) + log(fp) - beta_logpdf(R, share) + kernel_norm + ((off_r * off_r + off_c * off_c) / (2.0 * k2)) +
           T_children - T_parent;
}
__device__ __forceinline__ double rj_lr_merge(const RjParams& R, double kernel_norm, double f_merged, double share, double gap2,
                                              double T_pair, double T_merged) {
    const double k2 = R.K_split * R.K_split;
    return (3.0 / 2.0) - log(f_merged) + beta_logpdf(R, share) - kernel_norm - (gap2 / (2.0 * k2)) - T_pair + T_merged;
}

}  // namespace srhmc
