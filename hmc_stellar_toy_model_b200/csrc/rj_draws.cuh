// Device draws of the reversible-jump moves (field_kernel MODE_RUN_RJ): one fixed record of kRjDraws doubles per
// (field, iteration), so that a run is reproducible whatever the star count does and can be replayed record for record.
//   [0] u_move   [1] u_grow   [2] u_a (birth row, death victim, split parent, merge pick)   [3] u_b (birth column)
//   [4] u_c (birth flux)   [5] [6] split offset normals   [7] split share ~ Beta(beta_a, beta_b)
//   [8..13] normals: the newborn's or the merged star's momentum (8..10), or the two children's (8..10, 11..13)
// Philox4x32-10 counters (word, iteration, field, domain): the momentum uses domains 0 and 1, the accept test 2 and the
// mock data 3, so the jump draws take 4 (uniforms: words 0..2, normals: words 3..6) and 5 / 6 (the two gamma variates of
// the share).  A run with P_move = [1, 0, 0] therefore consumes exactly the draws of srhmc_run.
#pragma once
#include "common.cuh"

namespace srhmc {

constexpr uint32_t kGammaMaxAttempts = 64;   // Marsaglia-Tsang accepts > 95% of attempts: 64 rejections in a row ~ 1e-83

// Gamma(a, 1) by Marsaglia and Tsang (2000).  Attempt t draws its normal from word 2t and its uniform from word 2t + 1 of
// `domain`; shape a < 1 is boosted: Gamma(a + 1) * U^(1/a) with U from the last two words of word 1.
static __device__ __forceinline__ double gamma_philox(uint64_t seed, uint32_t fid, uint32_t l, uint32_t domain, double a) {
    const bool boost = a < 1.0;
    const double d = (boost ? a + 1.0 : a) - 1.0 / 3.0, cc = 1.0 / sqrt(9.0 * d);
    double out = d;
    for (uint32_t t = 0; t < kGammaMaxAttempts; ++t) {
        uint32_t r[4];
        Philox::block(seed, 2u * t, l, fid, domain, r);
        double s, co;
        sincospi(2.0 * u01(r[2], r[3]), &s, &co);
        const double x = sqrt(-2.0 * log(u01(r[0], r[1]))) * co;
        double v = 1.0 + cc * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        Philox::block(seed, 2u * t + 1u, l, fid, domain, r);
        const double u = u01(r[0], r[1]), x2 = x * x;
        if (u < 1.0 - 0.0331 * (x2 * x2) || log(u) < 0.5 * x2 + d * (1.0 - v + log(v))) {
            out = d * v;
            break;
        }
    }
    if (boost) {
        uint32_t r[4];
        Philox::block(seed, 1u, l, fid, domain, r);
        out *= pow(u01(r[2], r[3]), 1.0 / a);
    }
    return out;
}

static __device__ __noinline__ void rj_record(uint64_t seed, uint32_t fid, uint32_t l, double beta_a, double beta_b, double* o) {
    uint32_t r[4];
    Philox::block(seed, 0u, l, fid, 4u, r);
    o[0] = u01(r[0], r[1]);
    o[1] = u01(r[2], r[3]);
    Philox::block(seed, 1u, l, fid, 4u, r);
    o[2] = u01(r[0], r[1]);
    o[3] = u01(r[2], r[3]);
    Philox::block(seed, 2u, l, fid, 4u, r);
    o[4] = u01(r[0], r[1]);
    const int slot[8] = {5, 6, 8, 9, 10, 11, 12, 13};
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        Philox::block(seed, 3u + b, l, fid, 4u, r);
        const double rad = sqrt(-2.0 * log(u01(r[0], r[1])));
        double s, c;
        sincospi(2.0 * u01(r[2], r[3]), &s, &c);
        o[slot[2 * b]] = rad * c;
        o[slot[2 * b + 1]] = rad * s;
    }
    const double x = gamma_philox(seed, fid, l, 5u, beta_a), y = gamma_philox(seed, fid, l, 6u, beta_b);
    o[7] = x / (x + y);
}

}  // namespace srhmc
