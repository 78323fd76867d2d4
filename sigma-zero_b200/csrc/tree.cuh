// tree.cuh -- the exact fp32 arithmetic of the reference search, one IEEE operation at a time.
//
//   puct_score        <- mctsnode.py:33-37  Node.get_ucb as torch (CPU, fp32) evaluates it
//   cascade_lane/...  <- mcts.py:79         torch.sum over the masked fp32[4672] policy (ATen cascade_sum)
//   noisy_prior       <- mcts.py:91-96      learning=True: one-category Dirichlet == constant
//   dir_log_gamma/... <- szb_exploration    opt-in: AlphaZero's Dirichlet noise over the root's children (not the reference's rule)
//
// No FMA contraction is allowed anywhere in here: every operation goes through an explicit
// round-to-nearest intrinsic on the device (and the host harness is built with -ffp-contract=off).
#pragma once
#include <stdint.h>
#include <math.h>
#include "chess.cuh"

namespace szb {

#if defined(__CUDA_ARCH__)
SZB_HD float f_add(float a, float b) { return __fadd_rn(a, b); }
SZB_HD float f_sub(float a, float b) { return __fsub_rn(a, b); }
SZB_HD float f_mul(float a, float b) { return __fmul_rn(a, b); }
SZB_HD float f_div(float a, float b) { return __fdiv_rn(a, b); }
SZB_HD float d2f(double a) { return __double2float_rn(a); }
SZB_HD double d_sqrt(double a) { return __dsqrt_rn(a); }
SZB_HD double d_add(double a, double b) { return __dadd_rn(a, b); }
SZB_HD double d_mul(double a, double b) { return __dmul_rn(a, b); }
#else
SZB_HD float f_add(float a, float b) { volatile float r = a + b; return r; }
SZB_HD float f_sub(float a, float b) { volatile float r = a - b; return r; }
SZB_HD float f_mul(float a, float b) { volatile float r = a * b; return r; }
SZB_HD float f_div(float a, float b) { volatile float r = a / b; return r; }
SZB_HD float d2f(double a) { return (float)a; }
SZB_HD double d_sqrt(double a) { return sqrt(a); }
SZB_HD double d_add(double a, double b) { volatile double r = a + b; return r; }
SZB_HD double d_mul(double a, double b) { volatile double r = a * b; return r; }
#endif

// sqrt(N_parent) as the reference feeds it to torch: math.sqrt in double, then cast to fp32 by the
// scalar * tensor multiplication.
SZB_HD float sqrt_parent(int n_parent) { return d2f(d_sqrt((double)n_parent)); }

// q + C * (sqrt(N_p) / (n + 1)) * prior, with q = 1 - (W/(n + 1e-6) + 1)/2, in torch's op order.
SZB_HD float puct_score(int n, double w, float prior, float sqrt_np, float c) {
    const float wf = d2f(w);
    const float d = f_add((float)n, 1e-6f);
    const float q = f_sub(1.0f, f_div(f_add(f_div(wf, d), 1.0f), 2.0f));
    const float r = f_div(1.0f, (float)(n + 1));       // Tensor.__rtruediv__ = reciprocal() * other
    const float u = f_mul(r, sqrt_np);
    return f_add(q, f_mul(f_mul(c, u), prior));
}

constexpr int CASCADE_STEPS = N_ACTIONS / 32;            // 146

// Partial sum owned by lane t (= row*8 + vector lane) of ATen's cascade_sum over 4672 contiguous floats.
template <class Elem>
SZB_HD float cascade_lane(Elem elem, int t) {
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    int i = 0;
    for (; i + 16 <= CASCADE_STEPS;) {
        for (int j = 0; j < 16; j++, i++) a0 = f_add(a0, elem(i * 32 + t));
        a1 = f_add(a1, a0);
        a0 = 0.0f;                                       // (i & 0xF0) != 0 for every i < 256: no deeper carry
    }
    for (; i < CASCADE_STEPS; i++) a0 = f_add(a0, elem(i * 32 + t));
    a0 = f_add(a0, a1);
    a0 = f_add(a0, a2);
    a0 = f_add(a0, a3);
    return a0;
}

// The same partial sum when every element outside the bitset `mask` (73 x uint64 over the element index) is +0 and no
// element is negative -- the masked policy of mcts.py:77-79.  x + (+0) == x exactly, so only the set bits are visited, in
// ascending order, and the merge of a finished 16-step block into the next level is applied lazily when the first element
// of a later block shows up (merging an untouched +0 block is the identity).  ~35 legal moves instead of 4672 additions.
template <class Elem>
SZB_HD float cascade_lane_sparse(const uint64_t* mask, Elem elem, int t) {
    float a0 = 0.0f, a1 = 0.0f;
    int cur = 0;                                         // 16-step block the pending a0 belongs to
    for (int w = 0; w < MASK_WORDS; w++) {
        const uint64_t m = mask[w];
        if (((m >> t) & 0x100000001ull) == 0) continue;  // neither step 2w (bit t) nor step 2w+1 (bit 32+t)
#pragma unroll
        for (int h = 0; h < 2; h++) {
            if ((m >> (h * 32 + t)) & 1ull) {
                const int i = 2 * w + h, b = i >> 4;
                if (b != cur) { a1 = f_add(a1, a0); a0 = 0.0f; cur = b; }
                a0 = f_add(a0, elem(i * 32 + t));
            }
        }
    }
    if (cur < CASCADE_STEPS / 16) { a1 = f_add(a1, a0); a0 = 0.0f; }   // pending block was a complete one; the tail block stays in a0
    return f_add(a0, a1);                                // (+ the two deeper levels, which stay +0 for 146 steps)
}

// Final reduction of the 32 lane partials: rows first (per vector lane), then the 8 lanes in order.
template <class Lane>
SZB_HD float cascade_combine(Lane lane_value) {
    float total = 0.0f;
    for (int l = 0; l < 8; l++) {
        float p = lane_value(l);
        p = f_add(p, lane_value(8 + l));
        p = f_add(p, lane_value(16 + l));
        p = f_add(p, lane_value(24 + l));
        total = f_add(total, p);
    }
    return total;
}

// 0.25f * nextafter(1, 0): the only value torch's one-category Dirichlet ever samples
#define SZB_NOISE_CONST 0.24999998509883880615234375f
SZB_HD float noisy_prior(float p) { return f_add(f_mul(0.75f, p), SZB_NOISE_CONST); }

// splitmix-style evaluator used for exact-parity testing and tree-only benchmarking
// (host twin: oracle/hash_eval.py)
constexpr uint64_t HE_GOLDEN = 0x9E3779B97F4A7C15ull;
constexpr uint64_t HE_VALUE_SALT = 0xD6E8FEB86659FD93ull;
SZB_HD uint64_t he_fold(const uint64_t* words119) {
    uint64_t h = 0x243F6A8885A308D3ull;
    for (int i = 0; i < N_PLANES; i++) h = mix64((h ^ words119[i]) + HE_GOLDEN);
    return h;
}
SZB_HD float he_policy(uint64_t h, int i) {
    const uint64_t r = mix64(h + (uint64_t)(i + 1) * HE_GOLDEN) >> 40;
    if ((r & 255) == 0) return 0.0f;
    const float u = f_mul((float)(uint32_t)(r + 1), 5.9604644775390625e-08f);   // 2^-24
    return f_mul(f_mul(f_mul(u, u), u), u);
}
SZB_HD float he_value(uint64_t h) {
    const uint64_t r = mix64(h ^ HE_VALUE_SALT) >> 40;
    return f_sub(f_mul((float)(uint32_t)r, 1.1920928955078125e-07f), 1.0f);      // 2^-23
}


// ---- opt-in root exploration (szb_exploration): AlphaZero's Dirichlet(alpha) noise over the ROOT's children --------------------
// Keyed, not stateful: a child's draw is a function of (seed, global game id, root ply, the child's policy index) only, so it does
// not depend on the slot, the cohort split, the shard, leaves_per_tree or which other children the root has.  The stream is
// separated from k_pick's move-sampling RNG by DIR_SALT; the uniforms of one child come from a splitmix64 sequence (its counter
// drives the rejection loop).  Arithmetic in double; the engine is built with --fmad=false and its host build with
// -ffp-contract=off, so host and device agree up to the last bits of the libm functions.
constexpr uint64_t DIR_SALT = 0x6A09E667F3BCC908ull;
SZB_HD uint64_t dir_root_key(uint64_t seed, uint64_t game_id, int ply) {
    return mix64(mix64(seed ^ DIR_SALT ^ (HE_GOLDEN * (game_id + 1))) + (uint64_t)ply);
}
struct DirStream {
    uint64_t state;
    SZB_HD double uniform() {                              // in (0, 1): 52 random bits + 1/2, exact in double
        state += HE_GOLDEN;
        return ((double)(mix64(state) >> 12) + 0.5) * 2.220446049250313080847263336181640625e-16;    // 2^-52
    }
    SZB_HD double normal() {                               // Box-Muller, cosine branch
        const double r = d_sqrt(d_mul(-2.0, log(uniform())));
        return d_mul(r, cos(d_mul(6.283185307179586, uniform())));
    }
};
// log of a Gamma(alpha, 1) draw for the child with policy index `move`.  alpha >= 1: Marsaglia-Tsang; alpha < 1: the boost
// log G(alpha) = log G(alpha + 1) + log(U) / alpha, kept in the log domain because U^(1/alpha) underflows for small alpha.
// The rejection loop accepts with probability > 0.95 per try; after 64 rejected tries (probability < 1e-83) it returns log(d).
SZB_HD double dir_log_gamma(uint64_t root_key, int move, double alpha) {
    DirStream s{mix64(root_key + (uint64_t)(move + 1) * HE_GOLDEN)};
    const double a = alpha < 1.0 ? d_add(alpha, 1.0) : alpha;
    const double d = d_add(a, -1.0 / 3.0), c = 1.0 / d_sqrt(d_mul(9.0, d));
    double lg = log(d);
    for (int tries = 0; tries < 64; tries++) {
        const double x = s.normal();
        double v = d_add(1.0, d_mul(c, x));
        if (v <= 0.0) continue;
        v = d_mul(d_mul(v, v), v);
        const double u = s.uniform();
        const double x2 = d_mul(x, x);
        if (log(u) < d_add(d_mul(0.5, x2), d_mul(d, d_add(d_add(1.0, -v), log(v))))) { lg = d_add(log(d), log(v)); break; }
    }
    if (alpha < 1.0) lg = d_add(lg, log(s.uniform()) / alpha);
    return lg;
}
// eta_i = exp(l_i - max l) / sum_j exp(l_j - max l): the sum in the device's fixed order -- lane t = k mod 32 adds the children k of
// its lane in ascending k, then the 32 lane sums are added in lane order (dir_combine).
template <class Lane>
SZB_HD double dir_combine(Lane lane_value) {
    double total = 0.0;
    for (int t = 0; t < 32; t++) total = d_add(total, lane_value(t));
    return total;
}
// the mixed root prior fl32((1 - eps) p + eps fl32(eta)), in double, no contraction, one rounding
SZB_HD float dir_mix(float p, float eta32, float eps) {
    return d2f(d_add(d_mul(d_add(1.0, -(double)eps), (double)p), d_mul((double)eps, (double)eta32)));
}

}  // namespace szb
