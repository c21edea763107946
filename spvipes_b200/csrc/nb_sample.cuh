// Draws from the decoder's negative-binomial mixture (scvi 0.20 NegativeBinomialMixture.sample, theta2 = None):
//
//   mu    = mu1 if Bernoulli(sigmoid(pi)) else mu2
//   lam   = min(max(Gamma(theta, rate = theta / mu), FLT_MIN), 1e8)   (torch's Gamma.rsample clamp, scvi's clamp)
//   count = Poisson(lam)                                              (float32, as torch's sampler returns it)
//
// The algorithms are torch's (ATen Distributions.h): Gamma by Marsaglia-Tsang with the U^(1/alpha) boost for alpha < 1, Poisson
// by multiplication of uniforms below lambda = 10 and by Hoermann's PTRS transformed rejection above (in double, as torch's CPU
// sampler runs it).  The draws are equal in distribution to torch's, not bit for bit.
//
// Randomness: Philox4x32-10 (common.cuh) under key = seed, counter = (gene, row, NBS_STREAM | group << 24 | block, draw).  An
// element's draw is therefore a pure function of (seed, group, draw index, row of the minibatch, gene), whatever kernel, tile shape
// or launch produced it.  The reparameterisation noise (poe.cu) and the dropout masks (elementwise.cu, gemm_simt.cu) put a stream
// id below 16 in the third counter word, so the top bit of NBS_STREAM keeps these counters disjoint from theirs under every seed.
// Each attempt of a rejection loop takes its own block (a fresh counter); the block index has three phases of 2^20 blocks each.
//
// The common path (theta >= 1, the first Gamma attempt accepted, lam < 10) is inline; the rest is out of line, so that the fused
// epilogue stays small.  Both call sites (the tensor-core sampling sweep and the SIMT sampler, nb_tc_sample.cu) are in one
// translation unit and share the out-of-line functions, so they produce the same bits.
#pragma once
#include "common.cuh"

constexpr uint32_t NBS_STREAM = 0x80000000u;
constexpr uint32_t NBS_GAMMA = 0u << 20;  // attempt a of the Gamma loop: (x, y) normal, z acceptance uniform; block 0's w: Bernoulli
constexpr uint32_t NBS_BOOST = 1u << 20;  // block 0's x: the U^(1/alpha) boost of alpha < 1
constexpr uint32_t NBS_POIS = 2u << 20;   // Poisson: 4 uniforms per block (multiplication), or one block per PTRS attempt
constexpr int NBS_MAX_GROUP = 127;        // group fills bits 24..30 of the third counter word

struct NbsKey {
    uint2 seed;
    uint32_t gene, row, tag, draw;
};

__device__ __forceinline__ NbsKey nbs_key(unsigned long long seed, int group, uint32_t draw, uint32_t row, uint32_t gene) {
    NbsKey k;
    k.seed = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    k.gene = gene; k.row = row; k.draw = draw;
    k.tag = NBS_STREAM | ((uint32_t)group << 24);
    return k;
}

__device__ __forceinline__ uint4 nbs_block(const NbsKey& k, uint32_t phase, uint32_t i) {
    return philox4x32_10(make_uint4(k.gene, k.row, k.tag | phase | (i & 0xfffffu), k.draw), k.seed);
}

// standard normal from two words (Box-Muller, as philox_normal)
__device__ __forceinline__ float nbs_normal(uint32_t a, uint32_t b) {
    return sqrtf(-2.0f * logf(u32_to_unit(a))) * cospif(2.0f * u32_to_unit(b));
}

// Gamma(alpha, 1), the whole of torch's sample_gamma (attempt 0 again when called after the inline attempt rejected it)
__device__ __noinline__ float nbs_gamma(float alpha, NbsKey k) {
    if (!(alpha > 0.0f)) return alpha == 0.0f ? 0.0f : __int_as_float(0x7fffffff);  // NaN stays NaN (the loop would not end)
    float scale = 1.0f;
    if (alpha < 1.0f) {
        scale = powf(u32_to_unit(nbs_block(k, NBS_BOOST, 0).x), 1.0f / alpha);
        alpha += 1.0f;
    }
    const float d = alpha - 1.0f / 3.0f, c = 1.0f / sqrtf(9.0f * d);
    for (uint32_t a = 0;; ++a) {
        const uint4 r = nbs_block(k, NBS_GAMMA, a);
        const float x = nbs_normal(r.x, r.y), y = 1.0f + c * x;
        if (y <= 0.0f) continue;
        const float v = y * y * y, u = u32_to_unit(r.z), xx = x * x;
        if (u < 1.0f - 0.0331f * xx * xx) return scale * d * v;
        if (logf(u) < 0.5f * xx + d * (1.0f - v + logf(v))) return scale * d * v;
    }
}

// Poisson(lam) for lam >= 10 (or NaN, returned as is): PTRS (Hoermann 1993), torch's constants, in double
__device__ __noinline__ float nbs_poisson_ptrs(float lamf, NbsKey k) {
    if (!(lamf >= 10.0f)) return lamf;
    const double lam = lamf, slam = sqrt(lam), loglam = log(lam);
    const double b = 0.931 + 2.53 * slam, a = -0.059 + 0.02483 * b;
    const double invalpha = 1.1239 + 1.1328 / (b - 3.4), vr = 0.9277 - 3.6224 / (b - 2.0);
    for (uint32_t i = 0;; ++i) {
        const uint4 r = nbs_block(k, NBS_POIS, i);
        // uniforms strictly inside (0, 1) on a 2^-32 grid: us > 0 below
        const double U = ((double)r.x + 0.5) * 0x1p-32 - 0.5, V = ((double)r.y + 0.5) * 0x1p-32;
        const double us = 0.5 - fabs(U);
        const double kk = floor((2.0 * a / us + b) * U + lam + 0.43);
        if (us >= 0.07 && V <= vr) return (float)kk;
        if (kk < 0.0 || (us < 0.013 && V > us)) continue;
        if (log(V) + log(invalpha) - log(a / (us * us) + b) <= -lam + kk * loglam - lgamma(kk + 1.0)) return (float)kk;
    }
}

// one draw of the mixture for one element
__device__ __forceinline__ float nb_mixture_sample(float mu1, float mu2, float pi, float theta, const NbsKey& k) {
    const uint4 r0 = nbs_block(k, NBS_GAMMA, 0);
    const float w = 1.0f / (1.0f + __expf(-pi));
    const float mu = u32_to_unit(r0.w) <= w ? mu1 : mu2;  // u in (0, 1]: P(u <= w) = w on the 2^-24 grid
    if (mu == 0.0f) return 0.0f;
    float g = -1.0f;
    if (theta >= 1.0f) {  // the first Marsaglia-Tsang attempt, inline
        const float d = theta - 1.0f / 3.0f, c = 1.0f / sqrtf(9.0f * d);
        const float x = nbs_normal(r0.x, r0.y), y = 1.0f + c * x;
        const float v = y * y * y, xx = x * x, u = u32_to_unit(r0.z);
        if (y > 0.0f && u < 1.0f - 0.0331f * xx * xx) g = d * v;
    }
    if (g < 0.0f) g = nbs_gamma(theta, k);
    float lam = g / (theta / mu);
    lam = lam < 1.17549435e-38f ? 1.17549435e-38f : (lam > 1e8f ? 1e8f : lam);  // comparisons, not fminf / fmaxf: NaN stays NaN
    if (!(lam < 10.0f)) return nbs_poisson_ptrs(lam, k);
    const float enlam = expf(-lam);
    float prod = 1.0f, n = 0.0f;
    for (uint32_t i = 0;; ++i) {
        const uint4 r = nbs_block(k, NBS_POIS, i);
        prod *= u32_to_unit(r.x);
        if (prod <= enlam) return n;
        prod *= u32_to_unit(r.y);
        if (prod <= enlam) return n + 1.0f;
        prod *= u32_to_unit(r.z);
        if (prod <= enlam) return n + 2.0f;
        prod *= u32_to_unit(r.w);
        if (prod <= enlam) return n + 3.0f;
        n += 4.0f;
    }
}
