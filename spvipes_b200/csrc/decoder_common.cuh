// per-gene constant table shared by the decoder kernels: genec[GC_N][G] (SoA, stride G)
#pragma once
enum {
    GC_CP = 0,   // folded BatchNorm shift of the private branch: beta - mean * a
    GC_CS,       // ... shared branch
    GC_AP,       // folded scale gamma / sqrt(var + eps), private
    GC_AS,       // ... shared
    GC_ISTD_P,   // 1 / sqrt(var + eps)
    GC_ISTD_S,
    GC_MEAN_P,   // batch (or running) mean of z W^T
    GC_MEAN_S,
    GC_THETA,    // exp(px_r)
    GC_LTE,      // log(theta + eps)
    GC_LGT,      // lgamma(theta)
    GC_DGT,      // digamma(theta)
    // ready-made constants of the base-2 element math of the tensor-core likelihood kernels (nb_math.cuh, v3)
    GC_CPL,      // GC_CP * log2(e)
    GC_CSL,      // GC_CS * log2(e)
    GC_THE,      // theta + eps
    GC_K0,       // theta log(theta + eps) - lgamma(theta) + 0.5 log(2 pi)          (forward)
    GC_K1,       // log(theta + eps) + theta / (theta + eps) - digamma(theta)       (backward)
    // shifts of the CENTRED form y = W' (z - m) + c' used by the tensor-core kernels (m = batch mean of z when training, so
    // c' = beta exactly; m = 0 in eval mode), times log2(e)
    GC_CPLC,
    GC_CSLC,
    // v5 element math (r2): the lgamma / digamma terms that depend on the count come from per-gene tables (spv_dec_theta_tables)
    GC_KC,       // theta log(theta + eps)                                          (forward)
    GC_K1C,      // log(theta + eps) + theta / (theta + eps)                        (backward)
    GC_N
};

// Layout of the 64-wide branch k-block of the tensor-core likelihood kernels (fp16; zc_f16 [B, 64] against wz_f16 [2 Gp, 64]).
// Columns [0, P + S): centred latents against the folded weights times log2(e).  The last six columns carry every additive
// term of the base-2 logit as split-fp16 pairs (hi + lo: 2^-22 relative), so the accumulator IS log2(rho):
//   ZK_ONE, +1 : 1, 1 in zc            against (shift hi, shift lo) of the gene in wz (private rows: c'_p log2e, shared rows: c'_s log2e)
//   ZK_RP,  +1 : (Rp hi, Rp lo) in zc  against 1, 1 in the private rows of wz (0 in the shared rows);  Rp = (lib - logsumexp_p) log2e
//   ZK_RS,  +1 : (Rs hi, Rs lo) in zc  against 1, 1 in the shared rows
// spv_dec_fold writes the ones and zeroes the R columns (the statistics sweep must not see them); the row-statistics kernel
// fills the R columns once the normalisers are known.
#define ZK_ONE 58
#define ZK_RP 60
#define ZK_RS 62
#define ZK_MAX_LATENT 58   // P + S (+ covariate columns) must fit below ZK_ONE
#define DEC_MAX_LATENT 96  // P + S (+ covariate columns) of every decoder path: the per-gene kernels' shared-memory sizing

// Per-gene count tables (spv_dec_theta_tables): for raw counts c < NB_TAB, t = log1p(c) and
//   forward  tgf[g][c] = (t, lgamma(t + theta) - lgamma(theta) - lgamma(t + 1))
//   backward tb1[g][c] = digamma(t + theta) - digamma(theta)
// (both 0 at c = 0).  Larger or non-integer counts take an out-of-line path that evaluates the same terms directly.
#define NB_TAB 16
