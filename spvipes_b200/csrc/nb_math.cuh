// Element math of the NB-mixture likelihood for the tensor-core path (fast SFU intrinsics: ex2.approx / lg2.approx /
// rcp.approx; north_star's gate for this path is 1e-2 relative on the loss terms).  Measured on a B200 against float64
// (tests/test_gpu_decoder_f64.py, inputs at every edge branch): per-cell reconstruction terms within 1.7e-4; per element, ep / es
// of rho just above the EXACT threshold carry the plain form's relative error 1e-8 / rho (1 % at rho = 1e-6), and d px_r of
// genes with theta > e^6.5 loses digits to the cancellation in the d-theta form (3.1e-3 of the largest d px_r).
// scvi-tools 0.20.0 log_mixture_nb, shared-theta branch, eps = 1e-8; reference call sites module/spVIPESmodule.py:759, 823-824.
#pragma once
#include "common.cuh"
#include "decoder_common.cuh"

// single-MUFU transcendental forms (flush-to-zero, no denormal fix-up code): operands here are never denormal
#if defined(PTC_EXP) && PTC_EXP == 2  // timing experiment only: no SFU instructions (wrong numerics)
__device__ __forceinline__ float fast_lg2(float x) { return fmaf(x, 0.25f, -1.0f); }
__device__ __forceinline__ float fast_ex2(float x) { return fmaf(x, 0.01f, 1.0f); }
__device__ __forceinline__ float fast_rcp(float x) { return fmaf(x, -0.01f, 1.0f); }
#else
__device__ __forceinline__ float fast_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
#endif
__device__ __forceinline__ float fast_log(float x) { return fast_lg2(x) * 0.69314718056f; }
__device__ __forceinline__ float fast_exp(float x) { return fast_ex2(x * 1.44269504089f); }

// outputs of the element functions below
struct NbOut { float ll, ep, es; };

// ================================================================================================================
// v5 element math (r2).  Everything in the base-2 domain, and nothing in it depends on the minibatch except through its
// arguments:
//   xp, xs : log2(rho) of the two branches, COMPLETE - the folded BatchNorm shift and the row normaliser
//            (lib - logsumexp) log2e ride in the branch k-block of the MMA as split-fp16 columns (decoder_common.cuh ZK_*)
//   pi     : mixture logit (natural units, bias included by the caller)
//   t, Ct  : t = log1p(count) and the count-dependent lgamma (forward) / digamma (backward) term
//            forward  Ct = lgamma(t + theta) - lgamma(theta) - lgamma(t + 1)        backward  Ct = digamma(t + theta) - digamma(theta)
//            from the per-gene tables of spv_dec_theta_tables (counts < NB_TAB) - both vanish at t = 0, and they enter the
//            log-likelihood additively (the same term in both mixture components), so they never touch the logsumexp
//   per gene: th, thE = th + eps,  forward Kc = th log(th + eps),  backward K1c = log(th + eps) + th / (th + eps)
// 8 SFU operations per element (forward and backward): ex2 x4, lg2 x3 (x2 backward), ONE rcp shared by the four reciprocals
// 1/d1, 1/d2, 1/(1 + e), 1/(1 + epi) (r = rcp(d1 d2 o1 o2); products stay far inside fp32's range: d <= rho + theta, o <= 2).
// log2(rho + eps) = x (rho = 2^x) and rho / (rho + eps) = 1 unless rho < 1e-6 with a positive count, where the EXACT variant
// runs (the caller decides per group of elements).  History: v1 91 FP32 + 22 SFU, v3 59 + 16, v4 62 + 11, v5 ~45 + 8
// (profiles/r2_nb_v5.md).  Algebra checked against scvi's formula in float64 (tools/check_nb_math.py).
// ================================================================================================================
#define NB_LOG2E 1.4426950408889634f
#define NB_LN2 0.6931471805599453f
#define NB_X_RARE -19.931568f   // log2(1e-6)

template <bool EXACT>
__device__ __forceinline__ NbOut nb_forward_v5(float t, float Ct, float xp, float xs, float pi, float th, float thE, float Kc) {
    const float rp = fast_ex2(xp), rs = fast_ex2(xs);
    const float d1 = rp + thE, d2 = rs + thE;
    const float L1 = fast_lg2(d1), L2 = fast_lg2(d2);
    const float x = t + th;
    float Lap = xp, Las = xs, fp = 1.0f, fs = 1.0f;  // log2(rho + eps) and rho / (rho + eps)
    if (EXACT) {
        const float ap = rp + NB_EPS, as = rs + NB_EPS;
        Lap = fast_lg2(ap); Las = fast_lg2(as);
        fp = rp * fast_rcp(ap); fs = rs * fast_rcp(as);
    }
    // a = Kc + Ct - ln2 m1,  b = Kc + Ct - ln2 m2 - pi,  m = x log2(th + rho + eps) - t log2(rho + eps)
    const float m1 = fmaf(-t, Lap, x * L1), m2 = fmaf(-t, Las, x * L2);
    const float df = fmaf(m2 - m1, NB_LN2, pi);  // a - b
    const float e = fast_ex2(-NB_LOG2E * fabsf(df)), epi = fast_ex2(-NB_LOG2E * fabsf(pi));
    const float o1 = 1.0f + e, o2 = 1.0f + epi;
    const float d12 = d1 * d2, oo = o1 * o2;
    const float r = fast_rcp(d12 * oo);
    const float rd = r * oo, ro = r * d12;  // 1 / (d1 d2), 1 / (o1 o2)
    const float id1 = rd * d2, id2 = rd * d1, i1 = ro * o2, i2 = ro * o1;
    NbOut o;
    // logsumexp(a, b) - softplus(-pi) = a + max(0, -df) - max(-pi, 0) + log((1 + e) / (1 + epi))
    o.ll = (Kc + Ct) + fmaf(m1, -NB_LN2, fmaxf(-df, 0.0f)) - fmaxf(-pi, 0.0f) + NB_LN2 * fast_lg2(o1 * i2);
    const float wmin = e * i1;
    const float wa = df >= 0.0f ? 1.0f - wmin : wmin, wb = 1.0f - wa;
    o.ep = wa * fmaf(t, fp, -(x * id1) * rp);
    o.es = wb * fmaf(t, fs, -(x * id2) * rs);
    return o;
}

// Forward and backward of one element in one evaluation (the training sweep, nb_tc_train.cu): the log-likelihood, the two branch
// terms WITHOUT the softmax coupling (ep, es: d ll / d log rho at fixed normaliser; d ll / d y = e - rho exp(-lib) D with the row
// sum D known only after the sweep), rho of both branches, and the gradients w.r.t. the mixture logit and theta.
// Ctf / Ctb: the count-dependent lgamma / digamma terms (tables), Kc / K1c the per-gene forward / backward constants above.
struct NbTrain { float ll, ep, es, rp, rs, dpi, dth; };
template <bool EXACT>
__device__ __forceinline__ NbTrain nb_train_v5(float t, float Ctf, float Ctb, float xp, float xs, float pi, float th, float thE, float Kc,
                                               float K1c) {
    const float rp = fast_ex2(xp), rs = fast_ex2(xs);
    const float d1 = rp + thE, d2 = rs + thE;
    const float L1 = fast_lg2(d1), L2 = fast_lg2(d2);
    const float x = t + th;
    float Lap = xp, Las = xs, fp = 1.0f, fs = 1.0f;
    if (EXACT) {
        const float ap = rp + NB_EPS, as = rs + NB_EPS;
        Lap = fast_lg2(ap); Las = fast_lg2(as);
        fp = rp * fast_rcp(ap); fs = rs * fast_rcp(as);
    }
    const float m1 = fmaf(-t, Lap, x * L1), m2 = fmaf(-t, Las, x * L2);
    const float df = fmaf(m2 - m1, NB_LN2, pi);
    const float e = fast_ex2(-NB_LOG2E * fabsf(df)), epi = fast_ex2(-NB_LOG2E * fabsf(pi));
    const float o1 = 1.0f + e, o2 = 1.0f + epi;
    const float d12 = d1 * d2, oo = o1 * o2;
    const float r = fast_rcp(d12 * oo);
    const float rd = r * oo, ro = r * d12;
    const float id1 = rd * d2, id2 = rd * d1, i1 = ro * o2, i2 = ro * o1;
    NbTrain o;
    o.ll = (Kc + Ctf) + fmaf(m1, -NB_LN2, fmaxf(-df, 0.0f)) - fmaxf(-pi, 0.0f) + NB_LN2 * fast_lg2(o1 * i2);
    const float wmin = e * i1;
    const float wa = df >= 0.0f ? 1.0f - wmin : wmin, wb = 1.0f - wa;
    const float q1 = x * id1, q2 = x * id2;
    o.ep = wa * fmaf(t, fp, -q1 * rp);
    o.es = wb * fmaf(t, fs, -q2 * rs);
    o.rp = rp;
    o.rs = rs;
    const float sneg = (pi >= 0.0f ? epi : 1.0f) * i2;  // sigmoid(-pi)
    o.dpi = sneg - wb;
    o.dth = (K1c + Ctb) - wa * fmaf(L1, NB_LN2, q1) - wb * fmaf(L2, NB_LN2, q2);
    return o;
}

// ---- count terms outside the tables (counts >= NB_TAB, non-integer "counts" of a float32 source): out of line, accurate libm
// forms; lgt = lgamma(theta), dgt = digamma(theta) of the gene
static __device__ __noinline__ float2 nb_count_terms_fwd_slow(float xraw, float th, float lgt) {
    const float t = log1pf(xraw);
    return make_float2(t, xraw > 0.0f ? lgammaf(t + th) - lgt - lgammaf(t + 1.0f) : 0.0f);
}
// ... of a target value t given as it is (SPV_SRC_F32: px.log_prob(value) at an arbitrary value)
static __device__ __noinline__ float2 nb_target_terms_fwd(float t, float th, float lgt) {
    return make_float2(t, t != 0.0f ? lgammaf(t + th) - lgt - lgammaf(t + 1.0f) : 0.0f);
}
static __device__ __noinline__ float2 nb_count_terms_bwd_slow(float xraw, float th, float dgt) {
    const float t = log1pf(xraw);
    return make_float2(t, xraw > 0.0f ? digammaf_pos(t + th) - dgt : 0.0f);
}

// Count tile of the likelihood kernels in shared memory: one uint16 code per element, the byte offset into the gene's table row
// (count * 8) for tabulated counts, NB_CODE_SLOW for everything else (the element then re-reads its raw value from global memory)
#define NB_CODE_SLOW 0xFFF8u
__device__ __forceinline__ uint32_t nb_code_u16(uint32_t c) { return c < NB_TAB ? c << 3 : NB_CODE_SLOW; }
__device__ __forceinline__ uint32_t nb_code_f32(float v) {
    const int c = (int)v;
    return (v >= 0.0f && v < (float)NB_TAB && (float)c == v) ? (uint32_t)c << 3 : NB_CODE_SLOW;
}

// Two raw values of a row (genes g, g + 1) as one register pair, and their two 16-bit count codes.  SRC 1: uint16 counts,
// 2: float32 counts.  Load and conversion are separate, and the vector form has no branch, so that a caller can put a whole
// batch of loads in flight before the first one is used (nb_pair_vec_ok: decided once per thread, not per load).
template <int SRC>
__device__ __forceinline__ bool nb_pair_vec_ok(const void* X, long ldx, int g, int G) {
    const uintptr_t mask = SRC == 1 ? 3 : 7;
    return g + 1 < G && (ldx & 1) == 0 && (g & 1) == 0 && (reinterpret_cast<uintptr_t>(X) & mask) == 0;
}
template <int SRC>
__device__ __forceinline__ uint2 nb_load_pair_vec(const void* X, long row_off, int g) {
    if (SRC == 1 /* SPV_SRC_U16_LOG1P */) {
        return make_uint2(__ldg(reinterpret_cast<const uint32_t*>(reinterpret_cast<const unsigned short*>(X) + row_off + g)), 0u);
    } else {
        const float2 v = __ldg(reinterpret_cast<const float2*>(reinterpret_cast<const float*>(X) + row_off + g));
        return make_uint2(__float_as_uint(v.x), __float_as_uint(v.y));
    }
}
template <int SRC>
__device__ __forceinline__ uint2 nb_load_pair(const void* X, long row_off, int g, int G) {
    if (SRC == 1 /* SPV_SRC_U16_LOG1P */) {
        const unsigned short* src = reinterpret_cast<const unsigned short*>(X) + row_off + g;
        return make_uint2((g < G ? (uint32_t)__ldg(src) : 0u) | ((g + 1 < G ? (uint32_t)__ldg(src + 1) : 0u) << 16), 0u);
    } else {
        const float* src = reinterpret_cast<const float*>(X) + row_off + g;
        return make_uint2(__float_as_uint(g < G ? __ldg(src) : 0.0f), __float_as_uint(g + 1 < G ? __ldg(src + 1) : 0.0f));
    }
}
template <int SRC>
__device__ __forceinline__ uint32_t nb_pair_codes(uint2 raw) {
    if (SRC == 1 /* SPV_SRC_U16_LOG1P */) {
        const uint32_t w = raw.x;
        const uint32_t lo = (w & 0xfff0u) ? NB_CODE_SLOW : (w & 0xffffu) << 3;
        const uint32_t hi = (w & 0xfff00000u) ? NB_CODE_SLOW : (w >> 16) << 3;
        return lo | (hi << 16);
    } else if (SRC == 0 /* SPV_SRC_F32: target values t, not counts */) {
        // the tables are indexed by count (t = log1p(c)); a target hits them only at t = 0 = log1p(0), entry 0
        return (__uint_as_float(raw.x) == 0.0f ? 0u : NB_CODE_SLOW) | ((__uint_as_float(raw.y) == 0.0f ? 0u : NB_CODE_SLOW) << 16);
    } else {
        return nb_code_f32(__uint_as_float(raw.x)) | (nb_code_f32(__uint_as_float(raw.y)) << 16);
    }
}
template <int SRC>
__device__ __forceinline__ float nb_load_raw(const void* X, long idx) {
    return SRC == 1 /* SPV_SRC_U16_LOG1P */ ? (float)__ldg(reinterpret_cast<const unsigned short*>(X) + idx)
                                    : __ldg(reinterpret_cast<const float*>(X) + idx);
}
