// Per-gene stages of the decoder: closed-form BatchNorm statistics of the two "factor regressor" branches
// (u = z W^T, BatchNorm1d over the minibatch, eps 1e-3, momentum 0.01: scvi FCLayers; reference nn/networks.py:314-320),
// their fold into an affine map, the constants of the NB term (theta = exp(px_r), reference module/spVIPESmodule.py:758),
// and the matching backward.  Because u is linear in z, the batch mean / variance of u[:, g] are W[g] . mean(z) and
// W[g]^T Cov(z) W[g]: no [B, G] pass is needed, only the [KZ, KZ] covariance of the latent minibatch.
//
// Work split: one warp per gene (lanes over the latent dimension), 64 genes per CTA.
#include <cooperative_groups.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "common.cuh"
#include "decoder_common.cuh"
#include "../../include/spvipes_b200.h"

#define GENES_PER_CTA 32        // gene_bwd: 32 genes share one set of per-CTA partial sums (ncu r1: instruction bound, so
                                // more, smaller CTAs; spv_dec_gene_bwd_parts reports the resulting number of partials)
#define FOLD_GENES_PER_CTA 32   // fold: 8 warps x 4 genes for the quadratic forms, then one gene per lane for the NB constants
#define GENE_BWD_THREADS 256

// ---------------------------------------------------------------------------------------
// mean and (biased) covariance of the latent minibatch zz [B, KZ] in ONE launch: a cluster of 8 CTAs, each owning a
// contiguous slice of the rows.  Column sums are exchanged through distributed shared memory (every CTA adds the eight
// partials in rank order, so all see the same mean), the centred second moments of the slice are accumulated in shared
// memory, and CTA r adds the eight partials of every 8th covariance entry, again in rank order: deterministic, no
// global-memory partials, no atomics, two cluster barriers instead of a second launch + "last CTA" pass.
// ---------------------------------------------------------------------------------------
#define ZS_CTAS 8
// rows per shared-memory tile: template parameter ZS_ROWS = 64 / 128 / 256, the smallest that holds a CTA's slice (B / 8 rows) so
// that the slice is read from global memory once and the passes run without tile loops (64-row tiles at B = 2048: 46 us)
#define ZS_THREADS 256

// rows [r0, r0 + nr) of zz into tile [ZS_ROWS][ldt] (zero rows beyond nr); all loads of a thread in flight before the stores
template <int ZS_ROWS>
__device__ __forceinline__ void zs_load_tile(float* tile, int ldt, const float* __restrict__ zz, long ld, int r0, int nr, int KZ) {
    const int total = ZS_ROWS * KZ;
    for (int base = 0; base < total; base += 12 * ZS_THREADS) {
        float v[12];
#pragma unroll
        for (int u = 0; u < 12; ++u) {
            const int i = base + u * ZS_THREADS + (int)threadIdx.x;
            const int r = i / KZ, k = i - r * KZ;
            v[u] = (i < total && r < nr) ? __ldg(zz + (long)(r0 + r) * ld + k) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 12; ++u) {
            const int i = base + u * ZS_THREADS + (int)threadIdx.x;
            const int r = i / KZ, k = i - r * KZ;
            if (i < total) tile[r * ldt + k] = v[u];
        }
    }
}

template <int ZS_ROWS>
__global__ void __cluster_dims__(ZS_CTAS, 1, 1) __launch_bounds__(ZS_THREADS)
    zstats_kernel(const float* __restrict__ zz, long ld, int B, int KZ, float* __restrict__ zsum_out,
                  float* __restrict__ zmean_out, float* __restrict__ zcov_out) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ float zs_sh[];
    const int ldt = KZ + 1;
    float* tile = zs_sh;                    // [ZS_ROWS][KZ + 1]
    float* csum = tile + ZS_ROWS * ldt;     // [KZ]   column sums of this CTA's rows
    float* mean = csum + KZ;                // [KZ]
    float* scratch = mean + KZ;             // [8][KZ]
    float* cpart = scratch + 8 * KZ;        // [KZ * KZ] centred second moments of this CTA's rows
    const int rank = (int)cluster.block_rank();
    const int chunk = (B + ZS_CTAS - 1) / ZS_CTAS;
    const int r_begin = min(B, rank * chunk), r_end = min(B, r_begin + chunk);
    const bool single = chunk <= ZS_ROWS;  // the slice fits one tile: it is read from global memory once
    const float invB = 1.0f / (float)B;
    const int q = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // ---- column sums of the slice
    for (int k = threadIdx.x; k < KZ; k += ZS_THREADS) csum[k] = 0.0f;
    for (int i = threadIdx.x; i < KZ * KZ; i += ZS_THREADS) cpart[i] = 0.0f;
    for (int r0 = r_begin; r0 < r_end || r0 == r_begin; r0 += ZS_ROWS) {
        const int nr = max(0, min(ZS_ROWS, r_end - r0));
        __syncthreads();
        zs_load_tile<ZS_ROWS>(tile, ldt, zz, ld, r0, nr, KZ);
        __syncthreads();
        for (int k = lane; k < KZ; k += 32) {  // 8 row lanes per column, rows beyond nr are zero
            float s = 0.0f;
#pragma unroll
            for (int r = 0; r < ZS_ROWS / 8; ++r) s += tile[(q + 8 * r) * ldt + k];
            scratch[q * KZ + k] = s;
        }
        __syncthreads();
        for (int k = threadIdx.x; k < KZ; k += ZS_THREADS) {
            float s = csum[k];
#pragma unroll
            for (int i = 0; i < 8; ++i) s += scratch[i * KZ + k];
            csum[k] = s;
        }
        if (r0 + ZS_ROWS >= r_end) break;
    }
    cluster.sync();
    for (int k = threadIdx.x; k < KZ; k += ZS_THREADS) {
        float s = 0.0f;
#pragma unroll
        for (int c = 0; c < ZS_CTAS; ++c) s += cluster.map_shared_rank(csum, c)[k];
        mean[k] = s * invB;
        if (rank == 0) {
            zsum_out[k] = s;
            zmean_out[k] = s * invB;
        }
    }
    // ---- centred second moments of the slice
    for (int r0 = r_begin; r0 < r_end; r0 += ZS_ROWS) {
        const int nr = min(ZS_ROWS, r_end - r0);
        __syncthreads();
        if (!single) {
            zs_load_tile<ZS_ROWS>(tile, ldt, zz, ld, r0, nr, KZ);
            __syncthreads();
        }
        for (int i = threadIdx.x; i < ZS_ROWS * KZ; i += ZS_THREADS) {
            const int r = i / KZ, k = i - r * KZ;
            if (r < nr) tile[r * ldt + k] -= mean[k];
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < KZ * KZ; idx += ZS_THREADS) {
            const int i = idx / KZ, j = idx - i * KZ;
            float s = 0.0f;
#pragma unroll 8
            for (int r = 0; r < ZS_ROWS; ++r) s = fmaf(tile[r * ldt + i], tile[r * ldt + j], s);
            cpart[idx] += s;
        }
    }
    cluster.sync();
    for (int idx = rank + ZS_CTAS * threadIdx.x; idx < KZ * KZ; idx += ZS_CTAS * ZS_THREADS) {
        float s = 0.0f;
#pragma unroll
        for (int c = 0; c < ZS_CTAS; ++c) s += cluster.map_shared_rank(cpart, c)[idx];
        zcov_out[idx] = s * invB;
    }
    cluster.sync();  // no CTA may exit while its shared memory is still being read by the others
}

// Larger minibatches (B > 512): the eight-CTA cluster above is bound by its own serial work (35-47 us at 2048 rows, on the critical
// path before the decoders).  Instead: one CTA per 64 rows computes the tile's column sums and its second moments CENTRED ON THE
// TILE'S OWN MEAN, and a merge kernel combines the tiles exactly (Chan et al.):
//   Cov = [ sum_c M2_c + sum_c n_c (mean_c - mean)(mean_c - mean)^T ] / B.
// Deterministic (fixed order), no atomics; part [tiles][KZ + KZ * KZ] is caller-provided scratch.
__global__ void __launch_bounds__(ZS_THREADS) zstats_part_kernel(const float* __restrict__ zz, long ld, int B, int KZ, float* __restrict__ part) {
    extern __shared__ float zs_sh[];
    const int ldt = KZ + 1;
    float* tile = zs_sh;               // [64][KZ + 1]
    float* scratch = tile + 64 * ldt;  // [8][KZ]
    float* lmean = scratch + 8 * KZ;   // [KZ]
    const int r0 = blockIdx.x * 64, nr = min(64, B - r0);
    const int q = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* out = part + (long)blockIdx.x * (KZ + KZ * KZ);
    zs_load_tile<64>(tile, ldt, zz, ld, r0, nr, KZ);
    __syncthreads();
    for (int k = lane; k < KZ; k += 32) {  // 8 row lanes per column, rows beyond nr are zero
        float s = 0.0f;
#pragma unroll
        for (int r = 0; r < 8; ++r) s += tile[(q + 8 * r) * ldt + k];
        scratch[q * KZ + k] = s;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < KZ; k += ZS_THREADS) {
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += scratch[i * KZ + k];
        out[k] = s;
        lmean[k] = s / (float)nr;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * KZ; i += ZS_THREADS) {
        const int r = i / KZ, k = i - r * KZ;
        if (r < nr) tile[r * ldt + k] -= lmean[k];
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < KZ * KZ; idx += ZS_THREADS) {
        const int i = idx / KZ, j = idx - i * KZ;
        float s = 0.0f;
#pragma unroll 8
        for (int r = 0; r < 64; ++r) s = fmaf(tile[r * ldt + i], tile[r * ldt + j], s);
        out[KZ + idx] = s;
    }
}

__global__ void __launch_bounds__(ZS_THREADS) zstats_merge_kernel(const float* __restrict__ part, int tiles, int B, int KZ,
                                                                  float* __restrict__ zsum_out, float* __restrict__ zmean_out,
                                                                  float* __restrict__ zcov_out) {
    extern __shared__ float zm_sh[];
    float* tot = zm_sh;      // [KZ] column sums of the whole minibatch
    float* d = zm_sh + KZ;   // [tiles][KZ] tile mean - minibatch mean
    const long pitch = KZ + (long)KZ * KZ;
    const float invB = 1.0f / (float)B;
    for (int k = threadIdx.x; k < KZ; k += ZS_THREADS) {
        float s = 0.0f;
        for (int c = 0; c < tiles; ++c) s += part[c * pitch + k];
        tot[k] = s;
        if (blockIdx.x == 0) {
            zsum_out[k] = s;
            zmean_out[k] = s * invB;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < tiles * KZ; i += ZS_THREADS) {
        const int c = i / KZ, k = i - c * KZ;
        const float n = (float)min(64, B - 64 * c);
        d[i] = part[c * pitch + k] / n - tot[k] * invB;
    }
    __syncthreads();
    const int idx = blockIdx.x * ZS_THREADS + threadIdx.x;
    if (idx >= KZ * KZ) return;
    const int i = idx / KZ, j = idx - i * KZ;
    float s = 0.0f;
    for (int c = 0; c < tiles; ++c) {
        const float n = (float)min(64, B - 64 * c);
        s += part[c * pitch + KZ + idx] + n * d[c * KZ + i] * d[c * KZ + j];
    }
    zcov_out[idx] = s * invB;
}

struct FoldP {
    const float *Wp, *Ws;
    const float* vec[9];  // per-gene vectors: gamma_p, beta_p, gamma_s, beta_s, px_r, rm_p, rv_p, rm_s, rv_s
    float *rm_p, *rv_p, *rm_s, *rv_s;
    float *wfold, *genec;
    const float *zmean, *zcov;
    // optional: rows [Gp, 3 Gp) of the stacked bf16 operand [3 Gp, ld_wz] (private block then shared block); the folded weights
    // go into the latent columns HD .. HD + P + S of their block, every other entry of those rows stays zero
    __nv_bfloat16* wfold_bf16;
    long ld_wz;
    int Gp, HD;
    int stack_f16;  // the stacked operand holds fp16 (the fused tensor-core decoder) instead of bf16 values
    // optional fp16 operands of the branch-logit MMAs (forward / statistics / training sweeps): wz_f16 [2 Gp, 64] = folded
    // private weights in columns [0, P) of rows [0, G), folded shared weights in columns [P, P + S) of rows [Gp, Gp + G);
    // zc_f16 [B, 64] = zz - m (m = batch mean when training, else 0) in columns [0, P + S).  Centring makes the shift exactly
    // beta and keeps the operand rounding (2^-12) from acting on the common part of the latents.
    __half* wz_f16;
    __half* zc_f16;
    const float* zz;
    long ld_zz;
    int G, P, S, B, training;
    float eps, momentum;
};

// 32 genes per CTA.  All inputs of the CTA arrive in one round of loads; the quadratic forms W C W^T run as one thread per
// (gene, latent index) over T = W C, so every lane is busy (ncu r1: the one-gene-per-warp form used 10 resp. 25 of 32 lanes
// and ~1000 instructions per gene, 5 M warp instructions per launch).
__global__ void __launch_bounds__(256) fold_kernel(FoldP p) {
    extern __shared__ float sh[];
    const int KZ = p.P + p.S;
    const int g0 = blockIdx.x * FOLD_GENES_PER_CTA;
    const int ng = min(FOLD_GENES_PER_CTA, p.G - g0);
    float* scov = sh;                                   // [KZ][KZ]
    float* smean = scov + KZ * KZ;                      // [KZ]
    float* sWp = smean + KZ;                            // [32][P]
    float* sWs = sWp + FOLD_GENES_PER_CTA * p.P;        // [32][S]
    float* svec = sWs + FOLD_GENES_PER_CTA * p.S;       // [9][32]
    float* sT = svec + 9 * FOLD_GENES_PER_CTA;          // [32][KZ]   T = W C (block diagonal)
    float* sA = sT + FOLD_GENES_PER_CTA * KZ;           // [2][32]    folded scale a = gamma invstd; [2][32] centred shift (base 2)
    {
        StageArr<5> c;
        StageArr<1> m;
        StageArr<2> wp;
        StageArr<4> ws;
        float sc[2];
        c.load(p.training ? p.zcov : nullptr, KZ * KZ);
        m.load(p.training ? p.zmean : nullptr, KZ);
        wp.load(p.Wp + (long)g0 * p.P, ng * p.P);
        ws.load(p.Ws + (long)g0 * p.S, ng * p.S);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int i = u * 256 + (int)threadIdx.x, arr = i >> 5, gl = i & 31;
            sc[u] = (arr < 9 && gl < ng) ? __ldg(p.vec[arr] + g0 + gl) : 0.0f;
        }
        c.store(scov, KZ * KZ);
        m.store(smean, KZ);
        wp.store(sWp, ng * p.P);
        ws.store(sWs, ng * p.S);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int i = u * 256 + (int)threadIdx.x;
            if (i < 9 * 32) svec[i] = sc[u];
        }
        StageArr<5>::rest(scov, p.training ? p.zcov : nullptr, KZ * KZ);
        StageArr<1>::rest(smean, p.training ? p.zmean : nullptr, KZ);
        StageArr<2>::rest(sWp, p.Wp + (long)g0 * p.P, ng * p.P);
        StageArr<4>::rest(sWs, p.Ws + (long)g0 * p.S, ng * p.S);
    }
    __syncthreads();
    const long G = p.G;
    // T[gl][k] = sum_l C[k][l] W[gl][l]  (l within k's block)
    if (p.training) {
        for (int i = threadIdx.x; i < ng * KZ; i += 256) {
            const int gl = i / KZ, k = i - gl * KZ;
            const bool pr = k < p.P;
            const int K = pr ? p.P : p.S, off = pr ? 0 : p.P;
            const float* W = pr ? sWp + gl * p.P : sWs + gl * p.S;
            const float* C = scov + k * KZ + off;
            float t = 0.0f;
#pragma unroll 5
            for (int l = 0; l < K; ++l) t = fmaf(C[l], W[l], t);
            sT[i] = t;
        }
        __syncthreads();
    }
    // per (gene, branch): batch statistics of u = z W^T, running-statistics update, folded scale and shift
    if (threadIdx.x < 2 * FOLD_GENES_PER_CTA) {
        const int br = threadIdx.x >> 5, gl = threadIdx.x & 31;
        if (gl < ng) {
            const int g = g0 + gl;
            const int K = br == 0 ? p.P : p.S, off = br == 0 ? 0 : p.P;
            const float* W = br == 0 ? sWp + gl * p.P : sWs + gl * p.S;
            const float gamma = svec[(br == 0 ? 0 : 2) * 32 + gl], beta = svec[(br == 0 ? 1 : 3) * 32 + gl];
            float mean = svec[(br == 0 ? 5 : 7) * 32 + gl], var = svec[(br == 0 ? 6 : 8) * 32 + gl];  // running statistics
            if (p.training) {
                float bmean = 0.0f, bvar = 0.0f;
                for (int k = 0; k < K; ++k) {
                    bmean = fmaf(smean[off + k], W[k], bmean);
                    bvar = fmaf(W[k], sT[gl * KZ + off + k], bvar);
                }
                bvar = fmaxf(bvar, 0.0f);
                const float unb = bvar * ((float)p.B / (float)max(p.B - 1, 1));
                (br == 0 ? p.rm_p : p.rm_s)[g] = (1.0f - p.momentum) * mean + p.momentum * bmean;
                (br == 0 ? p.rv_p : p.rv_s)[g] = (1.0f - p.momentum) * var + p.momentum * unb;
                mean = bmean;
                var = bvar;
            }
            const float invstd = 1.0f / sqrtf(var + p.eps);
            const float a = gamma * invstd;
            sA[br * 32 + gl] = a;
            sA[64 + br * 32 + gl] = (p.training ? beta : beta - mean * a) * 1.4426950408889634f;
            p.genec[(br == 0 ? GC_CP : GC_CS) * G + g] = beta - mean * a;
            p.genec[(br == 0 ? GC_CPL : GC_CSL) * G + g] = (beta - mean * a) * 1.4426950408889634f;
            p.genec[(br == 0 ? GC_CPLC : GC_CSLC) * G + g] = (p.training ? beta : beta - mean * a) * 1.4426950408889634f;
            p.genec[(br == 0 ? GC_AP : GC_AS) * G + g] = a;
            p.genec[(br == 0 ? GC_ISTD_P : GC_ISTD_S) * G + g] = invstd;
            p.genec[(br == 0 ? GC_MEAN_P : GC_MEAN_S) * G + g] = mean;
        }
    } else if (threadIdx.x < 3 * FOLD_GENES_PER_CTA) {
        // NB constants of the inverse dispersion: one gene per lane
        const int gl = threadIdx.x - 2 * FOLD_GENES_PER_CTA;
        if (gl < ng) {
            const int g = g0 + gl;
            float th = expf(svec[4 * 32 + gl]);  // reference module/spVIPESmodule.py:758
            const float lte = logf(th + NB_EPS), lgt = lgammaf(th), dgt = digammaf_pos(th);
            p.genec[GC_THETA * G + g] = th;
            p.genec[GC_LTE * G + g] = lte;
            p.genec[GC_LGT * G + g] = lgt;
            p.genec[GC_DGT * G + g] = dgt;
            p.genec[GC_THE * G + g] = th + NB_EPS;
            p.genec[GC_K0 * G + g] = fmaf(th, lte, 0.91893853f - lgt);
            p.genec[GC_K1 * G + g] = lte + th / (th + NB_EPS) - dgt;
            p.genec[GC_KC * G + g] = th * lte;
            p.genec[GC_K1C * G + g] = lte + th / (th + NB_EPS);
        }
    }
    __syncthreads();
    // folded weights W' = a W: fp32 [G, KZ] and the bf16 copy inside the stacked tensor-core operand
    for (int i = threadIdx.x; i < ng * KZ; i += 256) {
        const int gl = i / KZ, k = i - gl * KZ;
        const bool pr = k < p.P;
        const float wf = sA[(pr ? 0 : 32) + gl] * (pr ? sWp[gl * p.P + k] : sWs[gl * p.S + (k - p.P)]);
        const int g = g0 + gl;
        p.wfold[(long)g * KZ + k] = wf;
        if (p.wfold_bf16) {
            const long at = ((long)(pr ? 0 : 1) * p.Gp + g) * p.ld_wz + p.HD + k;
            if (p.stack_f16) reinterpret_cast<__half*>(p.wfold_bf16)[at] = to_half_sat(wf);
            else p.wfold_bf16[at] = __float2bfloat16(wf);
        }
        // branch operand of the likelihood kernels: base-2 units (decoder_common.cuh, ZK_*)
        if (p.wz_f16) p.wz_f16[((long)(pr ? 0 : 1) * p.Gp + g) * 64 + k] = to_half_sat(wf * 1.4426950408889634f);
    }
    if (p.wz_f16) {  // the additive columns of the branch k-block: (shift hi, shift lo) against ones, ones against (R hi, R lo)
        for (int i = threadIdx.x; i < 2 * ng * 6; i += 256) {
            const int br = i / (ng * 6), r = i - br * ng * 6, gl = r / 6, c = r - gl * 6;
            const float sh = sA[64 + br * 32 + gl];
            const __half hi = to_half_sat(sh);
            __half v;
            if (c == 0) v = hi;
            else if (c == 1) v = to_half_sat(sh - __half2float(hi));
            else v = __float2half_rn(((c < 4) == (br == 0)) ? 1.0f : 0.0f);
            p.wz_f16[((long)br * p.Gp + g0 + gl) * 64 + ZK_ONE + c] = v;
        }
    }
    if (p.zc_f16) {  // centred latents: the CTAs share the rows; ones in the shift columns, zeros elsewhere (the R columns are
                     // filled by the row-statistics kernel after the normaliser sweep, which must see them as zero)
        for (long i = (long)blockIdx.x * 256 + threadIdx.x; i < (long)p.B * 64; i += (long)gridDim.x * 256) {
            const int b = (int)(i >> 6), k = (int)(i & 63);
            float v = 0.0f;
            if (k < KZ) v = __ldg(p.zz + (long)b * p.ld_zz + k) - (p.training ? smean[k] : 0.0f);
            else if (k == ZK_ONE || k == ZK_ONE + 1) v = 1.0f;
            p.zc_f16[i] = to_half_sat(v);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Count tables of the tensor-core likelihood kernels (decoder_common.cuh, NB_TAB): they depend on the inverse dispersion only,
// i.e. on a parameter, not on the minibatch, so they are computed beside the encoders, off the critical path.  Evaluated in
// double: lgamma(t + theta) - lgamma(theta) cancels badly in fp32 once theta is large.
// ---------------------------------------------------------------------------------------
__device__ double digamma_d(double x) {
    double r = 0.0;
    while (x < 8.0) {
        r -= 1.0 / x;
        x += 1.0;
    }
    const double f = 1.0 / (x * x);
    return r + log(x) - 0.5 / x - f * (1.0 / 12.0 - f * (1.0 / 120.0 - f * (1.0 / 252.0 - f * (1.0 / 240.0 - f * (1.0 / 132.0)))));
}

__global__ void __launch_bounds__(256) theta_tables_kernel(const float* __restrict__ px_r, int G, float2* __restrict__ tgf,
                                                           float* __restrict__ tb1) {
    const int i = blockIdx.x * 256 + threadIdx.x;  // entry (gene, count): 16 consecutive threads share a gene
    const int g = i / NB_TAB, c = i - g * NB_TAB;
    if (g >= G) return;
    const float thf = expf(__ldg(px_r + g));  // reference module/spVIPESmodule.py:758 (the same fp32 value as GC_THETA)
    float2 f = make_float2(0.0f, 0.0f);
    float b = 0.0f;
    if (c > 0) {
        const double th = (double)thf;
        const float tf = log1pf((float)c);  // the fp32 value the reference's log1p produces
        const double t = (double)tf;
        f = make_float2(tf, (float)(lgamma(t + th) - lgamma(th) - lgamma(t + 1.0)));
        b = (float)(digamma_d(t + th) - digamma_d(th));
    }
    if (tgf) tgf[i] = f;
    if (tb1) tb1[i] = b;
}

extern "C" int spv_dec_theta_tables(const float* px_r, int G, void* tgf, float* tb1, void* stream) {
    if (!px_r || G <= 0 || (!tgf && !tb1)) return SPV_ERR_ARG;
    theta_tables_kernel<<<(G * NB_TAB + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        px_r, G, reinterpret_cast<float2*>(tgf), tb1);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// ptrs: Wp, Ws, gamma_p, beta_p, gamma_s, beta_s, px_r, rm_p, rv_p, rm_s, rv_s, zz, zsum, (unused), wfold, genec, zmean, zcov
extern "C" int spv_dec_fold(const void* const* ptrs, long long ld_zz, int B, int G, int P, int S, int training, float eps,
                            float momentum, void* wz_bf16, long long ld_wz, int Gp, int HD, void* wz_f16, void* zc_f16, void* stream) {
    if (!ptrs || B <= 0 || G <= 0 || P <= 0 || S <= 0 || P + S > DEC_MAX_LATENT) return SPV_ERR_ARG;
    for (int i = 0; i < 18; ++i)
        if (!ptrs[i]) return SPV_ERR_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int KZ = P + S;
    const float* zz = (const float*)ptrs[11];
    if (training) {
        const int chunk = (B + ZS_CTAS - 1) / ZS_CTAS;
        const int zrows = chunk <= 64 ? 64 : (chunk <= 128 ? 128 : 256);
        const int tiles = (B + 63) / 64;
        const size_t sm_merge = (size_t)(KZ + tiles * KZ) * sizeof(float);
        if (B > 512 && sm_merge <= 200 * 1024) {  // one CTA per 64 rows + an exact merge (scratch: ptrs[13])
            float* part = (float*)ptrs[13];
            const size_t sm_part = (size_t)(64 * (KZ + 1) + 9 * KZ) * sizeof(float);
            zstats_part_kernel<<<tiles, ZS_THREADS, sm_part, st>>>(zz, ld_zz, B, KZ, part);
            SPV_CHECK_LAUNCH();
            if (sm_merge > 48 * 1024) cudaFuncSetAttribute(zstats_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_merge);
            zstats_merge_kernel<<<(KZ * KZ + ZS_THREADS - 1) / ZS_THREADS, ZS_THREADS, sm_merge, st>>>(part, tiles, B, KZ, (float*)ptrs[12],
                                                                                                   (float*)ptrs[16], (float*)ptrs[17]);
            SPV_CHECK_LAUNCH();
        } else {
            const size_t sm1 = (size_t)(zrows * (KZ + 1) + 10 * KZ + KZ * KZ) * sizeof(float);
            float *zsum = (float*)ptrs[12], *zmean = (float*)ptrs[16], *zcov = (float*)ptrs[17];
            if (zrows == 64) {
                if (sm1 > 48 * 1024) cudaFuncSetAttribute(zstats_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1);
                zstats_kernel<64><<<ZS_CTAS, ZS_THREADS, sm1, st>>>(zz, ld_zz, B, KZ, zsum, zmean, zcov);
            } else if (zrows == 128) {
                if (sm1 > 48 * 1024) cudaFuncSetAttribute(zstats_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1);
                zstats_kernel<128><<<ZS_CTAS, ZS_THREADS, sm1, st>>>(zz, ld_zz, B, KZ, zsum, zmean, zcov);
            } else {
                if (sm1 > 48 * 1024) cudaFuncSetAttribute(zstats_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1);
                zstats_kernel<256><<<ZS_CTAS, ZS_THREADS, sm1, st>>>(zz, ld_zz, B, KZ, zsum, zmean, zcov);
            }
            SPV_CHECK_LAUNCH();
        }
    }
    FoldP p;
    p.Wp = (const float*)ptrs[0]; p.Ws = (const float*)ptrs[1];
    for (int i = 0; i < 5; ++i) p.vec[i] = (const float*)ptrs[2 + i];
    for (int i = 0; i < 4; ++i) p.vec[5 + i] = (const float*)ptrs[7 + i];
    p.rm_p = (float*)ptrs[7]; p.rv_p = (float*)ptrs[8]; p.rm_s = (float*)ptrs[9]; p.rv_s = (float*)ptrs[10];
    p.wfold = (float*)ptrs[14]; p.genec = (float*)ptrs[15];
    p.zmean = (const float*)ptrs[16]; p.zcov = (const float*)ptrs[17];
    p.wfold_bf16 = reinterpret_cast<__nv_bfloat16*>(wz_bf16);
    p.ld_wz = ld_wz; p.Gp = Gp; p.HD = HD;
    if ((wz_f16 != nullptr) != (zc_f16 != nullptr) || (wz_f16 && KZ > ZK_MAX_LATENT)) return SPV_ERR_ARG;
    p.wz_f16 = reinterpret_cast<__half*>(wz_f16); p.zc_f16 = reinterpret_cast<__half*>(zc_f16);
    p.zz = zz; p.ld_zz = ld_zz;
    p.stack_f16 = wz_f16 != nullptr;  // fp16 branch operands requested: the whole decoder runs on fp16 operands
    p.G = G; p.P = P; p.S = S; p.B = B; p.training = training; p.eps = eps; p.momentum = momentum;
    size_t sm2 = (size_t)(KZ + KZ * KZ + FOLD_GENES_PER_CTA * (2 * KZ + 13)) * sizeof(float);
    if (sm2 > 48 * 1024) cudaFuncSetAttribute(fold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2);
    fold_kernel<<<(G + FOLD_GENES_PER_CTA - 1) / FOLD_GENES_PER_CTA, 256, sm2, st>>>(p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// ---------------------------------------------------------------------------------------
// per-gene backward of the two folded BatchNorm+Linear branches (closed form):
//   Q = dy^T z (from spv_gemm), sdy = colsum(dy):  S2 = (Q.W - sdy mean_u) invstd = dgamma,  dbeta = sdy,
//   dW = a (Q - sdy zbar - S2 invstd Cov W)
// and the per-CTA partial sums of the two operands of the d z correction (BatchNorm couples all cells of a gene):
//   v1[c]   = sum_g (a sdy / B) W[g, c]                 -> vpart[cta, c]
//   M[k, l] = sum_g (a S2 invstd / B) W[g, k] W[g, l]   -> mpart[cta, k * KZ + l]   (block diagonal: private, shared)
// also d px_r = theta * colsum(dtheta), d bm = colsum(dpi).
// ---------------------------------------------------------------------------------------
struct GeneBwdP {
    const float *Wp, *Ws, *Qp, *Qs, *zmean, *zcov;
    const float* vec[11];  // per-gene vectors: genec a_p, a_s, invstd_p, invstd_s, mean_p, mean_s, theta; colsum rows 0..3
    long vstride[11];      // element stride of each (1; ldq for the two branch column sums when they ride behind Qp / Qs)
    float *dWp, *dWs, *dgp, *dbp, *dgs, *dbs, *dpx_r, *dbm, *vpart, *mpart;
    int G, P, S, B;
    long ldq;  // row pitch of Qp / Qs (0: packed, P resp. S)
};

// 32 genes per CTA, 256 threads.  One round of loads brings in every input; T = W C runs as one thread per (gene, latent
// index); the per-CTA partial of M is a rank-32 update computed on its upper triangle only.
__global__ void __launch_bounds__(GENE_BWD_THREADS) gene_bwd_kernel(GeneBwdP p) {
    extern __shared__ float sh[];
    const int KZ = p.P + p.S;
    const int g0 = blockIdx.x * GENES_PER_CTA;
    const int ng = min(GENES_PER_CTA, p.G - g0);
    const long G = p.G;
    const int pitch_p = p.ldq > 0 ? (int)p.ldq : p.P, pitch_s = p.ldq > 0 ? (int)p.ldq : p.S;
    const int nQp = (ng - 1) * pitch_p + p.P, nQs = (ng - 1) * pitch_s + p.S;
    float* scov = sh;                                   // [KZ][KZ]
    float* smean = scov + KZ * KZ;                      // [KZ]
    float* sWp = smean + KZ;                            // [32][P]
    float* sWs = sWp + GENES_PER_CTA * p.P;             // [32][S]
    float* sQp = sWs + GENES_PER_CTA * p.S;             // [32][pitch_p]
    float* sQs = sQp + GENES_PER_CTA * pitch_p;         // [32][pitch_s]
    float* svec = sQs + GENES_PER_CTA * pitch_s;        // [11][32]
    float* sT = svec + 11 * GENES_PER_CTA;              // [32][KZ]   T = W C (block diagonal)
    float* sc1 = sT + GENES_PER_CTA * KZ;               // [2][32]    a S2 invstd          (scale of the T term of dW)
    float* scv = sc1 + 2 * GENES_PER_CTA;               // [2][32]    a sdy / B            (weights of v1)
    float* scm = scv + 2 * GENES_PER_CTA;               // [2][32]    a S2 invstd / B      (weights of M)
    {
        StageArr<5> c, qp, qs;
        StageArr<1> m;
        StageArr<2> wp;
        StageArr<4> ws;
        float sc[2];
        c.load(p.zcov, KZ * KZ);
        m.load(p.zmean, KZ);
        wp.load(p.Wp + (long)g0 * p.P, ng * p.P);
        ws.load(p.Ws + (long)g0 * p.S, ng * p.S);
        qp.load(p.Qp + (long)g0 * pitch_p, nQp);
        qs.load(p.Qs + (long)g0 * pitch_s, nQs);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int i = u * GENE_BWD_THREADS + (int)threadIdx.x, arr = i >> 5, gl = i & 31;
            sc[u] = (arr < 11 && gl < ng) ? __ldg(p.vec[arr] + (long)(g0 + gl) * p.vstride[arr]) : 0.0f;
        }
        c.store(scov, KZ * KZ);
        m.store(smean, KZ);
        wp.store(sWp, ng * p.P);
        ws.store(sWs, ng * p.S);
        qp.store(sQp, nQp);
        qs.store(sQs, nQs);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int i = u * GENE_BWD_THREADS + (int)threadIdx.x;
            if (i < 11 * 32) svec[i] = sc[u];
        }
        StageArr<5>::rest(scov, p.zcov, KZ * KZ);
        StageArr<1>::rest(smean, p.zmean, KZ);
        StageArr<2>::rest(sWp, p.Wp + (long)g0 * p.P, ng * p.P);
        StageArr<4>::rest(sWs, p.Ws + (long)g0 * p.S, ng * p.S);
        StageArr<5>::rest(sQp, p.Qp + (long)g0 * pitch_p, nQp);
        StageArr<5>::rest(sQs, p.Qs + (long)g0 * pitch_s, nQs);
    }
    __syncthreads();
    // T[gl][k] = sum_l C[k][l] W[gl][l]  (l within k's block)
    for (int i = threadIdx.x; i < ng * KZ; i += GENE_BWD_THREADS) {
        const int gl = i / KZ, k = i - gl * KZ;
        const bool pr = k < p.P;
        const int K = pr ? p.P : p.S, off = pr ? 0 : p.P;
        const float* W = pr ? sWp + gl * p.P : sWs + gl * p.S;
        const float* C = scov + k * KZ + off;
        float t = 0.0f;
#pragma unroll 5
        for (int l = 0; l < K; ++l) t = fmaf(C[l], W[l], t);
        sT[i] = t;
    }
    // per (gene, branch): S2 = (Q . W - sdy mean_u) invstd = dgamma, dbeta = sdy
    const float invB = 1.0f / (float)p.B;
    if (threadIdx.x < 2 * GENES_PER_CTA) {
        const int br = threadIdx.x >> 5, gl = threadIdx.x & 31;
        if (gl < ng) {
            const int g = g0 + gl;
            const int K = br == 0 ? p.P : p.S;
            const float* W = br == 0 ? sWp + gl * p.P : sWs + gl * p.S;
            const float* Q = br == 0 ? sQp + gl * pitch_p : sQs + gl * pitch_s;
            const float a = svec[(0 + br) * 32 + gl], invstd = svec[(2 + br) * 32 + gl], mean_u = svec[(4 + br) * 32 + gl];
            const float sdy = svec[(7 + br) * 32 + gl];
            float qw = 0.0f;
            for (int k = 0; k < K; ++k) qw = fmaf(Q[k], W[k], qw);
            const float S2 = (qw - sdy * mean_u) * invstd;
            (br == 0 ? p.dgp : p.dgs)[g] = S2;
            (br == 0 ? p.dbp : p.dbs)[g] = sdy;
            sc1[br * 32 + gl] = a * S2 * invstd;
            scv[br * 32 + gl] = a * sdy * invB;
            scm[br * 32 + gl] = a * S2 * invB * invstd;
        } else {
            sc1[br * 32 + gl] = 0.0f; scv[br * 32 + gl] = 0.0f; scm[br * 32 + gl] = 0.0f;
        }
    } else if (threadIdx.x < 3 * GENES_PER_CTA) {
        const int gl = threadIdx.x - 2 * GENES_PER_CTA;
        if (gl < ng) {
            p.dpx_r[g0 + gl] = svec[6 * 32 + gl] * svec[10 * 32 + gl];  // theta * colsum(d theta)
            p.dbm[g0 + gl] = svec[9 * 32 + gl];                         // colsum(d pi)
        }
    }
    __syncthreads();
    // dW[g, k] = a (Q[g, k] - sdy zbar[k]) - (a S2 invstd) T[g, k]
    for (int i = threadIdx.x; i < ng * KZ; i += GENE_BWD_THREADS) {
        const int gl = i / KZ, k = i - gl * KZ;
        const bool pr = k < p.P;
        const int br = pr ? 0 : 1, kr = pr ? k : k - p.P;
        const float a = svec[br * 32 + gl], sdy = svec[(7 + br) * 32 + gl];
        const float q = pr ? sQp[gl * pitch_p + kr] : sQs[gl * pitch_s + kr];
        const float v = a * (q - sdy * smean[k]) - sc1[br * 32 + gl] * sT[i];
        (pr ? p.dWp + (long)(g0 + gl) * p.P : p.dWs + (long)(g0 + gl) * p.S)[kr] = v;
    }
    // per-CTA partials: v1[c] = sum_g cv[g] W[g, c];  M[k, l] = sum_g cm[g] W[g, k] W[g, l] (symmetric: upper triangle, mirrored)
    for (int c = threadIdx.x; c < KZ; c += GENE_BWD_THREADS) {
        const bool pr = c < p.P;
        const float* cv = scv + (pr ? 0 : 32);
        const float* Wc = pr ? sWp + c : sWs + (c - p.P);
        const int K = pr ? p.P : p.S;
        float s = 0.0f;
        for (int gl = 0; gl < ng; ++gl) s = fmaf(cv[gl], Wc[gl * K], s);
        p.vpart[(long)blockIdx.x * KZ + c] = s;
    }
    const int nP = p.P * (p.P + 1) / 2, nS = p.S * (p.S + 1) / 2;
    for (int idx = threadIdx.x; idx < nP + nS; idx += GENE_BWD_THREADS) {
        const bool pr = idx < nP;
        const int K = pr ? p.P : p.S, o = pr ? 0 : p.P;
        int j = pr ? idx : idx - nP;
        // (k, l) with k <= l from the triangular index j = k K - k (k - 1) / 2 + (l - k)
        int k = 0;
        while (j >= K - k) { j -= K - k; ++k; }
        const int l = k + j;
        const float* cm = scm + (pr ? 0 : 32);
        const float* Wb = pr ? sWp : sWs;
        float s = 0.0f;
#pragma unroll 4
        for (int gl = 0; gl < ng; ++gl) s = fmaf(cm[gl] * Wb[gl * K + k], Wb[gl * K + l], s);
        float* M = p.mpart + (long)blockIdx.x * KZ * KZ;
        M[(o + k) * KZ + o + l] = s;
        M[(o + l) * KZ + o + k] = s;
    }
}

extern "C" int spv_dec_gene_bwd_parts(int G) { return G > 0 ? (G + GENES_PER_CTA - 1) / GENES_PER_CTA : 0; }

// ptrs: Wp, Ws, Qp, Qs, genec, colsum, zmean, zcov, dWp, dWs, dgamma_p, dbeta_p, dgamma_s, dbeta_s, dpx_r, dbm,
//       vpart [parts, KZ], mpart [parts, KZ*KZ]   with parts = spv_dec_gene_bwd_parts(G)
// colsum_in_q != 0 (needs ldq > 0): the column sums of dyp / dys are not rows 0 / 1 of colsum but the column right behind each Q
// block, Qp[g * ldq + P] and Qs[g * ldq + S] (the ones column of the single-sweep Q GEMM, spv_dec_zq4)
extern "C" int spv_dec_gene_bwd(const void* const* ptrs, long long ldq, int B, int G, int P, int S, int colsum_in_q, void* stream) {
    if (!ptrs || B <= 0 || G <= 0 || P <= 0 || S <= 0 || P + S > DEC_MAX_LATENT) return SPV_ERR_ARG;
    for (int i = 0; i < 18; ++i)
        if (!ptrs[i]) return SPV_ERR_ARG;
    GeneBwdP p;
    p.Wp = (const float*)ptrs[0]; p.Ws = (const float*)ptrs[1]; p.Qp = (const float*)ptrs[2]; p.Qs = (const float*)ptrs[3];
    const float* genec = (const float*)ptrs[4];
    const float* colsum = (const float*)ptrs[5];
    const int gc_rows[7] = {GC_AP, GC_AS, GC_ISTD_P, GC_ISTD_S, GC_MEAN_P, GC_MEAN_S, GC_THETA};
    for (int i = 0; i < 7; ++i) p.vec[i] = genec + (long)gc_rows[i] * G;
    for (int i = 0; i < 4; ++i) p.vec[7 + i] = colsum + (long)i * G;
    for (int i = 0; i < 11; ++i) p.vstride[i] = 1;
    if (colsum_in_q) {
        if (ldq <= 0) return SPV_ERR_ARG;
        p.vec[7] = p.Qp + P; p.vec[8] = p.Qs + S;
        p.vstride[7] = p.vstride[8] = ldq;
    }
    p.zmean = (const float*)ptrs[6];
    p.zcov = (const float*)ptrs[7]; p.dWp = (float*)ptrs[8]; p.dWs = (float*)ptrs[9]; p.dgp = (float*)ptrs[10];
    p.dbp = (float*)ptrs[11]; p.dgs = (float*)ptrs[12]; p.dbs = (float*)ptrs[13]; p.dpx_r = (float*)ptrs[14];
    p.dbm = (float*)ptrs[15]; p.vpart = (float*)ptrs[16]; p.mpart = (float*)ptrs[17];
    p.G = G; p.P = P; p.S = S; p.B = B; p.ldq = ldq;
    const int KZ = P + S;
    const int pitch = ldq > 0 ? (int)ldq : (P > S ? P : S);
    size_t smem = (size_t)(KZ + KZ * KZ + GENES_PER_CTA * (2 * KZ + 2 * pitch + 11 + 6)) * sizeof(float);
    if (smem > 48 * 1024) cudaFuncSetAttribute(gene_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    gene_bwd_kernel<<<(G + GENES_PER_CTA - 1) / GENES_PER_CTA, GENE_BWD_THREADS, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// dzz[b, c] = dmix[b, c] + dzraw[b, c] - v1[c] - sum_l M[c, l] (zz[b, l] - zbar[l])   (l within c's branch block)
//   dmix: the zz columns of d Amix (mixture GEMM);  dzraw: further addends (dy W' of the softmax branches when they are
//   not part of dmix already, and dah Wh of the mixing net's hidden layer), may be null;
//   v1 / M: sums over the `nparts` per-CTA partials written by spv_dec_gene_bwd (fixed order: deterministic).
// One latent column per CTA (blockIdx.x) and 256 rows (blockIdx.y): the CTA only needs row c of M, i.e. at most
// max(P, S) + 1 sums over the partials, taken by 8 part lanes x 32 entries and combined in lane order.
#define DZC_THREADS 256
__global__ void __launch_bounds__(DZC_THREADS) dzz_combine_kernel(const float* __restrict__ dmix, long ld_dmix,
                                                                  const float* __restrict__ dzraw, const float* __restrict__ vpart,
                                                                  const float* __restrict__ mpart, int nparts,
                                                                  const float* __restrict__ zz, long ld_zz,
                                                                  const float* __restrict__ zmean, float* __restrict__ dzz, int B,
                                                                  int P, int S, const float* __restrict__ raw_colsum) {
    __shared__ float red[8][100];
    __shared__ float srow[100];  // [0, n): M[c, lo + .],  [n]: v1[c]
    const int KZ = P + S;
    const int c = blockIdx.x;
    const int lo = c < P ? 0 : P, n = c < P ? P : S;
    const int lane = threadIdx.x & 31, q = threadIdx.x >> 5;
    for (int e0 = 0; e0 <= n; e0 += 32) {
        const int e = e0 + lane;
        float s = 0.0f;
        if (e <= n) {
            const float* src = e < n ? mpart + (long)c * KZ + lo + e : vpart + c;
            const long pitch = e < n ? (long)KZ * KZ : KZ;
#pragma unroll 4
            for (int t = q; t < nparts; t += 8) s += src[(long)t * pitch];
            red[q][e] = s;
        }
    }
    __syncthreads();
    if (threadIdx.x <= n) {
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += red[i][threadIdx.x];
        srow[threadIdx.x] = s;
    }
    __syncthreads();
    if (raw_colsum) {
        // v1 is the column mean of the uncorrected input gradient sum_g a dy W (BatchNorm backward: the corrected one sums to
        // zero over the minibatch).  dzraw came out of a reduced-precision GEMM while vpart is exact fp32, so subtracting the
        // exact v1 would leave the GEMM's coherent rounding error as a spurious column mean; the mean of dzraw itself cancels
        // exactly (its other addend, the hidden layer's BatchNorm backward, has zero column mean as well).
        if (threadIdx.x == 0) srow[n] = __ldg(raw_colsum + c) / (float)B;
        __syncthreads();
    }
    const int b = blockIdx.y * DZC_THREADS + threadIdx.x;
    if (b >= B) return;
    const float* zrow = zz + (long)b * ld_zz + lo;
    float corr = 0.0f;
    for (int l = 0; l < n; ++l) corr = fmaf(srow[l], zrow[l] - zmean[lo + l], corr);
    dzz[(long)b * KZ + c] = (dmix ? dmix[(long)b * ld_dmix + c] : 0.0f) + (dzraw ? dzraw[(long)b * KZ + c] : 0.0f) - srow[n] - corr;
}

extern "C" int spv_dec_dzz_combine(const float* dmix, long long ld_dmix, const float* dzraw, const float* vpart, const float* mpart,
                                   int nparts, const float* zz, long long ld_zz, const float* zmean, float* dzz, int B, int P,
                                   int S, const float* raw_colsum, void* stream) {
    if (!vpart || !mpart || !zz || !zmean || !dzz || B <= 0 || P <= 0 || S <= 0 || nparts <= 0 || P > 96 || S > 96)
        return SPV_ERR_ARG;
    if (raw_colsum && !dzraw) return SPV_ERR_ARG;
    dim3 grid(P + S, (B + DZC_THREADS - 1) / DZC_THREADS);
    dzz_combine_kernel<<<grid, DZC_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(dmix, ld_dmix, dzraw, vpart, mpart, nparts,
                                                                                         zz, ld_zz, zmean, dzz, B, P, S, raw_colsum);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}
