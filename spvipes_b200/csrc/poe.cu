// Product-of-experts stage: pairing indices (integer work, bit-exact), the Gaussian PoE merge of
// the shared posteriors, reparameterised sampling and the four KL terms in one warp-level pass,
// plus its backward.  Reference: module/spVIPESmodule.py:583-718 (_label_based_poe), :282-379
// (_poe2), :511-581 (_paired_poe, _product_of_experts), :474-482 (_get_batch_transport_plans),
// :184-280 (_cluster_based_poe), :841-868 (KL terms).
#include <cuda_bf16.h>
#include "common.cuh"
#include "../../include/spvipes_b200.h"

// ---------------------------------------------------------------------------------------
// label pairing: row i of group a (label L, rank r among the label-L rows of a, minibatch
// order) is paired with the rank-r label-L row of group b; PAD if b has the label but fewer
// rows, ABSENT if b's minibatch lacks the label (reference :599-659, :685-701, _poe2 :297-326)
// ---------------------------------------------------------------------------------------
__global__ void pair_label_kernel(const int* __restrict__ la, const int* __restrict__ lb, const int* __restrict__ rows_a,
                                  const int* __restrict__ rows_b, int Ba, int Bb, int* __restrict__ pa, int* __restrict__ pb) {
    extern __shared__ int sl[];
    int* sa = sl;
    int* sb = sl + Ba;
    for (int i = threadIdx.x; i < Ba; i += blockDim.x) sa[i] = la[rows_a ? rows_a[i] : i];
    for (int i = threadIdx.x; i < Bb; i += blockDim.x) sb[i] = lb[rows_b ? rows_b[i] : i];
    __syncthreads();
    // one warp per row: 32 labels are compared per step with a ballot
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= Ba + Bb) return;
    const bool side_a = row < Ba;
    const int i = side_a ? row : row - Ba;
    const int* own = side_a ? sa : sb;
    const int* oth = side_a ? sb : sa;
    const int n_oth = side_a ? Bb : Ba;
    const int l = own[i];
    int rank = 0;  // number of earlier rows of this group with the same label
    for (int k0 = 0; k0 < i; k0 += 32) {
        int k = k0 + lane;
        rank += __popc(__ballot_sync(0xffffffffu, k < i && own[k] == l));
    }
    int found = SPV_PARTNER_ABSENT, seen = 0;
    for (int j0 = 0; j0 < n_oth; j0 += 32) {
        int j = j0 + lane;
        unsigned m = __ballot_sync(0xffffffffu, j < n_oth && oth[j] == l);
        int c = __popc(m);
        if (c) found = SPV_PARTNER_PAD;
        if (seen + c > rank) {  // the (rank - seen)-th set bit of m is the partner
            found = j0 + __fns(m, 0, rank - seen + 1);
            break;
        }
        seen += c;
    }
    if (lane == 0) (side_a ? pa : pb)[i] = found;
}

extern "C" int spv_pair_label(const int* la, const int* lb, const int* rows_a, const int* rows_b, int Ba, int Bb, int* pa,
                              int* pb, void* stream) {
    if (!la || !lb || !pa || !pb || Ba <= 0 || Bb <= 0) return SPV_ERR_ARG;
    size_t smem = (size_t)(Ba + Bb) * sizeof(int);
    if (smem > 200 * 1024) return SPV_ERR_ARG;
    if (smem > 48 * 1024) cudaFuncSetAttribute(pair_label_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int blocks = (Ba + Bb + 7) / 8;  // 8 warps per CTA, one warp per row
    pair_label_kernel<<<blocks, 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(la, lb, rows_a, rows_b, Ba, Bb, pa, pb);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// ---------------------------------------------------------------------------------------
// transport plan: sub = T[idx0][:, idx1]  (reference :474-482), then
// row_arg[i] = argmax_j sub[i, j], col_arg[j] = argmax_i sub[i, j]  (reference :526-527;
// ties -> first index, as torch.argmax)
// ---------------------------------------------------------------------------------------
__global__ void plan_gather_kernel(const float* __restrict__ T, long ldT, const int* __restrict__ idx0,
                                   const int* __restrict__ idx1, int B0, int B1, float* __restrict__ sub) {
    int i = blockIdx.x;
    const float* row = T + (long)idx0[i] * ldT;
    for (int j = threadIdx.x; j < B1; j += blockDim.x) sub[(long)i * B1 + j] = __ldg(row + idx1[j]);
}

// the same from a plan stored as bf16 (a 200k x 200k plan is 160 GB in fp32, 80 GB in bf16: the cluster mode, which only
// uses row-normalised weights of the sub-plan, tolerates the 2^-9 rounding; the paired mode's bit-exact argmax keeps fp32)
__global__ void plan_gather_bf16_kernel(const __nv_bfloat16* __restrict__ T, long ldT, const int* __restrict__ idx0,
                                        const int* __restrict__ idx1, int B0, int B1, float* __restrict__ sub) {
    int i = blockIdx.x;
    const __nv_bfloat16* row = T + (long)idx0[i] * ldT;
    for (int j = threadIdx.x; j < B1; j += blockDim.x) sub[(long)i * B1 + j] = __bfloat162float(row[idx1[j]]);
}

extern "C" int spv_plan_gather_bf16(const void* T, long long ldT, const int* idx0, const int* idx1, int B0, int B1, float* sub,
                                    void* stream) {
    if (!T || !idx0 || !idx1 || !sub || B0 <= 0 || B1 <= 0) return SPV_ERR_ARG;
    plan_gather_bf16_kernel<<<B0, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(T), ldT, idx0,
                                                                                    idx1, B0, B1, sub);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

extern "C" int spv_plan_gather(const float* T, long long ldT, const int* idx0, const int* idx1, int B0, int B1, float* sub,
                               void* stream) {
    if (!T || !idx0 || !idx1 || !sub || B0 <= 0 || B1 <= 0) return SPV_ERR_ARG;
    plan_gather_kernel<<<B0, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(T, ldT, idx0, idx1, B0, B1, sub);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// strict "greater" of torch.argmax: NaN compares greater than every number, and the FIRST NaN wins
__device__ __forceinline__ bool arg_gt(float a, float b) { return a > b || (isnan(a) && !isnan(b)); }

__global__ void plan_argmax_kernel(const float* __restrict__ sub, int B0, int B1, int* __restrict__ row_arg,
                                   int* __restrict__ col_arg) {
    const int nrow_blocks = (B0 + 7) / 8;
    if ((int)blockIdx.x < nrow_blocks) {  // one warp per row
        int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
        if (i >= B0) return;
        float best = -INFINITY;
        int bj = 0x7fffffff;
        if (lane < B1) { best = sub[(long)i * B1 + lane]; bj = lane; }
        for (int j = lane + 32; j < B1; j += 32) {
            float v = sub[(long)i * B1 + j];
            if (arg_gt(v, best)) { best = v; bj = j; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            float ov = __shfl_xor_sync(0xffffffffu, best, o);
            int oj = __shfl_xor_sync(0xffffffffu, bj, o);
            if (arg_gt(ov, best) || ((ov == best || (isnan(ov) && isnan(best))) && oj < bj)) { best = ov; bj = oj; }
        }
        if (lane == 0) row_arg[i] = bj;
    } else {  // one thread per column
        int j = (blockIdx.x - nrow_blocks) * blockDim.x + threadIdx.x;
        if (j >= B1) return;
        float best = sub[j];
        int bi = 0;
        for (int i = 1; i < B0; ++i) {
            float v = sub[(long)i * B1 + j];
            if (arg_gt(v, best)) { best = v; bi = i; }
        }
        col_arg[j] = bi;
    }
}

extern "C" int spv_plan_argmax(const float* sub, int B0, int B1, int* row_arg, int* col_arg, void* stream) {
    if (!sub || !row_arg || !col_arg || B0 <= 0 || B1 <= 0) return SPV_ERR_ARG;
    int blocks = (B0 + 7) / 8 + (B1 + 255) / 256;
    plan_argmax_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(sub, B0, B1, row_arg, col_arg);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// ---------------------------------------------------------------------------------------
// cluster mode: masked, row-normalised sub-plans (reference :207-219)
//   P1[i, j] = [l0[i] == l1[j]] * norm_row_i(sub[i, j])          [B0, B1]
//   P2[j, i] = [l1[j] == l0[i]] * norm_row_j(sub^T[j, i])        [B1, B0]
//   norm(p) = where(p > 0, p / clamp(rowsum over the mask, 1e-10), p)
// ---------------------------------------------------------------------------------------
__global__ void plan_cluster_rows_kernel(const float* __restrict__ sub, int B0, int B1, const int* __restrict__ l0,
                                         const int* __restrict__ l1, float* __restrict__ P1) {
    __shared__ float red[8];
    int i = blockIdx.x;
    int li = l0[i];
    float s = 0.0f;
    for (int j = threadIdx.x; j < B1; j += blockDim.x)
        if (l1[j] == li) s += sub[(long)i * B1 + j];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    float rs = 0.0f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) rs += red[w];
    rs = fmaxf(rs, 1e-10f);
    for (int j = threadIdx.x; j < B1; j += blockDim.x) {
        float p = sub[(long)i * B1 + j];
        float v = 0.0f;
        if (l1[j] == li) v = p > 0.0f ? p / rs : p;
        P1[(long)i * B1 + j] = v;
    }
}

// Column direction: one CTA per 32 columns (the first version walked each column with one thread and wrote P2 with a stride of
// B0: 0.8 ms at 2048 x 2048).  Phase 1, masked column sums: lanes = columns (coalesced reads), the 8 warps stride the rows,
// partials combined in warp order (deterministic).  Phase 2: the strip is re-read (from L2) in 32 x 32 tiles, normalised and
// written transposed through shared memory, so both the reads of sub and the writes of P2 are coalesced.
__global__ void __launch_bounds__(256) plan_cluster_cols_kernel(const float* __restrict__ sub, int B0, int B1, const int* __restrict__ l0,
                                                                const int* __restrict__ l1, float* __restrict__ P2) {
    __shared__ float part[8][32];
    __shared__ float tile[32][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int j0 = blockIdx.x * 32, j = j0 + lane;
    const int lj = j < B1 ? l1[j] : -1;
    float s = 0.0f;
    if (j < B1)
        for (int i = w; i < B0; i += 8)
            if (l0[i] == lj) s += sub[(long)i * B1 + j];
    part[w][lane] = s;
    __syncthreads();
    float rs = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; ++k) rs += part[k][lane];
    rs = fmaxf(rs, 1e-10f);
    for (int i0 = 0; i0 < B0; i0 += 32) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int i = i0 + w + 8 * r;
            float v = 0.0f;
            if (i < B0 && j < B1 && l0[i] == lj) {
                const float p = sub[(long)i * B1 + j];
                v = p > 0.0f ? p / rs : p;
            }
            tile[w + 8 * r][lane] = v;  // [row of sub][column of sub]
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int jj = j0 + w + 8 * r, i = i0 + lane;
            if (i < B0 && jj < B1) P2[(long)jj * B0 + i] = tile[lane][w + 8 * r];
        }
        __syncthreads();
    }
}

extern "C" int spv_plan_cluster_norm(const float* sub, int B0, int B1, const int* l0, const int* l1, float* P1, float* P2,
                                     void* stream) {
    if (!sub || !l0 || !l1 || !P1 || !P2 || B0 <= 0 || B1 <= 0) return SPV_ERR_ARG;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    plan_cluster_rows_kernel<<<B0, 256, 0, st>>>(sub, B0, B1, l0, l1, P1);
    SPV_CHECK_LAUNCH();
    plan_cluster_cols_kernel<<<(B1 + 31) / 32, 256, 0, st>>>(sub, B0, B1, l0, l1, P2);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// ---------------------------------------------------------------------------------------
// merge + sampling + KL (forward).  One warp per minibatch row, lanes over latent dims.
// ---------------------------------------------------------------------------------------
struct PoeSide {
    // own / partner expert statistics for the shared posterior (loc and logvar, row-major with leading dim)
    const float* own_loc; const float* own_lv; long ld_own;
    const float* oth_loc; const float* oth_lv; long ld_oth;
    // this group's encoder output [B, 2P + 2S] = [loc_p | lv_p | loc_s | lv_s] (post BatchNorm)
    const float* stats; long ld_stats;
    const int* partner;
    const float* eps_p; const float* eps_q;  // explicit noise [B,P], [B,S] or null -> Philox
    float* zpriv; float* poe_loc; float* poe_lv; float* poe_scale; float* zpoe;  // [B,P], 4 x [B,S]
    float* klp; float* klq;  // [B]
    float* zz; long ld_zz;   // decoder input columns [z_private_arg (P) | z_shared_arg (S)]  (quirk Q1)
    int B;
};
struct PoeParams {
    PoeSide side[2];
    int S, P, mode;
    unsigned long long seed;
    const int* step;
};

__device__ __forceinline__ int zz_col_of_c(int ci, int S, int P) {  // c = [z_priv (P) | z_poe (S)];  zz = [c[S:S+P] | c[:S]]
    return ci >= S ? ci - S : P + ci;
}

__global__ void __launch_bounds__(256) poe_fwd_kernel(PoeParams p) {
    const PoeSide& s = p.side[blockIdx.y];
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= s.B) return;
    const int S = p.S, P = p.P;
    const unsigned int stp = p.step ? (unsigned int)*p.step : 0u;
    // ---- private posterior: sample + KL (reference nn/networks.py:125-127, module :841-856)
    float klp = 0.0f;
    for (int d = lane; d < P; d += 32) {
        float loc = s.stats[(long)row * s.ld_stats + d];
        float lv = s.stats[(long)row * s.ld_stats + P + d];
        float sc = expf(0.5f * lv);
        float e = s.eps_p ? s.eps_p[(long)row * P + d]
                          : philox_normal(p.seed, 2u * blockIdx.y, stp, (unsigned long long)row * P + d);
        float z = loc + sc * e;
        s.zpriv[(long)row * P + d] = z;
        s.zz[(long)row * s.ld_zz + zz_col_of_c(d, S, P)] = z;
        float vr = sc * sc;
        klp += 0.5f * (vr + loc * loc - 1.0f - logf(vr));
    }
    klp = warp_sum(klp);
    // ---- shared posterior: product of experts
    const int pr = s.partner ? s.partner[row] : SPV_PARTNER_ABSENT;
    float klq = 0.0f;
    for (int d = lane; d < S; d += 32) {
        float mu, jlv, sc;
        if (p.mode == SPV_POE_CLUSTER && pr == SPV_PARTNER_ABSENT) {
            // cluster present in this group only: own statistics pass through (reference :233-244)
            mu = s.stats[(long)row * s.ld_stats + 2 * P + d];
            jlv = s.stats[(long)row * s.ld_stats + 2 * P + S + d];
            sc = expf(0.5f * jlv);
        } else {
            float mua = s.own_loc[(long)row * s.ld_own + d];
            float lva = s.own_lv[(long)row * s.ld_own + d];
            float va = expf(lva);
            float ivp, mvp;
            if (pr >= 0) {
                float mub = s.oth_loc[(long)pr * s.ld_oth + d];
                float vb = expf(s.oth_lv[(long)pr * s.ld_oth + d]);
                ivp = 1.0f / vb;
                mvp = mub / vb;
            } else if (pr == SPV_PARTNER_PAD) {
                ivp = 1.0f;  // _poe2 pads the shorter group with precision 1, mean term 0 (reference :297-326)
                mvp = 0.0f;
            } else {
                ivp = 1.0f / expf(1.0f);  // synthetic partner mu = 0, logvar = 1 (reference :629-659)
                mvp = 0.0f;
            }
            float prec = 1.0f + 1.0f / va + ivp;  // prior expert N(0,1) always included (quirk Q4)
            float jv = 1.0f / prec;
            mu = (mua / va + mvp) * jv;
            jlv = logf(jv);
            sc = p.mode == SPV_POE_PAIRED ? expf(0.5f * jlv) : sqrtf(expf(jlv));
        }
        float scq = p.mode == SPV_POE_LABEL ? sc : fmaxf(sc, 1e-6f);  // clamp only in the OT modes (quirk Q6)
        float e = s.eps_q ? s.eps_q[(long)row * S + d]
                          : philox_normal(p.seed, 2u * blockIdx.y + 1u, stp, (unsigned long long)row * S + d);
        float z = mu + scq * e;
        s.poe_loc[(long)row * S + d] = mu;
        s.poe_lv[(long)row * S + d] = jlv;
        s.poe_scale[(long)row * S + d] = sc;
        s.zpoe[(long)row * S + d] = z;
        s.zz[(long)row * s.ld_zz + zz_col_of_c(P + d, S, P)] = z;
        float vr = scq * scq;
        klq += 0.5f * (vr + mu * mu - 1.0f - logf(vr));
    }
    klq = warp_sum(klq);
    if (lane == 0) {
        s.klp[row] = klp;
        s.klq[row] = klq;
    }
}

static int fill_side(PoeSide& s, const void* const* ptrs, const long long* lds, int B) {
    s.own_loc = (const float*)ptrs[0]; s.own_lv = (const float*)ptrs[1]; s.oth_loc = (const float*)ptrs[2];
    s.oth_lv = (const float*)ptrs[3]; s.stats = (const float*)ptrs[4]; s.partner = (const int*)ptrs[5];
    s.eps_p = (const float*)ptrs[6]; s.eps_q = (const float*)ptrs[7]; s.zpriv = (float*)ptrs[8];
    s.poe_loc = (float*)ptrs[9]; s.poe_lv = (float*)ptrs[10]; s.poe_scale = (float*)ptrs[11]; s.zpoe = (float*)ptrs[12];
    s.klp = (float*)ptrs[13]; s.klq = (float*)ptrs[14]; s.zz = (float*)ptrs[15];
    s.ld_own = lds[0]; s.ld_oth = lds[1]; s.ld_stats = lds[2]; s.ld_zz = lds[3];
    s.B = B;
    if (!s.own_loc || !s.own_lv || !s.oth_loc || !s.oth_lv || !s.stats || !s.zpriv || !s.poe_loc || !s.poe_lv ||
        !s.poe_scale || !s.zpoe || !s.klp || !s.klq || !s.zz || B <= 0)
        return SPV_ERR_ARG;
    return SPV_OK;
}

// ptrs0 / ptrs1: SPV_POE_FWD_NPTR pointers per group in the order documented in include/spvipes_b200.h
extern "C" int spv_poe_fwd(int mode, int S, int P, int B0, int B1, const void* const* ptrs0, const long long* lds0,
                           const void* const* ptrs1, const long long* lds1, unsigned long long seed, const int* step,
                           void* stream) {
    if (mode < 0 || mode > 2 || S <= 0 || P <= 0 || !ptrs0 || !ptrs1 || !lds0 || !lds1) return SPV_ERR_ARG;
    PoeParams p;
    if (fill_side(p.side[0], ptrs0, lds0, B0) != SPV_OK || fill_side(p.side[1], ptrs1, lds1, B1) != SPV_OK) return SPV_ERR_ARG;
    p.S = S; p.P = P; p.mode = mode; p.seed = seed; p.step = step;
    int Bmax = B0 > B1 ? B0 : B1;
    dim3 grid((Bmax + 7) / 8, 2);
    poe_fwd_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// ---------------------------------------------------------------------------------------
// backward.  Pass 1 (per row of each group): gradients w.r.t. the private statistics, the own
// expert and the contribution destined to the partner's expert.  Pass 2: each row adds the
// contributions of the rows that chose it as partner, in index order (deterministic).
// ---------------------------------------------------------------------------------------
struct PoeBwdSide {
    const float* own_loc; const float* own_lv; long ld_own;
    const float* oth_loc; const float* oth_lv; long ld_oth;
    const float* stats; long ld_stats;
    const int* partner;
    const float* eps_p; const float* eps_q;
    const float* dzz; long ld_dzz;  // gradient w.r.t. the decoder input columns
    float* dstats; long ld_dstats;  // [B, 2P+2S]: private columns written here; shared columns: pass-through rows (cluster)
    float* g_own;                   // [B, 2S] gradient w.r.t. own expert (loc | lv)
    float* g_contrib;               // [B, 2S] gradient destined to the partner row's expert
    int B;
};
struct PoeBwdParams {
    PoeBwdSide side[2];
    int S, P, mode;
    unsigned long long seed;
    const int* step;
    const float* kl_weight;  // device scalar
    float inv_batch;         // 1 / B of the loss mean
};

__global__ void __launch_bounds__(256) poe_bwd_kernel(PoeBwdParams p) {
    const PoeBwdSide& s = p.side[blockIdx.y];
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= s.B) return;
    const int S = p.S, P = p.P;
    const unsigned int stp = p.step ? (unsigned int)*p.step : 0u;
    const float kw = (*p.kl_weight) * p.inv_batch;
    for (int d = lane; d < P; d += 32) {
        float loc = s.stats[(long)row * s.ld_stats + d];
        float lv = s.stats[(long)row * s.ld_stats + P + d];
        float sc = expf(0.5f * lv);
        float e = s.eps_p ? s.eps_p[(long)row * P + d]
                          : philox_normal(p.seed, 2u * blockIdx.y, stp, (unsigned long long)row * P + d);
        float dz = s.dzz[(long)row * s.ld_dzz + zz_col_of_c(d, S, P)];
        float dloc = dz + kw * loc;
        float dsc = dz * e + kw * (sc - 1.0f / sc);
        s.dstats[(long)row * s.ld_dstats + d] = dloc;
        s.dstats[(long)row * s.ld_dstats + P + d] = dsc * 0.5f * sc;
    }
    const int pr = s.partner ? s.partner[row] : SPV_PARTNER_ABSENT;
    for (int d = lane; d < S; d += 32) {
        float e = s.eps_q ? s.eps_q[(long)row * S + d]
                          : philox_normal(p.seed, 2u * blockIdx.y + 1u, stp, (unsigned long long)row * S + d);
        float dz = s.dzz[(long)row * s.ld_dzz + zz_col_of_c(P + d, S, P)];
        float g_loc = 0.0f, g_lv = 0.0f, c_loc = 0.0f, c_lv = 0.0f, pass_loc = 0.0f, pass_lv = 0.0f;
        if (p.mode == SPV_POE_CLUSTER && pr == SPV_PARTNER_ABSENT) {
            float mu = s.stats[(long)row * s.ld_stats + 2 * P + d];
            float lv = s.stats[(long)row * s.ld_stats + 2 * P + S + d];
            float sc = expf(0.5f * lv);
            float scq = fmaxf(sc, 1e-6f);
            float dmu = dz + kw * mu;
            float dscq = dz * e + kw * (scq - 1.0f / scq);
            float dsc = sc >= 1e-6f ? dscq : 0.0f;
            pass_loc = dmu;
            pass_lv = dsc * 0.5f * sc;
        } else {
            float mua = s.own_loc[(long)row * s.ld_own + d];
            float lva = s.own_lv[(long)row * s.ld_own + d];
            float iva = 1.0f / expf(lva);
            float ivp, mvp, mub = 0.0f;
            if (pr >= 0) {
                mub = s.oth_loc[(long)pr * s.ld_oth + d];
                ivp = 1.0f / expf(s.oth_lv[(long)pr * s.ld_oth + d]);
                mvp = mub * ivp;
            } else if (pr == SPV_PARTNER_PAD) { ivp = 1.0f; mvp = 0.0f; }
            else { ivp = 1.0f / expf(1.0f); mvp = 0.0f; }
            float prec = 1.0f + iva + ivp;
            float jv = 1.0f / prec;
            float num = mua * iva + mvp;
            float mu = num * jv;
            float sc = sqrtf(jv);
            float scq = p.mode == SPV_POE_LABEL ? sc : fmaxf(sc, 1e-6f);
            float dmu = dz + kw * mu;
            float dscq = dz * e + kw * (scq - 1.0f / scq);
            float dsc = (p.mode == SPV_POE_LABEL || sc >= 1e-6f) ? dscq : 0.0f;
            float djlv = dsc * 0.5f * sc;
            float dnum = dmu * jv;
            float djv = dmu * num + djlv * prec;  // jlv = log(jv)
            float dprec = -djv * jv * jv;
            float diva = dnum * mua + dprec;
            g_loc = dnum * iva;
            g_lv = -iva * diva;
            if (pr >= 0) {
                float divb = dnum * mub + dprec;
                c_loc = dnum * ivp;
                c_lv = -ivp * divb;
            }
        }
        s.g_own[(long)row * 2 * S + d] = g_loc;
        s.g_own[(long)row * 2 * S + S + d] = g_lv;
        s.g_contrib[(long)row * 2 * S + d] = c_loc;
        s.g_contrib[(long)row * 2 * S + S + d] = c_lv;
        if (p.mode == SPV_POE_CLUSTER) {
            s.dstats[(long)row * s.ld_dstats + 2 * P + d] = pass_loc;
            s.dstats[(long)row * s.ld_dstats + 2 * P + S + d] = pass_lv;
        }
    }
}

// out[j, :] = g_own[j, :] + sum_{i : partner_oth[i] == j} contrib_oth[i, :]      ([B, 2S] -> out with leading dim)
struct PoeScatterSide {
    const float* g_own; const float* contrib_oth; const int* partner_oth;
    float* out; long ld_out;
    int B, B_oth;
};
struct PoeScatterParams { PoeScatterSide side[2]; int S; };

__global__ void __launch_bounds__(256) poe_bwd_scatter_kernel(PoeScatterParams p) {
    const PoeScatterSide& s = p.side[blockIdx.y];
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= s.B) return;
    const int W = 2 * p.S;
    float acc[4];  // supports 2S <= 128
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        int d = lane + 32 * q;
        acc[q] = d < W ? s.g_own[(long)row * W + d] : 0.0f;
    }
    // the other side's partner list is scanned 8 x 32 entries at a time: the eight loads are in flight together (one memory
    // round trip per 256 entries instead of one per 32), then the ballots; contributions are added in index order
    for (int c0 = 0; s.partner_oth && c0 < s.B_oth; c0 += 256) {
        int pv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = c0 + 32 * u + lane;
            pv[u] = i < s.B_oth ? __ldg(s.partner_oth + i) : -1;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            unsigned m = __ballot_sync(0xffffffffu, pv[u] == row);
            while (m) {
                int b = __ffs(m) - 1;
                m &= m - 1;
                int ii = c0 + 32 * u + b;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    int d = lane + 32 * q;
                    if (d < W) acc[q] += s.contrib_oth[(long)ii * W + d];
                }
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        int d = lane + 32 * q;
        if (d < W) s.out[(long)row * s.ld_out + d] = acc[q];
    }
}

// ptrs per group (SPV_POE_BWD_NPTR): own_loc, own_lv, oth_loc, oth_lv, stats, partner, eps_p, eps_q, dzz, dstats,
// g_own, g_contrib, out ; lds per group: ld_own, ld_oth, ld_stats, ld_dzz, ld_dstats, ld_out
extern "C" int spv_poe_bwd(int mode, int S, int P, int B0, int B1, const void* const* ptrs0, const long long* lds0,
                           const void* const* ptrs1, const long long* lds1, unsigned long long seed, const int* step,
                           const float* kl_weight, float inv_batch, void* stream) {
    if (mode < 0 || mode > 2 || S <= 0 || P <= 0 || 2 * S > 128 || !ptrs0 || !ptrs1 || !lds0 || !lds1 || !kl_weight)
        return SPV_ERR_ARG;
    PoeBwdParams p;
    PoeScatterParams q;
    const void* const* pp[2] = {ptrs0, ptrs1};
    const long long* ll[2] = {lds0, lds1};
    const int Bs[2] = {B0, B1};
    for (int g = 0; g < 2; ++g) {
        PoeBwdSide& s = p.side[g];
        s.own_loc = (const float*)pp[g][0]; s.own_lv = (const float*)pp[g][1]; s.oth_loc = (const float*)pp[g][2];
        s.oth_lv = (const float*)pp[g][3]; s.stats = (const float*)pp[g][4]; s.partner = (const int*)pp[g][5];
        s.eps_p = (const float*)pp[g][6]; s.eps_q = (const float*)pp[g][7]; s.dzz = (const float*)pp[g][8];
        s.dstats = (float*)pp[g][9]; s.g_own = (float*)pp[g][10]; s.g_contrib = (float*)pp[g][11];
        s.ld_own = ll[g][0]; s.ld_oth = ll[g][1]; s.ld_stats = ll[g][2]; s.ld_dzz = ll[g][3]; s.ld_dstats = ll[g][4];
        s.B = Bs[g];
        if (!s.own_loc || !s.own_lv || !s.oth_loc || !s.oth_lv || !s.stats || !s.dzz || !s.dstats || !s.g_own ||
            !s.g_contrib || !pp[g][12] || s.B <= 0)
            return SPV_ERR_ARG;
    }
    for (int g = 0; g < 2; ++g) {
        PoeScatterSide& s = q.side[g];
        s.g_own = p.side[g].g_own;
        s.contrib_oth = p.side[1 - g].g_contrib;
        s.partner_oth = p.side[1 - g].partner;
        s.out = (float*)pp[g][12];
        s.ld_out = ll[g][5];
        s.B = Bs[g];
        s.B_oth = Bs[1 - g];
    }
    p.S = S; p.P = P; p.mode = mode; p.seed = seed; p.step = step; p.kl_weight = kl_weight; p.inv_batch = inv_batch;
    q.S = S;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int Bmax = B0 > B1 ? B0 : B1;
    dim3 grid((Bmax + 7) / 8, 2);
    poe_bwd_kernel<<<grid, 256, 0, st>>>(p);
    SPV_CHECK_LAUNCH();
    poe_bwd_scatter_kernel<<<grid, 256, 0, st>>>(q);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// loss = mean_b(rec0 + rec1 + w (klp0 + klq0 + klp1 + klq1))   (reference :886-893); also the 4 KL means
// (extra_metrics :870-875) -> out[0] = loss, out[1..4] = mean klp0, klq0, klp1, klq1, out[5..6] = mean rec0, rec1
__global__ void loss_kernel(const float* __restrict__ rec0, const float* __restrict__ rec1, const float* __restrict__ klp0,
                            const float* __restrict__ klq0, const float* __restrict__ klp1, const float* __restrict__ klq1,
                            int B, const float* __restrict__ kl_weight, float* __restrict__ out) {
    __shared__ float red[7][32];
    float a[7] = {0, 0, 0, 0, 0, 0, 0};
    const float w = *kl_weight;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        a[0] += rec0[b] + rec1[b] + w * klp0[b] + w * klq0[b] + w * klp1[b] + w * klq1[b];
        a[1] += klp0[b]; a[2] += klq0[b]; a[3] += klp1[b]; a[4] += klq1[b]; a[5] += rec0[b]; a[6] += rec1[b];
    }
    for (int k = 0; k < 7; ++k) {
        float v = warp_sum(a[k]);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 7) {
        float v = 0.0f;
        for (int w2 = 0; w2 < (int)(blockDim.x >> 5); ++w2) v += red[threadIdx.x][w2];
        out[threadIdx.x] = v / (float)B;
    }
}

extern "C" int spv_loss(const float* rec0, const float* rec1, const float* klp0, const float* klq0, const float* klp1,
                        const float* klq1, int B, const float* kl_weight, float* out, void* stream) {
    if (!rec0 || !rec1 || !klp0 || !klq0 || !klp1 || !klq1 || !kl_weight || !out || B <= 0) return SPV_ERR_ARG;
    loss_kernel<<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(rec0, rec1, klp0, klq0, klp1, klq1, B, kl_weight, out);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// one evaluation pass's loss terms added to a float64 accumulator (validation epochs, get_elbo):
// acc[0..5] += sum rec0, sum rec1, sum klp0, sum klq0, sum klp1, sum klq1 (each group over its own B_g cells, fp32 as loss_kernel),
// acc[6] += B0 (n_obs of the minibatch: group 0's size), acc[7] += sum rec0 + sum rec1 + w (sum of the four KL sums).
// The groups may differ in size: nothing is paired across them.  float64 so that ~50 minibatch sums of an epoch do not drift.
__global__ void elbo_accumulate_kernel(const float* __restrict__ rec0, const float* __restrict__ rec1,
                                       const float* __restrict__ klp0, const float* __restrict__ klq0,
                                       const float* __restrict__ klp1, const float* __restrict__ klq1, int B0, int B1,
                                       const float* __restrict__ kl_weight, double* __restrict__ acc) {
    __shared__ float red[6][32];
    float a[6] = {0, 0, 0, 0, 0, 0};
    for (int b = threadIdx.x; b < B0; b += blockDim.x) {
        a[0] += rec0[b]; a[2] += klp0[b]; a[3] += klq0[b];
    }
    for (int b = threadIdx.x; b < B1; b += blockDim.x) {
        a[1] += rec1[b]; a[4] += klp1[b]; a[5] += klq1[b];
    }
    for (int k = 0; k < 6; ++k) {
        float v = warp_sum(a[k]);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s[6];
        for (int k = 0; k < 6; ++k) {
            float v = 0.0f;
            for (int w2 = 0; w2 < (int)(blockDim.x >> 5); ++w2) v += red[k][w2];
            s[k] = (double)v;
            acc[k] += s[k];
        }
        acc[6] += (double)B0;
        acc[7] += s[0] + s[1] + (double)*kl_weight * (s[2] + s[3] + s[4] + s[5]);
    }
}

extern "C" int spv_elbo_accumulate(const float* rec0, const float* rec1, const float* klp0, const float* klq0, const float* klp1,
                                   const float* klq1, int B0, int B1, const float* kl_weight, double* acc, void* stream) {
    if (!rec0 || !rec1 || !klp0 || !klq0 || !klp1 || !klq1 || !kl_weight || !acc || B0 <= 0 || B1 <= 0) return SPV_ERR_ARG;
    elbo_accumulate_kernel<<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(rec0, rec1, klp0, klq0, klp1, klq1, B0, B1,
                                                                                    kl_weight, acc);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}
