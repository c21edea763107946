// TRAINING sweep of the fused decoder + NB-mixture likelihood on the tensor-core path: the forward sweep (nb_tc.cu) that also emits
// everything the backward needs, so that a training step makes ONE pass over the [B, G] problem instead of two.
//
// The only cross-gene quantity of the backward is the softmax coupling D_b = sum_g (d ll / d rho) rho of each branch, known after
// the forward sweep:  d ll / d y_p[b, g] = ep[b, g] - rho_p[b, g] exp(-lib_b) Dp_b.  Both terms are per-element products of this
// sweep, and the correction is a row scaling, which commutes with the gradient GEMMs.  So the sweep writes, per (gene, cell),
//   E4T [Gp, 4 Bp] fp16, gene-major, four interleaved components per cell: (ep, rp', es, rs'),  r' = 4096 softmax value
//                                                                         (= rho exp(-lib) 4096: fp16-safe whatever the library size)
//   DPIT [Gp, Bp]  fp16: d ll / d pi
// and the consumers apply the coupling through their other operand:
//   [Qp | sum dyp | Qs | sum dys] = E4T . ZQ4,  ZQ4 [4 Bp, KZ + 2] rows (4b .. 4b+3) = [zp 1 0 0], -Dp'/1 [zp 1 0 0], [0 0 zs 1], -Ds' [0 0 zs 1]
//   T [4 Bp, KZ] = E4T^T . [W'p | W's],   d zz[b] = T[4b] - Dp' T[4b+1] (private columns), T[4b+2] - Ds' T[4b+3] (shared), D' = D / 4096
// (spv_dec_zq4, spv_dec_dz4_combine).  Column sums of d pi and d theta are reduced here; those of
// dyp / dys come out of the first GEMM's ones column.  Row partials (ll, sum ep, sum es) as the forward sweep.
// Tiling, pipeline and tensor-memory protocol: nb_tc_sweep.cuh.  8 SFU operations per element.
// Reference: nn/networks.py:314-325 + scvi log_mixture_nb (module/spVIPESmodule.py:759, 823-824) and their autograd.
#include <cuda_fp16.h>
#include "nb_tc_sweep.cuh"

namespace {

using namespace nbtc;

// Scratch behind the count tile in the drained operand stages: column sums (2 quantities), d-theta count table.  The column-sum
// scratch does NOT get its own 4 KB of shared memory (that made it 80 128 bytes and two CTAs per SM).
constexpr int COL_BYTES = 2 * 4 * BN * 4, TB_BYTES = BN * NB_TAB * 4;
static_assert(CNT_BYTES + COL_BYTES + TB_BYTES <= STAGES * STAGE_BYTES, "count tile + scratch must fit in the operand stages");

struct NbTcTrainParams : NbTcParams {  // tgf: (log1p(c), lgamma term)
    const float* lib;    // [B]
    const float* tb1;    // [G, NB_TAB] digamma term of the same counts
    float* part_nb;      // [2 nTG, B, 3] row partials (ll, sum ep, sum es), as the forward sweep
    __half* e4t; long ld_e4;     // [Gp, ld_e4 >= 4 B]: (ep, rp', es, rs') per cell, gene-major
    __half* dpit; long ld_dpi;   // [Gp, ld_dpi >= B]
    float* colpart;              // [nTB, 2, G]: column sums of d pi, d theta per 128-row tile
};

// CTAs of this kernel currently resident per SM (nb_tc_sweep.cuh mma_warp)
__device__ int g_resident_trn[256];

__device__ __forceinline__ void st_half4(unsigned long long addr, float a, float b, float c, float d) {
    const __half2 lo = __floats2half2_rn(a, b), hi = __floats2half2_rn(c, d);
    asm volatile("st.global.v2.b32 [%0], {%1, %2};" ::"l"(addr), "r"(*reinterpret_cast<const uint32_t*>(&lo)),
                 "r"(*reinterpret_cast<const uint32_t*>(&hi))
                 : "memory");
}
__device__ __forceinline__ void st_half(unsigned long long addr, float v) {
    const unsigned short h = __half_as_ushort(__float2half_rn(v));
    asm volatile("st.global.u16 [%0], %1;" ::"l"(addr), "h"(h) : "memory");
}

// one element off the fast path (a count outside the tables, a logit below the fast logarithm's range, an edge tile): out of line
template <int SRC>
__device__ __noinline__ NbTrain nb_train_general(uint32_t code, float xp, float xs, float acc_pi, float4 gc, const uint8_t* tg_row,
                                                 const float* tb_row, const void* X, long xidx, const float* lgt, const float* dgt) {
    float t, ctf, ctb;
    if (code == NB_CODE_SLOW) {
        const float xraw = nb_load_raw<SRC>(X, xidx);
        const float2 f = nb_count_terms_fwd_slow(xraw, gc.x, __ldg(lgt));
        t = f.x; ctf = f.y;
        ctb = nb_count_terms_bwd_slow(xraw, gc.x, __ldg(dgt)).y;
    } else {
        const float2 f = *reinterpret_cast<const float2*>(tg_row + code);
        t = f.x; ctf = f.y;
        ctb = tb_row[code >> 3];
    }
    const float pi = acc_pi + gc.w;
    if (t != 0.0f && fminf(xp, xs) < NB_X_RARE) return nb_train_v5<true>(t, ctf, ctb, xp, xs, pi, gc.x, gc.x + NB_EPS, gc.y, gc.z);
    return nb_train_v5<false>(t, ctf, ctb, xp, xs, pi, gc.x, gc.x + NB_EPS, gc.y, gc.z);
}

template <int SRC>
__global__ void __launch_bounds__(THREADS, 3) nb_tc_train_kernel(const __grid_constant__ CUtensorMap mapA,
                                                               const __grid_constant__ CUtensorMap mapB,
                                                               const __grid_constant__ CUtensorMap mapZ,
                                                               const __grid_constant__ CUtensorMap mapZc, NbTcTrainParams p) {
    const Smem sm = carve_smem();
    float* s_col = reinterpret_cast<float*>(sm.tiles + CNT_BYTES);  // [2 quantities][4 quarters][BN], behind the count tile
    float* s_tb = reinterpret_cast<float*>(sm.tiles + CNT_BYTES + COL_BYTES);  // [BN][NB_TAB] digamma terms, behind it
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    const int num_kb = (p.K + BK - 1) / BK;
    init_pipeline(sm, &mapA, &mapB, &mapZ, &mapZc, warp, lane);
    uint32_t tmem_base = 0, tmem_z = 0;  // mixture-logit accumulator [BN columns]; the two branch-logit accumulators [2 BN]

    if (warp == 0) {
        produce(sm, &mapA, &mapB, &mapZ, &mapZc, n0, m0, num_kb, p.Gp);
    } else if (warp == 1) {
        mma_warp(sm, g_resident_trn, num_kb, lane, tmem_base, tmem_z);
    } else {
        // ================= epilogue: 8 warps =================
        const int et = threadIdx.x - 64;
        const long G = p.G;
        const int e = warp - 2;
        const int q = warp & 3;
        const int half = e >> 2;
        const int rloc = q * 32 + lane;
        const int m = m0 + rloc;
        const bool mok = m < p.B;
        const int mm = mok ? m : 0;
        uint32_t cw[NGATHER];
        float libm;
        float4 tbv;
        // gene constants: theta, Kc, K1c, bm
        const int my_row = epi_prologue<SRC, GC_KC, GC_K1C>(p, sm, true, n0, m0, mm, cw, [&] {
            libm = __ldg(p.lib + mm);
            // the digamma terms of the tile's genes: BN * NB_TAB floats = one 16-byte word per epilogue thread (gene et / 4)
            static_assert(BN * NB_TAB * 4 == EPI_THREADS * 16, "one 16-byte word of the d-theta table per epilogue thread");
            tbv = n0 + (et >> 2) < p.G ? __ldg(reinterpret_cast<const float4*>(p.tb1 + (long)n0 * NB_TAB) + et) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        });
        const float c_row = 4096.0f * fast_exp(-libm);  // rho -> 4096 x softmax value: fp16-safe whatever the library size
        const long xrow = (long)my_row * p.ldx;
        // One epilogue warp polls the two mbarriers; the other seven block in a named barrier, where they cost no issue slots (a
        // CTA waiting for its tensor-memory grant spends most of its life here: eight polling warps took a quarter of the SM's
        // issued instructions away from the two CTAs doing the math - profiles/r2_nb_ncu.md)
        if (e == 0) {
            tc::mbar_wait(sm.tmem_ready, 0);
            tc::mbar_wait(sm.tmem_full, 0);  // accumulators complete; the operand stages are free from here on
            tc::fence_after_sync();
        }
        tc::fence_before_sync();
        asm volatile("bar.sync 2, %0;" ::"r"(EPI_THREADS) : "memory");
        tc::fence_after_sync();
        tmem_base = *reinterpret_cast<volatile uint32_t*>(sm.tmem_slot);
        tmem_z = *reinterpret_cast<volatile uint32_t*>(sm.tmem_slot + 1);
        stage_counts(sm, cw, true);
        reinterpret_cast<float4*>(s_tb)[et] = tbv;
        asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");
        const float4* s_gc = sm.s_gc;
        const uint8_t* s_tg = sm.s_tg;
        // running store addresses: this cell's slot in the row of the first gene of the current four (byte pitches are 32-bit)
        const uint32_t ldb_e = (uint32_t)p.ld_e4 * 2u, ldb_d = (uint32_t)p.ld_dpi * 2u;
        unsigned long long a_e = reinterpret_cast<unsigned long long>(p.e4t) + (unsigned long long)(n0 + half * WCOLS) * ldb_e + 8ull * (unsigned)m;
        unsigned long long a_d = reinterpret_cast<unsigned long long>(p.dpit) + (unsigned long long)(n0 + half * WCOLS) * ldb_d + 2ull * (unsigned)m;
        float sll = 0.0f, sep = 0.0f, ses = 0.0f;
        const bool full_tile = n0 + BN <= p.G && m0 + BM <= p.B;  // CTA-uniform
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16), lane_z = tmem_z + ((uint32_t)(q * 32) << 16);
        const uint32_t* cnt_row_p = sm.s_cnt + rloc * CNT_PITCH_W + half * (WCOLS / 2);
#pragma unroll 1
        for (int j4 = 0; j4 < WCOLS; j4 += 4) {
            const int c0 = half * WCOLS + j4;
            uint32_t rpi[4], rlp[4], rls[4];
            tc::tmem_ld4(lane_addr + (uint32_t)c0, rpi);
            tc::tmem_ld4(lane_z + (uint32_t)c0, rlp);
            tc::tmem_ld4(lane_z + (uint32_t)(BN + c0), rls);
            const uint2 cc = *reinterpret_cast<const uint2*>(cnt_row_p + (j4 >> 1));  // four count codes
            tc::tmem_ld_wait();
            const uint32_t call = cc.x | cc.y;
            const float xm = fminf(fminf(fminf(__uint_as_float(rlp[0]), __uint_as_float(rls[0])), fminf(__uint_as_float(rlp[1]), __uint_as_float(rls[1]))),
                                   fminf(fminf(__uint_as_float(rlp[2]), __uint_as_float(rls[2])), fminf(__uint_as_float(rlp[3]), __uint_as_float(rls[3]))));
            // every count tabulated, every column and row valid, the fast logarithm holds (as in nb_tc_fwd_kernel)
            const bool plain = full_tile && (call & 0x80008000u) == 0u && !(call != 0u && xm < NB_X_RARE);
            float vpi[4], vth[4];
            // E4T[gene, cell] = (ep, rp', es, rs') (8 bytes) and DPIT[gene, cell]: the 32 lanes of the warp are 32 consecutive cells,
            // so the two stores of a gene write 256 and 64 contiguous bytes
            if (plain) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int gl = c0 + jj;
                    const uint32_t w = jj < 2 ? cc.x : cc.y;
                    const uint32_t code = (jj & 1) ? (w >> 16) : (w & 0xffffu);
                    const float2 tcn = *reinterpret_cast<const float2*>(s_tg + gl * (NB_TAB * 8) + code);
                    const float ctb = *reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(s_tb) + gl * (NB_TAB * 4) + (code >> 1));
                    const float4 gc = s_gc[gl];
                    const NbTrain o = nb_train_v5<false>(tcn.x, tcn.y, ctb, __uint_as_float(rlp[jj]), __uint_as_float(rls[jj]),
                                                         __uint_as_float(rpi[jj]) + gc.w, gc.x, gc.x + NB_EPS, gc.y, gc.z);
                    sll += o.ll; sep += o.ep; ses += o.es;
                    vpi[jj] = o.dpi; vth[jj] = o.dth;
                    st_half4(a_e + jj * ldb_e, o.ep, o.rp * c_row, o.es, o.rs * c_row);
                    st_half(a_d + jj * ldb_d, o.dpi);
                }
            } else {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int gl = c0 + jj;
                    const uint32_t w = jj < 2 ? cc.x : cc.y;
                    const uint32_t code = (jj & 1) ? (w >> 16) : (w & 0xffffu);
                    vpi[jj] = vth[jj] = 0.0f;
                    if (mok && n0 + gl < p.G) {
                        const NbTrain o = nb_train_general<SRC>(code, __uint_as_float(rlp[jj]), __uint_as_float(rls[jj]), __uint_as_float(rpi[jj]),
                                                                s_gc[gl], s_tg + gl * (NB_TAB * 8), s_tb + gl * NB_TAB, p.X, xrow + n0 + gl,
                                                                p.genec + GC_LGT * G + n0 + gl, p.genec + GC_DGT * G + n0 + gl);
                        sll += o.ll; sep += o.ep; ses += o.es;
                        vpi[jj] = o.dpi; vth[jj] = o.dth;
                        st_half4(a_e + jj * ldb_e, o.ep, o.rp * c_row, o.es, o.rs * c_row);
                        st_half(a_d + jj * ldb_d, o.dpi);
                    }
                }
            }
            a_e += 4ull * ldb_e; a_d += 4ull * ldb_d;
            // column sums over this warp's 32 rows (lanes): transpose-reduce of the 8 values (2 quantities x 4 columns).  Each
            // butterfly step halves the values a lane carries (4 + 2 + 1 shuffles), two plain steps finish; lanes with the two low
            // bits clear end up with the total of value index (lane >> 2) and park it for the cross-quarter sum.
            {
                float v4[4], v2[2];
                const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float send = b4 ? vpi[i] : vth[i], keep = b4 ? vth[i] : vpi[i];
                    v4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                }
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const float send = b3 ? v4[i] : v4[i + 2], keep = b3 ? v4[i + 2] : v4[i];
                    v2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                }
                const float send = b2 ? v2[0] : v2[1], keep = b2 ? v2[1] : v2[0];
                float tot = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                tot += __shfl_xor_sync(0xffffffffu, tot, 2);
                tot += __shfl_xor_sync(0xffffffffu, tot, 1);
                if ((lane & 3) == 0) {
                    const int idx = lane >> 2;  // = 4 b4 + 2 b3 + b2: quantity idx >> 2 (0: d pi, 1: d theta), column idx & 3
                    s_col[((idx >> 2) * 4 + q) * BN + c0 + (idx & 3)] = tot;
                }
            }
        }
        if (mok) {
            float* o = p.part_nb + ((long)(blockIdx.x * 2 + half) * p.B + m) * 3;
            o[0] = sll; o[1] = sep; o[2] = ses;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");
        for (int i = et; i < 2 * BN; i += EPI_THREADS) {
            const int qty = i / BN, gl = i - qty * BN, g = n0 + gl;
            if (g < p.G) {
                const float* s = s_col + (qty * 4) * BN + gl;
                p.colpart[((long)blockIdx.y * 2 + qty) * G + g] = s[0] + s[BN] + s[2 * BN] + s[3 * BN];
            }
        }
    }
    release_tmem(warp, lane, tmem_base, tmem_z, g_resident_trn);
}

__global__ void colpart2_reduce_kernel(const float* __restrict__ colpart, int nTB, int G, float* __restrict__ colsum, float mult) {
    long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (i >= 2L * G) return;
    float s = 0.0f;
    for (int t = 0; t < nTB; ++t) s += colpart[(long)t * 2 * G + i];
    colsum[i] = s * mult;
}

// ZQ4 [4 Bp, ldq] (fp16): the other operand of Q = E4T . ZQ4 (header comment).  zb [B, ld_zb] = the regressors' inputs
// [z_private_arg (Pb) | z_shared_arg (Sb)], rowc [B, 4] = (Rp, Rs, Dp, Ds).
__global__ void zq4_kernel(const float* __restrict__ zb, long ld_zb, const float* __restrict__ rowc, __half* __restrict__ zq, long ldq, int B,
                           int Pb, int Sb) {
    const int W = Pb + Sb + 2;
    const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (i >= (long)B * W) return;
    const int b = (int)(i / W), c = (int)(i - (long)b * W);
    const bool priv = c <= Pb;
    const float v = priv ? (c < Pb ? zb[(long)b * ld_zb + c] : 1.0f) : (c < W - 1 ? zb[(long)b * ld_zb + c - 1] : 1.0f);
    const float dp = -rowc[4 * b + 2] * (1.0f / 4096.0f), ds = -rowc[4 * b + 3] * (1.0f / 4096.0f);
    __half* row = zq + (long)(4 * b) * ldq + c;
    row[0] = to_half_sat(priv ? v : 0.0f);
    row[ldq] = to_half_sat(priv ? dp * v : 0.0f);
    row[2 * ldq] = to_half_sat(priv ? 0.0f : v);
    row[3 * ldq] = to_half_sat(priv ? 0.0f : ds * v);
}

// d zz (softmax branches) from T [4 Bp, ld_t] = E4T^T [W'p | W's]:  out[b, c] = T[4b + k, c] - D' T[4b + k + 1, c],  k = 0 / D = Dp for
// the private columns c < Pb, k = 2 / D = Ds for the shared ones
__global__ void dz4_combine_kernel(const float* __restrict__ T, long ld_t, const float* __restrict__ rowc, float* __restrict__ out, long ld_out,
                                   int B, int Pb, int Sb) {
    const int W = Pb + Sb;
    const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (i >= (long)B * W) return;
    const int b = (int)(i / W), c = (int)(i - (long)b * W);
    const int k = c < Pb ? 0 : 2;
    const float d = rowc[4 * b + (c < Pb ? 2 : 3)] * (1.0f / 4096.0f);
    out[(long)b * ld_out + c] = T[(long)(4 * b + k) * ld_t + c] - d * T[(long)(4 * b + k + 1) * ld_t + c];
}

}  // namespace

// Training sweep (header comment).  ptrs: the SPV_DEC_NPTR list as spv_dec_nb_fwd_tc (X, rows, -, -, -, bm, genec, lib, -, -, -,
// part_nb, -, -, -, colpart [ceil(B/128), 2, G], -, tgf) + [18] = tb1, the [G, 16] float table of digamma terms (spv_dec_theta_tables).
// e4t [Gp, ld_e4 >= 4 B] and dpit [Gp, ld_dpi >= B] (fp16, pitches multiples of 8, zero-initialised by the caller: rows >= G and
// cells >= B are never written).  Follow with spv_dec_nb_rowreduce (rec, Dp, Ds) as after the forward sweep.
extern "C" int spv_dec_nb_train_tc(int src, const void* const* ptrs, long long ldx, const void* amix_f16, long long ld_amixb,
                                   const void* wstack_f16, long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, void* e4t,
                                   long long ld_e4, void* dpit, long long ld_dpi, int B, int G, int HD, int P, int S, int kmix,
                                   void* stream) {
    if (!sweep_args_ok(ptrs, amix_f16, wstack_f16, zc_f16, wz_f16, Gp, B, G, P, S) || !e4t || !dpit || ld_e4 < 4ll * B || ld_dpi < B ||
        (ld_e4 & 3) || ld_e4 >= (1ll << 28))
        return SPV_ERR_ARG;
    for (int i : {0, 7, 11, 15, 17, 18})
        if (!ptrs[i]) return SPV_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(ptrs[17]) | reinterpret_cast<uintptr_t>(ptrs[18]) | reinterpret_cast<uintptr_t>(e4t)) & 15) return SPV_ERR_ARG;
    const int K = kmix > 0 ? kmix : HD + P + S;
    NbTcTrainParams p{};
    NbTcMaps mp;
    const int rc = sweep_setup<nb_tc_train_kernel<SPV_SRC_U16_LOG1P>, nb_tc_train_kernel<SPV_SRC_F32_LOG1P>>(
        p, mp, ptrs, ldx, amix_f16, ld_amixb, wstack_f16, ld_w, Gp, zc_f16, wz_f16, B, G, K);
    if (rc != SPV_OK) return rc;
    p.lib = (const float*)ptrs[7]; p.tb1 = (const float*)ptrs[18]; p.part_nb = (float*)ptrs[11];
    p.colpart = (float*)ptrs[15];
    p.e4t = reinterpret_cast<__half*>(e4t); p.ld_e4 = ld_e4; p.dpit = reinterpret_cast<__half*>(dpit); p.ld_dpi = ld_dpi;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dim3 grid((G + BN - 1) / BN, (B + BM - 1) / BM);
    if (src == SPV_SRC_U16_LOG1P) nb_tc_train_kernel<SPV_SRC_U16_LOG1P><<<grid, THREADS, SMEM_BYTES, st>>>(mp.a, mp.b, mp.z, mp.zc, p);
    else if (src == SPV_SRC_F32_LOG1P) nb_tc_train_kernel<SPV_SRC_F32_LOG1P><<<grid, THREADS, SMEM_BYTES, st>>>(mp.a, mp.b, mp.z, mp.zc, p);
    else return SPV_ERR_ARG;
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// colsum[0:2, G] = scale x column sums of (d ll / d pi, d ll / d theta) from the per-row-tile partials of spv_dec_nb_train_tc
extern "C" int spv_dec_nb_train_colsum(const float* colpart, int B, int G, float scale, float* colsum, void* stream) {
    if (!colpart || !colsum || B <= 0 || G <= 0) return SPV_ERR_ARG;
    colpart2_reduce_kernel<<<(2 * G + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(colpart, (B + BM - 1) / BM, G, colsum, scale);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// the second operand of the Q GEMM of the single-sweep backward: zq [4 Bp, ldq] fp16 (rows beyond 4 B untouched), ldq >= Pb + Sb + 2
extern "C" int spv_dec_zq4(const float* zb, long long ld_zb, const float* rowc, void* zq, long long ldq, int B, int Pb, int Sb, void* stream) {
    if (!zb || !rowc || !zq || B <= 0 || Pb <= 0 || Sb <= 0 || ldq < Pb + Sb + 2) return SPV_ERR_ARG;
    const long n = (long)B * (Pb + Sb + 2);
    zq4_kernel<<<(unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(zb, ld_zb, rowc, reinterpret_cast<__half*>(zq), ldq, B, Pb, Sb);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// out [B, ld_out] (Pb + Sb columns) = the softmax-branch part of d zz from T [4 B, ld_t] (header comment)
extern "C" int spv_dec_dz4_combine(const float* T, long long ld_t, const float* rowc, float* out, long long ld_out, int B, int Pb, int Sb,
                                   void* stream) {
    if (!T || !rowc || !out || B <= 0 || Pb <= 0 || Sb <= 0) return SPV_ERR_ARG;
    const long n = (long)B * (Pb + Sb);
    dz4_combine_kernel<<<(unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(T, ld_t, rowc, out, ld_out, B, Pb, Sb);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}
