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
// Same tiling, pipeline and tensor-memory protocol as nb_tc.cu.  8 SFU operations per element.
// Reference: nn/networks.py:314-325 + scvi log_mixture_nb (module/spVIPESmodule.py:759, 823-824) and their autograd.
#include <cuda_fp16.h>
#include "tc_common.cuh"
#include "nb_math.cuh"
#include "decoder_common.cuh"
#include "../../include/spvipes_b200.h"

namespace {

constexpr int BM = 128, BN = 64, BK = 64, STAGES = 2;
constexpr int WCOLS = BN / 2;                 // gene columns per epilogue warp (two warps per TMEM lane quarter)
constexpr int GATHER_ROWS = 64 / BN;          // rows of the count tile one warp gathers per load: 32 lanes cover BN / 2 words each
constexpr int EPI_WARPS = 8, EPI_THREADS = 32 * EPI_WARPS;
constexpr int THREADS = 64 + EPI_THREADS;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int ACC_COLS = BN, Z_COLS = 2 * BN;  // tensor memory is allocated in two steps (powers of two >= 32)
static_assert(ACC_COLS == 32 || ACC_COLS == 64, "tensor-memory allocations are powers of two");
constexpr int CNT_PITCH_W = BN / 2 + 2;  // 34 words per row: thread = row reads 64 bits (four codes), aligned and conflict-free
// 76 032 bytes: three CTAs per SM (3 x (76 032 + 1 024 reserved) <= 233 472).  The column-sum scratch s_col does NOT get its own
// 4 KB (that made it 80 128 bytes and two CTAs per SM): it aliases the drained operand stages behind the count tile.
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 2 * B_BYTES + 1024 + BN * 16 + BN * NB_TAB * 8 + 256;
constexpr int COL_BYTES = 2 * 4 * BN * 4, TB_BYTES = BN * NB_TAB * 4;  // aliased scratch: column sums (2 quantities), d-theta count table
static_assert(3 * (SMEM_BYTES + 1024) <= 233472, "three resident CTAs per SM");

static_assert(BM * CNT_PITCH_W * 4 + COL_BYTES + TB_BYTES <= STAGES * STAGE_BYTES, "count tile + scratch must fit in the operand stages");

struct NbTcTrainParams {
    const void* X; long ldx; const int* rows;
    const float* bm;
    const float* genec;
    const float* lib;    // [B]
    const float2* tgf;   // [G, NB_TAB] forward count table (spv_dec_theta_tables): (log1p(c), lgamma term)
    const float* tb1;    // [G, NB_TAB] digamma term of the same counts
    float* part_nb;      // [2 nTG, B, 3] row partials (ll, sum ep, sum es), as the forward sweep
    __half* e4t; long ld_e4;     // [Gp, ld_e4 >= 4 B]: (ep, rp', es, rs') per cell, gene-major
    __half* dpit; long ld_dpi;   // [Gp, ld_dpi >= B]
    float* colpart;              // [nTB, 2, G]: column sums of d pi, d theta per 128-row tile
    int B, G, K, Gp;
};

// row of the count tile that lane `lane` of epilogue warp e loads in its i-th gather: a warp covers GATHER_ROWS rows per load
__device__ __forceinline__ int cnt_row(int e, int lane, int i) {
    return (e + EPI_WARPS * i) * GATHER_ROWS + lane / (BN / 2);
}

// CTAs of this kernel currently resident per SM (a scheduling hint only, see the allocation below; balanced by every CTA)
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
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = tc::smem_u32(smem_raw);
    const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
    uint8_t* tiles = smem_raw + pad;
    uint8_t* z_tiles = tiles + STAGES * STAGE_BYTES;
    float4* s_gc = reinterpret_cast<float4*>(z_tiles + 2 * B_BYTES);  // [BN]: theta, Kc, K1c, bm
    uint8_t* s_tg = reinterpret_cast<uint8_t*>(s_gc + BN);              // [BN][NB_TAB] float2: (log1p(c), lgamma term) per gene
    uint64_t* full = reinterpret_cast<uint64_t*>(s_tg + BN * NB_TAB * 8);
    uint64_t* empty = full + STAGES;
    uint64_t* z_full = empty + STAGES;
    uint64_t* tmem_full = z_full + 1;
    uint64_t* tmem_ready = tmem_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_ready + 1);
    uint32_t* s_cnt = reinterpret_cast<uint32_t*>(tiles);               // aliases the operand stages once the MMAs are done
    float* s_col = reinterpret_cast<float*>(tiles + BM * CNT_PITCH_W * 4);  // [2 quantities][4 quarters][BN], behind the count tile
    float* s_tb = reinterpret_cast<float*>(tiles + BM * CNT_PITCH_W * 4 + COL_BYTES);  // [BN][NB_TAB] digamma terms, behind it

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    const int num_kb = (p.K + BK - 1) / BK;

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&mapA);
        tc::tma_prefetch_desc(&mapB);
        tc::tma_prefetch_desc(&mapZ);
        tc::tma_prefetch_desc(&mapZc);
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(&full[s], 1);
            tc::mbar_init(&empty[s], 1);
        }
        tc::mbar_init(z_full, 1);
        tc::mbar_init(tmem_full, 1);
        tc::mbar_init(tmem_ready, 1);
        tc::fence_barrier_init();
    }
    __syncthreads();
    // tensor memory is allocated by the MMA warp when it is about to issue, so that a third resident CTA runs its prologue
    // while two others own the SM's 512 columns (see nb_tc_fwd_kernel)
    uint32_t tmem_base = 0, tmem_z = 0;  // mixture-logit accumulator [BN columns]; the two branch-logit accumulators [2 BN]

    if (warp == 0) {
        if (tc::elect_one()) {
            tc::mbar_expect_tx(z_full, 2 * B_BYTES);
            tc::tma_load_2d(&mapZ, z_full, z_tiles, 0, n0);  // folded branch weights, fp16 [2 Gp, 64]
            tc::tma_load_2d(&mapZ, z_full, z_tiles + B_BYTES, 0, p.Gp + n0);
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                tc::mbar_wait(&empty[s], ph ^ 1);
                uint8_t* a_dst = tiles + s * STAGE_BYTES;
                tc::mbar_expect_tx(&full[s], STAGE_BYTES);
                tc::tma_load_2d(&mapA, &full[s], a_dst, i * BK, m0);
                tc::tma_load_2d(&mapB, &full[s], a_dst + A_BYTES, i * BK, n0);
            }
            {  // the branch k-block: centred latents (fp16), A tile only, next slot of the ring
                const int s = num_kb % STAGES;
                const uint32_t ph = (num_kb / STAGES) & 1;
                tc::mbar_wait(&empty[s], ph ^ 1);
                tc::mbar_expect_tx(&full[s], A_BYTES);
                tc::tma_load_2d(&mapZc, &full[s], tiles + s * STAGE_BYTES, 0, m0);
            }
        }
    } else if (warp == 1) {
        // two-step allocation as in nb_tc_fwd_kernel: the mixture-logit accumulator is completed while the CTA still waits
        // for the 2 BN columns of the branch logits; one thread issues every MMA and commit
        // A CTA that has allocated without giving up its permit keeps the SM from launching further CTAs (measured: the second
        // and third CTA of an SM entered 5 and 9.5 us after the first), so the two-step path is only taken by a CTA that finds
        // two others resident - the SM is full then anyway; the first two allocate everything at once.
        unsigned int smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        int ahead = 0;
        if (lane == 0) ahead = atomicAdd(&g_resident_trn[smid & 255], 1);
        const bool at_once = __shfl_sync(0xffffffffu, ahead, 0) < 2;
        tc::tmem_alloc_keep_permit(tmem_slot, ACC_COLS);
        if (at_once) tc::tmem_alloc(tmem_slot + 1, Z_COLS);
        tc::fence_before_sync();
        __syncwarp();
        tc::fence_after_sync();
        tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
        constexpr uint32_t idesc = tc::idesc_f16(BM, BN);  // every operand of the fused decoder is fp16
        constexpr uint32_t idesc_z = tc::idesc_f16(BM, BN);
        const int s_z = num_kb % STAGES;  // ring slot of the branch k-block (the centred latents)
        if (lane == 0) {
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                tc::mbar_wait(&full[s], ph);
                tc::fence_after_sync();
                const uint32_t a_base = tc::smem_u32(tiles + s * STAGE_BYTES);
                const uint32_t b_base = a_base + A_BYTES;
#pragma unroll
                for (int kk = 0; kk < BK / 16; ++kk)
                    tc::umma_bf16(tmem_base, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(b_base + kk * 32, 16, 1024),
                                  idesc, (i > 0 || kk > 0) ? 1u : 0u);
                tc::umma_commit(&empty[s]);
            }
        }
        __syncwarp();
        if (!at_once) {
            tc::tmem_alloc(tmem_slot + 1, Z_COLS);  // whole warp; blocks while two other CTAs own their full sets
            tc::fence_before_sync();
            __syncwarp();
            tc::fence_after_sync();
        }
        tmem_z = *reinterpret_cast<volatile uint32_t*>(tmem_slot + 1);
        if (lane == 0) {
            tc::mbar_arrive(tmem_ready);  // release: the epilogue warps read the slots after acquiring this barrier
            tc::mbar_wait(z_full, 0);
            tc::mbar_wait(&full[s_z], (num_kb / STAGES) & 1);
            tc::fence_after_sync();
            const uint32_t a_base = tc::smem_u32(tiles + s_z * STAGE_BYTES);
            const uint32_t zp_base = tc::smem_u32(z_tiles), zs_base = zp_base + B_BYTES;
#pragma unroll
            for (int kk = 0; kk < BK / 16; ++kk) {
                tc::umma_bf16(tmem_z, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(zp_base + kk * 32, 16, 1024), idesc_z,
                              kk > 0 ? 1u : 0u);
                tc::umma_bf16(tmem_z + BN, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(zs_base + kk * 32, 16, 1024),
                              idesc_z, kk > 0 ? 1u : 0u);
            }
            tc::umma_commit(tmem_full);
        }
        __syncwarp();
    } else {
        // ================= epilogue: 8 warps =================
        const int et = threadIdx.x - 64;
        const long G = p.G;
        // Every global load of the prologue is issued before anything waits on one (as in nb_tc_fwd_kernel): the row indices
        // first, then the per-row and per-gene constants; the LUT is computed while they are in flight.
        const int e = warp - 2;
        const int q = warp & 3;
        const int half = e >> 2;
        const int rloc = q * 32 + lane;
        const int m = m0 + rloc;
        const bool mok = m < p.B;
        const int mm = mok ? m : 0;
        constexpr int NGATHER = BM / EPI_WARPS / GATHER_ROWS;
        int ridx[NGATHER];
#pragma unroll
        for (int i = 0; i < NGATHER; ++i) {
            const int gm = m0 + cnt_row(e, lane, i);
            ridx[i] = gm < p.B ? (p.rows ? __ldg(p.rows + gm) : gm) : -1;
        }
        const int my_row = p.rows ? __ldg(p.rows + mm) : mm;
        const float libm = __ldg(p.lib + mm);
        float4 gcv = make_float4(1.0f, 1.0f, 0.0f, 0.0f);
        static_assert(BN <= EPI_THREADS, "one thread per gene of the tile stages its constants");
        if (et < BN && n0 + et < p.G) {
            const int g = n0 + et;
            gcv.x = __ldg(p.genec + GC_THETA * G + g);
            gcv.y = __ldg(p.genec + GC_KC * G + g);
            gcv.z = __ldg(p.genec + GC_K1C * G + g);
            gcv.w = __ldg(p.bm + g);
        }
        float4 tgv[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int w16 = et + u * EPI_THREADS;
            const int g = n0 + (w16 >> 3);
            tgv[u] = g < p.G ? __ldg(reinterpret_cast<const float4*>(p.tgf + (long)n0 * NB_TAB) + w16) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        // the digamma terms of the tile's genes: BN * NB_TAB floats = one 16-byte word per epilogue thread (gene et / 4)
        static_assert(BN * NB_TAB * 4 == EPI_THREADS * 16, "one 16-byte word of the d-theta table per epilogue thread");
        const float4 tbv = n0 + (et >> 2) < p.G ? __ldg(reinterpret_cast<const float4*>(p.tb1 + (long)n0 * NB_TAB) + et) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        // coalesced row gather of the tile's counts into registers as count codes (overlaps the MMA phase)
        uint32_t cw[NGATHER];
        {
            const int g = n0 + 2 * (lane % (BN / 2));
#pragma unroll
            for (int i = 0; i < NGATHER; ++i) cw[i] = 0u;
            constexpr int BATCH = SRC == SPV_SRC_U16_LOG1P ? NGATHER : NGATHER / 2;  // every load of a batch in flight before any is used
            if (nb_pair_vec_ok<SRC>(p.X, p.ldx, g, p.G)) {
#pragma unroll
                for (int i0 = 0; i0 < NGATHER; i0 += BATCH) {
                    uint2 raw[BATCH];
#pragma unroll
                    for (int i = 0; i < BATCH; ++i) {
                        raw[i] = make_uint2(0u, 0u);
                        if (ridx[i0 + i] >= 0) raw[i] = nb_load_pair_vec<SRC>(p.X, (long)ridx[i0 + i] * p.ldx, g);
                    }
#pragma unroll
                    for (int i = 0; i < BATCH; ++i) cw[i0 + i] = nb_pair_codes<SRC>(raw[i]);
                }
            } else {  // odd pitch, unaligned base or the last gene of an odd-sized matrix: element loads
#pragma unroll
                for (int i = 0; i < NGATHER; ++i)
                    if (ridx[i] >= 0) cw[i] = nb_pair_codes<SRC>(nb_load_pair<SRC>(p.X, (long)ridx[i] * p.ldx, g, p.G));
            }
        }
        if (et < BN) s_gc[et] = gcv;
#pragma unroll
        for (int u = 0; u < 2; ++u) reinterpret_cast<float4*>(s_tg)[et + u * EPI_THREADS] = tgv[u];
        const float c_row = 4096.0f * fast_exp(-libm);  // rho -> 4096 x softmax value: fp16-safe whatever the library size
        const long xrow = (long)my_row * p.ldx;
        // One epilogue warp polls the two mbarriers; the other seven block in a named barrier, where they cost no issue slots (a
        // CTA waiting for its tensor-memory grant spends most of its life here: eight polling warps took a quarter of the SM's
        // issued instructions away from the two CTAs doing the math - profiles/r2_nb_ncu.md)
        if (e == 0) {
            tc::mbar_wait(tmem_ready, 0);
            tc::mbar_wait(tmem_full, 0);  // accumulators complete; the operand stages are free from here on
            tc::fence_after_sync();
        }
        tc::fence_before_sync();
        asm volatile("bar.sync 2, %0;" ::"r"(EPI_THREADS) : "memory");
        tc::fence_after_sync();
        tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
        tmem_z = *reinterpret_cast<volatile uint32_t*>(tmem_slot + 1);
#pragma unroll
        for (int i = 0; i < NGATHER; ++i) s_cnt[cnt_row(e, lane, i) * CNT_PITCH_W + lane % (BN / 2)] = cw[i];
        reinterpret_cast<float4*>(s_tb)[et] = tbv;
        asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");
        // running store addresses: this cell's slot in the row of the first gene of the current four (byte pitches are 32-bit)
        const uint32_t ldb_e = (uint32_t)p.ld_e4 * 2u, ldb_d = (uint32_t)p.ld_dpi * 2u;
        unsigned long long a_e = reinterpret_cast<unsigned long long>(p.e4t) + (unsigned long long)(n0 + half * WCOLS) * ldb_e + 8ull * (unsigned)m;
        unsigned long long a_d = reinterpret_cast<unsigned long long>(p.dpit) + (unsigned long long)(n0 + half * WCOLS) * ldb_d + 2ull * (unsigned)m;
        float sll = 0.0f, sep = 0.0f, ses = 0.0f;
        const bool full_tile = n0 + BN <= p.G && m0 + BM <= p.B;  // CTA-uniform
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16), lane_z = tmem_z + ((uint32_t)(q * 32) << 16);
        const uint32_t* cnt_row_p = s_cnt + rloc * CNT_PITCH_W + half * (WCOLS / 2);
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
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem_z, Z_COLS);
        tc::tmem_dealloc(tmem_base, ACC_COLS);
        unsigned int smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        if (lane == 0) atomicSub(&g_resident_trn[smid & 255], 1);
    }
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
    if (!ptrs || !amix_f16 || !wstack_f16 || !zc_f16 || !wz_f16 || !e4t || !dpit || Gp < G || B <= 0 || G <= 0 || P <= 0 || S <= 0 ||
        ld_e4 < 4ll * B || ld_dpi < B || (ld_e4 & 3) || ld_e4 >= (1ll << 28))
        return SPV_ERR_ARG;
    if (P + S > ZK_MAX_LATENT) return SPV_ERR_ARG;
    const int need[] = {0, 5, 6, 7, 11, 15, 17, 18};
    for (int i : need)
        if (!ptrs[i]) return SPV_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(ptrs[17]) | reinterpret_cast<uintptr_t>(ptrs[18]) | reinterpret_cast<uintptr_t>(e4t)) & 15) return SPV_ERR_ARG;
    const int K = kmix > 0 ? kmix : HD + P + S;
    CUtensorMap ma, mb, mz, mzc;
    int rc = spv_make_tensor_map_bf16(&ma, amix_f16, (unsigned long long)K, (unsigned long long)B, (unsigned long long)ld_amixb, 64, BM);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mb, wstack_f16, (unsigned long long)K, (unsigned long long)G, (unsigned long long)ld_w, 64, BN);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mz, wz_f16, 64ull, (unsigned long long)(2 * Gp), 64ull, 64, BN);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mzc, zc_f16, 64ull, (unsigned long long)B, 64ull, 64, BM);
    if (rc != SPV_OK) return rc;
    NbTcTrainParams p;
    p.X = ptrs[0]; p.ldx = ldx; p.rows = (const int*)ptrs[1]; p.bm = (const float*)ptrs[5]; p.genec = (const float*)ptrs[6];
    p.lib = (const float*)ptrs[7]; p.tgf = (const float2*)ptrs[17]; p.tb1 = (const float*)ptrs[18]; p.part_nb = (float*)ptrs[11];
    p.colpart = (float*)ptrs[15];
    p.e4t = reinterpret_cast<__half*>(e4t); p.ld_e4 = ld_e4; p.dpit = reinterpret_cast<__half*>(dpit); p.ld_dpi = ld_dpi;
    p.B = B; p.G = G; p.K = K; p.Gp = Gp;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
        if (cudaFuncSetAttribute(nb_tc_train_kernel<SPV_SRC_U16_LOG1P>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess ||
            cudaFuncSetAttribute(nb_tc_train_kernel<SPV_SRC_F32_LOG1P>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess)
            return SPV_ERR_LAUNCH;
        configured[dev & 63] = true;
    }
    dim3 grid((G + BN - 1) / BN, (B + BM - 1) / BM);
    if (src == SPV_SRC_U16_LOG1P) nb_tc_train_kernel<SPV_SRC_U16_LOG1P><<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, mz, mzc, p);
    else if (src == SPV_SRC_F32_LOG1P) nb_tc_train_kernel<SPV_SRC_F32_LOG1P><<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, mz, mzc, p);
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
