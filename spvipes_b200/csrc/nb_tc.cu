// Fused decoder GEMMs + NB-mixture log-likelihood, tensor-core path (the north-star kernel).
//
//   pi[b, g] = [hm | z_private_arg | z_shared_arg][b, :] . Wm[g, :] + bm[g]                 K = 256 + P + S
//   lp[b, g] = z_private_arg[b, :] . W'p[g, :] + cp[g],   ls[b, g] = z_shared_arg[b, :] . W's[g, :] + cs[g]
//                                      (W', c: BatchNorm folded into the factor regressors by spv_dec_fold)
//   rec_b    = - sum_g log_mixture_nb(log1p(x[b, g]); exp(lib) softmax(lp), exp(lib) softmax(ls), theta, pi)
//
// All three contractions run on tcgen05.mma (operands via TMA, fp32 accumulators in TMEM: 64 columns for pi, 2 x 64 for
// lp | ls, allocated separately).  pi: bf16 [hm | zz] against the bf16 mixture weight.  lp, ls: ONE extra 64-wide k-block of
// fp16 operands - the centred latents zz - mean(zz) against the folded weights (spv_dec_fold writes both) - streamed through
// the same shared-memory ring after the mixture k-blocks.  The softmax branches are where operand rounding hurts (it acts
// coherently on every cell of a gene and feeds sums that cancel over the minibatch: tools/diag_grad_noise.py), hence fp16
// (2^-12) and the centring (the shift of the centred form is exactly beta).
// One 128 (cells) x 64 (genes) tile per CTA, three CTAs resident per SM of which two own a full accumulator set (the third
// streams its operands and completes pi while it waits: see the allocation in the MMA warp).  warp 0: TMA producer, warp 1:
// TMEM allocator + MMA issuer, warps 2..9: epilogue (thread = cell row; two warps per TMEM lane quarter, 32 gene columns each).  Once the accumulators
// are complete the operand stages are reused for the tile's raw counts (coalesced row gather, uint16); the accumulators
// are streamed out of TMEM four columns at a time.  Nothing of size [B, G] is written unless store_pi is set.
// Reference: nn/networks.py:314-325, module/spVIPESmodule.py:751-759, 817-824; scvi log_mixture_nb.
#include "tc_common.cuh"
#include "nb_math.cuh"
#include "decoder_common.cuh"
#include "../../include/spvipes_b200.h"

// diagnostic hook (NB_TRACE builds, tools/nb_tile_trace*.py): per-CTA %globaltimer stamps go to this device buffer
static long long* g_trace_buf = nullptr;
extern "C" void spv_debug_trace(long long* buf) { g_trace_buf = buf; }
extern "C" long long* spv_debug_get_trace() { return g_trace_buf; }

namespace {

#ifndef NB_STAGES
#define NB_STAGES 2
#endif
constexpr int BM = 128, BN = 64, BK = 64, STAGES = NB_STAGES;
constexpr int WCOLS = BN / 2;                 // gene columns per epilogue warp (two warps per TMEM lane quarter)
constexpr int GATHER_ROWS = 64 / BN;          // rows of the count tile one warp gathers per load: 32 lanes cover BN / 2 words each
constexpr int EPI_WARPS = 8, EPI_THREADS = 32 * EPI_WARPS;
constexpr int THREADS = 64 + EPI_THREADS;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int ACC_COLS = BN, Z_COLS = 2 * BN;             // the likelihood kernels allocate in two steps (powers of two >= 32)
static_assert(ACC_COLS == 32 || ACC_COLS == 64, "tensor-memory allocations are powers of two");
constexpr int CNT_PITCH_W = BN / 2 + 2;  // count-code tile: 34 32-bit words per row - thread = row reads 64 bits (four codes) conflict-free
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 2 * B_BYTES + 1024 + BN * 16 + BN * NB_TAB * 8 + 256;

static_assert(BM * CNT_PITCH_W * 4 <= STAGES * STAGE_BYTES, "count tile must fit in the operand stages");
static_assert(3 * (SMEM_BYTES + 1024) <= 228 * 1024, "three CTAs per SM");

// Element sweep (ELEM variant): five optional fp32 outputs per element, in this order (spv_dec_nb_elems_tc)
enum { EO_LL = 0, EO_RATE_P, EO_RATE_S, EO_PI, EO_MEAN, EO_N };
// Each epilogue warp stages a 32-cell x EO_CH-gene slab per output in the operand stages and the folded-weight tiles (both free
// once the accumulators are complete), behind the count tile; lane -> (cell lane / EO_CH + 32 / EO_CH * k, gene lane % EO_CH)
// then makes every warp store four whole 32-byte sectors instead of 32 rows x 16 bytes.  Pitch EO_CH + 1: the thread = cell
// writes are conflict-free.
constexpr int EO_CH = 8, EO_PITCH = EO_CH + 1;
constexpr int EO_SLAB_OFF = BM * CNT_PITCH_W * 4;
constexpr int EO_WARP_FLOATS = EO_N * 32 * EO_PITCH;
static_assert(EO_SLAB_OFF + EPI_WARPS * EO_WARP_FLOATS * 4 <= STAGES * STAGE_BYTES + 2 * B_BYTES, "element slabs must fit");

struct NbTcParams {
    const void* X; long ldx; const int* rows;
    const float* bm;                   // [G]
    const float* genec;                // [GC_N, G]
    const float2* tgf;                 // [G, NB_TAB] forward count table (spv_dec_theta_tables)
    float* part_nb;                    // [nTG, B, 3]
    int B, G, K;
    int Gp;                            // row offset of the shared block inside the folded-weight operand
    long long* trace;                  // diagnostic (NB_TRACE builds): 6 globaltimer stamps per CTA
    float* eo[EO_N];                   // ELEM variant: the outputs [B, ld_out] (NULL = not written)
    long ld_out;
};

// row of the count tile that lane `lane` of epilogue warp e loads in its i-th gather: a warp covers GATHER_ROWS rows per load
__device__ __forceinline__ int cnt_row(int e, int lane, int i) {
    return (e + EPI_WARPS * i) * GATHER_ROWS + lane / (BN / 2);
}

// CTAs of this kernel currently resident per SM (a scheduling hint only, see the allocation below; balanced by every CTA)
__device__ int g_resident_fwd[256];

// one element off the fast path (a count outside the table, a logit below the fast logarithm's range, an edge tile): out of line
template <int SRC>
__device__ __noinline__ NbOut nb_fwd_general(uint32_t code, float xp, float xs, float acc_pi, float4 gc, const uint8_t* tg_row,
                                             const void* X, long xidx, const float* lgt) {
    float2 tcn;
    if (code == NB_CODE_SLOW) {
        if (SRC == SPV_SRC_F32) tcn = nb_target_terms_fwd(nb_load_raw<SRC>(X, xidx), gc.x, __ldg(lgt));
        else tcn = nb_count_terms_fwd_slow(nb_load_raw<SRC>(X, xidx), gc.x, __ldg(lgt));
    }
    else tcn = *reinterpret_cast<const float2*>(tg_row + code);
    const float pi = acc_pi + gc.w;
    if (tcn.x != 0.0f && fminf(xp, xs) < NB_X_RARE) return nb_forward_v5<true>(tcn.x, tcn.y, xp, xs, pi, gc.x, gc.y, gc.z);
    return nb_forward_v5<false>(tcn.x, tcn.y, xp, xs, pi, gc.x, gc.y, gc.z);
}

// ELEM = false: the reducing sweep (row partials of the log-likelihood).  ELEM = true: the element sweep - the same MMAs and the
// same element math, but the epilogue stores the per-element outputs selected in p.eo (no partials) and gathers the counts only
// when the log-likelihood is requested.  It is not on the training step and gives up the third resident CTA.
template <int SRC, bool ELEM = false>
__global__ void __launch_bounds__(THREADS, ELEM ? 2 : 3) nb_tc_fwd_kernel(const __grid_constant__ CUtensorMap mapA,
                                                               const __grid_constant__ CUtensorMap mapB,
                                                               const __grid_constant__ CUtensorMap mapZ,
                                                               const __grid_constant__ CUtensorMap mapZc, NbTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = tc::smem_u32(smem_raw);
    const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
    uint8_t* tiles = smem_raw + pad;
    uint8_t* z_tiles = tiles + STAGES * STAGE_BYTES;                    // folded private | shared weights, [BN][64] fp16 each
    float4* s_gc = reinterpret_cast<float4*>(z_tiles + 2 * B_BYTES);    // [BN]: theta, theta + eps, theta log(theta + eps), bm
    uint8_t* s_tg = reinterpret_cast<uint8_t*>(s_gc + BN);              // [BN][NB_TAB] float2: (log1p(c), count term) per gene
    uint64_t* full = reinterpret_cast<uint64_t*>(s_tg + BN * NB_TAB * 8);
    uint64_t* empty = full + STAGES;
    uint64_t* z_full = empty + STAGES;
    uint64_t* tmem_full = z_full + 1;
    uint64_t* tmem_ready = tmem_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_ready + 1);
    uint32_t* s_cnt = reinterpret_cast<uint32_t*>(tiles);  // aliases the operand stages once the MMAs are done

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    const int num_kb = (p.K + BK - 1) / BK;
#ifdef NB_TRACE
    long long* tr = (p.trace && (threadIdx.x == 64 || threadIdx.x == 32)) ? p.trace + ((long)blockIdx.y * gridDim.x + blockIdx.x) * 8 : nullptr;
    auto stamp = [&](int i) { if (tr) { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); tr[i] = t; } };
    if (tr && threadIdx.x == 64) { unsigned int smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); tr[7] = smid; }
    if (threadIdx.x == 64) stamp(0);
#else
    auto stamp = [&](int) {};
#endif

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
    // Tensor memory is allocated by the MMA warp only when it is about to issue: 3 x 64 accumulator columns round up to 256, so
    // two CTAs own an SM's 512 columns, while registers and shared memory admit a third.  That third CTA runs its whole
    // prologue (operand loads into both stages, count gather) while it waits in tcgen05.alloc for an owner to exit, which hides
    // most of the ~5 us load phase behind the other CTAs' likelihood math (profiles/r1_nb_persistent_notes.md).
    uint32_t tmem_base = 0, tmem_z = 0;  // mixture-logit accumulator [BN columns]; the two branch-logit accumulators [2 BN]

    if (warp == 0) {
        if (tc::elect_one()) {
            tc::mbar_expect_tx(z_full, 2 * B_BYTES);
            tc::tma_load_2d(&mapZ, z_full, z_tiles, 0, n0);                   // folded private weights (rows 0..G), fp16
            tc::tma_load_2d(&mapZ, z_full, z_tiles + B_BYTES, 0, p.Gp + n0);  // folded shared weights (rows Gp..)
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                tc::mbar_wait(&empty[s], ph ^ 1);
                uint8_t* a_dst = tiles + s * STAGE_BYTES;
                tc::mbar_expect_tx(&full[s], STAGE_BYTES);
                tc::tma_load_2d(&mapA, &full[s], a_dst, i * BK, m0);
                tc::tma_load_2d(&mapB, &full[s], a_dst + A_BYTES, i * BK, n0);
            }
            {  // the branch k-block: centred latents + additive columns (fp16), A tile only, next slot of the ring
                const int s = num_kb % STAGES;
                const uint32_t ph = (num_kb / STAGES) & 1;
                tc::mbar_wait(&empty[s], ph ^ 1);
                tc::mbar_expect_tx(&full[s], A_BYTES);
                tc::tma_load_2d(&mapZc, &full[s], tiles + s * STAGE_BYTES, 0, m0);
            }
        }
    } else if (warp == 1) {
        // Two-step allocation.  The BN columns of the mixture-logit accumulator are free whenever at most two other CTAs hold
        // their full 3 x BN, so this CTA streams all its k-blocks through the stages and finishes that accumulator while it
        // is still waiting for tensor memory; only the 8 MMAs of the two branch logits (one k-block against the resident
        // folded-weight tiles) are left once the second allocation is granted.  One thread issues every MMA and commit.
        // A CTA that has allocated without giving up its permit keeps the SM from launching further CTAs (measured: the second
        // and third CTA of an SM entered 5 and 9.5 us after the first), so the two-step path is only taken by a CTA that finds
        // two others resident - the SM is full then anyway; the first two allocate everything at once.
        unsigned int smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        int ahead = 0;
        if (lane == 0) ahead = atomicAdd(&g_resident_fwd[smid & 255], 1);
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
            stamp(6);  // tensor memory granted
            tc::mbar_arrive(tmem_ready);  // release: the epilogue warps read the slots after acquiring this barrier
            tc::mbar_wait(z_full, 0);
            tc::mbar_wait(&full[s_z], (num_kb / STAGES) & 1);
            tc::fence_after_sync();
            const uint32_t a_base = tc::smem_u32(tiles + s_z * STAGE_BYTES);
            const uint32_t zp_base = tc::smem_u32(z_tiles), zs_base = zp_base + B_BYTES;
#pragma unroll
            for (int kk = 0; kk < BK / 16; ++kk) {  // the two branch logits, complete: latents, shift and row normaliser (fp16)
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
        const int et = threadIdx.x - 64;  // 0..255
        const long G = p.G;
        // Every global load of the prologue is issued before anything waits on one: the row indices first (the count gather
        // depends on them), then the per-gene constants and the count table of the tile's genes.
        const int e = warp - 2;
        const int q = warp & 3;          // TMEM lane quarter this warp may access
        const int half = e >> 2;         // which 32 gene columns of the tile
        const int rloc = q * 32 + lane;  // row within the tile
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
        const bool counts = !ELEM || p.eo[EO_LL] != nullptr;  // CTA-uniform
        float4 gcv = make_float4(1.0f, 1.0f, 0.0f, 0.0f);
        static_assert(BN <= EPI_THREADS, "one thread per gene of the tile stages its constants");
        if (et < BN && n0 + et < p.G) {
            const int g = n0 + et;
            gcv.x = __ldg(p.genec + GC_THETA * G + g);
            gcv.y = __ldg(p.genec + GC_THE * G + g);
            gcv.z = __ldg(p.genec + GC_KC * G + g);
            gcv.w = __ldg(p.bm + g);
        }
        // the tile's slice of the count table: BN * NB_TAB * 8 bytes = 2 x 16 bytes per epilogue thread
        static_assert(BN * NB_TAB * 8 == EPI_THREADS * 32, "two 16-byte table words per epilogue thread");
        float4 tgv[2] = {};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (!counts) break;
            const int w16 = et + u * EPI_THREADS;          // 16-byte word of the slice: gene w16 / 8
            const int g = n0 + (w16 >> 3);
            tgv[u] = g < p.G ? __ldg(reinterpret_cast<const float4*>(p.tgf + (long)n0 * NB_TAB) + w16) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        // coalesced row gather of the tile's counts into registers as count codes (overlaps the MMA phase): warp e takes rows
        // e, e + 8, ...; lane l takes genes 2l, 2l + 1
        uint32_t cw[NGATHER];
        {
            const int g = n0 + 2 * (lane % (BN / 2));
#pragma unroll
            for (int i = 0; i < NGATHER; ++i) cw[i] = 0u;
            constexpr int BATCH = SRC == SPV_SRC_U16_LOG1P ? NGATHER : NGATHER / 2;  // every load of a batch in flight before any is used
            if (!counts) {
            } else if (nb_pair_vec_ok<SRC>(p.X, p.ldx, g, p.G)) {
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
        for (int u = 0; u < 2; ++u)
            if (counts) reinterpret_cast<float4*>(s_tg)[et + u * EPI_THREADS] = tgv[u];
        const long xrow = (long)my_row * p.ldx;
        stamp(2);  // count gather issued
        tc::mbar_wait(tmem_ready, 0);
        tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
        tmem_z = *reinterpret_cast<volatile uint32_t*>(tmem_slot + 1);
        tc::mbar_wait(tmem_full, 0);  // accumulators complete; the operand stages are free from here on
        tc::fence_after_sync();
        stamp(3);  // accumulators complete
#pragma unroll
        for (int i = 0; i < NGATHER; ++i)
            if (counts) s_cnt[cnt_row(e, lane, i) * CNT_PITCH_W + lane % (BN / 2)] = cw[i];
        asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");  // constants + counts staged (epilogue warps only)
        stamp(4);  // counts staged
        const uint32_t* cnt_row_p = s_cnt + rloc * CNT_PITCH_W + half * (WCOLS / 2);
        if constexpr (ELEM) {
            const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16), lane_z = tmem_z + ((uint32_t)(q * 32) << 16);
            float* slab = reinterpret_cast<float*>(tiles + EO_SLAB_OFF) + e * EO_WARP_FLOATS;
#pragma unroll 1
            for (int j8 = 0; j8 < WCOLS; j8 += EO_CH) {
#pragma unroll
                for (int j4 = j8; j4 < j8 + EO_CH; j4 += 4) {
                    const int c0 = half * WCOLS + j4;
                    uint32_t rpi[4], rlp[4], rls[4];
                    tc::tmem_ld4(lane_addr + (uint32_t)c0, rpi);
                    tc::tmem_ld4(lane_z + (uint32_t)c0, rlp);
                    tc::tmem_ld4(lane_z + (uint32_t)(BN + c0), rls);
                    const uint2 cc = counts ? *reinterpret_cast<const uint2*>(cnt_row_p + (j4 >> 1)) : make_uint2(0u, 0u);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int gl = c0 + jj, g = n0 + gl;
                        const float4 gc = s_gc[gl];
                        const float xp = __uint_as_float(rlp[jj]), xs = __uint_as_float(rls[jj]), pi = __uint_as_float(rpi[jj]) + gc.w;
                        float ll = 0.0f;
                        if (counts && mok && g < p.G) {  // the element form the reducing sweep takes for this element
                            const uint32_t w = jj < 2 ? cc.x : cc.y;
                            const uint32_t code = (jj & 1) ? (w >> 16) : (w & 0xffffu);
                            if (code == NB_CODE_SLOW) {
                                ll = nb_fwd_general<SRC>(code, xp, xs, __uint_as_float(rpi[jj]), gc, s_tg + gl * (NB_TAB * 8), p.X, xrow + g,
                                                         p.genec + GC_LGT * G + g).ll;
                            } else {
                                const float2 tcn = *reinterpret_cast<const float2*>(s_tg + gl * (NB_TAB * 8) + code);
                                if (tcn.x != 0.0f && fminf(xp, xs) < NB_X_RARE) ll = nb_forward_v5<true>(tcn.x, tcn.y, xp, xs, pi, gc.x, gc.y, gc.z).ll;
                                else ll = nb_forward_v5<false>(tcn.x, tcn.y, xp, xs, pi, gc.x, gc.y, gc.z).ll;
                            }
                        }
                        const float rp = fast_ex2(xp), rs = fast_ex2(xs);
                        // sigma(pi) and sigma(-pi) each in its accurate form (neither is 1 minus the other): mean keeps its digits
                        // at mixture logits of either sign
                        const float sg = 1.0f / (1.0f + __expf(-pi)), sn = 1.0f / (1.0f + __expf(pi));
                        float* s = slab + lane * EO_PITCH + (j4 - j8 + jj);
                        s[EO_LL * 32 * EO_PITCH] = ll;
                        s[EO_RATE_P * 32 * EO_PITCH] = rp;
                        s[EO_RATE_S * 32 * EO_PITCH] = rs;
                        s[EO_PI * 32 * EO_PITCH] = pi;
                        s[EO_MEAN * 32 * EO_PITCH] = fmaf(sg, rp, sn * rs);
                    }
                }
                __syncwarp();
                const int col = lane % EO_CH, g = n0 + half * WCOLS + j8 + col;
#pragma unroll
                for (int o = 0; o < EO_N; ++o) {
                    float* dst = p.eo[o];
                    if (dst == nullptr) continue;
#pragma unroll
                    for (int r = lane / EO_CH; r < 32; r += 32 / EO_CH) {
                        const int m = m0 + q * 32 + r;
                        if (m < p.B && g < p.G) dst[(long)m * p.ld_out + g] = slab[(o * 32 + r) * EO_PITCH + col];
                    }
                }
                __syncwarp();
            }
        } else {
        float sll = 0.0f, sep = 0.0f, ses = 0.0f;
        const bool full_tile = n0 + BN <= p.G && m0 + BM <= p.B;  // CTA-uniform
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16), lane_z = tmem_z + ((uint32_t)(q * 32) << 16);
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
            // smallest branch logit of the four elements: log2(rho + eps) = log2(rho) needs rho >= 1e-6 wherever the count is positive
            const float xm = fminf(fminf(fminf(__uint_as_float(rlp[0]), __uint_as_float(rls[0])), fminf(__uint_as_float(rlp[1]), __uint_as_float(rls[1]))),
                                   fminf(fminf(__uint_as_float(rlp[2]), __uint_as_float(rls[2])), fminf(__uint_as_float(rlp[3]), __uint_as_float(rls[3]))));
            const bool plain = full_tile && (call & 0x80008000u) == 0u && !(call != 0u && xm < NB_X_RARE);
            if (plain) {  // every count tabulated, every column and row valid, the fast logarithm holds
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int gl = c0 + jj;
                    const uint32_t w = jj < 2 ? cc.x : cc.y;
                    const uint32_t code = (jj & 1) ? (w >> 16) : (w & 0xffffu);
                    const float2 tcn = *reinterpret_cast<const float2*>(s_tg + gl * (NB_TAB * 8) + code);
                    const float4 gc = s_gc[gl];
                    const NbOut o = nb_forward_v5<false>(tcn.x, tcn.y, __uint_as_float(rlp[jj]), __uint_as_float(rls[jj]),
                                                         __uint_as_float(rpi[jj]) + gc.w, gc.x, gc.y, gc.z);
                    sll += o.ll; sep += o.ep; ses += o.es;
                }
            } else if (mok) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int gl = c0 + jj, g = n0 + gl;
                    if (g < p.G) {
                        const uint32_t w = jj < 2 ? cc.x : cc.y;
                        const uint32_t code = (jj & 1) ? (w >> 16) : (w & 0xffffu);
                        const NbOut o = nb_fwd_general<SRC>(code, __uint_as_float(rlp[jj]), __uint_as_float(rls[jj]), __uint_as_float(rpi[jj]),
                                                            s_gc[gl], s_tg + gl * (NB_TAB * 8), p.X, xrow + g, p.genec + GC_LGT * G + g);
                        sll += o.ll; sep += o.ep; ses += o.es;
                    }
                }
            }
        }
        if (mok) {
            float* o = p.part_nb + ((long)(blockIdx.x * 2 + half) * p.B + m) * 3;
            o[0] = sll; o[1] = sep; o[2] = ses;
        }
        }
        stamp(5);  // epilogue done
    }
    tc::fence_before_sync();
    __syncthreads();
    if (threadIdx.x == 64) stamp(1);  // every warp of the CTA done
    if (warp == 1) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem_z, Z_COLS);
        tc::tmem_dealloc(tmem_base, ACC_COLS);
        unsigned int smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        if (lane == 0) atomicSub(&g_resident_fwd[smid & 255], 1);
    }
}

// ---------------------------------------------------------------------------------------
// Softmax statistics of the two factor-regressor branches on the tensor cores: the base-2 logit y = zc . wz (latents against
// the folded weights, the shift riding in the ones columns, the R columns still zero: decoder_common.cuh ZK_*) is one 64-wide
// k-block, so a 128 x 64 tile costs 8 MMAs; each epilogue thread (= cell) reduces its 32 columns to (max, sum exp) per
// branch.  Using the same fp16 operands as the likelihood kernels makes the normaliser consistent with the rho they compute.
// part_stats [2 * ceil(G/64), B, 4] = (max_p, sum_p, max_s, sum_s), natural units.
// ---------------------------------------------------------------------------------------
constexpr int ST_SMEM = A_BYTES + 2 * B_BYTES + 1024 + 64;

__global__ void __launch_bounds__(THREADS, 3) nb_tc_stats_kernel(const __grid_constant__ CUtensorMap mapA,
                                                                 const __grid_constant__ CUtensorMap mapZ,
                                                                 float* __restrict__ part_stats, int B, int G, int Gp) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = tc::smem_u32(smem_raw);
    uint8_t* tiles = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
    uint8_t* z_tiles = tiles + A_BYTES;
    uint64_t* full = reinterpret_cast<uint64_t*>(z_tiles + 2 * B_BYTES);
    uint64_t* tmem_full = full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&mapA);
        tc::tma_prefetch_desc(&mapZ);
        tc::mbar_init(full, 1);
        tc::mbar_init(tmem_full, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, 128);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (tc::elect_one()) {
            tc::mbar_expect_tx(full, A_BYTES + 2 * B_BYTES);
            tc::tma_load_2d(&mapA, full, tiles, 0, m0);   // centred latents, fp16 [B, 64]
            tc::tma_load_2d(&mapZ, full, z_tiles, 0, n0);  // folded weights, fp16 [2 Gp, 64]
            tc::tma_load_2d(&mapZ, full, z_tiles + B_BYTES, 0, Gp + n0);
        }
    } else if (warp == 1) {
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::idesc_f16(BM, BN);
            tc::mbar_wait(full, 0);
            tc::fence_after_sync();
            const uint32_t a_base = tc::smem_u32(tiles), zp_base = tc::smem_u32(z_tiles), zs_base = zp_base + B_BYTES;
#pragma unroll
            for (int kk = 0; kk < BK / 16; ++kk) {
                tc::umma_bf16(tmem_base, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(zp_base + kk * 32, 16, 1024), idesc,
                              kk > 0 ? 1u : 0u);
                tc::umma_bf16(tmem_base + BN, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(zs_base + kk * 32, 16, 1024), idesc,
                              kk > 0 ? 1u : 0u);
            }
            tc::umma_commit(tmem_full);
        }
    } else {
        const int e = warp - 2, q = warp & 3, half = e >> 2;
        const int m = m0 + q * 32 + lane;
        tc::mbar_wait(tmem_full, 0);
        tc::fence_after_sync();
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        float yp[WCOLS], ys[WCOLS];  // this cell's 32 + 32 logits of the tile half, base-2 units
        float Mp = -INFINITY, Ms = -INFINITY;
#pragma unroll
        for (int j4 = 0; j4 < WCOLS; j4 += 4) {
            const int c0 = half * WCOLS + j4;
            uint32_t rp4[4], rs4[4];
            tc::tmem_ld4(lane_addr + (uint32_t)c0, rp4);
            tc::tmem_ld4(lane_addr + (uint32_t)(BN + c0), rs4);
            tc::tmem_ld_wait();
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const bool ok = n0 + c0 + jj < G;
                yp[j4 + jj] = ok ? __uint_as_float(rp4[jj]) : -INFINITY;
                ys[j4 + jj] = ok ? __uint_as_float(rs4[jj]) : -INFINITY;
                Mp = fmaxf(Mp, yp[j4 + jj]);
                Ms = fmaxf(Ms, ys[j4 + jj]);
            }
        }
        float Sp = 0.0f, Ss = 0.0f;
        if (Mp > -INFINITY) {  // at least one valid column in this half (the tile may end inside it)
#pragma unroll
            for (int j = 0; j < WCOLS; ++j) {
                Sp += fast_ex2(yp[j] - Mp);
                Ss += fast_ex2(ys[j] - Ms);
            }
        }
        if (m < B) {
            float4 o = make_float4(Mp * NB_LN2, Sp, Ms * NB_LN2, Ss);
            *reinterpret_cast<float4*>(part_stats + ((long)(blockIdx.x * 2 + half) * B + m) * 4) = o;
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem_base, 128);
    }
}

__global__ void rownb_tc_kernel(const float* __restrict__ part, int nPart, int B, float* __restrict__ rowc, float* __restrict__ rec) {
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    float ll = 0.0f, dp = 0.0f, ds = 0.0f;
#pragma unroll 8
    for (int t = lane; t < nPart; t += 32) {
        const float* o = part + ((long)t * B + b) * 3;
        ll += o[0]; dp += o[1]; ds += o[2];
    }
    ll = warp_sum(ll); dp = warp_sum(dp); ds = warp_sum(ds);
    if (lane == 0) {
        rec[b] = -ll;
        rowc[(long)b * 4 + 2] = dp;
        rowc[(long)b * 4 + 3] = ds;
    }
}

// wide variant for many gene tiles: one CTA per 32 rows, lanes over rows (each warp load is one contiguous 384-byte run of the
// [tile][row][3] layout), 8 warps split the tiles, fixed-order merge through shared memory
__global__ void __launch_bounds__(256) rownb_tc_wide_kernel(const float* __restrict__ part, int nPart, int B, float* __restrict__ rowc,
                                                            float* __restrict__ rec) {
    __shared__ float red[8][3][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * 32 + lane;
    const bool ok = b < B;
    float ll = 0.0f, dp = 0.0f, ds = 0.0f;
    const float* src = part + (long)(ok ? b : 0) * 3;
    constexpr int U = 8;
    for (int t0 = w; t0 < nPart; t0 += 8 * U) {
        float v[U][3];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int t = t0 + 8 * u;
            const bool in = ok && t < nPart;
            const float* o = src + (long)t * B * 3;
            v[u][0] = in ? __ldg(o) : 0.0f; v[u][1] = in ? __ldg(o + 1) : 0.0f; v[u][2] = in ? __ldg(o + 2) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) { ll += v[u][0]; dp += v[u][1]; ds += v[u][2]; }
    }
    red[w][0][lane] = ll; red[w][1][lane] = dp; red[w][2][lane] = ds;
    __syncthreads();
    if (w == 0 && ok) {
        float a = 0.0f, c = 0.0f, d = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) { a += red[i][0][lane]; c += red[i][1][lane]; d += red[i][2][lane]; }
        rec[b] = -a;
        rowc[(long)b * 4 + 2] = c;
        rowc[(long)b * 4 + 3] = d;
    }
}

}  // namespace

// per-device one-time kernel attribute (the attribute is per device; a process may drive several)
template <typename K>
static int set_smem_once(K kernel, int bytes, bool (&done)[64]) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (done[dev & 63]) return SPV_OK;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) return SPV_ERR_LAUNCH;
    done[dev & 63] = true;
    return SPV_OK;
}

// ptrs: the SPV_DEC_NPTR list of spv_dec_nb_fwd (X, rows, -, -, -, bm, genec, -, -, -, -, part_nb [>= 2 * ceil(G/64) * B * 3
// floats], ..., [17] = forward count table of spv_dec_theta_tables).  Operands (all fp16): amix_bf16 [B, ld_amixb] = [hm | zz];
// wstack_bf16 [>= G, ld_w]: rows [0, G) the mixture weight; zc_f16 [B, 64] / wz_f16 [2 Gp, 64]: the branch k-block of
// spv_dec_fold, completed by spv_dec_stats_tc (row normalisers).  Gp = G rounded up to a multiple of 8.
extern "C" int spv_dec_nb_fwd_tc(int src, const void* const* ptrs, long long ldx, const void* amix_bf16, long long ld_amixb,
                                 const void* wstack_bf16, long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, int B,
                                 int G, int HD, int P, int S, int store_pi, int kmix, void* stream) {
    if (!ptrs || !amix_bf16 || !wstack_bf16 || !zc_f16 || !wz_f16 || Gp < G || B <= 0 || G <= 0 || HD < 0 || P <= 0 || S <= 0)
        return SPV_ERR_ARG;
    if (P + S > ZK_MAX_LATENT) return SPV_ERR_ARG;  // the latent columns must fit the branch k-block below the additive columns
    const int need[] = {0, 5, 6, 11, 17};
    for (int i : need)
        if (!ptrs[i]) return SPV_ERR_ARG;
    if (store_pi) return SPV_ERR_ARG;  // the sweep keeps the mixture logits in tensor memory (the backward recomputes them)
    if (reinterpret_cast<uintptr_t>(ptrs[17]) & 15) return SPV_ERR_ARG;
    const int K = kmix > 0 ? kmix : HD + P + S;  // width of the mixing net's input ([hm | zz | covariates])
    CUtensorMap ma, mb, mz, mzc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = spv_make_tensor_map_bf16(&ma, amix_bf16, (unsigned long long)K, (unsigned long long)B, (unsigned long long)ld_amixb, 64, BM);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mb, wstack_bf16, (unsigned long long)K, (unsigned long long)G, (unsigned long long)ld_w, 64, BN);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mz, wz_f16, 64ull, (unsigned long long)(2 * Gp), 64ull, 64, BN);  // 16-bit elements: same map type
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mzc, zc_f16, 64ull, (unsigned long long)B, 64ull, 64, BM);
    if (rc != SPV_OK) return rc;
    NbTcParams p;
    p.Gp = Gp;
    p.X = ptrs[0]; p.ldx = ldx; p.rows = (const int*)ptrs[1]; p.bm = (const float*)ptrs[5]; p.genec = (const float*)ptrs[6];
    p.tgf = (const float2*)ptrs[17]; p.part_nb = (float*)ptrs[11];
    p.B = B; p.G = G; p.K = K;
    p.trace = spv_debug_get_trace();
#ifdef NB_TRACE
    {  // consecutive launches (the two groups of a step) stamp alternate halves of the buffer
        static int n_launch = 0;
        if (p.trace) p.trace += (long)(n_launch++ & 1) * 8 * ((G + BN - 1) / BN) * ((B + BM - 1) / BM);
    }
#endif
    static bool done_u16[64] = {}, done_f32[64] = {};
    if (set_smem_once(nb_tc_fwd_kernel<SPV_SRC_U16_LOG1P>, SMEM_BYTES, done_u16) != SPV_OK ||
        set_smem_once(nb_tc_fwd_kernel<SPV_SRC_F32_LOG1P>, SMEM_BYTES, done_f32) != SPV_OK)
        return SPV_ERR_LAUNCH;
    dim3 grid((G + BN - 1) / BN, (B + BM - 1) / BM);
    if (src == SPV_SRC_U16_LOG1P) nb_tc_fwd_kernel<SPV_SRC_U16_LOG1P><<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, mz, mzc, p);
    else if (src == SPV_SRC_F32_LOG1P) nb_tc_fwd_kernel<SPV_SRC_F32_LOG1P><<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, mz, mzc, p);
    else return SPV_ERR_ARG;
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// Element sweep: the operands and ptrs of spv_dec_nb_fwd_tc (ptrs[11], the row partials, unused), outputs in `outs` (a HOST array
// of EO_N device pointers, see the header).  The counts (ptrs[0], ptrs[1]) and the count table (ptrs[17]) are read only when the
// log-likelihood is requested; src SPV_SRC_F32 reads ptrs[0] as target values t (no log1p).
extern "C" int spv_dec_nb_elems_tc(int src, const void* const* ptrs, long long ldx, const void* amix_bf16, long long ld_amixb,
                                   const void* wstack_bf16, long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, int B,
                                   int G, int HD, int P, int S, int kmix, void* const* outs, long long ld_out, void* stream) {
    if (!ptrs || !outs || !amix_bf16 || !wstack_bf16 || !zc_f16 || !wz_f16 || Gp < G || B <= 0 || G <= 0 || HD < 0 || P <= 0 ||
        S <= 0 || ld_out < G)
        return SPV_ERR_ARG;
    if (P + S > ZK_MAX_LATENT) return SPV_ERR_ARG;
    if (src != SPV_SRC_F32 && src != SPV_SRC_U16_LOG1P && src != SPV_SRC_F32_LOG1P) return SPV_ERR_ARG;
    if (!ptrs[5] || !ptrs[6]) return SPV_ERR_ARG;
    bool any = false;
    for (int o = 0; o < EO_N; ++o) any = any || outs[o] != nullptr;
    if (!any) return SPV_ERR_ARG;
    if (outs[EO_LL] && (!ptrs[0] || !ptrs[17] || (reinterpret_cast<uintptr_t>(ptrs[17]) & 15))) return SPV_ERR_ARG;
    const int K = kmix > 0 ? kmix : HD + P + S;
    CUtensorMap ma, mb, mz, mzc;
    int rc = spv_make_tensor_map_bf16(&ma, amix_bf16, (unsigned long long)K, (unsigned long long)B, (unsigned long long)ld_amixb, 64, BM);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mb, wstack_bf16, (unsigned long long)K, (unsigned long long)G, (unsigned long long)ld_w, 64, BN);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mz, wz_f16, 64ull, (unsigned long long)(2 * Gp), 64ull, 64, BN);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mzc, zc_f16, 64ull, (unsigned long long)B, 64ull, 64, BM);
    if (rc != SPV_OK) return rc;
    NbTcParams p{};
    p.Gp = Gp;
    p.X = ptrs[0]; p.ldx = ldx; p.rows = (const int*)ptrs[1]; p.bm = (const float*)ptrs[5]; p.genec = (const float*)ptrs[6];
    p.tgf = (const float2*)ptrs[17]; p.part_nb = nullptr;
    p.B = B; p.G = G; p.K = K;
    p.trace = nullptr;
    for (int o = 0; o < EO_N; ++o) p.eo[o] = reinterpret_cast<float*>(outs[o]);
    p.ld_out = ld_out;
    static bool done[3][64] = {};
    if (set_smem_once(nb_tc_fwd_kernel<SPV_SRC_F32, true>, SMEM_BYTES, done[0]) != SPV_OK ||
        set_smem_once(nb_tc_fwd_kernel<SPV_SRC_U16_LOG1P, true>, SMEM_BYTES, done[1]) != SPV_OK ||
        set_smem_once(nb_tc_fwd_kernel<SPV_SRC_F32_LOG1P, true>, SMEM_BYTES, done[2]) != SPV_OK)
        return SPV_ERR_LAUNCH;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dim3 grid((G + BN - 1) / BN, (B + BM - 1) / BM);
    if (src == SPV_SRC_F32) nb_tc_fwd_kernel<SPV_SRC_F32, true><<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, mz, mzc, p);
    else if (src == SPV_SRC_U16_LOG1P) nb_tc_fwd_kernel<SPV_SRC_U16_LOG1P, true><<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, mz, mzc, p);
    else nb_tc_fwd_kernel<SPV_SRC_F32_LOG1P, true><<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, mz, mzc, p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

int spv_internal_rowstat(const float* part, int nparts, int B, const float* lib, float* rowc, void* zc_f16, cudaStream_t st);

// Softmax normalisers of the two branches on the tensor cores: rowc[b, 0:2] = lib[b] - logsumexp_g(y_p / y_s)   (phase 1 of
// spv_dec_nb_fwd for the tensor-core path), from the fp16 operands spv_dec_fold wrote: zc_f16 [B, 64] centred latents, wz_f16
// [2 Gp, 64] folded weights.  Also writes the normalisers into the R columns of zc_f16 (decoder_common.cuh ZK_RP / ZK_RS), which
// completes the branch operand for the likelihood sweeps.  part_stats needs 2 * ceil(G/64) * B * 4 floats.
extern "C" int spv_dec_stats_tc(void* zc_f16, const void* wz_f16, int Gp, const float* genec, const float* lib,
                                float* part_stats, float* rowc, int B, int G, int P, int S, void* stream) {
    if (!zc_f16 || !wz_f16 || !genec || !lib || !part_stats || !rowc || Gp < G || B <= 0 || G <= 0 || P <= 0 || S <= 0)
        return SPV_ERR_ARG;
    if (P + S > ZK_MAX_LATENT) return SPV_ERR_ARG;
    CUtensorMap ma, mz;
    int rc = spv_make_tensor_map_bf16(&ma, zc_f16, 64ull, (unsigned long long)B, 64ull, 64, BM);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mz, wz_f16, 64ull, (unsigned long long)(2 * Gp), 64ull, 64, BN);
    if (rc != SPV_OK) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    static bool done[64] = {};
    if (set_smem_once(nb_tc_stats_kernel, ST_SMEM, done) != SPV_OK) return SPV_ERR_LAUNCH;
    dim3 grid((G + BN - 1) / BN, (B + BM - 1) / BM);
    nb_tc_stats_kernel<<<grid, THREADS, ST_SMEM, st>>>(ma, mz, part_stats, B, G, Gp);
    SPV_CHECK_LAUNCH();
    return spv_internal_rowstat(part_stats, 2 * (int)grid.x, B, lib, rowc, zc_f16, st);
}

// floats spv_dec_nb_fwd_tc needs in part_nb
extern "C" long long spv_dec_nb_part_floats(int B, int G) {
    if (B <= 0 || G <= 0) return 0;
    return 2ll * ((G + BN - 1) / BN) * B * 3;
}

// rec[b] = - sum over the row partials of spv_dec_nb_fwd_tc (same B, G, HD); also the softmax-backward row sums rowc[:, 2:4]
extern "C" int spv_dec_nb_rowreduce(const float* part_nb, int G, int B, int HD, float* rowc, float* rec, void* stream) {
    if (!part_nb || !rowc || !rec || G <= 0 || B <= 0 || HD < 0) return SPV_ERR_ARG;
    const int nPart = 2 * ((G + BN - 1) / BN);
    if (nPart > 128) rownb_tc_wide_kernel<<<(B + 31) / 32, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(part_nb, nPart, B, rowc, rec);
    else rownb_tc_kernel<<<(B + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(part_nb, nPart, B, rowc, rec);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}
