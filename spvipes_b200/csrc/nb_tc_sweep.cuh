// The tile pipeline of the tensor-core likelihood sweeps: nb_tc_fwd_kernel (the forward-only and the element sweep, nb_tc.cu)
// and nb_tc_train_kernel (the training sweep, nb_tc_train.cu).  Each kernel keeps its own epilogue; this header holds what they
// share.
//
// One 128 (cells) x 64 (genes) tile per CTA, three CTAs resident per SM of which two own a full accumulator set (the third
// streams its operands and completes pi while it waits: see the allocation in mma_warp).  warp 0: TMA producer, warp 1: TMEM
// allocator + MMA issuer, warps 2..9: epilogue (thread = cell row; two warps per TMEM lane quarter, 32 gene columns each).
// Accumulators (fp32, TMEM): pi, 64 columns, over the mixture k-blocks (fp16 [hm | zz] against the mixture weight); lp | ls, 2 x 64
// columns, allocated separately, over ONE extra 64-wide k-block (the centred latents + additive columns against the folded
// weights) streamed through the same shared-memory ring after the mixture k-blocks.  Once the accumulators are complete the
// operand stages are reused for the tile's raw counts (coalesced row gather, uint16 codes) and the kernel's own scratch.
#pragma once
#include "tc_common.cuh"
#include "nb_math.cuh"
#include "decoder_common.cuh"
#include "../../include/spvipes_b200.h"

namespace nbtc {

constexpr int BM = 128, BN = 64, BK = 64, STAGES = 2;
constexpr int WCOLS = BN / 2;                 // gene columns per epilogue warp (two warps per TMEM lane quarter)
constexpr int GATHER_ROWS = 64 / BN;          // rows of the count tile one warp gathers per load: 32 lanes cover BN / 2 words each
constexpr int EPI_WARPS = 8, EPI_THREADS = 32 * EPI_WARPS;
constexpr int THREADS = 64 + EPI_THREADS;
constexpr int NGATHER = BM / EPI_WARPS / GATHER_ROWS;  // count-tile rows per epilogue thread
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int ACC_COLS = BN, Z_COLS = 2 * BN;  // tensor memory is allocated in two steps (powers of two >= 32)
static_assert(ACC_COLS == 32 || ACC_COLS == 64, "tensor-memory allocations are powers of two");
constexpr int CNT_PITCH_W = BN / 2 + 2;  // count-code tile: 34 32-bit words per row - thread = row reads 64 bits (four codes) conflict-free
constexpr int CNT_BYTES = BM * CNT_PITCH_W * 4;  // the count tile, at the start of the drained operand stages
// 76 032 bytes: three CTAs per SM (3 x (76 032 + 1 024 reserved) <= 233 472)
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 2 * B_BYTES + 1024 + BN * 16 + BN * NB_TAB * 8 + 256;
static_assert(CNT_BYTES <= STAGES * STAGE_BYTES, "count tile must fit in the operand stages");
static_assert(3 * (SMEM_BYTES + 1024) <= 228 * 1024, "three CTAs per SM");

// The parameters every sweep reads (spv_dec_nb_fwd_tc's ptrs[] slots in brackets); each kernel extends them.
struct NbTcParams {
    const void* X; long ldx; const int* rows;  // counts [0] (row pitch ldx) and the minibatch's rows of them [1] (NULL: 0..B-1)
    const float* bm;                   // [G] [5]
    const float* genec;                // [GC_N, G] [6]
    const float2* tgf;                 // [G, NB_TAB] forward count table [17] (spv_dec_theta_tables)
    int B, G, K;
    int Gp;                            // row offset of the shared block inside the folded-weight operand
};

// Shared memory (SMEM_BYTES, aligned here to the 1024 bytes of the 128-byte swizzle)
struct Smem {
    uint8_t* tiles;        // STAGES x [A BM x BK | B BN x BK] operand stages
    uint8_t* z_tiles;      // folded private | shared weights, [BN][64] fp16 each
    float4* s_gc;          // [BN]: theta, two genec rows (per kernel), bm
    uint8_t* s_tg;         // [BN][NB_TAB] float2: (log1p(c), count term) per gene
    uint64_t *full, *empty, *z_full, *tmem_full, *tmem_ready;
    uint32_t* tmem_slot;   // [2]: the mixture-logit accumulator, the two branch-logit accumulators
    uint32_t* s_cnt;       // [BM][CNT_PITCH_W] count codes: aliases the operand stages once the MMAs are done
};

__device__ __forceinline__ Smem carve_smem() {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = tc::smem_u32(smem_raw);
    Smem s;
    s.tiles = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
    s.z_tiles = s.tiles + STAGES * STAGE_BYTES;
    s.s_gc = reinterpret_cast<float4*>(s.z_tiles + 2 * B_BYTES);
    s.s_tg = reinterpret_cast<uint8_t*>(s.s_gc + BN);
    s.full = reinterpret_cast<uint64_t*>(s.s_tg + BN * NB_TAB * 8);
    s.empty = s.full + STAGES;
    s.z_full = s.empty + STAGES;
    s.tmem_full = s.z_full + 1;
    s.tmem_ready = s.tmem_full + 1;
    s.tmem_slot = reinterpret_cast<uint32_t*>(s.tmem_ready + 1);
    s.s_cnt = reinterpret_cast<uint32_t*>(s.tiles);
    return s;
}

// descriptor prefetch and barrier init by one thread, then a CTA barrier
__device__ __forceinline__ void init_pipeline(const Smem& s, const CUtensorMap* mapA, const CUtensorMap* mapB, const CUtensorMap* mapZ,
                                              const CUtensorMap* mapZc, int warp, int lane) {
    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(mapA);
        tc::tma_prefetch_desc(mapB);
        tc::tma_prefetch_desc(mapZ);
        tc::tma_prefetch_desc(mapZc);
        for (int st = 0; st < STAGES; ++st) {
            tc::mbar_init(&s.full[st], 1);
            tc::mbar_init(&s.empty[st], 1);
        }
        tc::mbar_init(s.z_full, 1);
        tc::mbar_init(s.tmem_full, 1);
        tc::mbar_init(s.tmem_ready, 1);
        tc::fence_barrier_init();
    }
    __syncthreads();
}

// warp 0: the folded-weight tiles, the num_kb mixture k-blocks through the ring, then the branch k-block into the next ring slot
__device__ __forceinline__ void produce(const Smem& s, const CUtensorMap* mapA, const CUtensorMap* mapB, const CUtensorMap* mapZ,
                                        const CUtensorMap* mapZc, int n0, int m0, int num_kb, int Gp) {
    if (tc::elect_one()) {
        tc::mbar_expect_tx(s.z_full, 2 * B_BYTES);
        tc::tma_load_2d(mapZ, s.z_full, s.z_tiles, 0, n0);                 // folded private weights (rows 0..G), fp16
        tc::tma_load_2d(mapZ, s.z_full, s.z_tiles + B_BYTES, 0, Gp + n0);  // folded shared weights (rows Gp..)
        for (int i = 0; i < num_kb; ++i) {
            const int st = i % STAGES;
            const uint32_t ph = (i / STAGES) & 1;
            tc::mbar_wait(&s.empty[st], ph ^ 1);
            uint8_t* a_dst = s.tiles + st * STAGE_BYTES;
            tc::mbar_expect_tx(&s.full[st], STAGE_BYTES);
            tc::tma_load_2d(mapA, &s.full[st], a_dst, i * BK, m0);
            tc::tma_load_2d(mapB, &s.full[st], a_dst + A_BYTES, i * BK, n0);
        }
        {  // the branch k-block: centred latents + additive columns (fp16), A tile only, next slot of the ring
            const int st = num_kb % STAGES;
            const uint32_t ph = (num_kb / STAGES) & 1;
            tc::mbar_wait(&s.empty[st], ph ^ 1);
            tc::mbar_expect_tx(&s.full[st], A_BYTES);
            tc::tma_load_2d(mapZc, &s.full[st], s.tiles + st * STAGE_BYTES, 0, m0);
        }
    }
}

// warp 1: tensor-memory allocation and every MMA; tmem_base / tmem_z receive the two allocations (for release_tmem).
// Tensor memory is allocated only when the warp is about to issue: 3 x 64 accumulator columns round up to 256, so two CTAs own
// an SM's 512 columns, while registers and shared memory admit a third.  That third CTA runs its whole prologue (operand loads
// into both stages, count gather) while it waits for tensor memory, which hides most of the ~5 us load phase behind the other
// CTAs' likelihood math.
// Two-step allocation.  The BN columns of the mixture-logit accumulator are free whenever at most two other CTAs hold their full
// 3 x BN, so this CTA streams all its k-blocks through the stages and finishes that accumulator while it is still waiting for
// tensor memory; only the 8 MMAs of the two branch logits (one k-block against the resident folded-weight tiles) are left once
// the second allocation is granted.  One thread issues every MMA and commit.
// A CTA that has allocated without giving up its permit keeps the SM from launching further CTAs (measured: the second and third
// CTA of an SM entered 5 and 9.5 us after the first), so the two-step path is only taken by a CTA that finds two others
// resident - the SM is full then anyway; the first two allocate everything at once.  `resident` counts the kernel's CTAs per SM
// (a scheduling hint only, balanced by release_tmem).  No deadlock: at most three of these CTAs fit an SM, a CTA that waits holds
// 64 columns, so at least one 128-column block of the 512 is free or held by a CTA that runs to completion; every other kernel
// that uses tensor memory allocates once (profiles/r1_nb_persistent_notes.md).
__device__ __forceinline__ void mma_warp(const Smem& s, int* resident, int num_kb, int lane, uint32_t& tmem_base, uint32_t& tmem_z) {
    unsigned int smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    int ahead = 0;
    if (lane == 0) ahead = atomicAdd(&resident[smid & 255], 1);
    const bool at_once = __shfl_sync(0xffffffffu, ahead, 0) < 2;
    tc::tmem_alloc_keep_permit(s.tmem_slot, ACC_COLS);
    if (at_once) tc::tmem_alloc(s.tmem_slot + 1, Z_COLS);
    tc::fence_before_sync();
    __syncwarp();
    tc::fence_after_sync();
    tmem_base = *reinterpret_cast<volatile uint32_t*>(s.tmem_slot);
    constexpr uint32_t idesc = tc::idesc_f16(BM, BN);  // every operand of the fused decoder is fp16
    constexpr uint32_t idesc_z = tc::idesc_f16(BM, BN);
    const int s_z = num_kb % STAGES;  // ring slot of the branch k-block (the centred latents)
    if (lane == 0) {
        for (int i = 0; i < num_kb; ++i) {
            const int st = i % STAGES;
            const uint32_t ph = (i / STAGES) & 1;
            tc::mbar_wait(&s.full[st], ph);
            tc::fence_after_sync();
            const uint32_t a_base = tc::smem_u32(s.tiles + st * STAGE_BYTES);
            const uint32_t b_base = a_base + A_BYTES;
#pragma unroll
            for (int kk = 0; kk < BK / 16; ++kk)
                tc::umma_bf16(tmem_base, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(b_base + kk * 32, 16, 1024),
                              idesc, (i > 0 || kk > 0) ? 1u : 0u);
            tc::umma_commit(&s.empty[st]);
        }
    }
    __syncwarp();
    if (!at_once) {
        tc::tmem_alloc(s.tmem_slot + 1, Z_COLS);  // whole warp; blocks while two other CTAs own their full sets
        tc::fence_before_sync();
        __syncwarp();
        tc::fence_after_sync();
    }
    tmem_z = *reinterpret_cast<volatile uint32_t*>(s.tmem_slot + 1);
    if (lane == 0) {
        tc::mbar_arrive(s.tmem_ready);  // release: the epilogue warps read the slots after acquiring this barrier
        tc::mbar_wait(s.z_full, 0);
        tc::mbar_wait(&s.full[s_z], (num_kb / STAGES) & 1);
        tc::fence_after_sync();
        const uint32_t a_base = tc::smem_u32(s.tiles + s_z * STAGE_BYTES);
        const uint32_t zp_base = tc::smem_u32(s.z_tiles), zs_base = zp_base + B_BYTES;
#pragma unroll
        for (int kk = 0; kk < BK / 16; ++kk) {  // the two branch logits, complete: latents, shift and row normaliser (fp16)
            tc::umma_bf16(tmem_z, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(zp_base + kk * 32, 16, 1024), idesc_z,
                          kk > 0 ? 1u : 0u);
            tc::umma_bf16(tmem_z + BN, tc::smem_desc(a_base + kk * 32, 16, 1024), tc::smem_desc(zs_base + kk * 32, 16, 1024),
                          idesc_z, kk > 0 ? 1u : 0u);
        }
        tc::umma_commit(s.tmem_full);
    }
    __syncwarp();
}

// every warp, at the end of the kernel: once all are done, warp 1 frees both allocations and leaves the residency count
__device__ __forceinline__ void release_tmem(int warp, int lane, uint32_t tmem_base, uint32_t tmem_z, int* resident) {
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem_z, Z_COLS);
        tc::tmem_dealloc(tmem_base, ACC_COLS);
        unsigned int smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        if (lane == 0) atomicSub(&resident[smid & 255], 1);
    }
}

// row of the count tile that lane `lane` of epilogue warp e loads in its i-th gather: a warp covers GATHER_ROWS rows per load
__device__ __forceinline__ int cnt_row(int e, int lane, int i) {
    return (e + EPI_WARPS * i) * GATHER_ROWS + lane / (BN / 2);
}

// The epilogue's prologue.  Every global load is issued before anything waits on one (they overlap the MMA phase): the row
// indices first (the count gather depends on them), then the constants of the tile's genes (theta, genec rows GC_Y and GC_Z, bm),
// the tile's slice of the count table and the kernel's own loads (own_loads()), then the coalesced row gather of the tile's
// counts into cw as count codes (warp e takes rows e, e + 8, ...; lane l takes genes 2l, 2l + 1).  The constants and the table
// slice are then stored to s_gc / s_tg.  counts (CTA-uniform) false: neither the table nor the counts are read.  mm: this
// thread's cell row (clamped into the minibatch); returns its row of X.
template <int SRC, int GC_Y, int GC_Z, typename OwnLoads>
__device__ __forceinline__ int epi_prologue(const NbTcParams& p, const Smem& s, bool counts, int n0, int m0, int mm, uint32_t (&cw)[NGATHER],
                                            OwnLoads&& own_loads) {
    const int lane = threadIdx.x & 31, e = (threadIdx.x >> 5) - 2, et = threadIdx.x - 64;
    const long G = p.G;
    int ridx[NGATHER];
#pragma unroll
    for (int i = 0; i < NGATHER; ++i) {
        const int gm = m0 + cnt_row(e, lane, i);
        ridx[i] = gm < p.B ? (p.rows ? __ldg(p.rows + gm) : gm) : -1;
    }
    const int my_row = p.rows ? __ldg(p.rows + mm) : mm;
    float4 gcv = make_float4(1.0f, 1.0f, 0.0f, 0.0f);
    static_assert(BN <= EPI_THREADS, "one thread per gene of the tile stages its constants");
    if ((et < BN) & (n0 + et < p.G)) {  // one predicate, not two branches: the element sweep needs 2-4 more registers with &&
        const int g = n0 + et;
        gcv.x = __ldg(p.genec + GC_THETA * G + g);
        gcv.y = __ldg(p.genec + GC_Y * G + g);
        gcv.z = __ldg(p.genec + GC_Z * G + g);
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
    own_loads();
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
    if (et < BN) s.s_gc[et] = gcv;
#pragma unroll
    for (int u = 0; u < 2; ++u)
        if (counts) reinterpret_cast<float4*>(s.s_tg)[et + u * EPI_THREADS] = tgv[u];
    return my_row;
}

// the gathered count codes into the count tile: only once the accumulators are complete (the tile aliases the operand stages)
__device__ __forceinline__ void stage_counts(const Smem& s, const uint32_t (&cw)[NGATHER], bool counts) {
    const int lane = threadIdx.x & 31, e = (threadIdx.x >> 5) - 2;
#pragma unroll
    for (int i = 0; i < NGATHER; ++i)
        if (counts) s.s_cnt[cnt_row(e, lane, i) * CNT_PITCH_W + lane % (BN / 2)] = cw[i];
}

// ---------------------------------------------------------------------------------------------------------------- host
struct NbTcMaps { CUtensorMap a, b, z, zc; };

// the branch operands of spv_dec_fold: wz_f16 [2 Gp, 64] in BN-row boxes, zc_f16 [B, 64] in BM-row boxes (16-bit elements: the
// bf16 map type serves fp16 as well)
inline int make_branch_maps(CUtensorMap* mz, CUtensorMap* mzc, const void* wz_f16, const void* zc_f16, int Gp, int B) {
    const int rc = spv_make_tensor_map_bf16(mz, wz_f16, 64ull, (unsigned long long)(2 * Gp), 64ull, 64, BN);
    if (rc != SPV_OK) return rc;
    return spv_make_tensor_map_bf16(mzc, zc_f16, 64ull, (unsigned long long)B, 64ull, 64, BM);
}

// the dynamic shared-memory attribute of Kernel, set once per device (the attribute is per device; a process may drive several)
template <auto Kernel>
int set_smem_once(int bytes) {
    static bool done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (done[dev & 63]) return SPV_OK;
    if (cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) return SPV_ERR_LAUNCH;
    done[dev & 63] = true;
    return SPV_OK;
}

// the argument checks every sweep's entry point makes
inline bool sweep_args_ok(const void* const* ptrs, const void* amix, const void* wstack, const void* zc_f16, const void* wz_f16, int Gp,
                          int B, int G, int P, int S) {
    return ptrs && amix && wstack && zc_f16 && wz_f16 && Gp >= G && B > 0 && G > 0 && P > 0 && S > 0 &&
           P + S <= ZK_MAX_LATENT &&  // the latent columns must fit the branch k-block below the additive columns
           ptrs[5] && ptrs[6];
}

// After the checks: the four operand maps (amix [B, K] and wstack [G, K] with pitches ld_amix / ld_w, the branch operands), the
// common parameters from ptrs[], and the shared-memory attribute of each kernel the entry point may launch.
template <auto... Kernels>
int sweep_setup(NbTcParams& p, NbTcMaps& m, const void* const* ptrs, long long ldx, const void* amix, long long ld_amix, const void* wstack,
                long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, int B, int G, int K) {
    int rc = spv_make_tensor_map_bf16(&m.a, amix, (unsigned long long)K, (unsigned long long)B, (unsigned long long)ld_amix, 64, BM);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&m.b, wstack, (unsigned long long)K, (unsigned long long)G, (unsigned long long)ld_w, 64, BN);
    if (rc != SPV_OK) return rc;
    rc = make_branch_maps(&m.z, &m.zc, wz_f16, zc_f16, Gp, B);
    if (rc != SPV_OK) return rc;
    p.X = ptrs[0]; p.ldx = ldx; p.rows = (const int*)ptrs[1]; p.bm = (const float*)ptrs[5]; p.genec = (const float*)ptrs[6];
    p.tgf = (const float2*)ptrs[17];
    p.B = B; p.G = G; p.K = K; p.Gp = Gp;
    if ((... || (set_smem_once<Kernels>(SMEM_BYTES) != SPV_OK))) return SPV_ERR_LAUNCH;
    return SPV_OK;
}

}  // namespace nbtc
