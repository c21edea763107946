// bf16 tensor-core GEMM for sm_100a: TMA (cp.async.bulk.tensor, 128B swizzle) -> shared memory ring -> tcgen05.mma with the
// fp32 accumulator in TMEM -> tcgen05.ld epilogue.  One 128 x BN output tile per CTA, warp-specialised:
//   warp 0: TMA producer (one elected lane)      warp 1: TMEM allocator + MMA issuer (one elected lane)
//   warps 2-5: epilogue (TMEM -> registers -> global), warp w owns TMEM lanes 32 * (w % 4) ..
// Both operands may be K-major ([rows][K]) or MN-major ([K][rows]), so weight / activation gradients
// (dW = dY^T X, dX = dY W) run without materialising transposes.
// This is the "bf16 tensor-core path" of BASELINE.json's north_star (parity gate 1e-2); the fp32 SIMT path of
// gemm_simt.cu is the 1e-4 mode.  Replaces the cuBLAS GEMMs behind nn.Linear in reference nn/networks.py:119, 323-325.
#include <cuda_fp16.h>
#include "tc_common.cuh"
#include "../../include/spvipes_b200.h"

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle row
constexpr int THREADS = 192;

struct TcParams {
    float* C;
    const float* bias;
    float* ws;
    long ldc;
    int M, N, K, relu, accumulate, splits, kb_per_split;
    uint32_t idesc;  // instruction descriptor (operand formats are a run-time choice: bf16 or fp16 per operand)
    float alpha;     // C = alpha * (A B^T) + bias
};

// SPLIT: both operands are given as a bf16 pair (hi, lo) with x ~ hi + lo (lo = bf16(x - hi)), and the product is
// hi.hi + hi.lo + lo.hi accumulated into the same TMEM tile: ~16 mantissa bits per operand, fp32-grade results from
// the bf16 tensor-core path (the dropped lo.lo term is 2^-18 relative).  A stage then holds four tiles.
template <int BN, bool SPLIT>
struct Smem {
    static constexpr int STAGES = SPLIT ? 3 : 4;
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = (SPLIT ? 2 : 1) * (A_BYTES + B_BYTES);
    static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BN, bool A_MN, bool B_MN, bool SPLIT>
__global__ void __launch_bounds__(THREADS, 1) tc_gemm_kernel(const __grid_constant__ CUtensorMap mapA,
                                                             const __grid_constant__ CUtensorMap mapB,
                                                             const __grid_constant__ CUtensorMap mapAlo,
                                                             const __grid_constant__ CUtensorMap mapBlo, TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    using S = Smem<BN, SPLIT>;
    constexpr int STAGES = S::STAGES;
    const uint32_t raw = tc::smem_u32(smem_raw);
    const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
    uint8_t* tiles = smem_raw + pad;  // 1024-byte aligned (SWIZZLE_128B atoms)
    uint64_t* full = reinterpret_cast<uint64_t*>(tiles + STAGES * S::STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tmem_full = empty + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int split = blockIdx.z;
    const int num_kb_total = (p.K + BK - 1) / BK;
    const int kb_begin = split * p.kb_per_split;
    const int kb_end = min(num_kb_total, kb_begin + p.kb_per_split);
    const int num_kb = max(kb_end - kb_begin, 0);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&mapA);
        tc::tma_prefetch_desc(&mapB);
        if (SPLIT) {
            tc::tma_prefetch_desc(&mapAlo);
            tc::tma_prefetch_desc(&mapBlo);
        }
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(&full[s], 1);
            tc::mbar_init(&empty[s], 1);
        }
        tc::mbar_init(tmem_full, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, BN);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        if (tc::elect_one()) {
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                tc::mbar_wait(&empty[s], ph ^ 1);
                uint8_t* a_dst = tiles + s * S::STAGE_BYTES;
                uint8_t* b_dst = a_dst + S::A_BYTES;
                tc::mbar_expect_tx(&full[s], S::STAGE_BYTES);
                const int k0 = (kb_begin + i) * BK;
                if (!A_MN) {
                    tc::tma_load_2d(&mapA, &full[s], a_dst, k0, m0);  // box {64 k, 128 rows}
                } else {
#pragma unroll
                    for (int h = 0; h < BM / 64; ++h) tc::tma_load_2d(&mapA, &full[s], a_dst + h * 8192, m0 + 64 * h, k0);
                }
                if (!B_MN) {
                    tc::tma_load_2d(&mapB, &full[s], b_dst, k0, n0);  // box {64 k, BN rows}
                } else {
#pragma unroll
                    for (int h = 0; h < BN / 64; ++h) tc::tma_load_2d(&mapB, &full[s], b_dst + h * 8192, n0 + 64 * h, k0);
                }
                if (SPLIT) {  // the residual planes, same boxes
                    uint8_t* al_dst = b_dst + S::B_BYTES;
                    uint8_t* bl_dst = al_dst + S::A_BYTES;
                    if (!A_MN) {
                        tc::tma_load_2d(&mapAlo, &full[s], al_dst, k0, m0);
                    } else {
#pragma unroll
                        for (int h = 0; h < BM / 64; ++h) tc::tma_load_2d(&mapAlo, &full[s], al_dst + h * 8192, m0 + 64 * h, k0);
                    }
                    if (!B_MN) {
                        tc::tma_load_2d(&mapBlo, &full[s], bl_dst, k0, n0);
                    } else {
#pragma unroll
                        for (int h = 0; h < BN / 64; ++h) tc::tma_load_2d(&mapBlo, &full[s], bl_dst + h * 8192, n0 + 64 * h, k0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (tc::elect_one()) {
            const uint32_t idesc = p.idesc;
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                tc::mbar_wait(&full[s], ph);
                tc::fence_after_sync();
                const uint32_t a_base = tc::smem_u32(tiles + s * S::STAGE_BYTES);
                const uint32_t b_base = a_base + S::A_BYTES;
#pragma unroll
                for (int kk = 0; kk < BK / 16; ++kk) {
                    // K-major: 16 k = 32 bytes along the swizzled 128-byte row; SBO = 1024 (8-row groups)
                    // MN-major: 16 k = 16 rows of 128 bytes = 2048 bytes; LBO = 8192 (next 64-wide block), SBO = 1024
                    const uint64_t da = A_MN ? tc::smem_desc(a_base + kk * 2048, 8192, 1024) : tc::smem_desc(a_base + kk * 32, 16, 1024);
                    const uint64_t db = B_MN ? tc::smem_desc(b_base + kk * 2048, 8192, 1024) : tc::smem_desc(b_base + kk * 32, 16, 1024);
                    tc::umma_bf16(tmem_base, da, db, idesc, (i > 0 || kk > 0) ? 1u : 0u);
                    if (SPLIT) {
                        const uint32_t al_base = b_base + S::B_BYTES, bl_base = al_base + S::A_BYTES;
                        const uint64_t dal = A_MN ? tc::smem_desc(al_base + kk * 2048, 8192, 1024) : tc::smem_desc(al_base + kk * 32, 16, 1024);
                        const uint64_t dbl = B_MN ? tc::smem_desc(bl_base + kk * 2048, 8192, 1024) : tc::smem_desc(bl_base + kk * 32, 16, 1024);
                        tc::umma_bf16(tmem_base, da, dbl, idesc, 1u);
                        tc::umma_bf16(tmem_base, dal, db, idesc, 1u);
                    }
                }
                tc::umma_commit(&empty[s]);  // frees the smem stage once these MMAs have read it
            }
            tc::umma_commit(tmem_full);  // accumulator complete
        }
    } else {
        // ================= epilogue (warps 2..5) =================
        const int lane_base = (warp & 3) * 32;
        const int m = m0 + lane_base + lane;
        if (num_kb > 0) {
            tc::mbar_wait(tmem_full, 0);
            tc::fence_after_sync();
        }
        float* out;
        long ld;
        if (p.splits > 1) {
            out = p.ws + (size_t)split * p.M * p.N;
            ld = p.N;
        } else {
            out = p.C;
            ld = p.ldc;
        }
        // All TMA loads have landed and all MMAs have read them once tmem_full fires, so the operand stages are free:
        // each warp transposes its 32 x 32 chunk through a private pitch-33 staging block so that global stores are
        // one full 128-byte row segment per instruction whatever ldc is (ldc = 291 for the mixing-net gradients).
        float* stage = reinterpret_cast<float*>(tiles) + (warp - 2) * (32 * 33);
        const bool acc = p.accumulate && p.splits == 1;
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
            const int nb = n0 + c0;
            if (nb >= p.N || m0 + lane_base >= p.M) break;  // warp-uniform
            uint32_t r[32];
            if (num_kb > 0) {
                tc::tmem_ld32(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)c0, r);
                tc::tmem_ld_wait();
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) r[j] = 0u;
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) stage[lane * 33 + j] = __uint_as_float(r[j]);
            __syncwarp();
            const int n = nb + lane;
            const bool n_ok = n < p.N;
            const float bv = (p.splits == 1 && p.bias && n_ok) ? __ldg(p.bias + n) : 0.0f;
            const int rows = min(32, p.M - (m0 + lane_base));
            float* dst = out + (size_t)(m0 + lane_base) * ld + n;
            if (n_ok) {
#pragma unroll 8
                for (int rr = 0; rr < rows; ++rr) {
                    float v = fmaf(stage[rr * 33 + lane], p.splits == 1 ? p.alpha : 1.0f, bv);
                    if (p.relu && p.splits == 1) v = fmaxf(v, 0.0f);
                    if (acc) v += dst[(size_t)rr * ld];
                    dst[(size_t)rr * ld] = v;
                }
            }
            __syncwarp();
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem_base, BN);
    }
}

__global__ void tc_splitk_reduce_kernel(TcParams p) {
    long total = (long)p.M * p.N;
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        int n = (int)(i % p.N);
        long m = i / p.N;
        float v = 0.0f;
        for (int s = 0; s < p.splits; ++s) v += p.ws[(size_t)s * total + i];
        v *= p.alpha;
        float* c = p.C + m * p.ldc + n;
        if (p.accumulate == 2) v += *c;  // pre-activation addend already in C
        if (p.bias) v += p.bias[n];
        if (p.relu) v = fmaxf(v, 0.0f);
        *c = p.accumulate == 1 ? (*c + v) : v;
    }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
    static EncodeFn fn = nullptr;
    if (fn) return fn;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess || !ptr) return nullptr;
    fn = reinterpret_cast<EncodeFn>(ptr);
    return fn;
}

template <int BN, bool A_MN, bool B_MN, bool SPLIT>
int launch(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mal, const CUtensorMap& mbl, const TcParams& p,
           cudaStream_t st) {
    using S = Smem<BN, SPLIT>;
    // the attribute is per device: set it once per device this process drives
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
        if (cudaFuncSetAttribute(tc_gemm_kernel<BN, A_MN, B_MN, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL) != cudaSuccess)
            return SPV_ERR_LAUNCH;
        configured[dev & 63] = true;
    }
    dim3 grid((p.N + BN - 1) / BN, (p.M + BM - 1) / BM, p.splits);
    tc_gemm_kernel<BN, A_MN, B_MN, SPLIT><<<grid, THREADS, S::TOTAL, st>>>(ma, mb, mal, mbl, p);
    SPV_CHECK_LAUNCH();
    if (p.splits > 1) {
        long total = (long)p.M * p.N;
        int blocks = (int)min((long)148 * 8, (total + 255) / 256);
        tc_splitk_reduce_kernel<<<blocks, 256, 0, st>>>(p);
        SPV_CHECK_LAUNCH();
    }
    return SPV_OK;
}

template <int BN, bool SPLIT>
int dispatch_major(int a_mn, int b_mn, const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mal, const CUtensorMap& mbl,
                   const TcParams& p, cudaStream_t st) {
    if (!a_mn && !b_mn) return launch<BN, false, false, SPLIT>(ma, mb, mal, mbl, p, st);
    if (!a_mn && b_mn) return launch<BN, false, true, SPLIT>(ma, mb, mal, mbl, p, st);
    if (a_mn && !b_mn) return launch<BN, true, false, SPLIT>(ma, mb, mal, mbl, p, st);
    return launch<BN, true, true, SPLIT>(ma, mb, mal, mbl, p, st);
}

int tc_gemm_impl(int a_mn, int b_mn, const void* A, const void* A_lo, long long lda, const void* B, const void* B_lo, long long ldb,
                 float* C, long long ldc, int M, int N, int K, const float* bias, int relu, int accumulate, int splits, float* ws,
                 void* stream, int fmt = 0, float alpha = 1.0f) {
    if (!A || !B || !C || M <= 0 || N <= 0 || K <= 0) return SPV_ERR_ARG;
    const bool split_ops = A_lo != nullptr;
    if (split_ops != (B_lo != nullptr)) return SPV_ERR_ARG;
    if (splits < 1) splits = 1;
    const int num_kb = (K + BK - 1) / BK;
    if (splits > num_kb) splits = num_kb;
    int kb_per = (num_kb + splits - 1) / splits;
    splits = (num_kb + kb_per - 1) / kb_per;
    if (splits > 1 && !ws) return SPV_ERR_ARG;
    const int BN = N <= 64 ? 64 : 128;
    CUtensorMap ma, mb, mal, mbl;
    auto map_a = [&](CUtensorMap* m, const void* base) {
        return !a_mn ? spv_make_tensor_map_bf16(m, base, (unsigned long long)K, (unsigned long long)M, (unsigned long long)lda, 64, BM)
                     : spv_make_tensor_map_bf16(m, base, (unsigned long long)M, (unsigned long long)K, (unsigned long long)lda, 64, 64);
    };
    auto map_b = [&](CUtensorMap* m, const void* base) {
        return !b_mn ? spv_make_tensor_map_bf16(m, base, (unsigned long long)K, (unsigned long long)N, (unsigned long long)ldb, 64, BN)
                     : spv_make_tensor_map_bf16(m, base, (unsigned long long)N, (unsigned long long)K, (unsigned long long)ldb, 64, 64);
    };
    int rc = map_a(&ma, A);
    if (rc != SPV_OK) return rc;
    rc = map_b(&mb, B);
    if (rc != SPV_OK) return rc;
    if (split_ops) {
        rc = map_a(&mal, A_lo);
        if (rc != SPV_OK) return rc;
        rc = map_b(&mbl, B_lo);
        if (rc != SPV_OK) return rc;
    } else {
        mal = ma;
        mbl = mb;
    }
    TcParams p;
    p.C = C; p.bias = bias; p.ws = ws; p.ldc = ldc; p.M = M; p.N = N; p.K = K; p.relu = relu; p.accumulate = accumulate;
    p.splits = splits; p.kb_per_split = kb_per;
    p.idesc = tc::idesc_16(BM, BN, a_mn != 0, b_mn != 0, !(fmt & 1), !(fmt & 2));
    p.alpha = alpha;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (split_ops) {
        if (BN == 64) return dispatch_major<64, true>(a_mn, b_mn, ma, mb, mal, mbl, p, st);
        return dispatch_major<128, true>(a_mn, b_mn, ma, mb, mal, mbl, p, st);
    }
    if (BN == 64) return dispatch_major<64, false>(a_mn, b_mn, ma, mb, mal, mbl, p, st);
    return dispatch_major<128, false>(a_mn, b_mn, ma, mb, mal, mbl, p, st);
}

}  // namespace

int spv_make_tensor_map_bf16(CUtensorMap* map, const void* base, unsigned long long inner, unsigned long long outer,
                             unsigned long long ld_elems, unsigned box_inner, unsigned box_outer) {
    EncodeFn enc = get_encode();
    if (!enc) return SPV_ERR_LAUNCH;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld_elems & 7) || box_inner * 2 > 128 || box_outer > 256) return SPV_ERR_ARG;
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {ld_elems * 2};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? SPV_OK : SPV_ERR_ARG;
}

// C[M, N] (+)= act(A B^T + bias), bf16 operands, fp32 accumulate / output.
//   a_mn == 0: A stored [M][K] (lda elements per row);  a_mn == 1: A stored [K][M]
//   b_mn == 0: B stored [N][K];                          b_mn == 1: B stored [K][N]
extern "C" int spv_tc_gemm(int a_mn, int b_mn, const void* A, long long lda, const void* B, long long ldb, float* C,
                           long long ldc, int M, int N, int K, const float* bias, int relu, int accumulate, int splits,
                           float* ws, void* stream) {
    return tc_gemm_impl(a_mn, b_mn, A, nullptr, lda, B, nullptr, ldb, C, ldc, M, N, K, bias, relu, accumulate, splits, ws, stream);
}

// general form: fmt 0 = both operands bf16, 3 = both fp16; C = alpha * A B^T (+ bias ...)
extern "C" int spv_tc_gemm_ex(int fmt, float alpha, int a_mn, int b_mn, const void* A, long long lda, const void* B, long long ldb,
                              float* C, long long ldc, int M, int N, int K, const float* bias, int relu, int accumulate, int splits,
                              float* ws, void* stream) {
    if (fmt != 0 && fmt != 3) return SPV_ERR_ARG;  // tcgen05 kind::f16 traps on mixed bf16 / fp16 operands (measured on B200)
    return tc_gemm_impl(a_mn, b_mn, A, nullptr, lda, B, nullptr, ldb, C, ldc, M, N, K, bias, relu, accumulate, splits, ws, stream, fmt, alpha);
}

// the same with split-bf16 operands: A ~ A + A_lo, B ~ B + B_lo (same layout and pitch as their hi planes); three MMAs per
// k-step (hi.hi + hi.lo + lo.hi) into one accumulator.  Used for the K = genes contractions of the encoder's first layer
// (forward and weight gradient), where bf16 operand rounding alone would miss the 1e-3 gate on the latent statistics.
extern "C" int spv_tc_gemm_split(int a_mn, int b_mn, const void* A, const void* A_lo, long long lda, const void* B, const void* B_lo,
                                 long long ldb, float* C, long long ldc, int M, int N, int K, const float* bias, int relu,
                                 int accumulate, int splits, float* ws, void* stream) {
    if (!A_lo || !B_lo) return SPV_ERR_ARG;
    return tc_gemm_impl(a_mn, b_mn, A, A_lo, lda, B, B_lo, ldb, C, ldc, M, N, K, bias, relu, accumulate, splits, ws, stream);
}

// ---------------------------------------------------------------------------------------
// bf16 operand staging for the tensor-core path
// ---------------------------------------------------------------------------------------
// split of an fp32 value into a bf16 pair: hi = bf16(x), lo = bf16(x - hi)  (x - hi is exact in fp32)
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16(x);
    lo = __float2bfloat16(x - __bfloat162float(hi));
}

// dst[r, c] = bf16(src[r, c]) for c < C, 0 for C <= c < ld_dst  (ld_dst = C rounded up to a multiple of 8);
// dst_lo (optional, same shape): the bf16 residual of the split-operand GEMM
__global__ void to_bf16_kernel(const float* __restrict__ src, long ld_src, __nv_bfloat16* __restrict__ dst,
                               __nv_bfloat16* __restrict__ dst_lo, long ld_dst, int R, int C) {
    long total = (long)R * ld_dst;
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        int c = (int)(i % ld_dst);
        long r = i / ld_dst;
        const float x = c < C ? src[r * ld_src + c] : 0.0f;
        __nv_bfloat16 hi, lo;
        split_bf16(x, hi, lo);
        dst[i] = hi;
        if (dst_lo) dst_lo[i] = lo;
    }
}

extern "C" int spv_to_bf16(const float* src, long long ld_src, void* dst, long long ld_dst, int R, int C, void* stream) {
    if (!src || !dst || R <= 0 || C <= 0 || ld_dst < C) return SPV_ERR_ARG;
    long total = (long)R * ld_dst;
    int blocks = (int)min((long)148 * 16, (total + 255) / 256);
    to_bf16_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, ld_src, reinterpret_cast<__nv_bfloat16*>(dst), nullptr,
                                                                               ld_dst, R, C);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

__global__ void to_f16_kernel(const float* __restrict__ src, long ld_src, __half* __restrict__ dst, long ld_dst, int R, int C) {
    long total = (long)R * ld_dst;
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        int c = (int)(i % ld_dst);
        long r = i / ld_dst;
        dst[i] = to_half_sat(c < C ? src[r * ld_src + c] : 0.0f);
    }
}

// fp16 staging (decoder operands of the tensor-core path): dst[r, :C] = half(src[r, :C]), zero padded up to ld_dst
extern "C" int spv_to_f16(const float* src, long long ld_src, void* dst, long long ld_dst, int R, int C, void* stream) {
    if (!src || !dst || R <= 0 || C <= 0 || ld_dst < C) return SPV_ERR_ARG;
    long total = (long)R * ld_dst;
    int blocks = (int)min((long)148 * 16, (total + 255) / 256);
    to_f16_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, ld_src, reinterpret_cast<__half*>(dst), ld_dst, R, C);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

extern "C" int spv_to_bf16_split(const float* src, long long ld_src, void* dst_hi, void* dst_lo, long long ld_dst, int R, int C,
                                 void* stream) {
    if (!src || !dst_hi || !dst_lo || R <= 0 || C <= 0 || ld_dst < C) return SPV_ERR_ARG;
    long total = (long)R * ld_dst;
    int blocks = (int)min((long)148 * 16, (total + 255) / 256);
    to_bf16_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, ld_src, reinterpret_cast<__nv_bfloat16*>(dst_hi),
                                                                               reinterpret_cast<__nv_bfloat16*>(dst_lo), ld_dst, R, C);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// T[b, g] = bf16(log1p(X[rows[b], g]))   (the encoder's input, reference module/spVIPESmodule.py:428-433), zero padded to ld_dst,
// optionally its bf16 residual T_lo (split-operand GEMM), and optionally library[b] = log(sum_g log1p(x[b, g]))
// (reference :433-435) from the same pass over the row.
// One CTA per cell.  uint16 counts: 8 genes per 16-byte load when the row is 16-byte aligned, log1p of counts < 256 from a
// shared-memory table filled with the same log1pf (bit-identical to computing it in place); the table also holds the packed
// (hi | lo << 16) bf16 pair of each entry.
#define ENC_IN_THREADS 256
__device__ __forceinline__ unsigned int pack_split(float f) {
    __nv_bfloat16 hi, lo;
    split_bf16(f, hi, lo);
    return (unsigned int)__bfloat16_as_ushort(hi) | ((unsigned int)__bfloat16_as_ushort(lo) << 16);
}
template <int SRC>
__global__ void __launch_bounds__(ENC_IN_THREADS) counts_to_bf16_kernel(const void* __restrict__ X, long ldx, const int* __restrict__ rows,
                                                                        __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dst_lo,
                                                                        long ld_dst, int B, int G, float* __restrict__ lib,
                                                                        const int* __restrict__ cov, int n_cov) {
    __shared__ float lut[256];
    __shared__ unsigned int lutp[256];
    __shared__ float red[ENC_IN_THREADS / 32];
    const int b = blockIdx.x;
    const long r = rows ? (long)rows[b] : (long)b;
    __nv_bfloat16* out = dst + (long)b * ld_dst;
    __nv_bfloat16* out_lo = dst_lo ? dst_lo + (long)b * ld_dst : nullptr;
    float sum = 0.0f;
    if (SRC == SPV_SRC_U16_LOG1P) {
        lut[threadIdx.x] = threadIdx.x == 0 ? 0.0f : log1pf((float)threadIdx.x);
        lutp[threadIdx.x] = pack_split(lut[threadIdx.x]);
        __syncthreads();
        const unsigned short* row = reinterpret_cast<const unsigned short*>(X) + r * ldx;
        const bool vec = (reinterpret_cast<uintptr_t>(row) & 15) == 0;  // dst rows are 16-byte aligned (ld_dst % 8 == 0)
        const int nvec = vec ? G / 8 : 0;
        for (int v = threadIdx.x; v < nvec; v += ENC_IN_THREADS) {
            uint4 raw = __ldg(reinterpret_cast<const uint4*>(row) + v);
            unsigned int w[4] = {raw.x, raw.y, raw.z, raw.w};
            uint4 o, ol;
            unsigned int* ow = &o.x;
            unsigned int* olw = &ol.x;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                unsigned int c0 = w[j] & 0xffffu, c1 = w[j] >> 16;
                float f0, f1;
                unsigned int e0, e1;
                if (c0 < 256u) { f0 = lut[c0]; e0 = lutp[c0]; } else { f0 = log1pf((float)c0); e0 = pack_split(f0); }
                if (c1 < 256u) { f1 = lut[c1]; e1 = lutp[c1]; } else { f1 = log1pf((float)c1); e1 = pack_split(f1); }
                sum += f0;
                sum += f1;
                ow[j] = __byte_perm(e0, e1, 0x5410);
                olw[j] = __byte_perm(e0, e1, 0x7632);
            }
            *(reinterpret_cast<uint4*>(out) + v) = o;
            if (out_lo) *(reinterpret_cast<uint4*>(out_lo) + v) = ol;
        }
        const int my_cov = cov ? __ldg(cov + b) : -1;  // columns G .. G + n_cov: one-hot batch code (not part of the library size)
        for (int g = nvec * 8 + threadIdx.x; g < ld_dst; g += ENC_IN_THREADS) {
            float f = 0.0f;
            if (g < G) {
                unsigned int c = row[g];
                f = c < 256u ? lut[c] : log1pf((float)c);
                sum += f;
            } else if (g - G < n_cov) {
                f = (g - G == my_cov) ? 1.0f : 0.0f;
            }
            __nv_bfloat16 hi, lo;
            split_bf16(f, hi, lo);
            out[g] = hi;
            if (out_lo) out_lo[g] = lo;
        }
    } else {
        const int my_cov = cov ? __ldg(cov + b) : -1;
        for (int g = threadIdx.x; g < ld_dst; g += ENC_IN_THREADS) {
            float f = 0.0f;
            if (g < G) {
                f = load_src<SRC>(X, r * ldx + g);
                sum += f;
            } else if (g - G < n_cov) {
                f = (g - G == my_cov) ? 1.0f : 0.0f;
            }
            __nv_bfloat16 hi, lo;
            split_bf16(f, hi, lo);
            out[g] = hi;
            if (out_lo) out_lo[g] = lo;
        }
    }
    if (!lib) return;
    sum = warp_sum(sum);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < ENC_IN_THREADS / 32; ++i) s += red[i];
        lib[b] = logf(s);
    }
}

extern "C" int spv_counts_to_bf16(int src, const void* X, long long ldx, const int* rows, void* dst, void* dst_lo, long long ld_dst,
                                  int B, int G, float* lib, const int* cov, int n_cov, void* stream) {
    if (!X || !dst || B <= 0 || G <= 0 || n_cov < 0 || ld_dst < G + n_cov || (ld_dst & 7) || (n_cov > 0 && !cov)) return SPV_ERR_ARG;
    if (n_cov == 0) cov = nullptr;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(dst);
    __nv_bfloat16* dl = reinterpret_cast<__nv_bfloat16*>(dst_lo);
    if (src == SPV_SRC_U16_LOG1P) counts_to_bf16_kernel<SPV_SRC_U16_LOG1P><<<B, ENC_IN_THREADS, 0, st>>>(X, ldx, rows, d, dl, ld_dst, B, G, lib, cov, n_cov);
    else if (src == SPV_SRC_F32_LOG1P) counts_to_bf16_kernel<SPV_SRC_F32_LOG1P><<<B, ENC_IN_THREADS, 0, st>>>(X, ldx, rows, d, dl, ld_dst, B, G, lib, cov, n_cov);
    else return SPV_ERR_ARG;
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

// Minibatch gather from a device-resident CSR count matrix (int64 row offsets, uint16 column indices) into a dense staging
// tile xs [B, ld_xs] that every count consumer then reads with rows = NULL.  One CTA per minibatch row: zero a row in dynamic
// shared memory, scatter the row's nonzeros into it (coalesced loads of indices / values), then write it out with 16-byte
// stores.  With dst != NULL the same CTA also does what counts_to_bf16_kernel does for a 16-byte aligned dense row (split-bf16
// pair, covariate columns, library size), with the same per-thread gene assignment, tables and reduction order: its outputs
// are bit-identical to spv_counts_to_bf16 on the gathered rows.  The CSR must be canonical (no duplicate column in a row).
#define CSR_SMEM_OPTIN (227 * 1024)  // largest dynamic + static shared memory of one CTA on sm_100
#define CSR_MAX_G_U16 65536          // range of the uint16 column index; the row takes 128 KB
#define CSR_MAX_G_F32 ((CSR_SMEM_OPTIN - (int)(ENC_IN_THREADS / 32 * sizeof(float))) / 4 / 4 * 4)  // static: the reduction slots
template <int SRC>
__global__ void __launch_bounds__(ENC_IN_THREADS) csr_gather_kernel(const long long* __restrict__ indptr,
                                                                    const unsigned short* __restrict__ indices,
                                                                    const void* __restrict__ values, const int* __restrict__ rows,
                                                                    int G, void* __restrict__ xs, long ld_xs,
                                                                    __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dst_lo,
                                                                    long ld_dst, float* __restrict__ lib, const int* __restrict__ cov,
                                                                    int n_cov) {
    constexpr bool U16 = SRC == SPV_SRC_U16_LOG1P;
    constexpr int PER_VEC = U16 ? 8 : 4;  // elements per 16-byte word
    extern __shared__ uint4 csr_row4[];
    __shared__ float red[ENC_IN_THREADS / 32];
    __shared__ float lut[256];          // uint16 instantiation only
    __shared__ unsigned int lutp[256];
    const int b = blockIdx.x;
    const long long r = rows ? (long long)rows[b] : (long long)b;
    const int nrow4 = (G + PER_VEC - 1) / PER_VEC;  // the row rounded up to whole 16-byte words; ld_xs covers it
    for (int v = threadIdx.x; v < nrow4; v += ENC_IN_THREADS) csr_row4[v] = make_uint4(0u, 0u, 0u, 0u);
    if constexpr (U16) {
        if (dst) {
            lut[threadIdx.x] = threadIdx.x == 0 ? 0.0f : log1pf((float)threadIdx.x);
            lutp[threadIdx.x] = pack_split(lut[threadIdx.x]);
        }
    }
    __syncthreads();
    const long long p0 = __ldg(indptr + r), p1 = __ldg(indptr + r + 1);
    if constexpr (U16) {
        unsigned short* srow = reinterpret_cast<unsigned short*>(csr_row4);
        const unsigned short* val = reinterpret_cast<const unsigned short*>(values);
        for (long long k = p0 + threadIdx.x; k < p1; k += ENC_IN_THREADS) srow[__ldg(indices + k)] = __ldg(val + k);
    } else {
        float* srow = reinterpret_cast<float*>(csr_row4);
        const float* val = reinterpret_cast<const float*>(values);
        for (long long k = p0 + threadIdx.x; k < p1; k += ENC_IN_THREADS) srow[__ldg(indices + k)] = __ldg(val + k);
    }
    __syncthreads();
    uint4* xrow4 = reinterpret_cast<uint4*>(reinterpret_cast<char*>(xs) + (long)b * ld_xs * (U16 ? 2 : 4));
    if (!dst) {
        for (int v = threadIdx.x; v < nrow4; v += ENC_IN_THREADS) xrow4[v] = csr_row4[v];
        return;
    }
    __nv_bfloat16* out = dst + (long)b * ld_dst;
    __nv_bfloat16* out_lo = dst_lo ? dst_lo + (long)b * ld_dst : nullptr;
    const int my_cov = cov ? __ldg(cov + b) : -1;
    float sum = 0.0f;
    if constexpr (U16) {
        // counts_to_bf16_kernel's vectorised path, the row read from shared memory
        const unsigned short* srow = reinterpret_cast<const unsigned short*>(csr_row4);
        const int nvec = G / 8;
        for (int v = threadIdx.x; v < nvec; v += ENC_IN_THREADS) {
            uint4 raw = csr_row4[v];
            xrow4[v] = raw;
            unsigned int w[4] = {raw.x, raw.y, raw.z, raw.w};
            uint4 o, ol;
            unsigned int* ow = &o.x;
            unsigned int* olw = &ol.x;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                unsigned int c0 = w[j] & 0xffffu, c1 = w[j] >> 16;
                float f0, f1;
                unsigned int e0, e1;
                if (c0 < 256u) { f0 = lut[c0]; e0 = lutp[c0]; } else { f0 = log1pf((float)c0); e0 = pack_split(f0); }
                if (c1 < 256u) { f1 = lut[c1]; e1 = lutp[c1]; } else { f1 = log1pf((float)c1); e1 = pack_split(f1); }
                sum += f0;
                sum += f1;
                ow[j] = __byte_perm(e0, e1, 0x5410);
                olw[j] = __byte_perm(e0, e1, 0x7632);
            }
            *(reinterpret_cast<uint4*>(out) + v) = o;
            if (out_lo) *(reinterpret_cast<uint4*>(out_lo) + v) = ol;
        }
        if (nvec < nrow4 && threadIdx.x == ENC_IN_THREADS - 1) xrow4[nvec] = csr_row4[nvec];  // last partial word (zero padded)
        for (int g = nvec * 8 + threadIdx.x; g < ld_dst; g += ENC_IN_THREADS) {
            float f = 0.0f;
            if (g < G) {
                unsigned int c = srow[g];
                f = c < 256u ? lut[c] : log1pf((float)c);
                sum += f;
            } else if (g - G < n_cov) {
                f = (g - G == my_cov) ? 1.0f : 0.0f;
            }
            __nv_bfloat16 hi, lo;
            split_bf16(f, hi, lo);
            out[g] = hi;
            if (out_lo) out_lo[g] = lo;
        }
    } else {
        // counts_to_bf16_kernel's scalar float path (load_src<SPV_SRC_F32_LOG1P>)
        for (int v = threadIdx.x; v < nrow4; v += ENC_IN_THREADS) xrow4[v] = csr_row4[v];
        const float* srow = reinterpret_cast<const float*>(csr_row4);
        for (int g = threadIdx.x; g < ld_dst; g += ENC_IN_THREADS) {
            float f = 0.0f;
            if (g < G) {
                const float c = srow[g];
                f = c == 0.0f ? 0.0f : logf(1.0f + c);
                sum += f;
            } else if (g - G < n_cov) {
                f = (g - G == my_cov) ? 1.0f : 0.0f;
            }
            __nv_bfloat16 hi, lo;
            split_bf16(f, hi, lo);
            out[g] = hi;
            if (out_lo) out_lo[g] = lo;
        }
    }
    if (!lib) return;
    sum = warp_sum(sum);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < ENC_IN_THREADS / 32; ++i) s += red[i];
        lib[b] = logf(s);
    }
}

extern "C" int spv_csr_max_genes(int src) {
    if (src == SPV_SRC_U16_LOG1P) return CSR_MAX_G_U16;
    if (src == SPV_SRC_F32_LOG1P) return CSR_MAX_G_F32;
    return SPV_ERR_ARG;
}

extern "C" int spv_csr_gather(int src, const long long* indptr, const unsigned short* indices, const void* values, const int* rows,
                              int B, int G, void* xs, long long ld_xs, void* dst, void* dst_lo, long long ld_dst, float* lib,
                              const int* cov, int n_cov, void* stream) {
    const int max_g = spv_csr_max_genes(src);
    if (max_g < 0 || !indptr || !indices || !values || !xs || B <= 0 || G <= 0 || G > max_g || n_cov < 0) return SPV_ERR_ARG;
    const int per_vec = src == SPV_SRC_U16_LOG1P ? 8 : 4;
    if (ld_xs < G || (ld_xs % per_vec) || (reinterpret_cast<uintptr_t>(xs) & 15)) return SPV_ERR_ARG;
    if (dst && (ld_dst < G + n_cov || (ld_dst & 7) || (reinterpret_cast<uintptr_t>(dst) & 15) ||
                (dst_lo && (reinterpret_cast<uintptr_t>(dst_lo) & 15))))
        return SPV_ERR_ARG;
    if (n_cov > 0 && !cov) return SPV_ERR_ARG;
    if (n_cov == 0) cov = nullptr;
    static bool done_u16[64] = {}, done_f32[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    bool& done = (src == SPV_SRC_U16_LOG1P ? done_u16 : done_f32)[dev & 63];
    if (!done) {
        cudaError_t e = src == SPV_SRC_U16_LOG1P
            ? cudaFuncSetAttribute(csr_gather_kernel<SPV_SRC_U16_LOG1P>, cudaFuncAttributeMaxDynamicSharedMemorySize, CSR_MAX_G_U16 * 2)
            : cudaFuncSetAttribute(csr_gather_kernel<SPV_SRC_F32_LOG1P>, cudaFuncAttributeMaxDynamicSharedMemorySize, CSR_MAX_G_F32 * 4);
        if (e != cudaSuccess) return SPV_ERR_LAUNCH;
        done = true;
    }
    const size_t smem = (size_t)((G + per_vec - 1) / per_vec) * 16;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(dst);
    __nv_bfloat16* dl = dst ? reinterpret_cast<__nv_bfloat16*>(dst_lo) : nullptr;
    float* lb = dst ? lib : nullptr;
    if (src == SPV_SRC_U16_LOG1P)
        csr_gather_kernel<SPV_SRC_U16_LOG1P><<<B, ENC_IN_THREADS, smem, st>>>(indptr, indices, values, rows, G, xs, ld_xs, d, dl, ld_dst, lb, cov, n_cov);
    else
        csr_gather_kernel<SPV_SRC_F32_LOG1P><<<B, ENC_IN_THREADS, smem, st>>>(indptr, indices, values, rows, G, xs, ld_xs, d, dl, ld_dst, lb, cov, n_cov);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}
