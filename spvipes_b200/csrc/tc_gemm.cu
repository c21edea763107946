// bf16 tensor-core GEMM for sm_100a: TMA (cp.async.bulk.tensor, 128B swizzle) -> shared memory ring -> tcgen05.mma with the
// fp32 accumulator in TMEM -> tcgen05.ld epilogue.  One 128 x BN output tile per CTA, warp-specialised:
//   warp 0: TMA producer (one elected lane)      warp 1: TMEM allocator + MMA issuer (one elected lane)
//   warps 2-5: epilogue (TMEM -> registers -> global), warp w owns TMEM lanes 32 * (w % 4) ..
// Both operands may be K-major ([rows][K]) or MN-major ([K][rows]), so weight / activation gradients
// (dW = dY^T X, dX = dY W) run without materialising transposes.
// This is the "bf16 tensor-core path" of BASELINE.json's north_star (parity gate 1e-2); the fp32 SIMT path of
// gemm_simt.cu is the 1e-4 mode.  Replaces the cuBLAS GEMMs behind nn.Linear in reference nn/networks.py:119, 323-325.
#include <cstdlib>
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

// column block: dst[r, c] = bf16(src[r, c]) for c < C, 0 for C <= c < width; columns beyond `width` of dst are left untouched
__global__ void to_bf16_block_kernel(const float* __restrict__ src, long ld_src, __nv_bfloat16* __restrict__ dst, long ld_dst, int R,
                                     int C, int width) {
    long total = (long)R * width;
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        int c = (int)(i % width);
        long r = i / width;
        dst[r * ld_dst + c] = __float2bfloat16(c < C ? src[r * ld_src + c] : 0.0f);
    }
}

extern "C" int spv_to_bf16_block(const float* src, long long ld_src, void* dst, long long ld_dst, int R, int C, int width,
                                 void* stream) {
    if (!src || !dst || R <= 0 || C <= 0 || width < C || ld_dst < width) return SPV_ERR_ARG;
    long total = (long)R * width;
    int blocks = (int)min((long)148 * 16, (total + 255) / 256);
    to_bf16_block_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, ld_src, reinterpret_cast<__nv_bfloat16*>(dst),
                                                                                     ld_dst, R, C, width);
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

// =======================================================================================================================
// Encoder first layer with the count transform fused into the GEMM's operand path (BASELINE.json north_star: "a tcgen05/TMEM GEMM
// fed by TMA that consumes raw counts and fuses log1p into its prologue"; reference module/spVIPESmodule.py:428-433 +
// nn/networks.py:119 and the weight gradient of that layer).
//
//   forward (DW = false):  C[b, n] = act( sum_g log1p(X[rows[b], g]) W1[n, g] + C_pre + bias )     A produced, B by TMA
//   gradient (DW = true):  C[m, g] = sum_b dh1[b, m] log1p(X[rows[b], g])                          A by TMA, B produced
//
// The produced operand tile is the same in both: rows = cells, 128 bytes = 64 genes per row and swizzle atom.  Eight producer
// warps gather the uint16 counts of the tile straight from the device-resident matrix (row indices = the minibatch), look
// log1p up in a shared-memory table that holds the split-bf16 pair (hi | lo << 16) of every count < 256, and write the hi and
// lo planes in the 128-byte-swizzled layout the UMMA descriptors expect; fence.proxy.async + an mbarrier hand the stage to the
// MMA warp, which issues hi.hi + hi.lo + lo.hi into one TMEM accumulator.  The other operand (W1 resp. dh1, as bf16 pairs)
// arrives by TMA.  Nothing [B, G]-sized is written: the bf16 copy of log1p(counts) that the separate staging pass produced
// (2 x 2 bytes per element written, read again by both GEMMs) is gone.  After the k-loop the producer warps turn into the
// epilogue (TMEM -> registers -> global).
// =======================================================================================================================
namespace fc1 {

constexpr int BM = 128, BN = 128, BK = 64, STAGES = 3;
constexpr int PROD_WARPS = 8, THREADS = 64 + 32 * PROD_WARPS;
constexpr int TILE = 128 * 64 * 2;                 // one 16 KB plane of either operand
constexpr int STAGE_BYTES = 4 * TILE;              // [A hi | A lo | B hi | B lo]
constexpr int ROWS_CACHE = 4096;                   // minibatch row indices staged in shared memory (gradient kernel)
constexpr int SMEM = STAGES * STAGE_BYTES + 1024 + 256 * 4 + 256 + ROWS_CACHE * 4;

__device__ __forceinline__ int s_rows_or_global(const int* __restrict__ rows, const int* s_rows, int cell, int n_cached) {
    return cell < n_cached ? s_rows[cell] : __ldg(rows + cell);
}

struct Params {
    const unsigned short* X; long ldx; const int* rows;   // counts, row gather
    float* C; long ldc;
    const float* bias; float* ws;
    int M, N, K;            // GEMM extents: forward M = cells, N = 2H, K = genes; gradient M = 2H, N = genes, K = cells
    int relu, pre_acc, splits, kb_per_split;
};

__device__ __forceinline__ unsigned int pack_split_dev(float f) {
    __nv_bfloat16 hi = __float2bfloat16(f);
    __nv_bfloat16 lo = __float2bfloat16(f - __bfloat162float(hi));
    return (unsigned int)__bfloat16_as_ushort(hi) | ((unsigned int)__bfloat16_as_ushort(lo) << 16);
}

// table miss (count >= 256): rare, kept out of line so that the producer loop stays small (inlined 32 x per k-block the libm
// log1pf bloated the kernel to 700 KB of code and the loop ran out of the instruction cache: 3.5 us per k-block instead of 0.5)
__device__ __noinline__ unsigned int lut_miss(unsigned int c) { return pack_split_dev(log1pf((float)c)); }
__device__ __noinline__ unsigned int lut_any(const unsigned int* lutp, unsigned int c) { return c < 256u ? lutp[c] : lut_miss(c); }

template <bool DW>
__global__ void __launch_bounds__(THREADS, 1) fc1_kernel(const __grid_constant__ CUtensorMap mapT, const __grid_constant__ CUtensorMap mapTlo,
                                                         Params p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = tc::smem_u32(smem_raw);
    uint8_t* tiles = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
    unsigned int* lutp = reinterpret_cast<unsigned int*>(tiles + STAGES * STAGE_BYTES);
    uint64_t* full_t = reinterpret_cast<uint64_t*>(lutp + 256);  // TMA operand landed
    uint64_t* full_p = full_t + STAGES;                           // produced operand written (one arrival per producer warp)
    uint64_t* empty = full_p + STAGES;
    uint64_t* tmem_full = empty + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
    int* s_rows = reinterpret_cast<int*>(tiles + STAGES * STAGE_BYTES + 256 * 4 + 256);
    const int s_rows_n = (DW && p.rows) ? min(p.K, ROWS_CACHE) : 0;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM, split = blockIdx.z;
    const int num_kb_total = (p.K + BK - 1) / BK;
    const int kb_begin = split * p.kb_per_split;
    const int num_kb = max(min(num_kb_total, kb_begin + p.kb_per_split) - kb_begin, 0);
    for (int i = threadIdx.x; i < s_rows_n; i += THREADS) s_rows[i] = __ldg(p.rows + i);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&mapT);
        tc::tma_prefetch_desc(&mapTlo);
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(&full_t[s], 1);
            tc::mbar_init(&full_p[s], PROD_WARPS);
            tc::mbar_init(&empty[s], 1);
        }
        tc::mbar_init(tmem_full, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, BN);
    if (warp >= 2) {  // the count table: split-bf16 pair of log1p(c), c < 256
        const int t = threadIdx.x - 64;
        lutp[t] = pack_split_dev(t == 0 ? 0.0f : log1pf((float)t));
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    // stage layout: the TMA operand's two planes first when it is A (gradient), last when it is B (forward)
    constexpr int OFF_PROD = DW ? 2 * TILE : 0, OFF_TMA = DW ? 0 : 2 * TILE;

    if (warp == 0) {
        if (tc::elect_one()) {
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % STAGES;
                tc::mbar_wait(&empty[s], ((i / STAGES) & 1) ^ 1);
                uint8_t* dst = tiles + s * STAGE_BYTES + OFF_TMA;
                tc::mbar_expect_tx(&full_t[s], 2 * TILE);
                const int k0 = (kb_begin + i) * BK;
                if (!DW) {  // W1 [n rows][k]: box {64 k, 128 rows}
                    tc::tma_load_2d(&mapT, &full_t[s], dst, k0, n0);
                    tc::tma_load_2d(&mapTlo, &full_t[s], dst + TILE, k0, n0);
                } else {    // dh1 [k rows][m]: two boxes {64 m, 64 k} per plane
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        tc::tma_load_2d(&mapT, &full_t[s], dst + h * 8192, m0 + 64 * h, k0);
                        tc::tma_load_2d(&mapTlo, &full_t[s], dst + TILE + h * 8192, m0 + 64 * h, k0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::idesc_bf16(BM, BN, DW, DW);
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                tc::mbar_wait(&full_t[s], ph);
                tc::mbar_wait(&full_p[s], ph);
                tc::fence_after_sync();
                const uint32_t st = tc::smem_u32(tiles + s * STAGE_BYTES);
                const uint32_t a_hi = st, a_lo = st + TILE, b_hi = st + 2 * TILE, b_lo = st + 3 * TILE;
#pragma unroll
                for (int kk = 0; kk < BK / 16; ++kk) {
                    // K-major (forward): 16 k = 32 bytes along the swizzled row; MN-major (gradient): 16 k = 16 rows = 2048 bytes
                    const uint32_t off = DW ? kk * 2048 : kk * 32;
                    const uint32_t lbo = DW ? 8192 : 16;
                    const uint64_t dah = tc::smem_desc(a_hi + off, lbo, 1024), dal = tc::smem_desc(a_lo + off, lbo, 1024);
                    const uint64_t dbh = tc::smem_desc(b_hi + off, lbo, 1024), dbl = tc::smem_desc(b_lo + off, lbo, 1024);
                    tc::umma_bf16(tmem_base, dah, dbh, idesc, (i > 0 || kk > 0) ? 1u : 0u);
                    tc::umma_bf16(tmem_base, dah, dbl, idesc, 1u);
                    tc::umma_bf16(tmem_base, dal, dbh, idesc, 1u);
                }
                tc::umma_commit(&empty[s]);
            }
            tc::umma_commit(tmem_full);
        }
    } else {
        // ================= producers (then epilogue): 8 warps =================
        const int t = threadIdx.x - 64;
        // forward: 128 cell rows x 64 genes, thread = (row, 32-gene half); gradient: 64 cell rows x 128 genes, thread = (row, quarter)
        const int r = DW ? (t >> 2) : (t >> 1);
        const int part = DW ? (t & 3) : (t & 1);           // 32 genes = 4 chunks of 8
        const int half = DW ? (part >> 1) : 0;             // 64-gene swizzle atom inside the 128-gene tile (gradient)
        const int chunk0 = DW ? (part & 1) * 4 : part * 4;  // first 16-byte chunk inside the atom's 128-byte row
        uint8_t* const prod_row = tiles + OFF_PROD + half * 8192 + r * 128;
        const int ncell = DW ? p.K : p.M, ngene = DW ? p.N : p.K;
        // forward: this thread's cell is fixed, its row pointer is resolved once
        const unsigned short* fwd_row = nullptr;
        if (!DW && m0 + r < ncell) fwd_row = p.X + (p.rows ? (long)__ldg(p.rows + m0 + r) : (long)(m0 + r)) * p.ldx;
        // The gather is latency bound (one scattered 64-byte read per thread and k-block, ~1.5 us from HBM, after the row-index
        // lookup in the gradient kernel): the raw counts of the next PF k-blocks are kept in flight in registers.
        constexpr int PF = 4;
        uint4 buf[PF][4];
        auto issue = [&](int i, uint4 (&dst)[4]) {
            const int kb = kb_begin + i;
            const int cell = DW ? kb * BK + r : m0 + r;
            const int gene0 = DW ? n0 + part * 32 : kb * BK + part * 32;
            const unsigned short* src = nullptr;
            if (DW) {
                if (cell < ncell) src = p.X + (p.rows ? (long)s_rows_or_global(p.rows, s_rows, cell, s_rows_n) : (long)cell) * p.ldx + gene0;
            } else if (fwd_row) {
                src = fwd_row + gene0;
            }
            if (!src || gene0 >= ngene) {
#pragma unroll
                for (int j = 0; j < 4; ++j) dst[j] = make_uint4(0u, 0u, 0u, 0u);
                return;
            }
            if (((reinterpret_cast<uintptr_t>(src) & 15) == 0) && gene0 + 32 <= ngene) {
#pragma unroll
                for (int j = 0; j < 4; ++j) dst[j] = __ldg(reinterpret_cast<const uint4*>(src) + j);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    unsigned int w[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int g = gene0 + j * 8 + q * 2;
                        const unsigned int c0 = g < ngene ? __ldg(src + j * 8 + q * 2) : 0u;
                        const unsigned int c1 = g + 1 < ngene ? __ldg(src + j * 8 + q * 2 + 1) : 0u;
                        w[q] = c0 | (c1 << 16);
                    }
                    dst[j] = make_uint4(w[0], w[1], w[2], w[3]);
                }
            }
        };
#pragma unroll
        for (int u = 0; u < PF; ++u)
            if (u < num_kb) issue(u, buf[u]);
        for (int i0 = 0; i0 < num_kb; i0 += PF) {
#pragma unroll
            for (int u = 0; u < PF; ++u) {
                const int i = i0 + u;
                if (i < num_kb) {
                    const int s = i % STAGES;
                    tc::mbar_wait(&empty[s], ((i / STAGES) & 1) ^ 1);
                    uint8_t* row_hi = prod_row + s * STAGE_BYTES;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const unsigned int w[4] = {buf[u][j].x, buf[u][j].y, buf[u][j].z, buf[u][j].w};
                        unsigned int e[8];
                        // one table-miss test per 16-byte chunk (any count >= 256 in its 8 genes): the common path is eight
                        // independent shared-memory lookups with no branch between them
                        if ((((w[0] | w[1]) | (w[2] | w[3])) & 0xff00ff00u) == 0u) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                e[2 * q] = lutp[w[q] & 0xffu];
                                e[2 * q + 1] = lutp[w[q] >> 16];
                            }
                        } else {
#pragma unroll  // (unrolled: a dynamically indexed e[] would live in local memory, on the common path too)
                            for (int q = 0; q < 4; ++q) {
                                const unsigned int c0 = w[q] & 0xffffu, c1 = w[q] >> 16;
                                e[2 * q] = lut_any(lutp, c0);
                                e[2 * q + 1] = lut_any(lutp, c1);
                            }
                        }
                        unsigned int hi[4], lo[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            hi[q] = __byte_perm(e[2 * q], e[2 * q + 1], 0x5410);
                            lo[q] = __byte_perm(e[2 * q], e[2 * q + 1], 0x7632);
                        }
                        const int sw = ((chunk0 + j) ^ (r & 7)) << 4;  // 128-byte swizzle: 16-byte chunk index XOR (row mod 8)
                        *reinterpret_cast<uint4*>(row_hi + sw) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<uint4*>(row_hi + TILE + sw) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    }
                    tc::fence_proxy_async();  // generic-proxy stores -> visible to the tensor core's async proxy
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&full_p[s]);
                    if (i + PF < num_kb) issue(i + PF, buf[u]);
                }
            }
        }
        // ---- epilogue: warp (w & 3) owns TMEM lanes 32 (w & 3) .., the two warps of a quarter split the 128 columns
        if (num_kb > 0) {
            tc::mbar_wait(tmem_full, 0);
            tc::fence_after_sync();
        }
        const int q = warp & 3, chalf = (warp - 2) >> 2;
        const int m = m0 + q * 32 + lane;
        float* out = p.splits > 1 ? p.ws + (size_t)split * p.M * p.N : p.C;
        const long ld = p.splits > 1 ? p.N : p.ldc;
        const bool fin = p.splits == 1;
#pragma unroll 1
        for (int c0 = chalf * 64; c0 < chalf * 64 + 64; c0 += 32) {
            if (n0 + c0 >= p.N) break;
            uint32_t v[32];
            if (num_kb > 0) {
                tc::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
                tc::tmem_ld_wait();
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = 0u;
            }
            if (m < p.M) {
                float* dst = out + (size_t)m * ld + n0 + c0;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int n = n0 + c0 + j;
                    if (n < p.N) {
                        float x = __uint_as_float(v[j]);
                        if (fin) {
                            if (p.pre_acc) x += dst[j];
                            if (p.bias) x += __ldg(p.bias + n);
                            if (p.relu) x = fmaxf(x, 0.0f);
                        }
                        dst[j] = x;
                    }
                }
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem_base, BN);
    }
}

template <bool DW>
int launch_fc1(const CUtensorMap& mt, const CUtensorMap& mtl, const Params& p, cudaStream_t st) {
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
        if (cudaFuncSetAttribute(fc1_kernel<DW>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM) != cudaSuccess) return SPV_ERR_LAUNCH;
        configured[dev & 63] = true;
    }
    dim3 grid((p.N + BN - 1) / BN, (p.M + BM - 1) / BM, p.splits);
    fc1_kernel<DW><<<grid, THREADS, SMEM, st>>>(mt, mtl, p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

}  // namespace fc1

int fc1t_launch(const CUtensorMap& mw, const CUtensorMap& mwl, const fc1::Params& p, cudaStream_t st);  // TMEM-A version, below

// h1[B, N] = act(log1p(X[rows, :G]) W^T (+ h1 as a pre-activation addend) + bias): uint16 counts, W given as a bf16 pair
// (W_hi, W_lo [N, ldw], spv_to_bf16_split / spv_adam staging).  splits > 1: split over the genes, partials in ws [splits, B, N],
// reduced by a second launch (bias / ReLU / addend applied there).
extern "C" int spv_enc_fc1_fwd(const void* X, long long ldx, const int* rows, const void* W_hi, const void* W_lo, long long ldw,
                               float* h1, long long ld_h1, int B, int N, int G, const float* bias, int relu, int pre_acc, int splits,
                               float* ws, void* stream) {
    if (!X || !W_hi || !W_lo || !h1 || B <= 0 || N <= 0 || G <= 0) return SPV_ERR_ARG;
    if (splits < 1) splits = 1;
    const int num_kb = (G + 63) / 64;
    if (splits > num_kb) splits = num_kb;
    const int kb_per = (num_kb + splits - 1) / splits;
    splits = (num_kb + kb_per - 1) / kb_per;
    if (splits > 1 && !ws) return SPV_ERR_ARG;
    CUtensorMap mt, mtl;
    int rc = spv_make_tensor_map_bf16(&mt, W_hi, (unsigned long long)G, (unsigned long long)N, (unsigned long long)ldw, 64, fc1::BN);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mtl, W_lo, (unsigned long long)G, (unsigned long long)N, (unsigned long long)ldw, 64, fc1::BN);
    if (rc != SPV_OK) return rc;
    fc1::Params p;
    p.X = reinterpret_cast<const unsigned short*>(X); p.ldx = ldx; p.rows = rows; p.C = h1; p.ldc = ld_h1; p.bias = bias; p.ws = ws;
    p.M = B; p.N = N; p.K = G; p.relu = relu; p.pre_acc = pre_acc; p.splits = splits; p.kb_per_split = kb_per;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    static const bool smem_version = getenv("SPV_FC1_SMEM") != nullptr;  // A/B switch: producers write shared-memory tiles
    rc = smem_version ? fc1::launch_fc1<false>(mt, mtl, p, st) : fc1t_launch(mt, mtl, p, st);
    if (rc != SPV_OK) return rc;
    if (splits > 1) {
        TcParams r;
        r.C = h1; r.bias = bias; r.ws = ws; r.ldc = ld_h1; r.M = B; r.N = N; r.K = G; r.relu = relu; r.accumulate = pre_acc ? 2 : 0;
        r.splits = splits; r.kb_per_split = kb_per; r.idesc = 0; r.alpha = 1.0f;
        const long total = (long)B * N;
        tc_splitk_reduce_kernel<<<(int)min((long)148 * 8, (total + 255) / 256), 256, 0, st>>>(r);
        SPV_CHECK_LAUNCH();
    }
    return SPV_OK;
}

// dW[M, :G] = dh1^T log1p(X[rows, :G]): dh1 given as a bf16 pair [B, ld_d] (the fused epilogue of the fc2 input-gradient GEMM
// writes it), dW row pitch ld_dw
extern "C" int spv_enc_fc1_dw(const void* X, long long ldx, const int* rows, const void* d_hi, const void* d_lo, long long ld_d,
                              float* dW, long long ld_dw, int B, int M, int G, void* stream) {
    if (!X || !d_hi || !d_lo || !dW || B <= 0 || M <= 0 || G <= 0) return SPV_ERR_ARG;
    CUtensorMap mt, mtl;
    int rc = spv_make_tensor_map_bf16(&mt, d_hi, (unsigned long long)M, (unsigned long long)B, (unsigned long long)ld_d, 64, 64);
    if (rc != SPV_OK) return rc;
    rc = spv_make_tensor_map_bf16(&mtl, d_lo, (unsigned long long)M, (unsigned long long)B, (unsigned long long)ld_d, 64, 64);
    if (rc != SPV_OK) return rc;
    fc1::Params p;
    p.X = reinterpret_cast<const unsigned short*>(X); p.ldx = ldx; p.rows = rows; p.C = dW; p.ldc = ld_dw; p.bias = nullptr; p.ws = nullptr;
    p.M = M; p.N = G; p.K = B; p.relu = 0; p.pre_acc = 0; p.splits = 1; p.kb_per_split = (B + 63) / 64;
    return fc1::launch_fc1<true>(mt, mtl, p, reinterpret_cast<cudaStream_t>(stream));
}

// =======================================================================================================================
// Forward of the encoder's first layer with the transformed counts written straight into TENSOR MEMORY as the MMA's A operand.
// The shared-memory version above is bound by shared-memory bandwidth: per 64-gene k-block the tensor core reads 3 x (A + B) =
// 96 KB of operands while producers and TMA write 64 KB more (measured: 2200 cycles per k-block in the producers' store phase,
// tools/bench_fc1.py).  Here thread = cell row = TMEM lane: the producer warps gather the row's counts, look the split-bf16 pair
// up and tcgen05.st the hi and lo halves of the A tile (2 x 32 columns per stage); only the weights go through shared memory
// (TMA, six stages), and the MMAs are issued in the TS form (A from TMEM).  Same arithmetic as fc1_kernel<false>.
// =======================================================================================================================
namespace fc1t {

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int B_STAGES = 6, A_STAGES = 4;
constexpr int PROD_WARPS = 8, THREADS = 64 + 32 * PROD_WARPS;
constexpr int TILE = 128 * 64 * 2;                    // one 16 KB plane of the weight tile
constexpr int B_STAGE_BYTES = 2 * TILE;               // [W hi | W lo]
constexpr int A_COLS = 64;                            // TMEM columns per A stage: hi (32) | lo (32)
constexpr int TMEM_COLS = 512;                        // accumulator 128 + 4 x 64 = 384 -> power of two
constexpr int SMEM = B_STAGES * B_STAGE_BYTES + 1024 + 256 * 4 + 512;

__global__ void __launch_bounds__(THREADS, 1) fc1_tmem_kernel(const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapWlo,
                                                              fc1::Params p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = tc::smem_u32(smem_raw);
    uint8_t* tiles = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
    unsigned int* lutp = reinterpret_cast<unsigned int*>(tiles + B_STAGES * B_STAGE_BYTES);
    uint64_t* full_b = reinterpret_cast<uint64_t*>(lutp + 256);
    uint64_t* empty_b = full_b + B_STAGES;
    uint64_t* full_a = empty_b + B_STAGES;
    uint64_t* empty_a = full_a + A_STAGES;
    uint64_t* tmem_full = empty_a + A_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM, split = blockIdx.z;
    const int num_kb_total = (p.K + BK - 1) / BK;
    const int kb_begin = split * p.kb_per_split;
    const int num_kb = max(min(num_kb_total, kb_begin + p.kb_per_split) - kb_begin, 0);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&mapW);
        tc::tma_prefetch_desc(&mapWlo);
        for (int s = 0; s < B_STAGES; ++s) { tc::mbar_init(&full_b[s], 1); tc::mbar_init(&empty_b[s], 1); }
        for (int s = 0; s < A_STAGES; ++s) { tc::mbar_init(&full_a[s], PROD_WARPS); tc::mbar_init(&empty_a[s], 1); }
        tc::mbar_init(tmem_full, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, TMEM_COLS);
    if (warp >= 2) {
        const int t = threadIdx.x - 64;
        lutp[t] = fc1::pack_split_dev(t == 0 ? 0.0f : log1pf((float)t));
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;          // accumulator: columns [0, 128)
    const uint32_t tmem_a0 = tmem_base + BN;        // A stages: columns [128, 128 + 4 x 64)

    if (warp == 0) {
        if (tc::elect_one()) {
            for (int i = 0; i < num_kb; ++i) {
                const int s = i % B_STAGES;
                tc::mbar_wait(&empty_b[s], ((i / B_STAGES) & 1) ^ 1);
                uint8_t* dst = tiles + s * B_STAGE_BYTES;
                tc::mbar_expect_tx(&full_b[s], B_STAGE_BYTES);
                const int k0 = (kb_begin + i) * BK;
                tc::tma_load_2d(&mapW, &full_b[s], dst, k0, n0);
                tc::tma_load_2d(&mapWlo, &full_b[s], dst + TILE, k0, n0);
            }
        }
    } else if (warp == 1) {
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::idesc_bf16(BM, BN, false, false);
            for (int i = 0; i < num_kb; ++i) {
                const int sb = i % B_STAGES, sa = i % A_STAGES;
                tc::mbar_wait(&full_b[sb], (i / B_STAGES) & 1);
                tc::mbar_wait(&full_a[sa], (i / A_STAGES) & 1);
                tc::fence_after_sync();
                const uint32_t b_hi = tc::smem_u32(tiles + sb * B_STAGE_BYTES), b_lo = b_hi + TILE;
                const uint32_t a_hi = tmem_a0 + sa * A_COLS, a_lo = a_hi + 32;
#pragma unroll
                for (int kk = 0; kk < BK / 16; ++kk) {
                    const uint64_t dbh = tc::smem_desc(b_hi + kk * 32, 16, 1024), dbl = tc::smem_desc(b_lo + kk * 32, 16, 1024);
                    tc::umma_bf16_ts(tmem_base, a_hi + kk * 8, dbh, idesc, (i > 0 || kk > 0) ? 1u : 0u);
                    tc::umma_bf16_ts(tmem_base, a_hi + kk * 8, dbl, idesc, 1u);
                    tc::umma_bf16_ts(tmem_base, a_lo + kk * 8, dbh, idesc, 1u);
                }
                tc::umma_commit(&empty_b[sb]);
                tc::umma_commit(&empty_a[sa]);
            }
            tc::umma_commit(tmem_full);
        }
    } else {
        // ================= producers: warp w owns TMEM lanes 32 (w & 3) .., the two warps of a quarter split the 64 genes
        const int q = warp & 3, khalf = (warp - 2) >> 2;
        const int r = q * 32 + lane;                 // row of the tile = TMEM lane
        const unsigned short* row = nullptr;
        if (m0 + r < p.M) row = p.X + (p.rows ? (long)__ldg(p.rows + m0 + r) : (long)(m0 + r)) * p.ldx;
        constexpr int PF = 4;
        uint4 buf[PF][4];
        auto issue = [&](int i, uint4 (&dst)[4]) {
            const int gene0 = (kb_begin + i) * BK + khalf * 32;
            if (!row || gene0 >= p.K) {
#pragma unroll
                for (int j = 0; j < 4; ++j) dst[j] = make_uint4(0u, 0u, 0u, 0u);
                return;
            }
            const unsigned short* src = row + gene0;
            if (((reinterpret_cast<uintptr_t>(src) & 15) == 0) && gene0 + 32 <= p.K) {
#pragma unroll
                for (int j = 0; j < 4; ++j) dst[j] = __ldg(reinterpret_cast<const uint4*>(src) + j);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    unsigned int w[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int g = gene0 + j * 8 + e * 2;
                        const unsigned int c0 = g < p.K ? __ldg(src + j * 8 + e * 2) : 0u;
                        const unsigned int c1 = g + 1 < p.K ? __ldg(src + j * 8 + e * 2 + 1) : 0u;
                        w[e] = c0 | (c1 << 16);
                    }
                    dst[j] = make_uint4(w[0], w[1], w[2], w[3]);
                }
            }
        };
#pragma unroll
        for (int u = 0; u < PF; ++u)
            if (u < num_kb) issue(u, buf[u]);
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        for (int i0 = 0; i0 < num_kb; i0 += PF) {
#pragma unroll
            for (int u = 0; u < PF; ++u) {
                const int i = i0 + u;
                if (i < num_kb) {
                    const int sa = i % A_STAGES;
                    uint32_t hi[16], lo[16];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const unsigned int w[4] = {buf[u][j].x, buf[u][j].y, buf[u][j].z, buf[u][j].w};
                        unsigned int e[8];
                        if ((((w[0] | w[1]) | (w[2] | w[3])) & 0xff00ff00u) == 0u) {
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                e[2 * c] = lutp[w[c] & 0xffu];
                                e[2 * c + 1] = lutp[w[c] >> 16];
                            }
                        } else {
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                e[2 * c] = fc1::lut_any(lutp, w[c] & 0xffffu);
                                e[2 * c + 1] = fc1::lut_any(lutp, w[c] >> 16);
                            }
                        }
#pragma unroll
                        for (int c = 0; c < 4; ++c) {  // column = two consecutive genes: low half = even gene
                            hi[4 * j + c] = __byte_perm(e[2 * c], e[2 * c + 1], 0x5410);
                            lo[4 * j + c] = __byte_perm(e[2 * c], e[2 * c + 1], 0x7632);
                        }
                    }
                    tc::mbar_wait(&empty_a[sa], ((i / A_STAGES) & 1) ^ 1);  // the conversion above overlaps the wait for the stage
                    tc::fence_after_sync();
                    const uint32_t a_hi = tmem_a0 + sa * A_COLS + lane_base + khalf * 16;
                    tc::tmem_st16(a_hi, hi);
                    tc::tmem_st16(a_hi + 32, lo);
                    tc::tmem_st_wait();
                    tc::fence_before_sync();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&full_a[sa]);
                    if (i + PF < num_kb) issue(i + PF, buf[u]);
                }
            }
        }
        // ---- epilogue
        if (num_kb > 0) {
            tc::mbar_wait(tmem_full, 0);
            tc::fence_after_sync();
        }
        const int m = m0 + r;
        float* out = p.splits > 1 ? p.ws + (size_t)split * p.M * p.N : p.C;
        const long ld = p.splits > 1 ? p.N : p.ldc;
        const bool fin = p.splits == 1;
#pragma unroll 1
        for (int c0 = khalf * 64; c0 < khalf * 64 + 64; c0 += 32) {
            if (n0 + c0 >= p.N) break;
            uint32_t v[32];
            if (num_kb > 0) {
                tc::tmem_ld32(tmem_base + lane_base + (uint32_t)c0, v);
                tc::tmem_ld_wait();
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = 0u;
            }
            if (m < p.M) {
                float* dst = out + (size_t)m * ld + n0 + c0;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int n = n0 + c0 + j;
                    if (n < p.N) {
                        float x = __uint_as_float(v[j]);
                        if (fin) {
                            if (p.pre_acc) x += dst[j];
                            if (p.bias) x += __ldg(p.bias + n);
                            if (p.relu) x = fmaxf(x, 0.0f);
                        }
                        dst[j] = x;
                    }
                }
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

int launch(const CUtensorMap& mw, const CUtensorMap& mwl, const fc1::Params& p, cudaStream_t st) {
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
        if (cudaFuncSetAttribute(fc1_tmem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM) != cudaSuccess) return SPV_ERR_LAUNCH;
        configured[dev & 63] = true;
    }
    dim3 grid((p.N + BN - 1) / BN, (p.M + BM - 1) / BM, p.splits);
    fc1_tmem_kernel<<<grid, THREADS, SMEM, st>>>(mw, mwl, p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

}  // namespace fc1t

int fc1t_launch(const CUtensorMap& mw, const CUtensorMap& mwl, const fc1::Params& p, cudaStream_t st) { return fc1t::launch(mw, mwl, p, st); }
