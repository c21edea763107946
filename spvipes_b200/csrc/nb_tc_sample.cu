// Count draws from the decoder's NB mixture (nb_sample.cuh): the tensor-core sampling sweep and the SIMT sampler over given
// parameters.  Both sample through the same device routine in this one translation unit, so for the same (rate_p, rate_s, pi,
// theta) and the same key they write the same bits.
//
// Sampling sweep: the operands, prologue and tensor-memory accumulators of the element sweep (nb_tc.cu, nb_tc_sweep.cuh) without
// the count gather.  The epilogue computes rate_p, rate_s and pi as the element sweep does, keeps them for eight genes at a time
// and, per draw, samples a 32-cell x 8-gene slab, stages it in the drained operand stages and stores it as four whole
// 32-byte sectors per warp store.  Nothing but the counts is written.
#include "nb_tc_sweep.cuh"
#include "nb_sample.cuh"

namespace {

using namespace nbtc;

constexpr int SO_CH = 8, SO_PITCH = SO_CH + 1;  // staging slab: 32 cells x SO_CH genes per epilogue warp, conflict-free thread = cell writes
constexpr int SO_WARP_FLOATS = 32 * SO_PITCH, SO_PAR_FLOATS = 3 * SO_CH * 32;
static_assert(EPI_WARPS * (SO_WARP_FLOATS + SO_PAR_FLOATS) * 4 <= STAGES * STAGE_BYTES, "slabs and parameters must fit in the operand stages");

struct NbTcSampleParams : NbTcParams {
    float* out;                        // [n_draws] x [B, ld_out], draw pitch draw_pitch
    long ld_out, draw_pitch;
    unsigned long long seed;
    int group, n_draws;
    uint32_t draw0;
};

// CTAs of this kernel currently resident per SM (nb_tc_sweep.cuh mma_warp)
__device__ int g_resident_sample[256];

__global__ void __launch_bounds__(THREADS, 2) nb_tc_sample_kernel(const __grid_constant__ CUtensorMap mapA,
                                                                  const __grid_constant__ CUtensorMap mapB,
                                                                  const __grid_constant__ CUtensorMap mapZ,
                                                                  const __grid_constant__ CUtensorMap mapZc, NbTcSampleParams p) {
    const Smem sm = carve_smem();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    const int num_kb = (p.K + BK - 1) / BK;
    init_pipeline(sm, &mapA, &mapB, &mapZ, &mapZc, warp, lane);
    uint32_t tmem_base = 0, tmem_z = 0;

    if (warp == 0) {
        produce(sm, &mapA, &mapB, &mapZ, &mapZc, n0, m0, num_kb, p.Gp);
    } else if (warp == 1) {
        mma_warp(sm, g_resident_sample, num_kb, lane, tmem_base, tmem_z);
    } else {
        const int e = warp - 2;
        const int q = warp & 3;          // TMEM lane quarter this warp may access
        const int half = e >> 2;         // which 32 gene columns of the tile
        const int m = m0 + q * 32 + lane;
        const bool mok = m < p.B;
        uint32_t cw[NGATHER];
        // gene constants: theta (x) and bm (w) are used; no counts are gathered
        epi_prologue<SPV_SRC_U16_LOG1P, GC_THE, GC_KC>(p, sm, false, n0, m0, mok ? m : 0, cw, [] {});
        tc::mbar_wait(sm.tmem_ready, 0);
        tmem_base = *reinterpret_cast<volatile uint32_t*>(sm.tmem_slot);
        tmem_z = *reinterpret_cast<volatile uint32_t*>(sm.tmem_slot + 1);
        tc::mbar_wait(sm.tmem_full, 0);  // accumulators complete; the operand stages are free from here on
        tc::fence_after_sync();
        asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");  // constants staged (epilogue warps only)
        const float4* s_gc = sm.s_gc;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16), lane_z = tmem_z + ((uint32_t)(q * 32) << 16);
        float* slab = reinterpret_cast<float*>(sm.tiles) + e * SO_WARP_FLOATS;
        // rate_p, rate_s, pi of the warp's SO_CH genes, [3][SO_CH][32 lanes]: kept in shared memory rather than registers, so that
        // one copy of the sampler serves the SO_CH genes
        float* par = reinterpret_cast<float*>(sm.tiles) + EPI_WARPS * SO_WARP_FLOATS + e * SO_PAR_FLOATS + lane;
#pragma unroll 1
        for (int j8 = 0; j8 < WCOLS; j8 += SO_CH) {
#pragma unroll
            for (int j4 = 0; j4 < SO_CH; j4 += 4) {
                const int c0 = half * WCOLS + j8 + j4;
                uint32_t rpi[4], rlp[4], rls[4];
                tc::tmem_ld4(lane_addr + (uint32_t)c0, rpi);
                tc::tmem_ld4(lane_z + (uint32_t)c0, rlp);
                tc::tmem_ld4(lane_z + (uint32_t)(BN + c0), rls);
                tc::tmem_ld_wait();
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {  // as the element sweep computes them
                    par[(0 * SO_CH + j4 + jj) * 32] = fast_ex2(__uint_as_float(rlp[jj]));
                    par[(1 * SO_CH + j4 + jj) * 32] = fast_ex2(__uint_as_float(rls[jj]));
                    par[(2 * SO_CH + j4 + jj) * 32] = __uint_as_float(rpi[jj]) + s_gc[c0 + jj].w;
                }
            }
            const int gl0 = half * WCOLS + j8;
            const int col = lane % SO_CH, gs = n0 + gl0 + col;  // the gene this lane stores
#pragma unroll 1
            for (int d = 0; d < p.n_draws; ++d) {
                const uint32_t draw = p.draw0 + (uint32_t)d;
#pragma unroll 1
                for (int jj = 0; jj < SO_CH; ++jj) {
                    const int g = n0 + gl0 + jj;
                    float c = 0.0f;
                    if (mok && g < p.G)
                        c = nb_mixture_sample(par[jj * 32], par[(SO_CH + jj) * 32], par[(2 * SO_CH + jj) * 32], s_gc[gl0 + jj].x,
                                              nbs_key(p.seed, p.group, draw, (uint32_t)m, (uint32_t)g));
                    slab[lane * SO_PITCH + jj] = c;
                }
                __syncwarp();
                float* dst = p.out + (long)d * p.draw_pitch;
#pragma unroll
                for (int r = lane / SO_CH; r < 32; r += 32 / SO_CH) {
                    const int mr = m0 + q * 32 + r;
                    if (mr < p.B && gs < p.G) dst[(long)mr * p.ld_out + gs] = slab[r * SO_PITCH + col];
                }
                __syncwarp();
            }
        }
    }
    release_tmem(warp, lane, tmem_base, tmem_z, g_resident_sample);
}

// SIMT sampler: thread = (cell, gene), every draw; the warp's stores of one draw are 32 consecutive genes
constexpr int SS_THREADS = 128;

__global__ void __launch_bounds__(SS_THREADS) nb_mixture_sample_kernel(const float* __restrict__ mu1, const float* __restrict__ mu2,
                                                                       const float* __restrict__ pi, long ld_in,
                                                                       const float* __restrict__ theta, int B, int G, int n_draws,
                                                                       float* __restrict__ out, long ld_out, long draw_pitch,
                                                                       unsigned long long seed, int group, uint32_t draw0) {
    const int g = blockIdx.x * SS_THREADS + threadIdx.x;
    if (g >= G) return;
    const float th = __ldg(theta + g);
    for (int b = blockIdx.y; b < B; b += gridDim.y) {
        const long i = (long)b * ld_in + g;
        const float r1 = __ldg(mu1 + i), r2 = __ldg(mu2 + i), pv = __ldg(pi + i);
        float* dst = out + (long)b * ld_out + g;
        for (int d = 0; d < n_draws; ++d)
            dst[(long)d * draw_pitch] = nb_mixture_sample(r1, r2, pv, th, nbs_key(seed, group, draw0 + (uint32_t)d, (uint32_t)b, (uint32_t)g));
    }
}

// the output arguments both entry points check: n_draws slabs [B, ld_out] that do not overlap, keys that fit the counter layout
bool sample_args_ok(int B, int G, int n_draws, const float* out, long long ld_out, long long draw_pitch, int group, unsigned int draw0) {
    if (!out || B <= 0 || G <= 0 || n_draws <= 0 || ld_out < G || group < 0 || group > NBS_MAX_GROUP) return false;
    if ((unsigned long long)draw0 + (unsigned long long)n_draws > 0x100000000ull) return false;  // draw indices are 32-bit
    return n_draws == 1 || draw_pitch >= (long long)(B - 1) * ld_out + G;
}

}  // namespace

// Sampling sweep: the operands and ptrs of spv_dec_nb_elems_tc (counts, count table and row partials unused: ptrs[5] bm and
// ptrs[6] genec are read), draws [draw0, draw0 + n_draws) into out[d - draw0] (see the header).
extern "C" int spv_dec_nb_sample_tc(const void* const* ptrs, const void* amix_bf16, long long ld_amixb, const void* wstack_bf16,
                                    long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, int B, int G, int HD, int P, int S,
                                    int kmix, unsigned long long seed, int group, unsigned int draw0, int n_draws, float* out,
                                    long long ld_out, long long draw_pitch, void* stream) {
    if (!sweep_args_ok(ptrs, amix_bf16, wstack_bf16, zc_f16, wz_f16, Gp, B, G, P, S) || HD < 0 ||
        !sample_args_ok(B, G, n_draws, out, ld_out, draw_pitch, group, draw0))
        return SPV_ERR_ARG;
    const int K = kmix > 0 ? kmix : HD + P + S;
    NbTcSampleParams p{};
    NbTcMaps mp;
    const int rc = sweep_setup<nb_tc_sample_kernel>(p, mp, ptrs, 0, amix_bf16, ld_amixb, wstack_bf16, ld_w, Gp, zc_f16, wz_f16, B, G, K);
    if (rc != SPV_OK) return rc;
    p.X = nullptr; p.rows = nullptr; p.tgf = nullptr;  // not read: no counts
    p.out = out; p.ld_out = ld_out; p.draw_pitch = draw_pitch;
    p.seed = seed; p.group = group; p.n_draws = n_draws; p.draw0 = draw0;
    dim3 grid((G + BN - 1) / BN, (B + BM - 1) / BM);
    nb_tc_sample_kernel<<<grid, THREADS, SMEM_BYTES, reinterpret_cast<cudaStream_t>(stream)>>>(mp.a, mp.b, mp.z, mp.zc, p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

extern "C" int spv_nb_mixture_sample(const float* mu1, const float* mu2, const float* pi, long long ld_in, const float* theta, int B,
                                     int G, int n_draws, float* out, long long ld_out, long long draw_pitch, unsigned long long seed,
                                     int group, unsigned int draw0, void* stream) {
    if (!mu1 || !mu2 || !pi || !theta || ld_in < G || !sample_args_ok(B, G, n_draws, out, ld_out, draw_pitch, group, draw0))
        return SPV_ERR_ARG;
    dim3 grid((G + SS_THREADS - 1) / SS_THREADS, B < 65535 ? B : 65535);
    nb_mixture_sample_kernel<<<grid, SS_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(mu1, mu2, pi, ld_in, theta, B, G, n_draws, out,
                                                                                              ld_out, draw_pitch, seed, group, draw0);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}
