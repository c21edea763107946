// Decoder + negative-binomial-mixture likelihood, fp32 SIMT path.
//   rho_p = exp(lib) softmax_g(BN_p(z_p Wp^T)),  rho_s = exp(lib) softmax_g(BN_s(z_s Ws^T)),
//   pi = [relu(BN_h(zz Wh^T + bh)) | zz] Wm^T + bm,  rec_b = -sum_g log_mixture_nb(log1p(x), rho_p, rho_s, theta, pi)
// Reference: nn/networks.py:314-325 (LinearDecoderSPVIPE.forward), module/spVIPESmodule.py:751-759 (generative),
// :817-824 (loss), scvi-tools 0.20.0 log_mixture_nb (eps 1e-8, shared theta) and FCLayers BatchNorm1d(eps 1e-3, mom 0.01).
//
// No [B, G] softmax / rate tensor is materialised: the per-gene BatchNorm statistics of z W^T are obtained in closed
// form from mean(z) and Cov(z) (spv_dec_fold), the gene-axis softmax normaliser by a first tile sweep
// (pass STATS), the likelihood and the row sums the backward needs by a second sweep (pass NB).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "gemm_simt.cuh"
#include "../../include/spvipes_b200.h"

#include "decoder_common.cuh"

// ---------------------------------------------------------------------------------------
// the NB-mixture element (scvi log_mixture_nb, shared theta).  t = log1p(count) (quirk Q3).
// ---------------------------------------------------------------------------------------
struct NbFwd { float ll, ep, es; };

__device__ __forceinline__ NbFwd nb_forward(float t, float lp, float ls, float pi, float th, float lte, float lgt,
                                            float Rp, float Rs) {
    float rp = expf(lp + Rp), rs = expf(ls + Rs);  // exp(lib) * softmax
    float d1 = th + rp + NB_EPS, d2 = th + rs + NB_EPS;
    float l1 = logf(d1), l2 = logf(d2);
    float a = th * (lte - l1), b = th * (lte - l2);
    float gp = 0.0f, gs = 0.0f;
    if (t != 0.0f) {
        float lg = lgammaf(t + th) - lgt - lgammaf(t + 1.0f);
        a += t * (logf(rp + NB_EPS) - l1) + lg;
        b += t * (logf(rs + NB_EPS) - l2) + lg;
        gp = t / (rp + NB_EPS);
        gs = t / (rs + NB_EPS);
    }
    b -= pi;
    float mx = fmaxf(a, b);
    float ea = expf(a - mx), eb = expf(b - mx);
    float se = ea + eb;
    float lse = mx + logf(se);
    NbFwd o;
    o.ll = lse - softplusf(-pi);
    float wa = ea / se, wb = eb / se;
    o.ep = wa * (gp - (th + t) / d1) * rp;  // d ll / d rho_p * rho_p
    o.es = wb * (gs - (th + t) / d2) * rs;
    return o;
}

// The same element in float64 from the fp32 rates: the per-element value of the element pass (PASS_ELEM).  Summed into a per-cell
// term, the fp32 form's absolute errors (lgamma(t + theta) - lgamma(theta) of a gene with theta ~ e^9 carries ~1e-2 of fp32
// rounding; theta (log(theta + eps) - log(theta + rho + eps)) cancels likewise) are small against the sum, but one element's
// value can be smaller than them.  Off the training step, so the float64 cost does not matter.
static __device__ __noinline__ float nb_ll_f64(double t, double rp, double rs, double pi, double th) {
    const double eps = 1e-8;
    const double lte = log(th + eps), l1 = log(th + rp + eps), l2 = log(th + rs + eps);
    const double lg = t != 0.0 ? lgamma(t + th) - lgamma(th) - lgamma(t + 1.0) : 0.0;
    const double a = th * (lte - l1) + t * (log(rp + eps) - l1) + lg;
    const double b = th * (lte - l2) + t * (log(rs + eps) - l2) + lg - pi;
    const double mx = fmax(a, b);
    const double lse = mx + log1p(exp(-fabs(a - b)));
    const double softplus_neg_pi = fmax(-pi, 0.0) + log1p(exp(-fabs(pi)));
    return (float)(lse - softplus_neg_pi);
}

struct NbBwd { float dyp, dys, dpi, dth; };

// scale = upstream d loss / d ll  (= -grad_scale / B)
__device__ __forceinline__ NbBwd nb_backward(float t, float lp, float ls, float pi, float th, float lte, float dgt, float Rp,
                                             float Rs, float Dp, float Ds, float inv_elib, float scale) {
    float rp = expf(lp + Rp), rs = expf(ls + Rs);
    float d1 = th + rp + NB_EPS, d2 = th + rs + NB_EPS;
    float l1 = logf(d1), l2 = logf(d2);
    float diff = th * (l2 - l1) + pi;  // log_nb_p - (log_nb_s - pi); the lgamma terms cancel
    float gp = 0.0f, gs = 0.0f, dg = 0.0f;
    if (t != 0.0f) {
        diff += t * (logf(rp + NB_EPS) - l1 - logf(rs + NB_EPS) + l2);
        gp = t / (rp + NB_EPS);
        gs = t / (rs + NB_EPS);
        dg = digammaf_pos(t + th) - dgt;
    }
    float wa = 1.0f / (1.0f + expf(-diff));
    float wb = 1.0f / (1.0f + expf(diff));
    float q1 = (th + t) / d1, q2 = (th + t) / d2;
    float ep = wa * (gp - q1) * rp;
    float es = wb * (gs - q2) * rs;
    NbBwd o;
    o.dyp = scale * (ep - rp * inv_elib * Dp);  // softmax backward: rho (g - D / exp(lib))
    o.dys = scale * (es - rs * inv_elib * Ds);
    o.dpi = scale * (1.0f / (1.0f + expf(pi)) - wb);
    o.dth = scale * (wa * (lte - l1 - q1) + wb * (lte - l2 - q2) + th / (th + NB_EPS) + dg);
    return o;
}

// ---------------------------------------------------------------------------------------
// tile sweeps over the [B, G] index space
// ---------------------------------------------------------------------------------------
struct DecP {
    const void* X; long ldx; const int* rows;           // counts (row-gathered minibatch)
    const float* amix; long ld_amix;                     // [B, HD + P + S] = [hm | z_private_arg | z_shared_arg]
    const float* wfold;                                  // [G, P + S]
    const float* wm; const float* bm;                    // [G, HD + P + S], [G]
    const float* genec;                                  // [GC_N, G]
    const float* lib;                                    // [B]
    float* part_stats;                                   // [nTG, B, 4]
    float* rowc;                                         // [B, 4] = Rp, Rs, Dp, Ds
    float* pi;                                           // [B, G]
    float* part_nb;                                      // [nTG, B, 3]
    float* dyp; float* dys; float* dpi;                  // [B, G]
    float* colpart;                                      // [nTB, 4, G]
    int B, G, HD, P, S;
    const float* zz; long ld_zz;                         // [B, P + S] inputs of the two factor regressors (default: amix + HD)
    int kmix;                                            // width of the mixing net's input (default HD + P + S)
    float scale;
    int pi_ready;                                        // PASS_NB: pi already holds the mixture logits (tensor-core GEMM)
    __nv_bfloat16* dpi_bf16; long ld_dpi_bf16;           // PASS_BWD: write d pi as bf16 (operand of the tensor-core GEMMs)
    float* eo[5]; long ld_out;                           // PASS_ELEM: ll, rate_p, rate_s, pi, mean [B, ld_out] (NULL = not written)
};

enum { PASS_STATS = 0, PASS_NB = 1, PASS_BWD = 2, PASS_ELEM = 3 };

template <int PASS, int SRC>
__global__ void __launch_bounds__(GT_THREADS) dec_tile_kernel(DecP p) {
    __shared__ GemmSmem sm;
    __shared__ float red[16][GT_BN + 1];
    const int n0 = blockIdx.x * GT_BN, m0 = blockIdx.y * GT_BM;
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    const int KMIX = p.kmix, KZ = p.P + p.S;
    const int G = p.G, B = p.B;
    float lp[4][4], ls[4][4], pi[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) lp[i][j] = ls[i][j] = pi[i][j] = 0.0f;
    const float* azz = p.zz;
    tile_mainloop<SPV_SRC_F32, false, SPV_SRC_F32, true>(lp, azz, p.ld_zz, nullptr, p.wfold, KZ, nullptr, B, G, 0, p.P, m0, n0, sm);
    tile_mainloop<SPV_SRC_F32, false, SPV_SRC_F32, true>(ls, azz + p.P, p.ld_zz, nullptr, p.wfold + p.P, KZ, nullptr, B, G, 0, p.S, m0, n0, sm);
    if ((PASS == PASS_NB || PASS == PASS_ELEM) && !p.pi_ready)
        tile_mainloop<SPV_SRC_F32, false, SPV_SRC_F32, true>(pi, p.amix, p.ld_amix, nullptr, p.wm, KMIX, nullptr, B, G, 0, KMIX, m0, n0, sm);

    // per-gene constants of this thread's 4 genes
    float cp[4], cs[4], th[4], lte[4], lgx[4], bm[4];
    bool nok[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int n = n0 + tx * 4 + j;
        nok[j] = n < G;
        int nn = nok[j] ? n : 0;
        cp[j] = p.genec[GC_CP * (long)G + nn];
        cs[j] = p.genec[GC_CS * (long)G + nn];
        if (PASS != PASS_STATS) {
            th[j] = p.genec[GC_THETA * (long)G + nn];
            lte[j] = p.genec[GC_LTE * (long)G + nn];
            lgx[j] = p.genec[(PASS != PASS_BWD ? GC_LGT : GC_DGT) * (long)G + nn];
            bm[j] = PASS != PASS_BWD ? p.bm[nn] : 0.0f;
        }
    }

    if (PASS == PASS_STATS) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int m = m0 + ty * 4 + i;
            float mp = -INFINITY, ms = -INFINITY;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (nok[j]) {
                    lp[i][j] += cp[j];
                    ls[i][j] += cs[j];
                    mp = fmaxf(mp, lp[i][j]);
                    ms = fmaxf(ms, ls[i][j]);
                }
            mp = half_warp_max(mp);
            ms = half_warp_max(ms);
            float sp = 0.0f, ss = 0.0f;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (nok[j]) {
                    sp += expf(lp[i][j] - mp);
                    ss += expf(ls[i][j] - ms);
                }
            sp = half_warp_sum(sp);
            ss = half_warp_sum(ss);
            if (tx == 0 && m < B) {
                float* o = p.part_stats + ((long)blockIdx.x * B + m) * 4;
                o[0] = mp; o[1] = sp; o[2] = ms; o[3] = ss;
            }
        }
        return;
    }

    if (PASS == PASS_ELEM) {  // the elements of the likelihood sweep, stored instead of reduced
        const int n = n0 + tx * 4;
        const bool vec = n + 3 < G && (p.ld_out & 3) == 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = m0 + ty * 4 + i;
            if (m >= B) break;
            const float Rp = p.rowc[(long)m * 4 + 0], Rs = p.rowc[(long)m * 4 + 1];
            const long xr = (p.rows ? (long)p.rows[m] : (long)m) * p.ldx;
            float v[5][4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float piv = p.pi_ready ? (nok[j] ? p.pi[(long)m * G + n + j] : 0.0f) : pi[i][j] + bm[j];
                const float lpj = lp[i][j] + cp[j], lsj = ls[i][j] + cs[j];
                v[1][j] = expf(lpj + Rp);  // the rates as nb_forward forms them
                v[2][j] = expf(lsj + Rs);
                v[0][j] = (p.eo[0] && nok[j]) ? nb_ll_f64(load_src<SRC>(p.X, xr + n + j), v[1][j], v[2][j], piv, th[j]) : 0.0f;
                v[3][j] = piv;
                v[4][j] = v[1][j] / (1.0f + expf(-piv)) + v[2][j] / (1.0f + expf(piv));
            }
#pragma unroll
            for (int o = 0; o < 5; ++o) {
                float* dst = p.eo[o];
                if (!dst) continue;
                dst += (long)m * p.ld_out + n;
                if (vec && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                    *reinterpret_cast<float4*>(dst) = make_float4(v[o][0], v[o][1], v[o][2], v[o][3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (nok[j]) dst[j] = v[o][j];
                }
            }
        }
        return;
    }

    float csum[4][4];  // [quantity][gene] column partial sums (PASS_BWD)
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int j = 0; j < 4; ++j) csum[q][j] = 0.0f;

#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int m = m0 + ty * 4 + i;
        const bool mok = m < B;
        const int mm = mok ? m : 0;
        const float Rp = p.rowc[(long)mm * 4 + 0], Rs = p.rowc[(long)mm * 4 + 1];
        const long xr = (p.rows ? (long)p.rows[mm] : (long)mm) * p.ldx;
        if (PASS == PASS_NB) {
            float sll = 0.0f, sep = 0.0f, ses = 0.0f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int n = n0 + tx * 4 + j;
                if (mok && nok[j]) {
                    float t = load_src<SRC>(p.X, xr + n);
                    float piv = p.pi_ready ? p.pi[(long)m * G + n] : pi[i][j] + bm[j];
                    NbFwd o = nb_forward(t, lp[i][j] + cp[j], ls[i][j] + cs[j], piv, th[j], lte[j], lgx[j], Rp, Rs);
                    sll += o.ll; sep += o.ep; ses += o.es;
                    if (!p.pi_ready) p.pi[(long)m * G + n] = piv;
                }
            }
            sll = half_warp_sum(sll);
            sep = half_warp_sum(sep);
            ses = half_warp_sum(ses);
            if (tx == 0 && mok) {
                float* o = p.part_nb + ((long)blockIdx.x * B + m) * 3;
                o[0] = sll; o[1] = sep; o[2] = ses;
            }
        } else {  // PASS_BWD
            const float Dp = p.rowc[(long)mm * 4 + 2], Ds = p.rowc[(long)mm * 4 + 3];
            const float inv_elib = expf(-p.lib[mm]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int n = n0 + tx * 4 + j;
                if (mok && nok[j]) {
                    float t = load_src<SRC>(p.X, xr + n);
                    float piv = p.pi[(long)m * G + n];
                    NbBwd o = nb_backward(t, lp[i][j] + cp[j], ls[i][j] + cs[j], piv, th[j], lte[j], lgx[j], Rp, Rs, Dp, Ds,
                                          inv_elib, p.scale);
                    p.dyp[(long)m * G + n] = o.dyp;
                    p.dys[(long)m * G + n] = o.dys;
                    if (p.dpi_bf16) p.dpi_bf16[(long)m * p.ld_dpi_bf16 + n] = __float2bfloat16(o.dpi);
                    else p.dpi[(long)m * G + n] = o.dpi;
                    csum[0][j] += o.dyp; csum[1][j] += o.dys; csum[2][j] += o.dpi; csum[3][j] += o.dth;
                }
            }
        }
    }
    if (PASS == PASS_BWD) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 4; ++j) red[ty][tx * 4 + j] = csum[q][j];
            __syncthreads();
            if (threadIdx.x < GT_BN) {
                int n = n0 + threadIdx.x;
                float s = 0.0f;
#pragma unroll
                for (int r = 0; r < 16; ++r) s += red[r][threadIdx.x];
                if (n < G) p.colpart[((long)blockIdx.y * 4 + q) * G + n] = s;
            }
        }
    }
}

// combine the per-gene-tile softmax partials: Rp = lib - logsumexp_g(y_p), Rs likewise
// R columns of the tensor-core branch operand (decoder_common.cuh ZK_RP / ZK_RS): the row normalisers in base-2 units as
// split-fp16 pairs, so that the likelihood kernels' accumulators are complete logits
__device__ __forceinline__ void store_row_normalisers(__half* zc, int b, float rp, float rs) {
    if (!zc) return;
    const float vp = rp * 1.4426950408889634f, vs = rs * 1.4426950408889634f;
    const __half ph = to_half_sat(vp), sh = to_half_sat(vs);
    __half2* dst = reinterpret_cast<__half2*>(zc + (long)b * 64 + ZK_RP);
    dst[0] = __halves2half2(ph, to_half_sat(vp - __half2float(ph)));
    dst[1] = __halves2half2(sh, to_half_sat(vs - __half2float(sh)));
}

__global__ void rowstat_kernel(const float* __restrict__ part, int nTG, int B, const float* __restrict__ lib,
                               float* __restrict__ rowc, __half* __restrict__ zc) {
    // one warp per row, lanes over the gene tiles; the row's partials are read once (16-byte loads, all in flight) and the
    // library size is fetched up front: one memory round trip instead of three dependent ones
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    const float l = __ldg(lib + b);
    constexpr int R = 4;
    const float4 none = make_float4(-INFINITY, 0.0f, -INFINITY, 0.0f);
    float4 o[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int t = lane + 32 * r;
        o[r] = t < nTG ? __ldg(reinterpret_cast<const float4*>(part) + (long)t * B + b) : none;
    }
    float Mp = -INFINITY, Ms = -INFINITY;
#pragma unroll
    for (int r = 0; r < R; ++r) { Mp = fmaxf(Mp, o[r].x); Ms = fmaxf(Ms, o[r].z); }
    for (int t = lane + 32 * R; t < nTG; t += 32) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(part) + (long)t * B + b);
        Mp = fmaxf(Mp, v.x); Ms = fmaxf(Ms, v.z);
    }
    Mp = warp_max(Mp);
    Ms = warp_max(Ms);
    float Sp = 0.0f, Ss = 0.0f;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        Sp += o[r].y * expf(o[r].x - Mp);
        Ss += o[r].w * expf(o[r].z - Ms);
    }
    for (int t = lane + 32 * R; t < nTG; t += 32) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(part) + (long)t * B + b);
        Sp += v.y * expf(v.x - Mp);
        Ss += v.w * expf(v.z - Ms);
    }
    Sp = warp_sum(Sp);
    Ss = warp_sum(Ss);
    if (lane == 0) {
        const float rp = l - (Mp + logf(Sp)), rs = l - (Ms + logf(Ss));
        rowc[(long)b * 4 + 0] = rp;
        rowc[(long)b * 4 + 1] = rs;
        store_row_normalisers(zc, b, rp, rs);
    }
}

// Many gene tiles (20k genes: 626 partials per row): one CTA per 32 rows, lanes over the rows so that every load of a warp is
// one contiguous 512-byte run of the [tile][row] layout, the 8 warps split the tiles and merge their running (max, sum) pairs
// through shared memory in warp order (deterministic).  The warp-per-row form above reads 16 useful bytes per 32-byte sector.
__global__ void __launch_bounds__(256) rowstat_wide_kernel(const float* __restrict__ part, int nTG, int B, const float* __restrict__ lib,
                                                           float* __restrict__ rowc, __half* __restrict__ zc) {
    __shared__ float4 red[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * 32 + lane;
    const bool ok = b < B;
    float Mp = -INFINITY, Ms = -INFINITY, Sp = 0.0f, Ss = 0.0f;
    const float4* src = reinterpret_cast<const float4*>(part) + (ok ? b : 0);
    constexpr int U = 8;
    for (int t0 = w; t0 < nTG; t0 += 8 * U) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int t = t0 + 8 * u;
            v[u] = (ok && t < nTG) ? __ldg(src + (long)t * B) : make_float4(-INFINITY, 0.0f, -INFINITY, 0.0f);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {  // online merge of (max, sum exp) pairs
            const float np = fmaxf(Mp, v[u].x), ns = fmaxf(Ms, v[u].z);
            if (np > -INFINITY) Sp = Sp * __expf(Mp - np) + v[u].y * __expf(v[u].x - np);
            if (ns > -INFINITY) Ss = Ss * __expf(Ms - ns) + v[u].w * __expf(v[u].z - ns);
            Mp = np; Ms = ns;
        }
    }
    red[w][lane] = make_float4(Mp, Sp, Ms, Ss);
    __syncthreads();
    if (w == 0 && ok) {
        float4 a = red[0][lane];
#pragma unroll
        for (int i = 1; i < 8; ++i) {
            const float4 c = red[i][lane];
            const float np = fmaxf(a.x, c.x), ns = fmaxf(a.z, c.z);
            if (np > -INFINITY) a.y = a.y * __expf(a.x - np) + c.y * __expf(c.x - np);
            if (ns > -INFINITY) a.w = a.w * __expf(a.z - ns) + c.w * __expf(c.z - ns);
            a.x = np; a.z = ns;
        }
        const float l = __ldg(lib + b);
        const float rp = l - (a.x + logf(a.y)), rs = l - (a.z + logf(a.w));
        rowc[(long)b * 4 + 0] = rp;
        rowc[(long)b * 4 + 1] = rs;
        store_row_normalisers(zc, b, rp, rs);
    }
}

// launch helper shared with the tensor-core statistics kernel (nb_tc.cu)
int spv_internal_rowstat(const float* part, int nparts, int B, const float* lib, float* rowc, void* zc_f16, cudaStream_t st) {
    __half* zc = reinterpret_cast<__half*>(zc_f16);
    if (nparts > 128) rowstat_wide_kernel<<<(B + 31) / 32, 256, 0, st>>>(part, nparts, B, lib, rowc, zc);
    else rowstat_kernel<<<(B + 7) / 8, 256, 0, st>>>(part, nparts, B, lib, rowc, zc);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

__global__ void rownb_kernel(const float* __restrict__ part, int nTG, int B, float* __restrict__ rowc, float* __restrict__ rec) {
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    float ll = 0.0f, dp = 0.0f, ds = 0.0f;
#pragma unroll 4
    for (int t = lane; t < nTG; t += 32) {
        const float* o = part + ((long)t * B + b) * 3;
        ll += o[0]; dp += o[1]; ds += o[2];
    }
    ll = warp_sum(ll); dp = warp_sum(dp); ds = warp_sum(ds);
    if (lane == 0) {
        rec[b] = -ll;  // reference :823-824
        rowc[(long)b * 4 + 2] = dp;
        rowc[(long)b * 4 + 3] = ds;
    }
}

static void fill_decp(DecP& p, const void* const* ptrs, long long ldx, long long ld_amix, int B, int G, int HD, int P, int S,
                      float scale, const float* zzb, long long ld_zzb, int kmix) {
    p.X = ptrs[0]; p.rows = (const int*)ptrs[1]; p.amix = (const float*)ptrs[2]; p.wfold = (const float*)ptrs[3];
    p.wm = (const float*)ptrs[4]; p.bm = (const float*)ptrs[5]; p.genec = (const float*)ptrs[6]; p.lib = (const float*)ptrs[7];
    p.part_stats = (float*)ptrs[8]; p.rowc = (float*)ptrs[9]; p.pi = (float*)ptrs[10]; p.part_nb = (float*)ptrs[11];
    p.dyp = (float*)ptrs[12]; p.dys = (float*)ptrs[13]; p.dpi = (float*)ptrs[14]; p.colpart = (float*)ptrs[15];
    p.ldx = ldx; p.ld_amix = ld_amix; p.B = B; p.G = G; p.HD = HD; p.P = P; p.S = S; p.scale = scale;
    p.pi_ready = 0; p.dpi_bf16 = nullptr; p.ld_dpi_bf16 = 0;
    for (float*& o : p.eo) o = nullptr;
    p.ld_out = 0;
    p.zz = zzb ? zzb : p.amix + HD;
    p.ld_zz = zzb ? ld_zzb : ld_amix;
    p.kmix = kmix > 0 ? kmix : HD + P + S;
}

// ptrs (SPV_DEC_NPTR = 17): X, rows, amix, wfold, wm, bm, genec, lib, part_stats, rowc, pi, part_nb, dyp, dys, dpi,
// colpart, rec.   Forward: rec[b], rowc and pi are produced.
extern "C" int spv_dec_nb_fwd(int src, const void* const* ptrs, long long ldx, long long ld_amix, int B, int G, int HD, int P,
                              int S, int phases, const float* zzb, long long ld_zzb, int kmix, void* stream) {
    if (!ptrs || (phases & 3) == 0 || B <= 0 || G <= 0 || HD < 0 || P <= 0 || S <= 0) return SPV_ERR_ARG;
    const int need[] = {0, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 16};
    for (int i : need)
        if (!ptrs[i]) return SPV_ERR_ARG;
    DecP p;
    fill_decp(p, ptrs, ldx, ld_amix, B, G, HD, P, S, 0.0f, zzb, ld_zzb, kmix);
    p.pi_ready = (phases & 4) ? 1 : 0;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dim3 grid((G + GT_BN - 1) / GT_BN, (B + GT_BM - 1) / GT_BM);
    const int nTG = grid.x;
    if (src != SPV_SRC_U16_LOG1P && src != SPV_SRC_F32_LOG1P) return SPV_ERR_ARG;
    if (phases & 1) {  // gene-axis softmax normalisers
        if (src == SPV_SRC_U16_LOG1P) dec_tile_kernel<PASS_STATS, SPV_SRC_U16_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
        else dec_tile_kernel<PASS_STATS, SPV_SRC_F32_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
        SPV_CHECK_LAUNCH();
        rowstat_kernel<<<(B + 7) / 8, 256, 0, st>>>(p.part_stats, nTG, B, p.lib, p.rowc, nullptr);
        SPV_CHECK_LAUNCH();
    }
    if (phases & 2) {  // mixture GEMM + NB log-likelihood
        if (src == SPV_SRC_U16_LOG1P) dec_tile_kernel<PASS_NB, SPV_SRC_U16_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
        else dec_tile_kernel<PASS_NB, SPV_SRC_F32_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
        SPV_CHECK_LAUNCH();
        rownb_kernel<<<(B + 7) / 8, 256, 0, st>>>(p.part_nb, nTG, B, p.rowc, (float*)ptrs[16]);
        SPV_CHECK_LAUNCH();
    }
    return SPV_OK;
}

// Element pass: the per-element outputs of phase 2, stored into `outs` (a HOST array of 5 device pointers [B, ld_out], NULL = not
// written: ll, rate_p, rate_s, pi, mean) after phase 1 has left the normalisers in rowc.  pi_ready: the mixture logits are in
// ptrs[10] (tensor-core GEMM), else they are computed here.  src SPV_SRC_F32 reads ptrs[0] as target values (no log1p).
extern "C" int spv_dec_nb_elems(int src, const void* const* ptrs, long long ldx, long long ld_amix, int B, int G, int HD, int P,
                                int S, int pi_ready, const float* zzb, long long ld_zzb, int kmix, void* const* outs,
                                long long ld_out, void* stream) {
    if (!ptrs || !outs || B <= 0 || G <= 0 || HD < 0 || P <= 0 || S <= 0 || ld_out < G) return SPV_ERR_ARG;
    if (src != SPV_SRC_F32 && src != SPV_SRC_U16_LOG1P && src != SPV_SRC_F32_LOG1P) return SPV_ERR_ARG;
    const int need[] = {2, 3, 5, 6, 9};
    for (int i : need)
        if (!ptrs[i]) return SPV_ERR_ARG;
    if (pi_ready ? !ptrs[10] : !ptrs[4]) return SPV_ERR_ARG;
    bool any = false;
    for (int o = 0; o < 5; ++o) any = any || outs[o] != nullptr;
    if (!any || (outs[0] && !ptrs[0])) return SPV_ERR_ARG;
    DecP p;
    fill_decp(p, ptrs, ldx, ld_amix, B, G, HD, P, S, 0.0f, zzb, ld_zzb, kmix);
    p.pi_ready = pi_ready ? 1 : 0;
    for (int o = 0; o < 5; ++o) p.eo[o] = reinterpret_cast<float*>(outs[o]);
    p.ld_out = ld_out;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dim3 grid((G + GT_BN - 1) / GT_BN, (B + GT_BM - 1) / GT_BM);
    if (src == SPV_SRC_F32) dec_tile_kernel<PASS_ELEM, SPV_SRC_F32><<<grid, GT_THREADS, 0, st>>>(p);
    else if (src == SPV_SRC_U16_LOG1P) dec_tile_kernel<PASS_ELEM, SPV_SRC_U16_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
    else dec_tile_kernel<PASS_ELEM, SPV_SRC_F32_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}

__global__ void colpart_reduce_kernel(const float* __restrict__ colpart, int nTB, int G, float* __restrict__ colsum) {
    long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (i >= 4L * G) return;
    float s = 0.0f;
    for (int t = 0; t < nTB; ++t) s += colpart[(long)t * 4 * G + i];
    colsum[i] = s;
}

// Backward sweep: writes dyp, dys, dpi [B, G] (gradients w.r.t. the two BatchNorm outputs and the mixture logits)
// and colsum [4, G] = column sums of dyp, dys, dpi and d loss / d theta.   scale = -grad_scale / B.
extern "C" int spv_dec_nb_bwd(int src, const void* const* ptrs, long long ldx, long long ld_amix, int B, int G, int HD, int P,
                              int S, float scale, float* colsum, void* dpi_bf16, long long ld_dpi_bf16, const float* zzb,
                              long long ld_zzb, int kmix, void* stream) {
    if (!ptrs || !colsum || B <= 0 || G <= 0 || HD < 0 || P <= 0 || S <= 0) return SPV_ERR_ARG;
    const int need[] = {0, 2, 3, 6, 7, 9, 10, 12, 13, 15};
    for (int i : need)
        if (!ptrs[i]) return SPV_ERR_ARG;
    if (!ptrs[14] && !dpi_bf16) return SPV_ERR_ARG;
    DecP p;
    fill_decp(p, ptrs, ldx, ld_amix, B, G, HD, P, S, scale, zzb, ld_zzb, kmix);
    p.dpi_bf16 = reinterpret_cast<__nv_bfloat16*>(dpi_bf16);
    p.ld_dpi_bf16 = ld_dpi_bf16;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dim3 grid((G + GT_BN - 1) / GT_BN, (B + GT_BM - 1) / GT_BM);
    if (src == SPV_SRC_U16_LOG1P) dec_tile_kernel<PASS_BWD, SPV_SRC_U16_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
    else if (src == SPV_SRC_F32_LOG1P) dec_tile_kernel<PASS_BWD, SPV_SRC_F32_LOG1P><<<grid, GT_THREADS, 0, st>>>(p);
    else return SPV_ERR_ARG;
    SPV_CHECK_LAUNCH();
    colpart_reduce_kernel<<<(4 * G + 255) / 256, 256, 0, st>>>(p.colpart, grid.y, G, colsum);
    SPV_CHECK_LAUNCH();
    return SPV_OK;
}
