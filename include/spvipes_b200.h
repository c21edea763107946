/* spvipes_b200 — C ABI of the B200-native spVIPES training hot path.
 *
 * The reference (nrclaudio/spVIPES) is pure Python/PyTorch and has no FFI of its own; these entry points are what a
 * binding for its per-minibatch path (spVIPESmodule inference -> generative -> loss, forward and backward) binds instead
 * of the ATen library calls listed in SURVEY.md section 2.2.  Each function cites the reference code it replaces.
 *
 * Conventions: every pointer is a DEVICE pointer unless said otherwise; matrices are row-major with an explicit leading
 * dimension in elements; `stream` is a cudaStream_t passed as void*; functions only enqueue work (no allocation, no
 * synchronisation, CUDA-graph capturable) and return SPV_OK (0) or a negative error code.  `rows` arguments are optional
 * row-gather indices into a device-resident count matrix (the minibatch), NULL meaning rows 0..B-1.
 */
#ifndef SPVIPES_B200_H
#define SPVIPES_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define SPV_ABI_VERSION 1

/* error codes */
#define SPV_OK 0
#define SPV_ERR_ARG -1
#define SPV_ERR_LAUNCH -2
#define SPV_ERR_ARCH -3

/* operand source kinds (srcA / srcB / src arguments) */
#define SPV_SRC_F32_ 0       /* float values                                                       */
#define SPV_SRC_U16_LOG1P_ 1 /* uint16 counts, consumed as log(1 + x)  (module/spVIPESmodule.py:432-433) */
#define SPV_SRC_F32_LOG1P_ 2 /* float counts,  consumed as log(1 + x)                                */

/* PoE modes (module/spVIPESmodule.py:484-509) and partner codes */
#define SPV_POE_LABEL_ 0
#define SPV_POE_PAIRED_ 1
#define SPV_POE_CLUSTER_ 2

int spv_abi_version(void);
/* kernels launched (or captured) by this library so far in this process; host-side counter */
long long spv_launch_count(void);
/* 0 if device `dev` is sm_100 (B200), SPV_ERR_ARCH otherwise, SPV_ERR_LAUNCH if no CUDA device. Host-side query. */
int spv_arch_check(int dev);

/* host -> device copy (cudaMemcpy2DAsync; asynchronous when the host matrix is pinned) of `rows` rows of `width` bytes from a
 * host matrix with row pitch `spitch` into a device buffer with row pitch `dpitch`: one group's own gene columns out of the
 * scvi minibatch matrix X [B, G0 + G1] (module/spVIPESmodule.py:428-430).  src is a HOST pointer. */
int spv_copy2d_h2d(void* dst, long long dpitch, const void* src, long long spitch, long long width, long long rows, void* stream);

/* C[b] (+)= act(op(A[b]) op(B[b]) + bias[b]) in fp32, batched over `batch` (element strides sA/sB/sC/sBias), optional
 * split-K (`ws` holds batch*splits*M*N floats).  transA: A stored [K][M]; transB: B stored [N][K] (y = x W^T).
 * accumulate: 0 = overwrite, 1 = add the result to C, 2 = C holds a PRE-activation addend (C <- act(A B + C + bias)).
 * Replaces nn.Linear forward/backward GEMMs: nn/networks.py:119-125 (Encoder), :314-325 (decoder, scvi FCLayers). */
int spv_gemm(int srcA, int transA, int srcB, int transB, const void* A, long long lda, const int* rowsA, const void* B,
             long long ldb, const int* rowsB, float* C, long long ldc, int M, int N, int K, int batch, long long sA,
             long long sB, long long sC, const float* bias, long long sBias, int relu, int accumulate, int splits, float* ws,
             void* stream);
/* spv_gemm with fused epilogue stages, applied after bias / ReLU / accumulate to element (m, n') of the full output
 * (n' = batch * sC + n): gate_y != NULL: multiply by (gate_y[m, n'] > 0 ? (gate_mask ? gate_mask[m, n'] : gate_scale) : 0)
 * (ReLU [+ dropout] backward, nn/networks.py:119-125 reversed); drop_mask / drop_p > 0: dropout forward with an explicit
 * multiplier matrix or the Philox keep mask of spv_dropout (seed, stream id, *drop_step, index m * drop_ld + n');
 * c_bf16 != NULL: also store the result as bf16 (operand of the tensor-core weight-gradient GEMM), c_bf16_lo (optional): its
 * bf16 residual bf16(v - hi) for the split-operand GEMM.  The fused stages
 * exist in the whole-K kernel only (fp32 operands, A not transposed, no row gather, K <= 256, splits == 1); -1 otherwise. */
int spv_gemm_fused(int srcA, int transA, int srcB, int transB, const void* A, long long lda, const int* rowsA, const void* B,
                   long long ldb, const int* rowsB, float* C, long long ldc, int M, int N, int K, int batch, long long sA,
                   long long sB, long long sC, const float* bias, long long sBias, int relu, int accumulate, int splits,
                   float* ws, const float* gate_y, long long ld_gate, const float* gate_mask, long long ld_mask,
                   float gate_scale, float drop_p, const float* drop_mask, unsigned long long drop_seed,
                   unsigned int drop_stream, const int* drop_step, long long drop_ld, void* c_bf16, void* c_bf16_lo,
                   long long ld_cbf16, void* stream);

/* bf16 tensor-core GEMM (tcgen05.mma, TMEM accumulator, TMA-fed): C[M,N] (+)= act(A B^T + bias), fp32 output.
 * a_mn = 0: A stored [M][K], 1: A stored [K][M];  b_mn = 0: B stored [N][K], 1: B stored [K][N]; lda / ldb in bf16
 * elements, multiples of 8, bases 16-byte aligned.  Same call sites as spv_gemm, for the "bf16 tensor-core path". */
int spv_tc_gemm(int a_mn, int b_mn, const void* A, long long lda, const void* B, long long ldb, float* C, long long ldc, int M,
                int N, int K, const float* bias, int relu, int accumulate, int splits, float* ws, void* stream);
/* general form of spv_tc_gemm: fmt 0 = bf16 operands, 3 = fp16 operands (mixed formats trap on sm_100: SPV_ERR_ARG);
 * C (+)= act(alpha * A B^T + bias) */
int spv_tc_gemm_ex(int fmt, float alpha, int a_mn, int b_mn, const void* A, long long lda, const void* B, long long ldb, float* C,
                   long long ldc, int M, int N, int K, const float* bias, int relu, int accumulate, int splits, float* ws,
                   void* stream);
/* the same with split-bf16 operands x ~ hi + lo (lo = bf16(x - hi), same layout and pitch as hi): hi.hi + hi.lo + lo.hi on
 * tcgen05 into one TMEM accumulator, ~16 mantissa bits per operand.  The K = genes contractions of the encoder's first layer
 * (nn/networks.py:119 forward and its weight gradient): north_star's 1e-3 gate on the latent statistics holds on this path. */
int spv_tc_gemm_split(int a_mn, int b_mn, const void* A, const void* A_lo, long long lda, const void* B, const void* B_lo,
                      long long ldb, float* C, long long ldc, int M, int N, int K, const float* bias, int relu, int accumulate,
                      int splits, float* ws, void* stream);
/* bf16 staging of GEMM operands: dst[r, :C] = bf16(src[r, :C]), zero padded up to ld_dst */
int spv_to_bf16(const float* src, long long ld_src, void* dst, long long ld_dst, int R, int C, void* stream);
/* fp16 staging (decoder operands of the fused tensor-core path) */
int spv_to_f16(const float* src, long long ld_src, void* dst, long long ld_dst, int R, int C, void* stream);
/* ... as a (hi, lo) pair for spv_tc_gemm_split */
int spv_to_bf16_split(const float* src, long long ld_src, void* dst_hi, void* dst_lo, long long ld_dst, int R, int C, void* stream);
/* T[b, :G] = bf16(log1p(X[rows[b], :G])), zero padded to ld_dst (a multiple of 8)   module/spVIPESmodule.py:428-433;
 * dst_lo (optional): the bf16 residual plane for spv_tc_gemm_split;
 * lib (optional, [B]): library size log(sum_g log1p(x[b,g])) from the same pass   module/spVIPESmodule.py:433-435 */
/* cov (optional, [B] batch codes) / n_cov: columns G .. G + n_cov of dst receive the one-hot batch code (batch covariates
 * appended to the encoders' input, nn/networks.py:110-118); they do not enter the library size */
int spv_counts_to_bf16(int src, const void* X, long long ldx, const int* rows, void* dst, void* dst_lo, long long ld_dst, int B,
                       int G, float* lib, const int* cov, int n_cov, void* stream);
/* minibatch gather from a device-resident CSR count matrix [N, G]: indptr int64 [N + 1], indices uint16 [nnz] (canonical: no
 * column twice in a row), values [nnz] uint16 (src = SPV_SRC_U16_LOG1P) or float (SPV_SRC_F32_LOG1P).  xs[b, :] = dense row
 * rows[b] (rows NULL: b) in the dtype of `values`, zero padded to the next 16-byte boundary; ld_xs >= G, a multiple of 8 (uint16)
 * resp. 4 (float), xs 16-byte aligned.  dst != NULL: also T / T_lo / lib / covariate columns exactly as spv_counts_to_bf16 on
 * the gathered rows (bit-identical to it on a 16-byte aligned dense row; ld_dst a multiple of 8); dst == NULL: xs only (lib and
 * cov unused).  G <= spv_csr_max_genes(src): the row is assembled in shared memory (65536 for uint16, the range of the column
 * index; 58104 for float, 227 KB).  Host-side query. */
int spv_csr_max_genes(int src);
int spv_csr_gather(int src, const long long* indptr, const unsigned short* indices, const void* values, const int* rows, int B,
                   int G, void* xs, long long ld_xs, void* dst, void* dst_lo, long long ld_dst, float* lib, const int* cov,
                   int n_cov, void* stream);

/* batch covariates (n_batch > 1; nn/utils.py:9-13, scvi FCLayers inject_covariates).  spv_one_hot: out[b, 0:nb] = one_hot(code[b]).
 * spv_cov_expand: zzb[b] = [zz[b, 0:P] | oh | zz[b, P:P+S] | oh] (the inputs of the two factor regressors, whose weights are
 * [G, P + nb] and [G, S + nb]) and oh_tail[b, 0:nb] = oh (optional: the covariate columns behind [hm | zz] in the mixing net's
 * input).  spv_cov_compact: the reverse selection for gradients (covariate columns dropped), plus an optional addend
 * add[b, 0 : P + S] (the mixture layer's input gradient, which has the plain [zz] layout). */
int spv_one_hot(const int* code, float* out, long long ld, int B, int nb, void* stream);
int spv_cov_expand(const float* zz, long long ld_zz, const int* code, float* zzb, long long ld_zzb, float* oh_tail, long long ld_oh,
                   int B, int P, int S, int nb, void* stream);
int spv_cov_compact(const float* dzzb, long long ld_in, float* dzz, long long ld_out, int B, int P, int S, int nb, const float* add,
                    long long ld_add, void* stream);

/* lib[b] = log(sum_g log1p(x[b,g]))   module/spVIPESmodule.py:433-435 */
int spv_library_size(int src, const void* X, long long ldx, const int* rows, int B, int G, float* lib, void* stream);

/* h *= mask (explicit multipliers) or a Philox keep-mask scaled by 1/(1-p)   nn/networks.py:121 */
int spv_dropout(float* h, long long ld, int B, int C, const float* mask, long long ldm, float p, unsigned long long seed,
                unsigned int stream_id, const int* step, void* stream);
/* dy <- y > 0 ? dy * (mask ? mask : scale) : 0   (ReLU + dropout backward) */
int spv_relu_bwd(float* dy, long long lddy, const float* y, long long ldy, int B, int C, const float* mask, long long ldm,
                 float scale, void* stream);

/* BatchNorm1d over the minibatch (training: batch statistics + running-stat update; eval: running statistics).
 * nn/networks.py:74-83 (eps 1e-5, momentum 0.1) and scvi FCLayers (eps 1e-3, momentum 0.01). */
int spv_bn_fwd(const float* x, long long ldx, float* y, long long ldy, int B, int C, const float* gamma, const float* beta,
               float eps, float momentum, float* running_mean, float* running_var, float* save_mean, float* save_invstd,
               int training, int relu, void* stream);
int spv_bn_bwd(const float* dy, long long lddy, const float* x, long long ldx, const float* y_relu, long long ldy, float* dx,
               long long lddx, int B, int C, const float* gamma, const float* save_mean, const float* save_invstd,
               float* dgamma, float* dbeta, void* stream);
int spv_colsum(const float* x, long long ldx, int B, int C, float* out, void* stream);

/* label-rank pairing, bit-exact integer contract   module/spVIPESmodule.py:599-659, 685-701, 297-326.
 * rows_a / rows_b (optional): the minibatch's labels are la[rows_a[i]] / lb[rows_b[i]] (gather from per-cell arrays). */
int spv_pair_label(const int* la, const int* lb, const int* rows_a, const int* rows_b, int Ba, int Bb, int* pa, int* pb,
                   void* stream);
/* sub = T[idx0][:, idx1]   :474-482 ;  row/col argmax (ties -> first)   :526-527 */
int spv_plan_gather(const float* T, long long ldT, const int* idx0, const int* idx1, int B0, int B1, float* sub, void* stream);
/* ... from a plan stored as bf16 (halves the residency of a large plan; cluster mode) */
int spv_plan_gather_bf16(const void* T, long long ldT, const int* idx0, const int* idx1, int B0, int B1, float* sub, void* stream);
/* NaN entries compare greater than any number and the first one wins, as torch.argmax */
int spv_plan_argmax(const float* sub, int B0, int B1, int* row_arg, int* col_arg, void* stream);
/* masked row-normalised sub-plans of the cluster mode   :207-219 */
int spv_plan_cluster_norm(const float* sub, int B0, int B1, const int* l0, const int* l1, float* P1, float* P2, void* stream);

/* PoE merge + reparameterised sampling + KL terms, both groups in one launch.
 * ptrs per group (SPV_POE_FWD_NPTR): own_loc, own_lv, oth_loc, oth_lv, stats, partner, eps_p, eps_q, zpriv, poe_loc,
 * poe_lv, poe_scale, zpoe, klp, klq, zz ;  lds per group: ld_own, ld_oth, ld_stats, ld_zz.
 * module/spVIPESmodule.py:282-379, 511-581, 583-718, 841-868; nn/networks.py:125-127. */
#define SPV_POE_FWD_NPTR 16
int spv_poe_fwd(int mode, int S, int P, int B0, int B1, const void* const* ptrs0, const long long* lds0,
                const void* const* ptrs1, const long long* lds1, unsigned long long seed, const int* step, void* stream);
/* ptrs per group (SPV_POE_BWD_NPTR): own_loc, own_lv, oth_loc, oth_lv, stats, partner, eps_p, eps_q, dzz, dstats, g_own,
 * g_contrib, out ;  lds per group: ld_own, ld_oth, ld_stats, ld_dzz, ld_dstats, ld_out */
#define SPV_POE_BWD_NPTR 13
int spv_poe_bwd(int mode, int S, int P, int B0, int B1, const void* const* ptrs0, const long long* lds0,
                const void* const* ptrs1, const long long* lds1, unsigned long long seed, const int* step,
                const float* kl_weight, float inv_batch, void* stream);
/* out[0] = loss (:886-893), out[1..4] = mean KL private0, poe0, private1, poe1 (:870-875), out[5..6] = mean rec0, rec1 */
int spv_loss(const float* rec0, const float* rec1, const float* klp0, const float* klq0, const float* klp1, const float* klq1,
             int B, const float* kl_weight, float* out, void* stream);
/* one evaluation pass added to a float64 accumulator acc[8] (validation epochs, get_elbo); the groups may differ in size:
 * acc[0..5] += sum rec0, sum rec1, sum klp0, sum klq0, sum klp1, sum klq1 (each group over its own B_g cells, fp32 sums),
 * acc[6] += B0 (n_obs), acc[7] += sum rec0 + sum rec1 + (*kl_weight) * (sum of the four KL sums).  One CTA, graph-capturable */
int spv_elbo_accumulate(const float* rec0, const float* rec1, const float* klp0, const float* klq0, const float* klp1,
                        const float* klq1, int B0, int B1, const float* kl_weight, double* acc, void* stream);

/* decoder: closed-form per-gene BatchNorm fold + NB constants.
 * ptrs (18): Wp, Ws, gamma_p, beta_p, gamma_s, beta_s, px_r, rm_p, rv_p, rm_s, rv_s, zz, zsum, scratch [ceil(B/64), (P+S) + (P+S)^2]
 * (used when B > 512), wfold, genec,
 * zmean, zcov.  training != 0: zsum / zmean / zcov [P+S], [P+S], [P+S, P+S] are OUTPUTS (column sums, mean and biased
 * covariance of the latent minibatch zz [B, P+S], one cluster launch).   nn/networks.py:314-320, scvi FCLayers;
 * module/spVIPESmodule.py:758 */
#define SPV_DEC_GENEC_ROWS 19
/* wz_bf16 (optional): rows [Gp, 3 Gp) of the stacked bf16 tensor-core operand [3 Gp, ld_wz] (rows [0, G): mixture weight,
 * [Gp, Gp + G): folded private weights in the latent columns HD .., [2 Gp, 2 Gp + G): folded shared weights) - the B operand
 * of the input-gradient GEMM of the two branches; written as FP16 when wz_f16 / zc_f16 are given (the fused tensor-core
 * decoder runs on fp16 operands throughout), else as bf16.
 * wz_f16 / zc_f16 (optional, both or none): fp16 operands of the branch-logit MMAs of the tensor-core sweeps: wz_f16
 * [2 Gp, 64] folded weights (private rows, columns [0, P); shared rows from Gp, columns [P, P + S)), zc_f16 [B, 64] the
 * CENTRED latents zz - mean(zz) (eval mode: zz); genec rows GC_CPLC / GC_CSLC hold the matching shifts. */
int spv_dec_fold(const void* const* ptrs, long long ld_zz, int B, int G, int P, int S, int training, float eps, float momentum,
                 void* wz_bf16, long long ld_wz, int Gp, int HD, void* wz_f16, void* zc_f16, void* stream);
/* fused decoder + NB-mixture likelihood sweeps.  ptrs (SPV_DEC_NPTR): X, rows, amix, wfold, wm, bm, genec, lib, part_stats,
 * rowc, pi, part_nb, dyp, dys, dpi, colpart, rec, tgf, tb1 (the last two: spv_dec_theta_tables, tensor-core sweeps only;
 * tb1 only for the training sweep).
 * nn/networks.py:314-325; module/spVIPESmodule.py:759, 817-824 */
#define SPV_DEC_NPTR 19
/* phases: bit 0 = gene-axis softmax normaliser sweep, bit 1 = mixture GEMM + NB log-likelihood sweep (3 = both),
 * bit 2 = the mixture logits are already in `pi` (written by spv_tc_gemm), skip the in-kernel fp32 GEMM */
/* zzb (optional, [B, P + S] with row pitch ld_zzb): the inputs of the two factor regressors when they are not the latent columns
 * of amix (batch covariates: P and S then include the covariate columns, spv_cov_expand); kmix (0 = HD + P + S): width of the
 * mixing net's input amix / of a row of wm. */
int spv_dec_nb_fwd(int src, const void* const* ptrs, long long ldx, long long ld_amix, int B, int G, int HD, int P, int S,
                   int phases, const float* zzb, long long ld_zzb, int kmix, void* stream);
int spv_dec_nb_bwd(int src, const void* const* ptrs, long long ldx, long long ld_amix, int B, int G, int HD, int P, int S,
                   float scale, float* colsum, void* dpi_bf16, long long ld_dpi_bf16, const float* zzb, long long ld_zzb, int kmix,
                   void* stream);
/* tensor-core version of phase 2 of spv_dec_nb_fwd: the mixture GEMM and the two softmax-branch logit GEMMs on tcgen05
 * (operands via TMA, fp32 accumulators in TMEM) with the NB-mixture log-likelihood fused into the TMEM epilogue.
 * amix_bf16 [B, ld_amixb] = [hm | zz] and wstack_bf16 [>= G, ld_w] (the mixture weight) hold FP16 values (spv_to_f16 /
 * spv_adam staging; the parameter names predate the switch); zc_f16 [B, 64], wz_f16 [2 Gp, 64]: the fp16 branch operands
 * written by spv_dec_fold.  part_nb (ptrs[11]) needs spv_dec_nb_part_floats(B, G) floats.
 * store_pi must be 0 (any other value: SPV_ERR_ARG): the mixture logits stay in tensor memory. */
int spv_dec_nb_fwd_tc(int src, const void* const* ptrs, long long ldx, const void* amix_bf16, long long ld_amixb,
                      const void* wstack_bf16, long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, int B, int G,
                      int HD, int P, int S, int store_pi, int kmix, void* stream);
/* per-element outputs of the likelihood sweeps (scvi NegativeBinomialMixture: px.log_prob, mu1, mu2, mixture_logits, mean),
 * stored instead of reduced.  outs: HOST array of 5 device pointers, each [B, ld_out] fp32 row-major or NULL (not written):
 *   outs[0] ll      log_mixture_nb(t; rate_p, rate_s, theta, pi) per element (eps 1e-8), t = log1p(count) or, for src
 *                   SPV_SRC_F32, the value in ptrs[0] as given (px.log_prob(value))
 *   outs[1] rate_p  exp(lib) softmax_g(BN_p(z_private_arg Wp^T))          (px_rate_private)
 *   outs[2] rate_s  exp(lib) softmax_g(BN_s(z_shared_arg Ws^T))           (px_rate_shared)
 *   outs[3] pi      mixing logit, bias included                           (px_mixing)
 *   outs[4] mean    sigmoid(pi) rate_p + (1 - sigmoid(pi)) rate_s
 * Counts / targets (ptrs[0], ptrs[1]) and the count table are read only when outs[0] is requested.  module/spVIPESmodule.py:751-759
 * spv_dec_nb_elems_tc: the element sweep of spv_dec_nb_fwd_tc (same operands, state of the same pass; part_nb unused).
 * spv_dec_nb_elems: the element pass of spv_dec_nb_fwd's phase 2, after phase 1 (rowc); pi_ready: the mixture logits are in
 * ptrs[10] (spv_tc_gemm) - else the pass computes them from amix / wm as phase 2 does. */
int spv_dec_nb_elems_tc(int src, const void* const* ptrs, long long ldx, const void* amix_bf16, long long ld_amixb,
                        const void* wstack_bf16, long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, int B, int G,
                        int HD, int P, int S, int kmix, void* const* outs, long long ld_out, void* stream);
int spv_dec_nb_elems(int src, const void* const* ptrs, long long ldx, long long ld_amix, int B, int G, int HD, int P, int S,
                     int pi_ready, const float* zzb, long long ld_zzb, int kmix, void* const* outs, long long ld_out, void* stream);
/* count draws from the NB mixture (scvi NegativeBinomialMixture.sample, theta2 = None), per element and draw:
 *   mu = rate_p if Bernoulli(sigmoid(pi)) else rate_s;  lam = min(Gamma(theta, rate theta / mu), 1e8);  count = Poisson(lam)
 * (0 where mu = 0).  Draws d = draw0 .. draw0 + n_draws - 1 go to out + (d - draw0) * draw_pitch, each [B, ld_out] fp32 row-major
 * (draw_pitch >= (B - 1) * ld_out + G unless n_draws = 1).  A draw is a function of (seed, group, d, row b of the minibatch,
 * gene g) only; group in [0, 127], draw0 + n_draws <= 2^32.  The counters are disjoint from those of the reparameterisation noise
 * and the dropout masks under the same seed.
 * spv_dec_nb_sample_tc: the tensor-core sampling sweep on the operands of spv_dec_nb_elems_tc (state of the same pass; counts,
 * count table and part_nb unused); rate_p, rate_s and pi are those spv_dec_nb_elems_tc writes and are not stored.
 * spv_nb_mixture_sample: the same draws from given parameters mu1 = rate_p, mu2 = rate_s, pi ([B, ld_in] fp32 each) and
 * theta [G] (exp(px_r)); bitwise equal to the sweep's on the sweep's own rates. */
int spv_dec_nb_sample_tc(const void* const* ptrs, const void* amix_bf16, long long ld_amixb, const void* wstack_bf16, long long ld_w,
                         int Gp, const void* zc_f16, const void* wz_f16, int B, int G, int HD, int P, int S, int kmix,
                         unsigned long long seed, int group, unsigned int draw0, int n_draws, float* out, long long ld_out,
                         long long draw_pitch, void* stream);
int spv_nb_mixture_sample(const float* mu1, const float* mu2, const float* pi, long long ld_in, const float* theta, int B, int G,
                          int n_draws, float* out, long long ld_out, long long draw_pitch, unsigned long long seed, int group,
                          unsigned int draw0, void* stream);
/* tensor-core version of phase 1 of spv_dec_nb_fwd: softmax normalisers rowc[b, 0:2] = lib[b] - logsumexp_g(y_p), (y_s)
 * from the fp16 branch operands (spv_dec_fold); part_stats: scratch of 2 * ceil(G/64) * B * 4 floats.
 * nn/networks.py:318-320, module/spVIPESmodule.py:751-757 */
int spv_dec_stats_tc(void* zc_f16, const void* wz_f16, int Gp, const float* genec, const float* lib, float* part_stats,
                     float* rowc, int B, int G, int P, int S, void* stream);
/* count tables of the tensor-core likelihood sweeps (csrc/decoder_common.cuh NB_TAB = 16 entries per gene):
 * tgf [G, 16] float2: tgf[g][c] = (log1p(c), lgamma(log1p(c) + theta_g) - lgamma(theta_g) - lgamma(log1p(c) + 1)),
 * tb1 [G, 16] float: tb1[g][c] = digamma(log1p(c) + theta_g) - digamma(theta_g) (training sweep), theta = exp(px_r)
 * (module/spVIPESmodule.py:758).  They depend on the parameter only; either pointer may be NULL.  16-byte aligned. */
int spv_dec_theta_tables(const float* px_r, int G, void* tgf, float* tb1, void* stream);
/* floats spv_dec_nb_fwd_tc needs in part_nb (ptrs[11]) for a [B, G] problem */
long long spv_dec_nb_part_floats(int B, int G);
/* rec[b] (ptrs[16] of the forward) and the softmax-backward row sums rowc[:, 2:4] from the row partials part_nb that
 * spv_dec_nb_fwd_tc wrote for the same B, G, HD */
int spv_dec_nb_rowreduce(const float* part_nb, int G, int B, int HD, float* rowc, float* rec, void* stream);
/* ptrs (18): Wp, Ws, Qp, Qs, genec, colsum, zmean, zcov, dWp, dWs, dgamma_p, dbeta_p, dgamma_s, dbeta_s, dpx_r, dbm,
 * vpart [parts, P+S], mpart [parts, (P+S)^2] with parts = spv_dec_gene_bwd_parts(G)
 * (backward of nn/networks.py:314-320 through the folded BatchNorm) */
int spv_dec_gene_bwd_parts(int G);
int spv_dec_gene_bwd(const void* const* ptrs, long long ldq, int B, int G, int P, int S, int colsum_in_q, void* stream);
/* d zz = dmix (latent columns of d [hm | zz]; NULL = none) + dzraw (optional further addends [B, P+S]: softmax-branch and hidden-layer
 * input gradients when they are not in dmix) - BatchNorm coupling terms, the latter summed from the `nparts` per-CTA
 * partials (vpart [nparts, P+S], mpart [nparts, (P+S)^2]) that spv_dec_gene_bwd writes (its last two ptrs).
 * raw_colsum != NULL (tensor-core path; [P+S] column sums of dzraw, spv_colsum): the mean-coupling term is taken as the column
 * mean of dzraw itself instead of vpart, so that the coherent operand-rounding error of the GEMM that produced dzraw cancels
 * instead of surviving as a column mean. */
int spv_dec_dzz_combine(const float* dmix, long long ld_dmix, const float* dzraw, const float* vpart, const float* mpart,
                        int nparts, const float* zz, long long ld_zz, const float* zmean, float* dzz, int B, int P, int S,
                        const float* raw_colsum, void* stream);

/* *step += 1 on the stream: the optimiser's step count, and (a separate counter) the Philox stream position that the noise /
 * dropout kernels read - the two must not share a counter, the backward regenerates its noise from the forward's value. */
/* Adam with the scvi TrainingPlan defaults restated by the caller (training_mixin.py:93-111); *step is a device counter of
 * completed optimiser steps.  ticket == NULL: *step already holds this step's 1-based index (spv_adam_tick first);
 * ticket != NULL (zeroed device int): the launch uses *step + 1 and its last CTA stores it back.
 * nseg (<= 8) staging segments, host arrays: the parameter block [seg_begin, seg_begin + seg_rows * seg_cols) viewed as
 * [seg_rows, seg_cols] is also written, updated, as bf16 into seg_dst (row pitch seg_ld): the tensor-core operand copies of
 * the large weights, so that the next step does not start with conversion kernels; seg_dst_lo (optional array, entries may
 * be NULL): the bf16 residual plane of a segment (split-operand GEMM), same pitch; seg_f16 (optional array): non-zero = the
 * segment's destination holds fp16 values (decoder operands).  p, g, m, v 16-byte aligned.
 * max_blocks > 0 caps the grid (an update overlapped with other kernels should not occupy every SM). */
int spv_adam_tick(int* step, void* stream);
int spv_adam(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps, float wd,
             float grad_scale, int* step, int* ticket, int nseg, const long long* seg_begin, const int* seg_rows,
             const int* seg_cols, void* const* seg_dst, void* const* seg_dst_lo, const int* seg_f16, const long long* seg_ld,
             int max_blocks, void* stream);

/* TRAINING sweep of the tensor-core decoder + likelihood (csrc/nb_tc_train.cu): spv_dec_nb_fwd_tc's outputs (row partials ->
 * spv_dec_nb_rowreduce) plus everything the backward needs, so that a training step sweeps the [B, G] problem once:
 *   e4t  [Gp, ld_e4 >= 4 B] fp16, gene-major, per cell (ep, rp', es, rs'): the branch gradients without the softmax coupling
 *        and 4096 x the softmax values;  d ll / d y_p = ep - rp' Dp / 4096 (Dp = rowc[:, 2] once the row reduction has run)
 *   dpit [Gp, ld_dpi >= B] fp16: d ll / d pi
 *   ptrs[15] = colpart [ceil(B/128), 2, G]: per-row-tile column sums of d pi and d theta -> spv_dec_nb_train_colsum
 * ptrs as spv_dec_nb_fwd_tc plus [7] = lib, [18] = tb1 (spv_dec_theta_tables).  The buffers must be zero-initialised once (rows
 * >= G and cells >= B are never written); pitches multiples of 8.  Autograd of nn/networks.py:314-325 + scvi log_mixture_nb. */
int spv_dec_nb_train_tc(int src, const void* const* ptrs, long long ldx, const void* amix_f16, long long ld_amixb,
                        const void* wstack_f16, long long ld_w, int Gp, const void* zc_f16, const void* wz_f16, void* e4t,
                        long long ld_e4, void* dpit, long long ld_dpi, int B, int G, int HD, int P, int S, int kmix, void* stream);
/* colsum [2, G] = scale x column sums of (d ll / d pi, d ll / d theta) from colpart of spv_dec_nb_train_tc */
int spv_dec_nb_train_colsum(const float* colpart, int B, int G, float scale, float* colsum, void* stream);
/* zq [4 Bp, ldq] fp16, rows 4b .. 4b+3 = [zp 1 0 0], -Dp' [zp 1 0 0], [0 0 zs 1], -Ds' [0 0 zs 1] (zp / zs: the regressors' inputs
 * zb[b, 0:Pb] / zb[b, Pb:Pb+Sb], D' = rowc[b, 2 or 3] / 4096): E4T . zq = [Qp | colsum dyp | Qs | colsum dys] with the softmax
 * coupling applied */
int spv_dec_zq4(const float* zb, long long ld_zb, const float* rowc, void* zq, long long ldq, int B, int Pb, int Sb, void* stream);
/* out [B, Pb + Sb] = softmax-branch part of d zz from T [4 B, ld_t] = E4T^T [W'p | W's]: T[4b + k] - D' T[4b + k + 1] */
int spv_dec_dz4_combine(const float* T, long long ld_t, const float* rowc, float* out, long long ld_out, int B, int Pb, int Sb,
                        void* stream);

/* Data-parallel gradient all-reduce as ONE kernel per parameter range over NVLink 5 / NVSwitch, capturable inside the step's
 * CUDA graph (SURVEY.md section 8e; the reference is single-device).  In-place sum over ranks of floats
 * [offset, offset + n) of a gradient buffer that lives at the same offset of a symmetric allocation on every rank.
 * peer_bufs / peer_flags: HOST arrays of `world` device addresses (each rank's buffer / flag buffer as mapped into this
 * process; entry `rank` is the local one).  mc_buf: this rank's multicast (NVLS) address of the buffer - the switch then
 * reduces (multimem.ld_reduce) and replicates (multimem.st) - or NULL: peer loads summed in rank order + peer stores.
 * Rank r reduces slice r of the range and writes the sums into every rank's buffer, so all ranks end with bitwise
 * identical values.  CTA b of every rank handshakes with CTA b of every peer before (peers' gradients complete) and after
 * (all writes landed, all reads done) through release / acquire flags carrying an epoch; `state` = 12 ints on this device,
 * zeroed once (per channel: epoch, ticket; state[8] = 1 + rank of a peer that did not answer within 20 s, 0 = healthy: the
 * kernel then gives up instead of hanging the GPU); the flag buffer holds spv_xgpu_flag_ints() ints, zeroed on every rank before the
 * first launch anywhere.  channel 0..3: launches that may overlap in time use different channels.  Every rank must launch
 * the same (offset, n, channel, blocks) sequence per channel.  offset, n multiples of 4; buffers 16-byte aligned. */
int spv_xgpu_allreduce(void* const* peer_bufs, void* const* peer_flags, void* mc_buf, long long offset, long long n, int rank,
                       int world, int channel, int* state, int blocks, void* stream);
int spv_xgpu_flag_ints(void);

#ifdef __cplusplus
}
#endif
#endif /* SPVIPES_B200_H */
