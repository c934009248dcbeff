/* libhba — C-ABI of the B200 (sm_100a) CLIP-HBA-Behavior hot path.
 *
 * Every entry point is `extern "C"`, takes plain device pointers + sizes + a CUDA stream
 * (`cudaStream_t` passed as void*), is asynchronous and stream-ordered, performs no hidden
 * synchronisation or persistent device allocation, and is safe under CUDA-graph capture.
 * Return value: 0 = ok, negative = error (see HBA_ERR_*); the message is in hba_last_error().
 * The library never aborts the process and has NO CPU fallback.
 *
 * Reference interfaces replaced (paths relative to the reference repo):
 *   NEW  = Training/functions/new_cvpr_train_behavior_things_pipeline.py
 *   VIT  = Training/vit_training/baseline/train_vit_sgd.py
 *   TORCH= torch/nn/functional.py (multi_head_attention_forward, the code the reference reaches)
 */
#ifndef HBA_H_
#define HBA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HBA_OK 0
#define HBA_ERR_ARG (-22)         /* EINVAL: shape / alignment / null-pointer violation   */
#define HBA_ERR_CUDA (-5)         /* EIO:    a CUDA runtime / driver call failed          */
#define HBA_ERR_UNSUPPORTED (-38) /* ENOSYS: device is not sm_100 / feature not built     */

#define HBA_ABI_VERSION 1

/* thread-local message of the last failing call */
const char* hba_last_error(void);
int hba_abi_version(void);
/* 0 when the current CUDA device is compute capability 10.x, HBA_ERR_UNSUPPORTED otherwise */
int hba_device_check(void);

/* ------------------------------------------------------------------------------------------
 * tcgen05 / TMEM / TMA GEMM:   C[M,N] = epilogue( A[M,K] . B[N,K]^T )
 * Replaces every nn.Linear / in_proj / out_proj / conv1-as-GEMM of the un-vendored CLIP towers
 * reached through NEW:298 (F.linear at TORCH functional.py:6244 in_proj, :6690 out_proj) and the
 * timm ViT-B/16 linears of VIT:138-140.
 *   A, B are bf16, K-major (row-major [rows, ld]) by default; lda/ldb % 8 == 0.  With a_mn_major /
 *   b_mn_major the operand is stored [K, M] / [K, N] instead (MN-major UMMA descriptors), which gives
 *   dW = dY^T X and dX = dY W without any transposed copy.  Any K > 0: TMA zero-fills a ragged last
 *   k-block past K, except where the hi part of a K-major fp32-mode operand lies inside the tensor map - that
 *   hi part must be zero in columns [K, ceil64(K)), and its lo offset at least ceil64(K).
 *   nsplit == 1: plain bf16 product.
 *   nsplit == 3: "fp32 mode" — A and B each hold a hi part at column 0 and a lo part at column
 *     offset a_lo_off / b_lo_off (x ~= hi + lo, both bf16; the offset is at least ceil64(K) for a
 *     K-major operand, at least M resp. N for an MN-major one); the kernel accumulates
 *     hi.hi + lo.hi + hi.lo in fp32 (error ~2^-16 relative per product).
 * Epilogue, applied per element v = alpha * acc (+ bias[n]):
 *   pre_out (optional) receives v (the pre-activation, for the backward pass)
 *   act: HBA_ACT_*  (QuickGELU: NEW's CLIP MLP; GELU_ERF: timm ViT-B/16 MLP;
 *        *_GRAD multiply v by act'(aux[m,n]) for the backward pass)
 *   v += residual[m,n] (optional, fp32)
 *   out_f32 / out_bf16 (hi at column n, lo at column n + out_lo_off when out_lo_off > 0)
 *   transpose_out != 0 writes the outputs as [N, M] (ld* are then row strides of that layout);
 *     only alpha and bias apply in that mode (no act / residual / pre_out)
 * Scheduling (no effect on results): persistent CTA pairs, 256 x 256 tiles; the tiles of a partial last round are
 * cut into 2 or 4 column slabs when that shortens the round; every element still accumulates its K products
 * in the same order, so the output bits do not depend on M, on max_ctas or on the split.
 */
enum {
  HBA_ACT_NONE = 0,
  HBA_ACT_QUICKGELU = 1,
  HBA_ACT_GELU_ERF = 2,
  HBA_ACT_QUICKGELU_GRAD = 3,
  HBA_ACT_GELU_ERF_GRAD = 4
};
enum { HBA_DT_F32 = 0, HBA_DT_BF16 = 1 };

typedef struct hba_gemm_params {
  const void* A;
  const void* B;
  int32_t M, N, K;
  int32_t lda, ldb;
  int32_t nsplit;
  int32_t a_lo_off, b_lo_off;
  float alpha;
  const float* bias;     /* [N] or NULL */
  const float* residual; /* [M, ldr] fp32 or NULL */
  int32_t ldr;
  int32_t act;
  const void* aux; /* [M, ld_aux] pre-activation for *_GRAD; with ld_aux % 4 == 0 16-byte (f32) / 8-byte (bf16)
                      aligned */
  int32_t ld_aux;
  int32_t aux_dtype; /* HBA_DT_* */
  void* pre_out;     /* [M, ld_pre] or NULL */
  int32_t ld_pre;
  int32_t pre_dtype;
  float* out_f32; /* or NULL */
  int32_t ld_f32;
  void* out_bf16; /* or NULL */
  int32_t ld_bf16;
  int32_t out_lo_off;
  int32_t transpose_out;
  int32_t max_ctas; /* 0 = one persistent CTA per SM */
  int32_t a_mn_major; /* A stored as [K, lda] (M contiguous): C = A^T-layout product, no transpose pass */
  int32_t b_mn_major; /* B stored as [K, ldb] (N contiguous), e.g. dX = dY . W with W [out, in] as is */
  int32_t k_slices;   /* > 1: split-K for problems with few output tiles (weight gradients: K = rows of the batch;
                         the CLS / EOT row GEMMs, M = 32 / 66): every (tile, K slice) is a work item writing fp32
                         partial sums into k_workspace; the slices are summed in a fixed order (deterministic) by a
                         reduction that runs this struct's whole epilogue (bias, pre_out, act / aux, residual,
                         out_f32, out_bf16 hi / lo).  Needs k_workspace, N % 4 == 0, no transpose_out / colsum */
  float* k_workspace; /* >= k_slices * M * N floats, 16-byte aligned */
  float* colsum_partial; /* or NULL: [ceil(M / 32), N] fp32 receiving, per 32-row group, the column sums
                            of the bf16 output's hi part (in fp32 mode too: the lo part is not summed) - the
                            bias gradient of the previous Linear fused into the GEMM that produces its dY
                            (VIT:143); sum the groups with hba_colsum */
} hba_gemm_params;

int hba_gemm_bf16(const hba_gemm_params* p, void* stream);

/* fp32 [rows, cols] (ld_in) -> bf16 hi at column c, lo at column c + lo_off (lo_off == 0: hi only)
 * transpose != 0 writes out[c, r] instead (out is then [cols, ld_out]). Weight / operand staging. */
int hba_split_bf16(const float* in, int64_t rows, int64_t cols, int64_t ld_in, void* out,
                   int64_t ld_out, int64_t lo_off, int transpose, void* stream);

/* ------------------------------------------------------------------------------------------
 * LayerNorm (un-vendored CLIP ln_1/ln_2/ln_pre/ln_post/ln_final, eps 1e-5; timm eps 1e-6)
 * x [rows, ldx] fp32 -> y_f32 (optional) and y_bf16 hi/lo (optional), biased variance, fp32.
 * row_stride_sel: processes rows r*row_step (row_step > 1 selects e.g. the CLS row of each image)
 */
int hba_layernorm_fwd(const float* x, int64_t rows, int32_t cols, int64_t ldx, int64_t row_step,
                      const float* gamma, const float* beta, float eps, float* y_f32,
                      int64_t ld_yf, void* y_bf16, int64_t ld_yb, int64_t lo_off, void* stream);
/* dx[r,:] (+)= LN backward of dy through (x, gamma); accumulate != 0 adds into dx.
 * dy, dx fp32 with leading dims ld_dy, ld_dx; x rows taken at r*row_step */
int hba_layernorm_bwd(const float* dy, int64_t ld_dy, const float* x, int64_t rows, int32_t cols,
                      int64_t ldx, int64_t row_step, const float* gamma, float eps, float* dx,
                      int64_t ld_dx, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------
 * Patch embedding front end of the vision tower (un-vendored visual.conv1 + class/positional
 * embedding + ln_pre, reached via NEW:298).
 * im2col: image [B,3,H,W] fp32 NCHW -> patches [B*gh*gw, ld_out] bf16 hi/lo, column index
 *         = c*P*P + py*P + px (conv weight [width, 3, P, P] flattened), zero padded to ld.
 * assemble: x[b,0,:] = cls + pos[0]; x[b,1+p,:] = conv[b*np+p,:] + pos[1+p]; then ln_pre
 *           (gamma == NULL: no LayerNorm, the timm ViT-B/16 layout of VIT:283).
 */
int hba_im2col_patches(const float* image, int32_t B, int32_t H, int32_t W, int32_t P, void* out,
                       int64_t ld_out, int64_t lo_off, void* stream);
int hba_assemble_tokens_ln(const float* conv, int32_t B, int32_t n_patches, int32_t width,
                           const float* cls, const float* pos, const float* gamma,
                           const float* beta, float eps, float* x_out, void* stream);
/* text front end: x[s, t, :] = token_embedding[tokens[s,t]] + pos[t]  (fp32) */
int hba_embed_tokens(const int64_t* tokens, int32_t S, int32_t T, int32_t width,
                     const float* table, const float* pos, float* x_out, void* stream);
/* gather rows: out[i,:] = in[idx[i],:] (fp32), used for the EOT rows (text.argmax(-1)) */
int hba_gather_rows(const float* in, int64_t ld_in, const int64_t* idx, int32_t n, int32_t cols,
                    float* out, int64_t ld_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused softmax attention (F.multi_head_attention_forward -> SDPA, TORCH functional.py:6682).
 * qkv: [B*T, 3*H*64] (q | k | v column blocks, head h at columns h*64..), dtype HBA_DT_*.
 * out: [B*T, H*64] bf16 hi/lo (lo_off > 0 adds the lo part).  causal != 0 applies the CLIP text
 * mask (key j visible to query i iff j <= i).  head_dim is fixed at 64 (ViT-L/14, ViT-B/16, text).
 * q_rows_only_first != 0 computes query row 0 of every sequence only (CLS pruning); out is then
 * [B, H*64].
 */
int hba_attention_fwd(const void* qkv, int32_t qkv_dtype, int64_t ld_qkv, int32_t B, int32_t T,
                      int32_t H, int32_t causal, int32_t first_row_only, void* out, int64_t ld_out,
                      int64_t lo_off, float* out_f32, int64_t ld_of, void* stream);
/* backward for the CLS query row only (all that the pruned live sub-graph needs):
 * d_out [B, H*64] fp32 -> d_qkv [B*T, 3*H*64] fp32 (fully written: dq on row 0 of each sequence,
 * zeros on other rows; dk, dv on all rows). qkv as in the forward. */
int hba_attention_bwd_row0(const void* qkv, int32_t qkv_dtype, int64_t ld_qkv, int32_t B,
                           int32_t T, int32_t H, const float* d_out, int64_t ld_do, float* d_qkv,
                           int64_t ld_dqkv, void* stream);

/* ------------------------------------------------------------------------------------------
 * DoRA merge (DoRALayer.weight, NEW:447-463) and its backward (autograd of the same lines).
 *   V = D + scale * Bm @ A;  n_j = ||V[:,j]||_2 + eps;  Wt[i,j] = V[i,j] / n_j * m[j]
 *   D [in,out] fp32, A [r,out], Bm [in,r], m [out].
 * Outputs (each optional): w_t_f32 [in,out] (the reference's pre-transpose matrix; `.weight` is
 * its transposed view), w_bf16 [out, ld_w] hi/lo (GEMM B operand for y = x W^T), wt_bf16
 * [in, ld_wt] hi/lo (GEMM B operand for dX = dY W), norm_out [out] (= n_j, saved for backward).
 */
int hba_dora_merge_fwd(const float* D, const float* A, const float* Bm, const float* m,
                       int32_t in_f, int32_t out_f, int32_t r, float scale, float eps,
                       float* w_t_f32, void* w_bf16, int64_t ld_w, int64_t w_lo_off, void* wt_bf16,
                       int64_t ld_wt, int64_t wt_lo_off, float* norm_out, void* stream);
/* G = dL/dW given in [out, ld_g] layout (W = Wt^T).  Produces dm [out], dA [r,out], dB [in,r].
 * workspace: in_f*out_f floats (holds dV). */
int hba_dora_merge_bwd(const float* G, int64_t ld_g, const float* D, const float* A,
                       const float* Bm, const float* m, int32_t in_f, int32_t out_f, int32_t r,
                       float scale, float eps, float* dm, float* dA, float* dB, float* workspace,
                       void* stream);

/* ------------------------------------------------------------------------------------------
 * Cosine-logit head (un-vendored CLIP.forward tail; contract NEW:298-300) + nn.MSELoss
 * (BDRV:31 applied at NEW:994):
 *   pred[b,c] = exp(logit_scale) * <img[b]/|img[b]|, txt[c]/|txt[c]|>
 *   loss = mean((pred - target)^2)   (target / loss optional)
 * bwd: d_pred [B,C] -> d_img [B,E], d_txt [C,E].  When d_pred == NULL the MSE gradient
 * 2 (pred - target) / (B C) * loss_scale is used (fused loss backward).
 */
int hba_cos_head_fwd(const float* img, const float* txt, int32_t B, int32_t C, int32_t E,
                     const float* logit_scale, float* pred, const float* target, float* loss,
                     void* stream);
int hba_cos_head_bwd(const float* img, const float* txt, int32_t B, int32_t C, int32_t E,
                     const float* logit_scale, const float* d_pred, const float* pred,
                     const float* target, float* d_img, float* d_txt, void* stream);
/* The same head with nn.MSELoss(reduction='mean') (BDRV:31; applied NEW:994 / NEW:597) and the loop's
 * per-batch bookkeeping (NEW:989-1004) fused into ONE launch, for `groups` independent problems
 * (lock-stepped sweep conditions; groups = 1 for a single run).  Group g owns img [B,E], txt [C,E],
 * pred [B,C] (contiguous per group) and target + g * target_group_stride (stride 0 = shared targets).
 *   loss[g]       = mean((pred - target)^2)
 *   bad_step[g]   = loss not finite   (the isnan(pred) / isnan(target) / isnan|isinf(loss) `continue`s
 *                   of NEW:932-935, 989-998: any of them makes the loss non-finite)        (optional)
 *   bad_total[g] += bad_step[g]                                                            (optional)
 *   total[g]     += loss * B, skipped for a bad batch when bad_step is given (NEW:1003-1004; evaluate_model
 *                   NEW:599-601 passes bad_step = NULL)                                     (optional)
 * workspace: groups * (B + 1) floats, zero before the first use (the kernel leaves it ready for the next).
 * target == NULL: plain forward (loss / bad_* / total / workspace must be NULL).
 * hba_cos_mse_bwd: d_img / d_txt of the fused loss, dL/dpred = 2 (pred - target) / (B C) * d_loss[g]
 * (d_loss optional device array of `groups` upstream gradients; 1 when NULL). */
int hba_cos_mse_fwd(const float* img, const float* txt, int32_t B, int32_t C, int32_t E, int32_t groups,
                    const float* logit_scale, float* pred, const float* target,
                    int64_t target_group_stride, float* loss, int32_t* bad_step, int32_t* bad_total,
                    double* total, float* workspace, void* stream);
int hba_cos_mse_bwd(const float* img, const float* txt, int32_t B, int32_t C, int32_t E, int32_t groups,
                    const float* logit_scale, const float* pred, const float* target,
                    int64_t target_group_stride, const float* d_loss, float* d_img, float* d_txt,
                    void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimisers. Multi-tensor, one launch.  AdamW(model.parameters(), lr) of NEW:1181 (betas
 * (0.9, 0.999), eps 1e-8, weight_decay 0.01, decoupled; torch.optim.AdamW arithmetic) and
 * SGD(momentum, weight_decay, dampening 0, no nesterov) of VIT:294-299.
 * ptrs: device array of 4*n pointers (param, grad, exp_avg, exp_avg_sq) resp. 3*n (param, grad,
 * momentum_buf); sizes: device array of n int64.  step is the 1-based step count AFTER this
 * update; when step_dev (optional, device int32) is given the count is read from the device instead
 * (a captured CUDA graph then replays with the right bias corrections).  skip_flag (optional, device
 * int32): when *skip_flag != 0 the update is skipped (the NaN/Inf guard of NEW:989-998 evaluated on
 * the device).
 */
int hba_adamw_multi(void* const* ptrs, const int64_t* sizes, int32_t n, int64_t total,
                    float lr, float beta1, float beta2, float eps, float weight_decay,
                    int64_t step, const int32_t* step_dev, const int32_t* skip_flag, void* stream);
int hba_sgd_multi(void* const* ptrs, const int64_t* sizes, int32_t n, int64_t total, float lr,
                  float momentum, float weight_decay, int32_t first_step,
                  const int32_t* skip_flag, void* stream);
/* Vectorised SGD of the fully trained ViT-B/16 with the bf16 GEMM operand of each weight refreshed in the
 * same pass.  ptrs: device array of 4*n pointers (param, grad, momentum_buf, bf16 copy or NULL), all 16-byte
 * aligned (the bf16 copy 8-byte), every tensor's element count a multiple of 4; prefix4: device array of n
 * int64 = exclusive prefix of the element counts / 4; total4 = sum of the element counts / 4. */
int hba_sgd_staged(void* const* ptrs, const int64_t* prefix4, int32_t n, int64_t total4, float lr,
                   float momentum, float weight_decay, int32_t first_step,
                   const int32_t* skip_flag, void* stream);

/* ------------------------------------------------------------------------------------------
 * RSA evaluation (behavioral_RSA tail, NEW:625-652; ViT variant MEAS:298-355):
 *   rdm = 1 - corrcoef(E) (float64, diagonal 0); upper triangle k=1 row-major;
 *   ranks with ties averaged (scipy.stats.rankdata 'average'); rho = Pearson(ranks, ref_ranks).
 * hba_rdm_f64: E [N, Dm] fp32 (ld = Dm) -> rdm [N,N] f64 (optional) and tri [N(N-1)/2] f64.
 * hba_rank_avg_f64: x [n] f64 -> ranks [n] f64 (1-based, ties averaged).
 *   workspace bytes needed: hba_rank_workspace_bytes(n).
 * hba_pearson_f64: rho (device double) of two f64 vectors, deterministic reduction.
 */
int hba_rdm_f64(const float* E, int32_t N, int32_t Dm, double* rdm, double* tri, void* stream);
int64_t hba_rank_workspace_bytes(int64_t n);
int hba_rank_avg_f64(const double* x, int64_t n, double* ranks, void* workspace,
                     int64_t workspace_bytes, void* stream);
int hba_pearson_f64(const double* a, const double* b, int64_t n, double* rho_out,
                    double* workspace /* >= 5*1024 doubles */, void* stream);
/* RSA at scale (BASELINE config 5: 1,854 x 66 embeddings per checkpoint -> P = 1,717,731 pairs), the whole
 * chain of NEW:625-652 for one checkpoint in 11 stream-ordered launches: E [N, Dm] fp32 -> RDM entries written
 * directly as sortable 64-bit keys -> all eight digit histograms in one pass -> one radix kernel per non-constant
 * digit (decoupled look-back) -> tie-averaged ranks consumed in sorted order by the Pearson sums against
 * ref_ranks [P] (the average ranks of the reference RDM's upper triangle) -> rho_out (device double).
 * rdm [N,N] f64 and ranks [P] f64 are optional outputs.  NaN semantics are numpy's / scipy's: a NaN or constant
 * embedding row gives rho = NaN.  Needs N(N-1)/2 > 2048; workspace: hba_rank_workspace_bytes(N(N-1)/2). */
int hba_rdm_spearman(const float* E, int32_t N, int32_t Dm, const double* ref_ranks, double* rdm,
                     double* ranks, double* rho_out, void* workspace, int64_t workspace_bytes, void* stream);
/* hba_rank_order_f64: as hba_rank_avg_f64 (same keys, passes and NaN ordering; ranks all NaN when any x is NaN)
 *   and also order [n] uint32, the stable sorted order: x[order[0]] <= x[order[1]] <= ..., equal values in
 *   index order, NaN at the ends.  Workspace: hba_rank_workspace_bytes(n). */
int hba_rank_order_f64(const double* x, int64_t n, uint32_t* order, double* ranks, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stimulus-resampling statistics of RSA for N stimuli, P = N(N-1)/2 upper-triangle pairs (k=1, row-major).
 * Sums are exact int64 sums of centred doubled ranks 2r - (M+1), so outputs are bit-identical run to run;
 * exact while 2 P^3 / 3 < 2^63: 3 <= N <= 2191.  Outputs are NaN where scipy.stats.spearmanr returns NaN.
 * hba_rsa_perm_null (Mantel permutation test): for p < n_perm and pi_p = perms[p, :] (int32, a permutation
 *   of 0..N-1; an entry outside [0, N) gives NaN),
 *     rho_out[p] = Pearson over i<j of (ref_ranks[i,j], model_ranks[pi_p(i), pi_p(j)])
 *   = scipy.stats.spearmanr(ref_tri, model_rdm[pi_p][:, pi_p][triu]).  ref_ranks, model_ranks: [P] f64 average
 *   ranks (hba_rank_avg_f64) of the two triangles.  Workspace: hba_rsa_perm_workspace_bytes(N, n_perm).
 * hba_rsa_bootstrap (stimulus bootstrap, Nili et al. 2014): for b < n_boot and counts c = counts[b, :] (int32,
 *   values in [0, N] summing to N; otherwise NaN), every pair {i,j}, i != j, enters with multiplicity c_i c_j
 *   and pairs of a stimulus with itself are dropped:
 *     rho_a[b] = spearmanr of (ref, model a) over that expanded multiset of pairs, with the average ranks of
 *     scipy.stats.rankdata on the expanded multiset = the weighted Pearson of the weighted average ranks.
 *   NaN when a pair of weight > 0 is NaN in either RDM or a side is constant (fewer than 3 distinct stimuli).
 *   tri_*: [P] f64 upper triangles; order_*: their sorted order (hba_rank_order_f64).  Model b (tri_b, order_b,
 *   rho_b: all given or all NULL) is evaluated on the same resamples, for a paired difference rho_a - rho_b.
 *   Workspace: hba_rsa_boot_workspace_bytes(N, n_boot).
 */
int64_t hba_rsa_perm_workspace_bytes(int32_t N, int32_t n_perm);
int hba_rsa_perm_null(const double* ref_ranks, const double* model_ranks, int32_t N, const int32_t* perms,
                      int32_t n_perm, double* rho_out, void* workspace, int64_t workspace_bytes, void* stream);
int64_t hba_rsa_boot_workspace_bytes(int32_t N, int32_t n_boot);
int hba_rsa_bootstrap(const double* ref_tri, const uint32_t* ref_order, const double* tri_a,
                      const uint32_t* order_a, const double* tri_b, const uint32_t* order_b, int32_t N,
                      const int32_t* counts, int32_t n_boot, double* rho_a, double* rho_b, void* workspace,
                      int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Kendall's tau-a and tau-b, the RDM comparator Nili et al. 2014 recommend when either RDM has ties (tau-a does not
 * favour models that predict tied dissimilarities).  For x [n] (model triangle) and y [n] (reference triangle),
 * n0 = n(n-1)/2, with values equal as in numpy (-0.0 == +0.0):
 *   n1 = sum t(t-1)/2 over the tie groups of x, n2 the same over y, n3 = pairs tied in both x and y,
 *   S  = concordant - discordant = n0 - n1 - n2 + n3 - 2 D   (D = discordant pairs),
 *   counts[0..3] = S, n1, n2, n3  (exact int64: outputs are bit-identical run to run),
 *   tau[0] = tau_a = S / n0,
 *   tau[1] = tau_b = S / sqrt(n0 - n1) / sqrt(n0 - n2) clipped to [-1, 1]  (= scipy.stats.kendalltau, variant 'b').
 * A NaN in x or y gives counts -1 and NaN taus; so does a y_order with an entry outside [0, n) or that does not sort
 * y.  A constant side (n1 == n0 or n2 == n0) gives NaN taus with the counts written.
 * y_order: the stable sorted order of y (hba_rank_order_f64; any permutation that sorts y will do).  2 <= n < 2^30
 * (the bound of hba_rank_order_f64).  n <= 2048 runs in one CTA without workspace; larger n needs
 * hba_kendall_workspace_bytes(n) bytes, 256-byte aligned: x[y_order] sorted by the radix passes of
 * hba_rank_order_f64, then a merge sort of the y-ranks that counts D as it merges (Knight's method, O(n log n)).
 */
int64_t hba_kendall_workspace_bytes(int64_t n);
int hba_kendall_tau_f64(const double* x, const double* y, const uint32_t* y_order, int64_t n, int64_t* counts,
                        double* tau, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Softmax cross-entropy (nn.CrossEntropyLoss at VIT:291, applied VIT:139) forward + backward:
 * logits [B, C] fp32, labels int64 -> loss (mean, device float) and d_logits = (softmax - 1hot)/B
 */
int hba_softmax_ce_fwd_bwd(const float* logits, int64_t ld, const int64_t* labels, int32_t B,
                           int32_t C, float* loss, float* d_logits, int64_t ld_d,
                           int32_t* correct_top1, float* workspace /* >= 2*B floats */,
                           void* stream);

/* ------------------------------------------------------------------------------------------
 * Extra kernels of the fully-trained ViT-B/16 data-parallel baseline (VIT:125-165: every parameter
 * receives a gradient).
 * hba_colsum: out[c] (+)= sum_r x[r, c]  (bias gradients of every Linear / the conv);
 *   workspace >= 128 * cols floats.
 * hba_layernorm_param_grad: dgamma_dbeta[0:cols] (+)= sum_r dy * xhat, [cols:2cols] (+)= sum_r dy;
 *   workspace >= 2*rows + 256*cols floats.
 * hba_attention_bwd: full softmax-attention backward, d_out [B*T, H*64] -> d_qkv [B*T, 3*H*64]
 *   (dtypes HBA_DT_*: (bf16, bf16|f32, bf16) or (f32, f32, f32); with bf16 qkv an f32 d_out is rounded to
 *   bf16 on load, like qkv); T <= 288, and T <= 203 with f32 qkv
 *   (its tiles must fit 227 KB of shared memory); HBA_ERR_ARG otherwise.
 */
int hba_colsum(const void* x, int32_t dtype, int64_t rows, int32_t cols, int64_t ld, float* out,
               int32_t accumulate, float* workspace, void* stream);
int hba_layernorm_param_grad(const float* dy, int64_t ld_dy, const float* x, int64_t rows,
                             int32_t cols, int64_t ldx, int64_t row_step, float eps,
                             float* dgamma_dbeta, int32_t accumulate, float* workspace, void* stream);
/* Fused LayerNorm backward of the trained ViT: dx (+)= LN'(dy), optional bf16 hi[/lo] copy of the
 * resulting dx (operand of the next GEMMs), dgamma_dbeta [2*cols] (+)=, and dx_colsum [cols] = column
 * sums of the resulting dx (bias gradient of the Linear feeding this residual stream); one pass over
 * HBM.  cols in {128, 256, 512, 768, 1024}; workspace >= 2 * #SM * 3 * cols floats. */
int hba_layernorm_bwd_fused(const float* dy, int64_t ld_dy, const float* x, int64_t rows,
                            int32_t cols, int64_t ldx, const float* gamma, float eps, float* dx,
                            int64_t ld_dx, int32_t accumulate, void* dx_bf16, int64_t ld_b,
                            int64_t lo_off, float* dgamma_dbeta, int32_t accumulate_params,
                            float* dx_colsum, float* workspace, void* stream);
int hba_attention_bwd(const void* qkv, int32_t qkv_dtype, int64_t ld_qkv, int32_t B, int32_t T,
                      int32_t H, int32_t causal, const void* d_out, int32_t do_dtype, int64_t ld_do,
                      void* d_qkv, int32_t dq_dtype, int64_t ld_dqkv, void* stream);
/* Tensor-core (tcgen05) pair for the bf16 training step, T <= 256 (ViT-B/16: T = 197), all matrices
 * bf16 with leading dimensions that are multiples of 8:
 * hba_attention_fwd_lse: as hba_attention_fwd (out [B*T, H*64] bf16) and additionally writes
 *   lse [B, H, T] fp32 = log2(sum_j exp(s_ij / 8)) (log2 domain), the only softmax statistic the
 *   backward needs.
 * hba_attention_bwd_lse: d_out [B*T, H*64] -> d_qkv [B*T, 3*H*64] from qkv, the forward's out and lse
 *   (autograd of SDPA as reached by VIT:138-145; dS = P o (dP - rowsum(dO o O)), FlashAttention-2 form).
 */
int hba_attention_fwd_lse(const void* qkv, int64_t ld_qkv, int32_t B, int32_t T, int32_t H,
                          int32_t causal, void* out, int64_t ld_out, float* lse, void* stream);
int hba_attention_bwd_lse(const void* qkv, int64_t ld_qkv, int32_t B, int32_t T, int32_t H,
                          int32_t causal, const void* out, int64_t ld_out, const void* d_out,
                          int64_t ld_do, const float* lse, void* d_qkv, int64_t ld_dqkv,
                          void* stream);

/* misc elementwise helpers used by the host-side engine */
int hba_add_rows(float* dst, int64_t ld_dst, int64_t dst_row_step, const float* src,
                 int64_t ld_src, int64_t rows, int32_t cols, void* stream);
int hba_nonfinite_flag(const float* x, int64_t n, int32_t* flag, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HBA_H_ */
