/* vitk.h — C ABI of libvitk.so, the B200 (sm_100a) kernel library behind the ViT training hot path.
 *
 * The reference (TaiMingLu/vision_transformers_torch_xla) has no FFI of its own: its operator seam
 * is Python (`models/_compat.py:27-172` resolves Attention/Mlp/PatchEmbed/LayerNorm by name, and
 * `engine.py:257-274` drives model -> criterion -> backward -> optimizer.step).  Each entry point
 * below replaces the PyTorch *library* op that those call sites dispatch to (SURVEY.md §2.4), and
 * is what a binding on the reference side would call (INTEGRATION.md shows the ctypes stub).
 *
 * Conventions
 *  - Plain pointers + sizes only.  All pointers are DEVICE pointers unless stated otherwise.
 *  - `stream` is a cudaStream_t passed as void*.  Every call only enqueues work; no host sync.
 *  - The library never allocates, frees or retains device memory.
 *  - Return 0 on success, a negative vitk_status otherwise; vitk_last_error() returns a
 *    thread-local message.  Nothing throws across the ABI.
 *  - bf16 buffers are passed as void* (raw __nv_bfloat16 storage).
 */
#ifndef VITK_H_
#define VITK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VITK_ABI_VERSION 4

enum vitk_status {
  VITK_STATUS_OK = 0,
  VITK_STATUS_SHAPE = -1,
  VITK_STATUS_ALIGN = -2,
  VITK_STATUS_DTYPE = -3,
  VITK_STATUS_CUDA = -4,
  VITK_STATUS_DRIVER = -5,
  VITK_STATUS_UNSUPPORTED = -6
};

int vitk_abi_version(void);
const char* vitk_last_error(void);
/* Compile-time target of the device code in this library, e.g. "sm_100a". */
const char* vitk_arch(void);
/* First 16 hex digits of the sha256 over the sources the library was built from (csrc/Makefile); a binding
 * recomputes it over the sources next to the library and refuses a stale binary. */
const char* vitk_build_id(void);

/* ------------------------------------------------------------------------------------------------
 * GEMM — tcgen05/TMEM bf16 GEMM with fused epilogues.   D[M,N] = opA(A)[M,K] * opB(B)[N,K]^T
 * Replaces: nn.Linear fwd/dgrad/wgrad for attn.qkv / attn.proj / mlp.fc1 / mlp.fc2 / head
 *   (reference models/vision_transformer.py:149-171, 618; timm Attention/Mlp), and the
 *   Conv2d(k=s=16) patchify of PatchEmbed (vision_transformer.py:552-560).
 * ---------------------------------------------------------------------------------------------- */
enum vitk_epilogue {
  VITK_EPI_BF16 = 0,   /* out_bf16[m,n]  = rowscale[m/g] * (acc + bias[n])                         */
  VITK_EPI_GELU = 1,   /* h = acc + bias; out_bf16 = gelu_erf(h); aux_bf16 = gelu_erf'(h)   (mlp.fc1) */
  VITK_EPI_RESID = 2,  /* out_f32 = resid_f32 + rowscale[m/g]*colscale[n]*(acc+bias)  (proj, fc2)  */
  VITK_EPI_F32 = 3,    /* out_f32 = acc + bias                                        (head)       */
  VITK_EPI_DGELU = 4,  /* out_bf16 = rowscale[m/g] * acc * aux_bf16[m,n], aux = gelu'(h) (fc2 dgrad)  */
  VITK_EPI_ATOMIC = 5, /* out_f32 += acc   via red.global.add (split-K)               (wgrad)      */
  VITK_EPI_PATCH = 6,  /* out_f32[b*(P+prefix)+prefix+t, n] = acc + bias[n] + pos[prefix+t, n]; rows are patches (b, t), or
                          the padded rows (b, gy, gx') of an a_image operand                         */
  /* GELU / x GELU' with the derivative kept in ONE byte per element: aux_u8 = round(200 * gelu'(h)) + 27, i.e. a fixed
   * grid of step 0.005 over [-0.135, 1.14] that represents gelu'(h) = 0 and 1 exactly (|error| <= 0.0025: what a bf16
   * rounding costs at gelu' ~ 1); fc1 writes 3 instead of 4 bytes per hidden element, fc2's dgrad reads 1 instead of 2.
   * N must be a multiple of 256; aux is uint8 [M, N] with ld_aux in elements (= bytes, multiple of 16). */
  VITK_EPI_GELU_Q8 = 7,
  VITK_EPI_DGELU_Q8 = 8
};

typedef struct vitk_gemm_args {
  const void* A;       /* bf16.  K-major: [M, K] row pitch lda.  MN-major: [K, M] row pitch lda.   */
  const void* B;       /* bf16.  K-major: [N, K] row pitch ldb.  MN-major: [K, N] row pitch ldb.   */
  int64_t lda, ldb;    /* in elements, multiples of 8                                              */
  int32_t a_mn_major, b_mn_major;
  int32_t M, N, K;
  int32_t epilogue;    /* enum vitk_epilogue                                                       */
  void* out;           /* bf16 or f32 depending on the epilogue                                    */
  int64_t ld_out;
  void* aux;           /* GELU: activation-derivative output (bf16; uint8 for the _Q8 codes); DGELU: the same buffer as input */
  int64_t ld_aux;
  const float* bias;   /* [N] or NULL                                                              */
  const float* resid;  /* RESID: fp32 [M, N] residual stream input                                 */
  int64_t ld_resid;
  const float* rowscale; /* per-sample DropPath scale (mask/keep_prob), indexed by m/rows_per_group, or NULL */
  int32_t rows_per_group;
  const float* colscale; /* LayerScale gamma [N] or NULL                                           */
  const float* pos;    /* PATCH: pos_embed fp32 [(P+prefix), N]                                    */
  int32_t tokens_per_img; /* PATCH: P                                                              */
  int32_t prefix;      /* PATCH: number of prefix (cls/dist) tokens                                */
  int32_t splits;      /* ATOMIC: split-K factor, 0 = choose to fill 148 SMs                       */
  int32_t block_n;     /* 0 = auto; otherwise 128, 192 or 256                                      */
  float* colsum_out;   /* ATOMIC with MN-major A: colsum_out[m] += sum_k A[k, m] (the bias gradient of the same
                          wgrad, summed out of the staged smem tiles by the epilogue warps), or NULL */
  /* im2col-free patch embedding (PatchEmbed = Conv2d(k = s = patch), vision_transformer.py:552-560): an operand may be a
   * bf16 NCHW image batch [B, img_c, img_h, img_w] read through TMA AS its patch matrix, never materialised:
   *   row    = (b * (img_h / patch) + gy) * img_gwp + gx'   gx' in [0, img_gwp); gx' >= img_w / patch are zero rows
   *   column = (c * patch + py) * patch + px                == proj.weight.view(D, -1) column order
   * img_gwp = the patch-grid width rounded up to a multiple of 8 (TMA boxes cover 8 neighbouring patches); patch = 16.
   * a_image: A is such an image (K-major use; with VITK_EPI_PATCH the epilogue maps row -> token and skips the pad rows),
   *          M = B * (img_h / patch) * img_gwp, K = img_c * patch * patch.
   * b_image: B is such an image in MN-major use (the weight gradient dW[D, K'] += gp^T patches), K = rows as above. */
  int32_t a_image, b_image;
  int32_t img_c, img_h, img_w, img_patch, img_gwp;
  /* Dropout in the epilogue (timm Attention.proj_drop, Mlp.drop1 / drop2; vision_transformer.py:149-171): keep-mask bytes
   * [M, N] (1 = keep, 0 = drop; written by vitk_dropout_mask or by the caller), row pitch ld_mask (multiple of 4), or NULL.
   *   VITK_EPI_GELU : out = gelu(h) * m * mask_scale, aux = gelu'(h) * m * mask_scale (the backward multiply is unchanged)
   *   VITK_EPI_RESID: out = resid + rowscale * colscale * m * mask_scale * (acc + bias)
   * mask_scale = 1 / (1 - p). */
  const uint8_t* mask;
  int64_t ld_mask;
  float mask_scale;
} vitk_gemm_args;

int vitk_gemm_bf16(const vitk_gemm_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LayerNorm (eps = 1e-6 in the reference: timm LayerNorm; vision_transformer.py:148,163,603,616)
 * fwd: y_bf16 = (x - mean) * rstd * gamma + beta over the last dim; x is the fp32 residual stream.
 *      Row r of x starts at x + r*ld_x (lets the 'token' pool normalise only the cls rows).
 * bwd: dx = LN'(dy); g_out = (g_in ? g_in : 0) + dx; gb_out = bf16(rowscale * g_out) (optional);
 *      dgamma/dbeta are ACCUMULATED (atomicAdd) into fp32 [dim] buffers.
 * ---------------------------------------------------------------------------------------------- */
int vitk_layernorm_fwd(const float* x, int64_t ld_x, const float* gamma, const float* beta,
                       void* y_bf16, int64_t ld_y, float* mean, float* rstd, int64_t rows,
                       int32_t dim, float eps, void* stream);
int vitk_layernorm_bwd(const void* dy_bf16, int64_t ld_dy, const float* x, int64_t ld_x,
                       const float* mean, const float* rstd, const float* gamma, const float* g_in,
                       float* g_out, int64_t ld_g, void* gb_out_bf16, const float* rowscale,
                       int32_t rows_per_group, float* dgamma, float* dbeta, int64_t rows,
                       int32_t dim, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention (timm Attention fused path = F.scaled_dot_product_attention, dropout 0, no mask)
 * qkv: bf16 [B, N, 3, H, hd] (exactly the qkv Linear output), out: bf16 [B, N, H*hd],
 * lse: fp32 [B, H, N] (natural-log sum-exp of scaled scores).  hd: a multiple of 8 in [16, 80]; N <= 4224
 * (N <= 256 when hd > 64); a longer sequence returns VITK_ERR_UNSUPPORTED.
 * ---------------------------------------------------------------------------------------------- */
int vitk_attn_fwd(const void* qkv, void* out, float* lse, int32_t B, int32_t N, int32_t H,
                  int32_t head_dim, float scale, void* stream);
/* bwd needs a caller-owned fp32 workspace of vitk_attn_bwd_workspace_bytes(): D = rowsum(O * dO) [B, H, N], plus - when
 * N > 256, or 128 < N <= 256 with hd > 64 - the dQ accumulator the kv tiles red.add their partials into. */
int64_t vitk_attn_bwd_workspace_bytes(int32_t B, int32_t N, int32_t H, int32_t head_dim);
int vitk_attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse,
                  void* dqkv, void* workspace, int32_t B, int32_t N, int32_t H, int32_t head_dim,
                  float scale, void* stream);
/* Attention dropout (timm Attention.attn_drop: softmax -> Dropout -> @ v; dropout_p of the fused SDPA call): keep_mask holds
 * keep bytes [B, H, N, N] (1 = keep; vitk_dropout_mask), keep_scale = 1 / (1 - p).  out = (softmax(S) * m * keep_scale) V, lse is
 * the log-sum-exp of the undropped scores; the backward sees the same mask.  Runs on the streaming forward and backward for
 * every N (the mask is read per element); the backward workspace holds the fp32 dQ accumulator when N > 128. */
int vitk_attn_fwd_dropout(const void* qkv, void* out, float* lse, const uint8_t* keep_mask, float keep_scale, int32_t B,
                          int32_t N, int32_t H, int32_t head_dim, float scale, void* stream);
int64_t vitk_attn_bwd_dropout_workspace_bytes(int32_t B, int32_t N, int32_t H, int32_t head_dim);
int vitk_attn_bwd_dropout(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, void* workspace,
                          const uint8_t* keep_mask, float keep_scale, int32_t B, int32_t N, int32_t H, int32_t head_dim,
                          float scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Patch embedding helpers (PatchEmbed + _pos_embed: vision_transformer.py:552-560, 743-780)
 * patchify: fp32 NCHW image -> bf16 [B*P, C*ps*ps] rows in (c, ph, pw) order == proj.weight.view(D,-1)
 * prefix_rows: x[b, j, :] = prefix_tok[j, :] + pos[j, :] for j < prefix (cls / dist tokens)
 * embed_bwd: from g fp32 [B, N, D]: gp_bf16 [B*P, D] (patch rows; with gw > 0 the padded row order of an image operand:
 *            [B * (P / gw) * gwp, D], row (b, gy, gx'), zeros for gx' >= gw), dpos[N, D] += sum_b g,
 *            dprefix0[D] += sum_b g[b, 0, :] (cls_token), dprefix1[D] += sum_b g[b, 1, :] (dist_token, prefix == 2);
 *            either may be NULL (frozen token)
 * ---------------------------------------------------------------------------------------------- */
int vitk_patchify(const float* img, void* patches_bf16, int32_t B, int32_t C, int32_t H, int32_t W,
                  int32_t ps, void* stream);
int vitk_prefix_rows(float* x, const float* prefix_tok, const float* pos, int32_t B, int32_t N,
                     int32_t D, int32_t prefix, void* stream);
int vitk_embed_bwd(const float* g, void* gp_bf16, float* dpos, float* dprefix0, float* dprefix1, int32_t B,
                   int32_t N, int32_t D, int32_t prefix, int32_t gw, int32_t gwp, void* stream);

/* DropPath (timm drop_path as called by Block, vision_transformer.py:160-161, 172-178): all per-sample keep masks of one
 * forward pass in one launch.  rs fp32 [rows, B]: rs[r, b] = Bernoulli(1 - drop_probs[r]) / (1 - drop_probs[r]).
 * drop_probs is a HOST array of `rows` <= 128 probabilities (copied by value into the launch), rows ordered as the
 * reference draws them (block 0 attention branch, block 0 MLP branch, block 1 ...).  Philox4x32-10 keyed by
 * (seed, offset): same (seed, offset) -> same masks. */
int vitk_droppath_masks(float* rs, const float* drop_probs, int32_t rows, int32_t B, uint64_t seed,
                        uint64_t offset, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Pooling (global_pool_nlc: vision_transformer.py:419-441).  mode 0 = 'avg' over non-prefix
 * tokens, mode 1 = 'token' (x[:, 0]).  bwd writes the full g [B, N, D] (zeros elsewhere).
 * ---------------------------------------------------------------------------------------------- */
int vitk_pool_fwd(const float* x, float* pooled, int32_t B, int32_t N, int32_t D, int32_t prefix,
                  int32_t mode, void* stream);
int vitk_pool_bwd(const float* dpooled, float* g, int32_t B, int32_t N, int32_t D, int32_t prefix,
                  int32_t mode, void* stream);

/* out[c] += sum_r x[r, c]   (bias gradients).  x bf16 [rows, cols] pitch ld. */
int vitk_colsum_bf16(const void* x_bf16, int64_t ld, float* out, int64_t rows, int32_t cols,
                     void* stream);

/* ------------------------------------------------------------------------------------------------
 * Losses (timm SoftTargetCrossEntropy / LabelSmoothingCrossEntropy selected at reference
 * main.py:926-935; DistillationLoss main.py:939-968).  One fused forward+backward kernel:
 *   base   = mean_b sum_c -t[b,c] * log_softmax(x)[b,c]
 *            (t = soft_targets, or the smoothed one-hot of labels when soft_targets == NULL)
 *   kd     = T^2 * mean_b KL(softmax(teacher/T) || softmax(x/T))          (teacher != NULL)
 *   loss   = (1 - alpha) * base + alpha * kd           (alpha = 0 when teacher == NULL)
 * Writes loss[0] (fp32 scalar, overwritten) and dlogits fp32 [B, C] = d loss / d x.
 * ---------------------------------------------------------------------------------------------- */
int vitk_ce_fwd_bwd(const float* logits, const float* soft_targets, const int64_t* labels,
                    float smoothing, const float* teacher_logits, float kd_alpha, float kd_temp,
                    float* loss, float* dlogits, float* row_loss_scratch, int32_t B, int32_t C,
                    void* stream);
/* x[i] *= scale_dev[0] in place (the upstream gradient of the loss applied to dlogits, no host sync) */
int vitk_scale_f32(float* x, const float* scale_dev, int64_t n, void* stream);

/* Dropout (nn.Dropout sites of the reference model: pos_drop, proj_drop, Mlp.drop1/2, head_drop).
 * vitk_dropout_mask: mask[i] = 1 with probability 1 - p, else 0 (Philox4x32-10 keyed by seed, counter = (i / 8, offset), 16 bits per element;
 *   n bytes, any n).  The masks feed the GEMM epilogues above and the two multiplies below (the backward of a site, and the
 *   sites that have no GEMM in front of them).
 * vitk_mask_mul_bf16 / _f32: x[r, c] *= mask[r, c] ? scale : 0 in place; x: [rows, cols] with row pitch ld_x, mask: [rows, cols]
 *   with row pitch ld_mask; cols a multiple of 4 (f32) / 8 (bf16). */
int vitk_dropout_mask(uint8_t* mask, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream);
int vitk_mask_mul_bf16(void* x, int64_t ld_x, const uint8_t* mask, int64_t ld_mask, int64_t rows, int32_t cols, float scale,
                       void* stream);
int vitk_mask_mul_f32(float* x, int64_t ld_x, const uint8_t* mask, int64_t ld_mask, int64_t rows, int32_t cols, float scale,
                      void* stream);
/* out_bf16[i] = in_f32[i] * scale_dev[0] */
int vitk_scale_cast_bf16(const float* in, const float* scale_dev, void* out_bf16, int64_t n,
                         void* stream);
/* out_bf16[i] = in_f32[i] * rowscale[i / elems_per_group]  (DropPath scale on a gradient stream; rowscale may be NULL) */
int vitk_rowscale_cast_bf16(const float* in, const float* rowscale, int64_t elems_per_group,
                            void* out_bf16, int64_t n, void* stream);
/* out_bf16[i] = in_f32[i] */
int vitk_cast_bf16(const float* in, void* out_bf16, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused multi-tensor AdamW over flat buffers (torch.optim.AdamW semantics, reference
 * optim_factory.py:248-249; stepped at engine.py:185/271).  All parameters live in one flat fp32
 * buffer; `chunk_group[i]` gives the param-group id of elements [i*chunk, (i+1)*chunk).
 *   g' = g * grad_scale * (grad_scale_dev ? grad_scale_dev[0] : 1)
 *   p *= 1 - lr*wd;  m = b1 m + (1-b1) g';  v = b2 v + (1-b2) g'^2
 *   p -= lr / bc1 * m / (sqrt(v) / sqrt(bc2) + eps);   shadow_bf16 = bf16(p);  ema = d ema + (1-d) p
 * lr[] / wd[] are HOST arrays of length num_groups (copied by value into the launch).
 * g_bf16 (optional): read the gradient from this bf16 copy instead of g (the copy the data-parallel layer all-reduces
 * at half the bytes); g is then only zeroed (zero_grad).  grad_scale_dev (optional): device scalar multiplied into the
 * gradient, e.g. the clip coefficient vitk_clip_coef left on the device.
 * ---------------------------------------------------------------------------------------------- */
int vitk_adamw_flat(float* p, float* g, const void* g_bf16, const float* grad_scale_dev, float* m, float* v,
                    void* shadow_bf16, float* ema, int64_t n, const uint8_t* chunk_group, int32_t chunk,
                    int32_t num_groups, const float* lr, const float* wd, float beta1, float beta2, float eps,
                    int64_t step, float grad_scale, float ema_decay, int32_t zero_grad, void* stream);
/* Tuning aid: when non-NULL, the first CTA of the persistent attention kernels (attn_fwd4 / attn_fwd6 / attn_bwd4) stamps
 * clock64() at its phase boundaries into this device buffer of >= 128 int64 (tools/attn_trace3.py and tools/attn_trace6.py
 * print the timelines).  NULL (default) disables it. */
void vitk_debug_set_trace(long long* device_buf);

/* Gradient clipping (engine.py:175-177; torch.nn.utils.clip_grad_norm_) without a host sync or an extra pass:
 * vitk_sumsq / vitk_sumsq_bf16: out[0] += sum_i x[i]^2, DETERMINISTIC (fixed grid and summation order, no floating-point
 * atomics: data-parallel ranks must get bit-identical coefficients from bit-identical gradients); `scratch` is a
 * caller-owned fp32 buffer of vitk_sumsq_scratch_floats() elements.  vitk_clip_coef: norm[0] = sqrt(sumsq[0]) * grad_scale (optional output),
 * coef[0] = min(1, max_norm / (norm + 1e-6)), which vitk_adamw_flat multiplies in through grad_scale_dev. */
int32_t vitk_sumsq_scratch_floats(void);
int vitk_sumsq(const float* x, int64_t n, float* out, float* scratch, void* stream);
int vitk_sumsq_bf16(const void* x_bf16, int64_t n, float* out, float* scratch, void* stream);
int vitk_clip_coef(const float* sumsq, float grad_scale, float max_norm, float* coef, float* norm, void* stream);

/* Mixup / CutMix, batch mode, in place on fp32 NCHW images (image b mixes with image B-1-b); replaces
 * timm.data.Mixup._mix_batch as constructed at /root/reference/main.py:622-629 and applied at engine.py:259-262.
 * lam and the CutMix box are drawn on the host exactly as timm does (no device sync); lam is a double so that
 * (float)lam and (float)(1 - lam) round exactly like the reference's Python scalars. */
int vitk_mixup_batch(float* x, int32_t B, int32_t C, int32_t H, int32_t W, double lam, int32_t use_cutmix,
                     int32_t yl, int32_t yh, int32_t xl, int32_t xh, void* stream);
/* out[b, c] = onehot_smooth(labels[b])[c] * lam + onehot_smooth(labels[B-1-b])[c] * (1 - lam)   (timm mixup_target) */
int vitk_mixup_target(const int64_t* labels, float* out, int32_t B, int32_t C, double lam, double smoothing,
                      void* stream);

/* LayerScale backward (/root/reference/models/vision_transformer.py:80-106; the forward is the `colscale` of the
 * residual GEMM epilogue).  vitk_colscale_bf16: x[r, c] *= gamma[c] in place on the bf16 branch gradient.
 * vitk_layerscale_grad: dgamma[c] = (sum_k W[c,k] dW[c,k] + bias[c] dbias[c]) / gamma[c]  (SET, not accumulated; W / dW are
 * the [C, K] weight of the branch's last Linear and its gradient computed from the gamma-scaled branch gradient). */
int vitk_colscale_bf16(void* x_bf16, const float* gamma, int64_t rows, int32_t dim, void* stream);
int vitk_layerscale_grad(const float* W, const float* dW, const float* bias, const float* dbias, const float* gamma,
                         float* dgamma, int32_t C, int32_t K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VITK_H_ */
