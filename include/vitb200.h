/*
 * vitb200.h — C ABI of libvitb200.so: hand-written sm_100a kernels for the training hot path of
 * mahbodnr/ViT-CIFAR (vit.ViT + layers.TransformerEncoder / MultiHeadSelfAttention + label-smoothing
 * cross-entropy + Adam).
 *
 * The reference has no native layer (SURVEY.md §2.1): every entry point below replaces a run of
 * PyTorch/ATen calls in the reference's Python, cited as `file:line` into the reference repository.
 * The Python host (vit-cifar_b200/) binds these with ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - All pointers are DEVICE pointers owned by the caller, alive until `stream` has passed the call.
 *  - Nothing allocates, nothing synchronises the host; every kernel runs on the `stream` argument
 *    (a cudaStream_t passed as void*), so calls can be captured into a CUDA graph.
 *  - Return value: 0 = ok; < 0 = bad argument (vitb_last_error() has the text); > 0 = cudaError_t.
 *  - `dt` selects the ACTIVATION storage type: VITB_F32 (check mode: fp32 storage, SIMT fp32 math)
 *    or VITB_BF16 (bf16 storage, fp32 accumulation; tcgen05 tensor-core GEMMs, mma.sync attention).
 *    Parameters, gradients and optimiser state are always fp32; `w_act` arguments are the weight
 *    in the activation type (the bf16 shadow written by vitb_adam_multi / vitb_cast_f32_to_bf16,
 *    or the fp32 master itself in check mode).
 *  - Row-major everywhere. "rows" is B*T (tokens of the whole batch).
 */
#ifndef VITB200_H_
#define VITB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VITB_F32 0
#define VITB_BF16 1

#define VITB_ABI_VERSION 1

/* ABI version of the loaded library (== VITB_ABI_VERSION). */
int vitb_version(void);
/* Text of the last error raised on the calling thread ("" if none). */
const char* vitb_last_error(void);
/* Number of kernels this library has launched (or recorded into a CUDA graph) in this process so far. */
unsigned long long vitb_launch_count(void);
/* 1 if the current device is compute capability 10.x, else 0 (the kernels are sm_100a only). */
int vitb_device_supported(void);

/* ---- L2 residency hint for the weights (host function; no kernel): every kernel launched through this library while a window is
 * set carries it as cudaLaunchAttributeAccessPolicyWindow (so captured CUDA-graph nodes keep it): reads of [base, base + bytes)
 * are persisting in a carve-out of `carve_out_bytes` of L2, everything else is streaming.  Intended for the bf16 weight shadow
 * (12.5 MB for the 7-layer model): the resident GEMMs then find their weight block in L2 at kernel start instead of in HBM.
 * base = NULL clears the window.  Values are clamped to the device limits. ---- */
int vitb_set_l2_persisting_window(void* base, size_t bytes, size_t carve_out_bytes);

/* fp32 -> bf16 copy of a flat buffer (weight shadow refresh after an external optimiser step). */
int vitb_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream);

/* ---- patch embedding: vit.py:79-89 (_to_words), vit.py:67 (emb), vit.py:68-70 (cls cat + pos_emb) ----
 * img   fp32 (B,3,S,S) NCHW;   w fp32 (H, K) with K = (S/P)^2*3, feature index (kh*ps+kw)*3+c
 * bias  fp32 (H);  cls fp32 (H) or NULL when has_cls == 0;  pos fp32 (T,H), T = P*P + has_cls
 * out   act  (B,T,H):  out[b,0] = cls+pos[0];  out[b,has_cls+n] = words[b,n]·wᵀ + bias + pos[has_cls+n]
 * P is the number of patches per side (the reference's `patch`, vit.py:37). */
size_t vitb_patch_embed_fwd_ws_bytes(int B, int S, int P, int H, int dt);
/* w_act: emb.weight in the activation type (bf16 shadow) or NULL; words: act (B*P*P, K) or NULL.  When both are given in
 * bf16 mode (and the shape allows) the product runs on the tensor cores: the patch matrix is written to `words` (kept
 * for backward), multiplied by tcgen05 and assembled with cls/pos; ws: vitb_patch_embed_fwd_ws_bytes().  Otherwise
 * (fp32 check mode) an fp32 FFMA kernel reads the image directly. */
int vitb_patch_embed_fwd(const float* img, const float* w, const void* w_act, const float* bias,
                         const float* cls, const float* pos, void* out, void* words, void* ws,
                         size_t ws_bytes, int B, int S, int P, int H, int has_cls, int dt, void* stream);
/* Backward of the above (autograd of vit.py:66-70). dout act (B,T,H); words as written by the forward (or NULL).
 * Writes (overwrites) dw (H,K), dbias (H), dcls (H) (may be NULL), dpos (T,H).  ws: vitb_patch_embed_bwd_ws_bytes(). */
size_t vitb_patch_embed_bwd_ws_bytes(int B, int S, int P, int H, int has_cls);
int vitb_patch_embed_bwd(const float* img, const void* words, const void* dout, float* dw, float* dbias,
                         float* dcls, float* dpos, void* ws, size_t ws_bytes, int B, int S, int P,
                         int H, int has_cls, int dt, void* stream);

/* ---- LayerNorm: layers.py:26,30,45,47 (la1/la2), vit.py:62 (fc[0]); eps 1e-5, affine ----
 * x act, row r at x + r*x_row_stride elements (lets the head read out[:,0], vit.py:73); y act (rows,H)
 * mean/rstd fp32 (rows) saved for backward. */
int vitb_layernorm_fwd(const void* x, int64_t x_row_stride, const float* gamma, const float* beta,
                       void* y, float* mean, float* rstd, int rows, int H, float eps, int dt,
                       void* stream);
/* dx = LN'(dy) (+ dres if dres != NULL: the residual branch of layers.py:45/47).
 * dx row r at dx + r*dx_row_stride.  dgamma/dbeta fp32 (H) overwritten.  If dx_colsum != NULL it
 * receives sum over rows of dx (H) = bias gradient of the Linear that produced the LN input.
 * ws: vitb_layernorm_bwd_ws_bytes(rows, H). */
size_t vitb_layernorm_bwd_ws_bytes(int rows, int H);
int vitb_layernorm_bwd(const void* dy, const void* x, int64_t x_row_stride, const float* gamma,
                       const float* mean, const float* rstd, const void* dres, void* dx,
                       int64_t dx_row_stride, float* dgamma, float* dbeta, float* dx_colsum,
                       void* ws, size_t ws_bytes, int rows, int H, int dt, void* stream);

/* ---- Linear layers: layers.py:81-85,92-94,102 (Wq/Wk/Wv/out_project), layers.py:33-37 (mlp),
 *      vit.py:63,76 (fc[1]).  GELU is exact/erf (nn.GELU default).
 * C[M,N] = act(A[M,K] · W[N,K]ᵀ + bias[N]) (+ residual[M,N]);  if preact != NULL the value before
 * GELU is stored there (needed by backward).  flags: VITB_GEMM_GELU.  A,W,residual,C,preact: act type.
 * bf16: tcgen05 path, needs N % 128 == 0 and K % 64 == 0 (else falls to the SIMT kernel). */
#define VITB_GEMM_GELU 1
#define VITB_GEMM_OUT_F32 2 /* C is fp32 regardless of dt (head logits) */
int vitb_gemm_bias_act_fwd(const void* a, const void* w_act, const float* bias, const void* residual,
                           void* c, void* preact, int M, int N, int K, int flags, int dt, void* stream);
/* dX[M,K] = dY[M,N] · W[N,K]  (* gelu'(z[M,K]) if z != NULL: fuses the GELU backward of the layer
 * that produced this Linear's input, layers.py:34/37). */
int vitb_gemm_dgrad(const void* dy, const void* w_act, const void* z, void* dx, int M, int N, int K,
                    int flags, int dt, void* stream);
/* dW[N,K] (fp32) = dY[M,N]ᵀ · X[M,K];  dbias[N] (fp32) = column sums of dY (if dbias != NULL).
 * Overwrites.  Split over M with a fixed-order second pass (deterministic).
 * flags: VITB_GEMM_DY_F32: dY is fp32 regardless of dt (head dlogits). */
#define VITB_GEMM_DY_F32 4
size_t vitb_gemm_wgrad_ws_bytes(int M, int N, int K, int dt);
int vitb_gemm_wgrad_dbias(const void* dy, const void* x, float* dw, float* dbias, void* ws,
                          size_t ws_bytes, int M, int N, int K, int flags, int dt, void* stream);

/* ---- attention core: layers.py:92-101.  qkv act (B,T,3H) = [Q | K | V] per token, head h owns
 * columns h*d..h*d+d-1 of each third;  o act (B,T,H) (= attn.flatten(2), layers.py:102)
 * lse fp32 (B,heads,T): log-sum-exp of the scaled scores (saved instead of the (B,h,T,T) map).
 * attn_map fp32 (B,heads,T,T) or NULL: the softmax map itself (save_attn_map, layers.py:99-100).
 * scale = 1/sqrt(features) (layers.py:79,97).  d in {32,64}, T <= 128. */
int vitb_attn_fwd(const void* qkv, void* o, float* lse, float* attn_map, int B, int T, int heads,
                  int d, float scale, int dt, void* stream);
/* dqkv act (B,T,3H) from d_o act (B,T,H): dP = dO·Vᵀ; dS = P∘(dP − D), D_i = rowsum(P∘dP)_i = sum_d dO_id·O_id;
 * dQ = dS·K·scale; dK = dSᵀ·Q·scale; dV = Pᵀ·dO (autograd of layers.py:96-101).  P is recomputed from lse;
 * o is the forward output (B,T,H) saved by vitb_attn_fwd (used for D). */
int vitb_attn_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, void* dqkv, int B,
                  int T, int heads, int d, float scale, int dt, void* stream);

/* ---- GELU backward + column sums: dz = dy * gelu'(z); colsum fp32 (cols) = sum over rows of dz
 * (bias gradient of the Linear before the GELU, layers.py:36-37) if colsum != NULL. ---- */
size_t vitb_colsum_ws_bytes(int rows, int cols);
int vitb_gelu_bwd_colsum(const void* dy, const void* z, void* dz, float* colsum, void* ws,
                         size_t ws_bytes, int rows, int cols, int dt, void* stream);
/* colsum fp32 (cols) = sum over rows of x act (rows, cols). */
int vitb_colsum(const void* x, float* colsum, void* ws, size_t ws_bytes, int rows, int cols, int dt,
                void* stream);

/* ---- training input pipeline on the device, utils.py:337-355: RandomCrop(S, padding=pad) + RandomHorizontalFlip + ToTensor +
 * Normalize(mean, std) as one gather.  img_u8 uint8 (B,S,S,3) HWC device; dx, dy int32 (B) crop offsets in [0, 2*pad] (NULL = centre);
 * flip uint8 (B) (NULL = none); mean3 / std3: 3 HOST floats each; out fp32 (B,3,S,S).  Out-of-image pixels are black before
 * normalisation, as torchvision pads.  The caller draws dx, dy, flip. ---- */
int vitb_augment_crop_flip_normalize(const uint8_t* img_u8, const int32_t* dx, const int32_t* dy, const uint8_t* flip,
                                     const float* mean3, const float* std3, float* out, int B, int S, int pad, void* stream);

/* AutoAugment sub-policies (the reference's autoaugment.py) fused with RandomCrop + flip + ToTensor + Normalize.
 * code int32 (B): bits 0-7 sub-policy index, bit 8/9 apply op 1/2, bit 10/11 negative sign of op 1/2 (the caller draws them).
 * op_ids int32 / mags double: 2*n_sub HOST entries (op code, raw reference magnitude); baked into the launch, graph-capturable.
 * Op codes: 0 shearX, 1 shearY, 2 translateX, 3 translateY, 4 rotate, 5 color, 6 posterize, 7 solarize, 8 contrast, 9 sharpness,
 * 10 brightness, 11 autocontrast, 12 equalize, 13 invert.  1 <= n_sub <= 32, S <= 64; other arguments as in
 * vitb_augment_crop_flip_normalize (dx, dy, flip may be NULL).  An image whose code indexes past the table is written as NaN. */
int vitb_augment_autoaugment(const uint8_t* img_u8, const int32_t* dx, const int32_t* dy, const uint8_t* flip, const int32_t* code,
                             const int32_t* op_ids, const double* mags, int n_sub, const float* mean3, const float* std3,
                             float* out, int B, int S, int pad, void* stream);

/* ---- the same two transforms reading from a dataset resident in device memory: what the reference's DataLoader does per batch
 * (RandomSampler / DistributedSampler order, default_collate of the transformed images and their labels; utils.py:452-470 and the
 * loaders main.py:220-231 passes to Lightning), fused with the transform of utils.py:337-355.
 * data_u8 uint8 (N,S,S,3) HWC, labels_src int64 (N), idx int32 (B): the dataset row of each batch row (repeats allowed).
 * Writes out fp32 (B,3,S,S) and labels_dst[b] = labels_src[idx[b]] (int64, B) in the same launch.  For the same draws, out is
 * bit-identical to vitb_augment_crop_flip_normalize / vitb_augment_autoaugment run on the gathered batch data_u8[idx].  A row
 * idx[b] outside [0, N) is never dereferenced: that image is written as NaN and its label as -1 (no host round trip).
 * N >= 1, B >= 1; the policy form takes S <= 64.  Other arguments as in the contiguous forms. ---- */
int vitb_augment_crop_flip_normalize_gather(const uint8_t* data_u8, const int64_t* labels_src, int N, const int32_t* idx,
                                            const int32_t* dx, const int32_t* dy, const uint8_t* flip, const float* mean3,
                                            const float* std3, float* out, int64_t* labels_dst, int B, int S, int pad, void* stream);
int vitb_augment_autoaugment_gather(const uint8_t* data_u8, const int64_t* labels_src, int N, const int32_t* idx,
                                    const int32_t* dx, const int32_t* dy, const uint8_t* flip, const int32_t* code,
                                    const int32_t* op_ids, const double* mags, int n_sub, const float* mean3, const float* std3,
                                    float* out, int64_t* labels_dst, int B, int S, int pad, void* stream);

/* ---- RandomCropPaste: the reference's da.RandomCropPaste(size) (alpha = 1, flip_p = 0.5), which utils.get_transform appends after
 * ToTensor + Normalize with --rcpaste; it replaces, per image,
 *     front = img[:, fy1:fy1+fh, fx1:fx1+fw].clone(); [front = front.flip(-1)]; [img = img.flip(-1)]
 *     img[:, y1:y1+fh, x1:x1+fw] *= a;  img[:, y1:y1+fh, x1:x1+fw] += front * (1 - a)
 * In place on img fp32 (B,3,S,S) device.  params int32 (B,8) device: [fx1, fy1, fw, fh, x1, y1, flip_front, flip_img] per image;
 * alpha double (B) device: a.  The caller draws and derives them.  As in the reference, whose a is a float64 array, the blend is fp64:
 * out = (float)((double)(float)(base * a) + front * (1 - a)).  fw = 0 or fh = 0: only the whole-image flip.  A box that does not lie
 * inside the image makes that image NaN.  1 <= S <= 64 (the image is staged in 3*S*S floats of shared memory). ---- */
int vitb_random_crop_paste(float* img, const int32_t* params, const double* alpha, int B, int S, void* stream);

/* ---- batch-level CutMix / MixUp (da.py:51-93; network.py:149-158) on a normalised fp32 (B, C, S, S) device batch; perm int32 (B) =
 * the shuffled partner of every image (the caller draws it, with lam and the box, like the reference does on the host).
 * mode 0: out[b, :, i, j] = img[perm[b], :, i, j] inside rows x1 <= i < x2, columns y1 <= j < y2 (the reference's own index order,
 * da.py:68), img[b] elsewhere; mode 1: out = lam * img[b] + (1 - lam) * img[perm[b]] with lam and 1 - lam rounded to fp32 from the
 * double, as torch does for a Python scalar.  out must not alias img; S % 4 == 0. ---- */
int vitb_batch_mix(const float* img, const int32_t* perm, float* out, int B, int C, int S, int mode, double lam, int x1, int x2, int y1, int y2,
                   void* stream);

/* ---- nn.Dropout of the encoder block (layers.py:35, 38, 102; replaces torch's native_dropout on this path):
 *   out[i] = x[i] * keep[i] / (1 - p)  (+ residual[i] if residual != NULL);  x / residual / out act, n elements, n % 8 == 0; in place allowed.
 * keep is not stored: it is Philox4x32-10 with key = seed and counter = (i / 8 as 64 bits, site, step); element i takes the 16-bit
 * field (i % 8) of the 128-bit output (word (i % 8) / 2, low half first) and is kept iff field >= vitb_dropout_threshold(p)
 * = round(p * 65536) (host function, no GPU).  The backward pass is the same call on the gradient with the same (seed, site, step).
 * step_dev != NULL: the step is read from that device word instead of `step` (CUDA-graph replays draw fresh masks). 0 <= p < 1. ---- */
uint32_t vitb_dropout_threshold(float p);
int vitb_dropout(const void* x, const void* residual, void* out, int64_t n, float p, uint64_t seed, uint32_t site, uint32_t step,
                 const uint32_t* step_dev, int dt, void* stream);

/* ---- nn.Dropout fused into the kernel that produces (forward) or consumes (backward) the tensor it acts on, instead of a
 * separate elementwise pass per site: the three Dropouts of an encoder block sit right behind a Linear / GELU (layers.py:35, 38,
 * 102), and their backward right in front of the next backward kernel.  A site is described by a vitb_dropout_t; the mask is the
 * one vitb_dropout draws for the same (p, seed, site, step) over the flattened output tensor, so fused and unfused calls are
 * interchangeable element for element.  drop == NULL or p == 0: no dropout (the call equals its plain namesake).
 *   vitb_gemm_bias_act_fwd_drop:  C = dropout(act(A W^T + bias)) + residual   (the pre-activation is stored before GELU, undropped)
 *   vitb_gemm_dgrad_drop:         dX = dropout(dY W * gelu'(z))               (mask and gelu' commute: backward of GELU -> Dropout)
 *   vitb_gelu_bwd_colsum_drop:    dz = dropout(dy) * gelu'(z); colsum over dz (backward of GELU -> Dropout, layers.py:37-38)
 *   vitb_layernorm_bwd_fused:     dx as vitb_layernorm_bwd (dres required), plus a second output
 *                                 dx2 (rows, H) = dropout(dx [* gelu'(z) if z != NULL]) and dx2_colsum (H) = its column sums:
 *                                 z == NULL: the gradient entering out_project through its Dropout (layers.py:102) with out_project's
 *                                 bias gradient; z != NULL: the gradient entering the PREVIOUS block's second MLP Linear through
 *                                 Dropout and GELU (layers.py:36-38) with that Linear's bias gradient — dx is that block's output gradient.
 * bf16 tensor-core shapes apply the mask in the epilogue; every other shape / fp32 runs the plain kernel followed by vitb_dropout
 * (same result, one more launch). ---- */
typedef struct vitb_dropout {
  float p;                  /* drop probability, 0 <= p < 1 */
  uint64_t seed;            /* Philox key */
  uint32_t site;            /* which Dropout module (counter word 2) */
  uint32_t step;            /* optimisation step (counter word 3) ... */
  const uint32_t* step_dev; /* ... read from this device word instead when != NULL (CUDA-graph replays) */
} vitb_dropout_t;
int vitb_gemm_bias_act_fwd_drop(const void* a, const void* w_act, const float* bias, const void* residual, void* c, void* preact,
                                int M, int N, int K, int flags, int dt, const vitb_dropout_t* drop, void* stream);
int vitb_gemm_dgrad_drop(const void* dy, const void* w_act, const void* z, void* dx, int M, int N, int K, int flags, int dt,
                         const vitb_dropout_t* drop, void* stream);
int vitb_gelu_bwd_colsum_drop(const void* dy, const void* z, void* dz, float* colsum, void* ws, size_t ws_bytes, int rows, int cols,
                              int dt, const vitb_dropout_t* drop, void* stream);
int vitb_layernorm_bwd_fused(const void* dy, const void* x, int64_t x_row_stride, const float* gamma, const float* mean,
                             const float* rstd, const void* dres, void* dx, int64_t dx_row_stride, float* dgamma, float* dbeta,
                             const void* z, void* dx2, float* dx2_colsum, const vitb_dropout_t* drop, void* ws, size_t ws_bytes,
                             int rows, int H, int dt, void* stream);

/* ---- token pooling for the head: vit.py:72-75.  mode 0: y[b] = x[b,0] (cls); mode 1: mean over T.
 * bwd: dx (B,T,H) fully written (zeros where no gradient flows); mode 2 = cls pooling into a dx whose other rows the caller
 * keeps zero (a static buffer zeroed once): only the B cls rows are written. */
int vitb_pool_fwd(const void* x, void* y, int B, int T, int H, int mode, int dt, void* stream);
int vitb_pool_bwd(const void* dy, void* dx, int B, int T, int H, int mode, int dt, void* stream);

/* ---- label-smoothing cross-entropy: criterions.py:13-19.  logits fp32 (B,C), labels int64 (B).
 * loss (1 float) = mean_i sum_j -q_ij log_softmax(z_i)_j, q_iy = 1-s, q_ij = s/(C-1) otherwise.
 * dlogits fp32 (B,C) = (softmax(z) - q) * (grad_scale / B)  (may be NULL: forward only). ---- */
int vitb_ls_ce_fwd_bwd(const float* logits, const int64_t* labels, float* loss, float* dlogits,
                       int B, int C, float smoothing, float grad_scale, void* stream);

/* ---- the same loss with two targets per image, network.py:149-167 (CutMix da.py:51-72, MixUp da.py:75-93):
 * loss = lam * L(z, labels_a) + (1 - lam) * L(z, labels_b);  dlogits = (softmax(z) - (lam q_a + (1-lam) q_b)) * (grad_scale / B).
 * labels_b NULL = plain loss.  lam_dev (device float, may be NULL) overrides lam, so a captured graph can change it per step. ---- */
int vitb_ls_ce_mix_fwd_bwd(const float* logits, const int64_t* labels_a, const int64_t* labels_b, float lam,
                           const float* lam_dev, float* loss, float* dlogits, int B, int C, float smoothing,
                           float grad_scale, void* stream);

/* ---- the same for a fixed-size step fed a PARTIAL batch (the reference's DataLoader has no drop_last: the last batch of an
 * epoch is 50000 % 128 = 80 images, main.py:43, utils.py:452-470): n_valid_dev (device int, may be NULL = B) is the number of
 * real images in rows [0, n_valid); the loss is their mean (criterions.py:19 on the smaller batch), dlogits of the other rows
 * is zero and the scale is grad_scale / n_valid. ---- */
int vitb_ls_ce_batch_fwd_bwd(const float* logits, const int64_t* labels_a, const int64_t* labels_b, float lam,
                             const float* lam_dev, const int* n_valid_dev, float* loss, float* dlogits, int B, int C,
                             float smoothing, float grad_scale, void* stream);

/* The same loss over many thread blocks (the single-block form above takes 57 us for 100 classes at B = 1024): per-block partial
 * sums and the arrival counter live in `ws` (vitb_ls_ce_ws_bytes() bytes of device memory, 4-byte aligned, ZERO before the first
 * call; the kernel leaves the counter at zero, so the buffer is reusable by the next call on the same stream — not by concurrent
 * calls).  The partials are added in block order: deterministic.  ws == NULL or C > 256: falls back to the single-block kernel. */
size_t vitb_ls_ce_ws_bytes(void);
int vitb_ls_ce_blocks_fwd_bwd(const float* logits, const int64_t* labels_a, const int64_t* labels_b, float lam,
                              const float* lam_dev, const int* n_valid_dev, float* loss, float* dlogits, int B, int C,
                              float smoothing, float grad_scale, void* ws, size_t ws_bytes, void* stream);

/* ---- validation metrics of one batch (network.py:388-395): logits fp32 (B,C), labels int64 (B), n_valid_dev device int (NULL = B):
 * rows >= n_valid are ignored.  totals: 3 device doubles [loss_sum, correct, count], ADDED to (not overwritten), so that one record
 * accumulates a whole validation pass.  loss per row = the label-smoothing CE of criterions.py:13-19 with `smoothing` (the value
 * the loss kernels above average); correct = (argmax_j logits[i,j] == label[i]), argmax as torch: the first index of the maximum,
 * NaN above any number.  A label outside [0, C) is never read through: its row is not correct and adds NaN to loss_sum.
 * Any C >= 2.  Per-block partial sums in fp64, added in block order: two identical calls give bit-identical totals.
 * ws: vitb_eval_metrics_ws_bytes() bytes, 8-byte aligned, ZERO before the first call and left zeroed (self-resetting counter;
 * reusable by the next call on the same stream, not by concurrent calls). ---- */
size_t vitb_eval_metrics_ws_bytes(void);
int vitb_eval_metrics(const float* logits, const int64_t* labels, const int* n_valid_dev, int B, int C,
                      float smoothing, double* totals, void* ws, size_t ws_bytes, void* stream);

/* ---- training-epoch loss record (network.py:206 logs the step loss; the epoch value is its batch-size-weighted mean):
 * acc[0] += loss[0] * n, in fp64, n = n_valid_dev clamped to [1, B] as the loss kernels do (NULL = B).  loss: the 1-float result of
 * the loss kernels above; acc: one device double, ADDED to.  One thread; graph-capturable. ---- */
int vitb_train_loss_accumulate(const float* loss, const int* n_valid_dev, int B, double* acc, void* stream);

/* ---- backward of one nn.Linear y = x W^T (W: [N, K] bf16) in a single pass over dY — what autograd runs as two GEMMs
 * (layers.py:33-37, 85, 102):  dx [M, K] = dy [M, N] W  (times gelu'(z) when z [M, K] != NULL: the Linear's input was GELU(z),
 * layers.py:34);  dw [N, K] fp32 = dy^T x;  dx_colsum [K] fp32 (may be NULL) = column sums of dx as stored, i.e. the bias gradient
 * of the Linear that produced z.  dy is read from HBM once and feeds both tensor-core products from the same shared-memory
 * bytes (csrc/gemm_bwd_fused.cuh).  bf16 only, N in {128, 256, 384}, K a multiple of 128: vitb_gemm_bwd_fused_ws_bytes returns 0
 * for anything else and the caller uses vitb_gemm_dgrad + vitb_gemm_wgrad_dbias.  ws: fp32 partials (honours vitb_defer_begin). ---- */
size_t vitb_gemm_bwd_fused_ws_bytes(int M, int N, int K, int dt);
int vitb_gemm_bwd_fused(const void* dy, const void* x, const void* w, const void* z, void* dx, float* dw, float* dx_colsum,
                        void* ws, size_t ws_bytes, int M, int N, int K, int dt, void* stream);

/* ---- deferred second passes of split reductions.  Every gradient that is a sum over the batch rows (wgrad dW / db, LayerNorm
 * dgamma / dbeta and the column sums that are a Linear's bias gradient, GELU-backward column sums) is computed as per-CTA fp32
 * partials followed by a fixed-order second pass.  Between vitb_defer_begin and vitb_defer_flush (same host thread) the calls
 * vitb_gemm_wgrad_dbias, vitb_layernorm_bwd and vitb_gelu_bwd_colsum place their partials in `arena` (device memory the caller
 * keeps alive until the flush has run; 256-byte aligned) and record the second pass instead of launching it; the flush runs all
 * recorded passes in one launch per kernel class with the SAME summation order, so results are bit-identical to the immediate
 * path.  The outputs of the deferred calls are undefined until the flush has executed.  A call whose partials do not fit in what is
 * left of the arena runs its second pass immediately, as without deferral.  vitb_defer_used: bytes a large enough arena would
 * have held in the last begin..flush window. ---- */
int vitb_defer_begin(void* arena, size_t arena_bytes);
int vitb_defer_flush(void* stream);
/* runs the second passes recorded so far on `stream` (which the caller has ordered after every kernel that produced those
 * partials) and keeps the window open: lets a training step reduce layer i's gradients on a side stream while layer i - 1's
 * backward runs */
int vitb_defer_flush_partial(void* stream);
size_t vitb_defer_used(void);

/* ---- Adam with coupled L2 over a flat buffer: torch.optim.Adam as configured at network.py:71-77
 * (lr main.py:48, betas :51-52, weight_decay :56, eps 1e-8).  g is multiplied by grad_scale first
 * (1/world_size after a sum all-reduce).  hyper: 16 HOST floats {step_size = lr/(1-b1^t),
 * bc2_sqrt = sqrt(1-b2^t), beta1, beta2, eps, weight_decay, grad_scale, 1-beta1, 1-beta2, 0...}
 * (computed in double by the caller, as torch does).  If hyper_dev != NULL the 16 floats are read
 * from device memory instead (so a captured CUDA graph sees new values every replay).
 * w_shadow (bf16, n) may be NULL; else it receives the updated parameters rounded to bf16. ---- */
int vitb_adam_multi(float* p, const float* g, float* m, float* v, void* w_shadow, int64_t n,
                    const float* hyper_host, const float* hyper_dev, void* stream);

/* ---- SGD with momentum over a flat buffer: torch.optim.SGD as configured at network.py:78-84 (momentum = beta1, dampening 0, no
 * Nesterov, coupled weight decay): g = g*grad_scale + wd*p; buf = momentum*buf + g; p -= lr*buf.  buf starts at zero.
 * hyper: the same 16-float block as vitb_adam_multi, of which SGD reads [0] = lr, [2] = momentum, [5] = weight_decay,
 * [6] = grad_scale (host, or device memory if hyper_dev != NULL).  w_shadow as in vitb_adam_multi. ---- */
int vitb_sgd_multi(float* p, const float* g, float* buf, void* w_shadow, int64_t n, const float* hyper_host, const float* hyper_dev, void* stream);

/* ---- Data-parallel step over NVLink peer memory: what Lightning's DDP all-reduce (main.py:220-231) followed by
 * torch.optim.Adam (network.py:71-77) does for the reference, as ONE kernel per rank and step:
 *   barrier (all ranks finished backward) -> rank r sums elements [r*ceil(n/4/W)*4, ...) of ALL ranks' gradient buffers in rank
 *   order (P2P loads) -> Adam on that slice (same arithmetic and hyper block as vitb_adam_multi; m, v are only maintained for
 *   the owned slice) -> stores the new fp32 parameters and bf16 shadow into EVERY rank's buffers (P2P stores) -> barrier.
 * g_peers / p_peers / shadow_peers / flag_peers: HOST arrays of `world` device pointers (index = rank; the own buffers at [rank];
 * shadow_peers may be NULL).  flag buffers: >= world uint32 each, zeroed once; sync: 4 uint32 of this rank, zeroed once.
 * optimizer: 0 = Adam; 1 = SGD with momentum as vitb_sgd_multi (m is the momentum buffer, v may be NULL).
 * Peer pointers come from vitb_ipc_open.  world <= 8, n % 4 == 0.  Every rank must issue the same sequence of calls; a rank that
 * waits longer than the flag-wait bound for a peer traps (default 600 s; VITB_DP_TIMEOUT_S in the environment or
 * vitb_dp_set_timeout(seconds) change it: all ranks must enter the step within that time of each other).  Replicas end
 * bit-identical. ---- */
int vitb_dp_reduce_adam(const void* const* g_peers, void* const* p_peers, void* const* shadow_peers, void* const* flag_peers, float* m, float* v,
                        uint32_t* sync, int64_t n, int rank, int world, int optimizer, const float* hyper_host, const float* hyper_dev, void* stream);
/* CUDA IPC plumbing for the above (host functions; no kernels).  export: 64-byte handle of the allocation that contains dev_ptr and
 * dev_ptr's byte offset inside it (the caller ships both to the other ranks, e.g. with torch.distributed.all_gather_object).
 * open: maps a peer's allocation into this process (once per handle, cached) with peer access enabled; returns base + offset. */
int vitb_dp_set_timeout(double seconds);
int vitb_ipc_export(const void* dev_ptr, void* handle64, int64_t* offset);
int vitb_ipc_open(const void* handle64, int64_t offset, void** dev_ptr);

#ifdef __cplusplus
}
#endif
#endif /* VITB200_H_ */
