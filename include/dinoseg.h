/* dinoseg.h — C ABI of libdinoseg.so: the B200 (sm_100a) implementation of the DINOSeg
 * inference hot path of sachaMorin/dino.
 *
 * The reference has no FFI layer: its boundary for this path is the Python method surface of
 * `DINOSeg` (dt_segmentation/src/pl_torch_modules.py).  Each entry point below names the
 * reference interface it replaces; `dino_b200/model.py` is the Python host that binds them
 * with ctypes and re-creates that method surface (see INTEGRATION.md).
 *
 * Conventions
 *  - plain pointers and sizes only; `stream` is a cudaStream_t passed as void* (NULL = legacy
 *    default stream); every call is asynchronous on that stream unless stated otherwise.
 *  - return value 0 = ok, negative = error; dinoseg_last_error(h) gives the message
 *    (stored per handle; for a failed dinoseg_create use dinoseg_last_error(NULL)).
 *  - one handle per (GPU, stream); a handle is not thread-safe, independent handles are.
 *  - there is NO CPU path: dinoseg_create fails unless the device is compute capability 10.x.
 */
#ifndef DINOSEG_H_
#define DINOSEG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dinoseg dinoseg_t;

/* Architecture of the truncated ViT + head.
 * Replaces: DINOSeg.__init__ vit branch (pl_torch_modules.py:173-183, heads :219-222) and
 * vit_small / vit_base (vision_transformer.py:300-311). */
typedef struct dinoseg_cfg {
  int32_t embed_dim;  /* 384 (ViT-S) or 768 (ViT-B); multiple of 128 */
  int32_t num_heads;  /* embed_dim / 64 */
  int32_t mlp_hidden; /* 4 * embed_dim */
  int32_t n_blocks;   /* number of leading transformer blocks kept (pl_torch_modules.py:177) */
  int32_t patch;      /* 8 */
  int32_t pos_grid;   /* side of the stored positional grid: 28 (img 224 / patch 8) */
  int32_t n_classes;  /* <= 16 */
  int32_t head_h1;    /* 200 (MLP head, pl_torch_modules.py:113) */
  int32_t head_h2;    /* 100 (pl_torch_modules.py:114) */
  int32_t head_kind;  /* 0 = 'mlp' head: layer_1 / layer_2 / layer_3 (pl_torch_modules.py:108-124);
                       * 1 = 'linear' head: one Linear(embed_dim, n_classes) stored as clf.layer_1,
                       *     head_h1 / head_h2 are ignored (pl_torch_modules.py:127-138) */
  float ln_eps;       /* 1e-6 (vision_transformer.py:303) */
} dinoseg_cfg;

/* Replaces DINOSeg.__init__ (pl_torch_modules.py:144-237) for the vit backbone. */
int dinoseg_create(const dinoseg_cfg* cfg, int device, dinoseg_t** out);
void dinoseg_destroy(dinoseg_t* h);
const char* dinoseg_last_error(const dinoseg_t* h);

/* Copy one fp32 parameter (device pointer) into the handle, keyed by its reference
 * state_dict name ("dino.blocks.0.attn.qkv.weight", "clf.layer_1.bias", ...).
 * Replaces: load_state_dict inside LightningModule.load_from_checkpoint (README.md:31). */
int dinoseg_set_weight(dinoseg_t* h, const char* key, const float* dev_ptr, const int64_t* shape, int ndim,
                       void* stream);
/* number of parameters still missing (0 = ready) */
int dinoseg_missing_weights(const dinoseg_t* h);

/* Replaces DINOSeg.set_resolution (pl_torch_modules.py:270-274); also builds the cached
 * bicubic positional table (vision_transformer.py:202-222).  resolution % 8 != 0 -> error
 * "Resolution should be a multiple of 8."  Same as dinoseg_set_resolution_hw(h, resolution, resolution). */
int dinoseg_set_resolution(dinoseg_t* h, int resolution, void* stream);
/* Frames of height x width pixels: a (height/8) x (width/8) patch grid, tokens = CLS then the patches row by row.  The
 * positional table is resampled per axis as the reference's interpolate_pos_encoding does for [B,3,height,width] input
 * (scale factors ((height/8 + 0.1)/G0, (width/8 + 0.1)/G0)); it is used unchanged only for a G0 x G0 grid.  Either side
 * <= 0 or not a multiple of 8 -> "Resolution should be a multiple of 8."; either grid side > 480 -> error.
 * With height != width: forward, features and CLS attention work (logprobs [batch*gh*gw, C], lowres [batch, gh, gw]);
 * int64 label maps (labels != NULL) and the host entry points (dinoseg_predict_host*) are predict()'s semantics, which
 * exist for square grids only: they return an error and enqueue nothing. */
int dinoseg_set_resolution_hw(dinoseg_t* h, int height, int width, void* stream);

size_t dinoseg_workspace_bytes(const dinoseg_t* h, int batch);

/* Replaces DINOSeg.forward (pl_torch_modules.py:239-256) + the argmax / np.kron tail of
 * DINOSeg.predict (:294-298), batched.
 *   frames   : device, fp32 [batch,3,H,W] NCHW, already normalised (H x W as set by dinoseg_set_resolution[_hw])
 *   logprobs : device, fp32 [batch*P, C] or NULL        (forward's return value; P = gh*gw, gh = H/8, gw = W/8)
 *   lowres   : device, uint8 [batch, gh, gw] or NULL     (argmax per patch)
 *   labels   : device, int64 [batch, g*p, g*p] or NULL   (square grids only, g = gh = gw, p = 480 / g; predict's return
 *                                                         value)
 *   workspace: device scratch of at least dinoseg_workspace_bytes(h, batch) bytes, 1024-aligned */
int dinoseg_forward(dinoseg_t* h, const float* frames, int batch, float* logprobs, uint8_t* lowres,
                    int64_t* labels, void* workspace, size_t workspace_bytes, void* stream);

/* Same computation with HOST buffers (pinned memory recommended): copies the frames to the
 * device, runs dinoseg_forward, copies the label maps back and SYNCHRONISES the stream.
 * This is the call that replaces a loop of DINOSeg.predict() (pl_torch_modules.py:276-300)
 * after preprocessing.  host_lowres / host_labels may be NULL individually.  Internally the batch is
 * pipelined in chunks over three library-owned streams and staging buffers. */
int dinoseg_predict_host(dinoseg_t* h, const float* host_frames, int batch, uint8_t* host_lowres,
                         int64_t* host_labels, void* stream);

/* Asynchronous form: dinoseg_predict_host_submit enqueues the whole submission (copies and kernels on the library's
 * streams) and returns a ticket (> 0; < 0 = error) without waiting for the GPU; the host buffers (frames in, label
 * maps out) must stay valid and untouched until dinoseg_predict_host_wait(h, ticket) has returned 0 (ticket 0 waits for
 * everything outstanding, oldest first).  Up to 4 submissions may be outstanding; they queue behind each other on the
 * same streams, so the first H2D copy of one overlaps the last kernels / D2H copy of the one before - what a caller
 * that streams batches (a camera, a folder of images) wants.  dinoseg_predict_host == submit + wait.
 * Replaces the boundaries `x.to(self.device)` / `.cpu()` of DINOSeg.predict (pl_torch_modules.py:292, :295). */
int64_t dinoseg_predict_host_submit(dinoseg_t* h, const float* host_frames, int batch, uint8_t* host_lowres,
                                    int64_t* host_labels, void* stream);
int64_t dinoseg_predict_host_submit_u8(dinoseg_t* h, const uint8_t* host_frames_u8, int batch, int src_h, int src_w,
                                       const float* mean, const float* std_, uint8_t* host_lowres, int64_t* host_labels,
                                       void* stream);
int dinoseg_predict_host_wait(dinoseg_t* h, int64_t ticket);

/* The same two calls on RAW camera frames: uint8 RGB, HWC, [batch, src_h, src_w, 3].  Replaces the inference
 * transforms of DINOSeg.predict (pl_torch_modules.py:33-41, :291: albumentations Resize(r, r) -> Normalize(mean, std)
 * -> ToTensorV2) on the GPU, fused into the patch-embed im2col: the bilinear resize reproduces cv2.resize(INTER_LINEAR)
 * on 8-bit images bit for bit (11-bit fixed-point weights, result rounded to uint8), the normalisation is
 * (pix - mean*255) * (1 / (std*255)) in fp32.  mean / std: 3 host floats each (ImageNet values in the reference).
 * The frames are resized to the H x W set by dinoseg_set_resolution[_hw] (cv2.resize(img, (W, H)), each axis with its
 * own scale); frames of exactly H x W pass through unchanged. */
int dinoseg_forward_u8(dinoseg_t* h, const uint8_t* frames_u8, int batch, int src_h, int src_w, const float* mean,
                       const float* std_, float* logprobs, uint8_t* lowres, int64_t* labels, void* workspace,
                       size_t workspace_bytes, void* stream);
int dinoseg_predict_host_u8(dinoseg_t* h, const uint8_t* host_frames_u8, int batch, int src_h, int src_w,
                            const float* mean, const float* std_, uint8_t* host_lowres, int64_t* host_labels,
                            void* stream);

/* Frames per pipeline chunk of dinoseg_predict_host (0 = automatic, the default): the host batch is processed in chunks
 * whose H2D copy, kernels and D2H copy overlap across two internal streams. */
int dinoseg_set_host_chunk(dinoseg_t* h, int frames_per_chunk);

/* How the host entry points produce the int64 label maps.  0: the maps are replicated on the GPU and copied out whole
 * (8*(g*p)^2 bytes per frame).  1: the low-res maps (g*g bytes per frame) are copied to the host and expanded there by
 * worker threads into the caller's buffer while later chunks / submissions compute - what the reference does with
 * np.kron (pl_torch_modules.py:297-298), 512x fewer bytes over PCIe.  Identical bytes either way.  -1 (default):
 * automatic - host expansion when this rank has at least 8 host cores to itself (cores of the process / ranks per
 * host), the DMA path otherwise.  dinoseg_get_host_expand returns the mode in effect (0 / 1). */
int dinoseg_set_host_expand(dinoseg_t* h, int on);
int dinoseg_get_host_expand(const dinoseg_t* h);
/* The host-side expansion itself (pure CPU, no device needed): lowres host uint8 [batch, g, g] -> labels host int64
 * [batch, g*p, g*p], out[b, y, x] = lowres[b, y / p, x / p] (np.kron with ones((p, p))); g*p <= 480. */
int dinoseg_expand_labels_host(const uint8_t* lowres, int batch, int g, int p, int64_t* labels);

/* CTA-pair (tcgen05 cta_group::2) forms of the fused MLP and of the qkv / patch-embed (ViT-B: fc1, fc2) GEMMs: M = 256
 * MMAs issued by the leader CTA of a 2-CTA cluster, weights split between the two SMs.  Bit-identical results, about
 * +2 % frames/s (ViT-B: +5 %).  On by default; 0 selects the single-CTA kernels (also DINOSEG_PAIR=0 in the
 * environment at dinoseg_create time). */
int dinoseg_set_pair_kernels(dinoseg_t* h, int on);
int dinoseg_get_pair_kernels(const dinoseg_t* h);   /* bit 0: GEMMs, bit 1: fused MLP */

/* CLS-query attention of the last kept block: attn [batch, heads, N] fp32 = softmax(q_cls k^T * dh^-0.5) per head,
 * i.e. row 0 of what VisionTransformer.get_last_selfattention returns (vision_transformer.py:273-280) — the only
 * row its caller reads (visualize_attention.py:46-54).  frames: device fp32 [batch,3,H,W]; N = gh*gw + 1. */
int dinoseg_cls_attention(dinoseg_t* h, const float* frames, int batch, float* attn, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Backbone features: VisionTransformer.get_intermediate_layers(x, n_last) (vision_transformer.py:282-290) in one pass
 * over the blocks, without the head.  out: device fp32 [min(n_last, n_blocks), batch, N, D], N = gh*gw + 1 (CLS
 * token first); slice k = dino.norm (eps ln_eps) applied to the residual stream after block
 * n_blocks - min(n_last, n_blocks) + k, so the last slice is what VisionTransformer.forward returns for all tokens.
 * frames: device fp32 [batch,3,H,W] (normalised).  Workspace as for dinoseg_forward (dinoseg_workspace_bytes).
 * n_last < 1, out == NULL, no resolution set, a model without blocks or a too small workspace: error. */
int dinoseg_features(dinoseg_t* h, const float* frames, int batch, int n_last, float* out, void* workspace,
                     size_t workspace_bytes, void* stream);
/* The same on raw uint8 HWC frames [batch, src_h, src_w, 3], resized and normalised as in dinoseg_forward_u8. */
int dinoseg_features_u8(dinoseg_t* h, const uint8_t* frames_u8, int batch, int src_h, int src_w, const float* mean,
                        const float* std_, int n_last, float* out, void* workspace, size_t workspace_bytes,
                        void* stream);

/* Image embeddings: one vector per frame instead of the token tensor, in one pass over the blocks (no head).
 * cls_out: device fp32 [min(n_last, n_blocks), batch, D] or NULL; slice k = dino.norm of the CLS row after block
 * n_blocks - min(n_last, n_blocks) + k (dinoseg_features without the token axis).  patch_mean: device fp32
 * [batch, D] or NULL = the mean over the patch tokens (not CLS) of dino.norm of the last block's output.
 * With patch_mean == NULL the last block runs for the CLS row only after its qkv GEMM (LayerNorm1 and the qkv GEMM
 * still cover every token); the last cls_out slice then agrees with dinoseg_features' CLS row to bf16 rounding of
 * the attention / MLP operands, and every earlier slice is bit-identical to it.  With patch_mean, the last block
 * runs in full and every cls_out slice is bit-identical to dinoseg_features' CLS rows.  Workspace as for
 * dinoseg_forward.  Both outputs NULL, n_last < 1, no resolution set, a model without blocks or a too small
 * workspace: error, nothing enqueued. */
int dinoseg_embeddings(dinoseg_t* h, const float* frames, int batch, int n_last, float* cls_out, float* patch_mean,
                       void* workspace, size_t workspace_bytes, void* stream);
/* The same on raw uint8 HWC frames [batch, src_h, src_w, 3], resized and normalised as in dinoseg_forward_u8. */
int dinoseg_embeddings_u8(dinoseg_t* h, const uint8_t* frames_u8, int batch, int src_h, int src_w, const float* mean,
                          const float* std_, int n_last, float* cls_out, float* patch_mean, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Controller-side reduction on the label map (the step after predict() in the robot pipeline, reference
 * docs/index.html "Controller": left / right obstacle masks for the potential-field controller).
 * lowres: device uint8 [batch, g, g] as written by dinoseg_forward; the output map is (g*p) x (g*p).
 * counts: device int32 [batch, 2, n_classes] = pixels of each class with x < g*p/2 (side 0) and x >= g*p/2 (side 1). */
int dinoseg_half_counts(const uint8_t* lowres, int batch, int g, int p, int n_classes, int32_t* counts, void* stream);

/* Output side of predict() on given log-probs: argmax (first max wins, NaN counts as max)
 * then p x p block replication.  Bit-exact w.r.t. torch.argmax + np.kron.
 * (pl_torch_modules.py:295-298).  rows = batch*g*g. */
int dinoseg_argmax_replicate(const float* logprobs, int batch, int g, int n_classes, int p, uint8_t* lowres,
                             int64_t* labels, void* stream);

/* ---- introspection (used by tests and bench) ------------------------------------------ */
/* Copy an internal device buffer of the LAST forward into dst (device pointer).
 * names: "pos" fp32 [N,D] | "x" fp32 [B*N,D] residual stream after the last executed stage |
 * "abuf" bf16 [B*N,D] | "qkv" bf16 [B*N,3D].  Returns the number of bytes copied or <0. */
int64_t dinoseg_copy_buffer(dinoseg_t* h, const char* name, void* dst, size_t dst_bytes, void* stream);
/* Stop the next forwards after stage k (debug): 0 = run everything, 1 = after prepare_tokens,
 * 2+3*i = after block i's qkv GEMM, 3+3*i = after block i's attention+proj, 4+3*i = after block i */
int dinoseg_set_debug_stop(dinoseg_t* h, int stage);
/* number of kernels launched by the last dinoseg_forward */
int dinoseg_last_launch_count(const dinoseg_t* h);
/* Per-kernel-kind device timing: when enabled, every launch of the following forwards is
 * bracketed by a pair of cudaEvents on the launching stream; dinoseg_profile_read waits for
 * them, sums the elapsed milliseconds and launch counts per kind (since enable / last read)
 * and resets the accumulation. */
int dinoseg_profile_enable(dinoseg_t* h, int on);
/* restrict the events to the kinds whose bit is set (default: all kinds) */
int dinoseg_profile_set_mask(dinoseg_t* h, uint32_t kind_mask);
/* Diagnostic for work that does not finish; may be called from another host thread while the launching thread is
 * blocked: the profiled launches (dinoseg_profile_enable) that have started and not ended, i.e. the kernels running or
 * stuck right now (kinds[] as in dinoseg_profile_kind_name, slots[] = launch index since profiling was enabled).
 * Returns the number written (<= max_out), -2 if profiling is off; *not_started = launches still queued behind them. */
int dinoseg_debug_pending_kinds(dinoseg_t* h, int* kinds, int* slots, int max_out, int* not_started);
/* Diagnostic: per-SM marks of the tcgen05 kernels (entry [sm] = kernel code * 10 + stage while a CTA of that kernel
 * sits on the SM, negative once it has left; codes and stages: csrc/ptx.cuh hb_mark, csrc/dinoseg_api.cu).  Copied on a
 * stream of its own: usable from another thread while the data streams are stuck.  Returns n or < 0. */
int dinoseg_debug_heartbeat(int* host_out, int n);
int dinoseg_profile_num_kinds(void);
const char* dinoseg_profile_kind_name(int kind);
int dinoseg_profile_read(dinoseg_t* h, float* ms_by_kind, int* launches_by_kind, int n_kinds);
/* Call before dinoseg_profile_read: span_ms = first launch's start -> last launch's end, gap_ms = the part of it that
 * lies between launches (measurement hook) */
int dinoseg_profile_gaps(dinoseg_t* h, float* span_ms, float* gap_ms);

/* ---- kernel-level entry points (parity tests of the individual CUDA kernels) ----------- */
/* C[M,N] = A[M,K] bf16 x W[N,K]^T bf16 with epilogue `epi` (see csrc/gemm.cuh EPI_*) */
int dinoseg_op_gemm(const void* A_bf16, const void* W_bf16, const float* bias, void* out, int M, int N, int K,
                    int ldo, int epi, float col_scale, int scale_cols, const float* pos, int P, int Ntok,
                    void* stream);
/* dinoseg_op_gemm (epilogues 0 bf16, 1 GELU bf16, 2 residual fp32) run by CTA pairs (tcgen05 cta_group::2: 256 x 192
 * tiles, the W tile split between the two SMs) - how the qkv GEMM (and ViT-B's fc1 / fc2) of the forward are launched */
int dinoseg_op_gemm_pair(const void* A, const void* W, const float* bias, void* out, int M, int N, int K, int ldo, int epi,
                         float col_scale, int scale_cols, void* stream);
/* out[B*N, D] bf16 = softmax(q k^T) v over qkv[B, N, 3D] bf16; q carries dh^-0.5 * log2(e) already (the qkv GEMM's
 * epilogue applies it), i.e. the kernel computes P = 2^(q k^T) */
int dinoseg_op_attention(const void* qkv_bf16, void* out_bf16, int B, int N, int H, void* stream);
/* Test hook: synchronises the device; 1 if the process's most recent attention launch left the range of the kernel
 * without row maxima and was redone by the classic kernel, 0 if not, -1 on a CUDA error. */
int dinoseg_debug_attn_redone(void);
/* Test hook (pure CPU): worker pool of the host entry points with n threads where the creation of thread fail_at fails
 * (< 0: none); returns the threads the pool ended up with (0: none, the caller falls back to the DMA path), -1 on error. */
int dinoseg_debug_host_pool(int n, int fail_at);
/* Host-side copy of the attention kernel's work-item plan (pure CPU): item i -> {bh0, q0_0, bh1, q0_1, active1, dual}
 * (frame*H + head and first query row of warpgroup 0 / 1).  items == NULL returns the item count. */
int dinoseg_debug_attn_items(int B, int H, int N, int32_t* items, int max_items);
/* Debug builds only (-DDSG_ATTN_TIMING): device buffer [grid][2][8] of int64 receiving the per-phase
 * cycle totals of the attention kernel's softmax warpgroups; returns -1 in regular builds. */
int dinoseg_debug_set_attn_timing(long long* dev_ptr);
/* x[M,384] fp32 (in place) += fc2(gelu(fc1(A))) with A [M,384] bf16 (= LayerNorm2(x)), W1 [1536,384], W2 [384,1536]
 * bf16: the fused transformer-MLP kernel (reference vision_transformer.py:135, :59-65) */
int dinoseg_op_mlp(float* x, const void* A_bf16, const void* W1_bf16, const float* b1, const void* W2_bf16,
                   const float* b2, int M, void* stream);
/* the same kernel run by CTA pairs (tcgen05 cta_group::2, M = 256 per MMA, weights split between the two SMs) when pair != 0 */
int dinoseg_op_mlp_ex(float* x, const void* A_bf16, const void* W1_bf16, const float* b1, const void* W2_bf16,
                      const float* b2, int M, int pair, void* stream);
/* LayerNorm folded into the Linear layer that consumes it: W [N,K] fp32, bias [N], gamma / beta [K] ->
 * W_out bf16 = W * gamma (per input column), bias_out = bias + W . beta.  Linear(LN(x)) = W_out xhat + bias_out with
 * xhat = (x - mean) * rstd: how the fused MLP kernel gets LayerNorm2's affine transform (vision_transformer.py:118). */
int dinoseg_op_fold_ln(const float* W, const float* bias, const float* gamma, const float* beta, int N, int K,
                       void* W_out_bf16, float* bias_out, void* stream);
/* x[M,384] fp32 (in place) += fc2(gelu(fc1'(xhat(x)))): the fused MLP kernel in the form the forward uses, normalising
 * the fp32 residual stream itself; W1f / b1f carry LayerNorm2's gamma / beta (dinoseg_op_fold_ln)
 * (vision_transformer.py:118, :135) */
int dinoseg_op_mlp_ln(float* x, float eps, const void* W1f_bf16, const float* b1f, const void* W2_bf16, const float* b2,
                      int M, int pair, void* stream);
/* 0: unfused LN / fc1 / fc2 kernels; 1: fused MLP kernel, one CTA per row block; 2: fused MLP kernel run by CTA pairs
 * (cta_group::2); 2 is the default where the fused kernel applies (embed_dim 384, mlp_hidden 1536) */
int dinoseg_set_fused_mlp(dinoseg_t* h, int on);
/* 1 (default where it applies: 'mlp' head, embed_dim 384): final LayerNorm -> layer_1 -> layer_2 -> layer_3 -> log_softmax
 * -> argmax -> p x p replication in ONE kernel (csrc/head.cuh); 0: the separate LayerNorm / GEMM / GEMM / tail kernels */
int dinoseg_set_fused_head(dinoseg_t* h, int on);
int dinoseg_op_layernorm(const float* x, const float* gamma, const float* beta, void* y_bf16, int M, int D,
                         float eps, void* stream);
/* y[M,D] fp32 = LayerNorm(x) * gamma + beta, D = 384 or 768: the kernel behind dinoseg_features */
int dinoseg_op_layernorm_f32(const float* x, const float* gamma, const float* beta, float* y, int M, int D,
                             float eps, void* stream);
int dinoseg_op_posembed(const float* pos_src, float* out, int G0, int g, int D, void* stream);
int dinoseg_op_im2col(const float* frames, void* A_bf16, int B, int g, void* stream);
int dinoseg_op_f32_to_bf16(const float* in, void* out_bf16, size_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DINOSEG_H_ */
