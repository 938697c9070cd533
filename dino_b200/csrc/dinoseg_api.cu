// libdinoseg.so — C-ABI implementation (see include/dinoseg.h).
// Host-side orchestration only: weight packing, tensor-map construction, launch sequence.
// The kernels are in gemm.cuh (tcgen05 GEMM), attention.cuh (tcgen05 flash attention) and
// kernels.cuh (memory-bound pieces).
#include "../../include/dinoseg.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <mutex>
#include <thread>
#include <sched.h>
#include <emmintrin.h>
#include <set>
#include <string>
#include <system_error>
#include <vector>

#include "attention.cuh"
#include "gemm.cuh"
#include "head.cuh"
#include "kernels.cuh"
#include "mlp.cuh"

using namespace dsg;

namespace {

// -----------------------------------------------------------------------------------------
// errors
// -----------------------------------------------------------------------------------------
thread_local std::string g_create_error;

#define DSG_FAIL(h, ...)                                 \
  do {                                                   \
    char _buf[512];                                      \
    snprintf(_buf, sizeof(_buf), __VA_ARGS__);           \
    if (h) (h)->err = _buf; else g_create_error = _buf;  \
    return -1;                                           \
  } while (0)

#define DSG_CUDA(h, call)                                                                     \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess) DSG_FAIL(h, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), \
                                    __FILE__, __LINE__);                                      \
  } while (0)

// -----------------------------------------------------------------------------------------
// TMA tensor maps (driver entry point fetched through the runtime: no -lcuda needed)
// -----------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

// bf16 2-D row-major matrix [rows, cols] (cols contiguous, row pitch ld elements); box {64, box_rows}, SWIZZLE_128B
bool make_tmap_2d(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t es[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// generic 3-D view {cols, rows, batches} of a row-major buffer (row pitch ld elements, batch pitch
// rows*ld unless given); box {box_cols, box_rows, 1}, SWIZZLE_128B (box_cols * elem size must be 128 B)
bool make_tmap_3d(CUtensorMap* m, const void* ptr, bool f32, uint64_t cols, uint64_t rows, uint64_t batches,
                  uint64_t ld, uint32_t box_cols, uint32_t box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return false;
  const uint64_t es_bytes = f32 ? 4 : 2;
  cuuint64_t dims[3] = {cols, rows, batches};
  cuuint64_t strides[2] = {ld * es_bytes, rows * ld * es_bytes};
  cuuint32_t box[3] = {box_cols, box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  return enc(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr),
             dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// A operand of the GEMM: bf16 {K, rows, batches}, box {64, 128, 1}
bool make_tmap_gemm_a(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t batches, uint64_t K) {
  return make_tmap_3d(m, ptr, false, K, rows, batches, K, 64, GEMM_BM);
}
// output / addend of the GEMM: {N, rows, batches} with row pitch ld; box = one staging chunk (128 B x 128 rows)
bool make_tmap_gemm_out(CUtensorMap* m, const void* ptr, bool f32, uint64_t N, uint64_t rows, uint64_t batches,
                        uint64_t ld) {
  return make_tmap_3d(m, ptr, f32, N, rows, batches, ld, f32 ? 32 : 64, GEMM_BM);
}

// qkv [B, N, ld] bf16 viewed as {ld, N, B}; box {64, 128, 1}: rows >= N of a frame read as zeros
bool make_tmap_qkv(CUtensorMap* m, const void* ptr, uint64_t B, uint64_t N, uint64_t ld) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[3] = {ld, N, B};
  cuuint64_t strides[2] = {ld * 2, N * ld * 2};
  cuuint32_t box[3] = {64, 128, 1};
  cuuint32_t es[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// -----------------------------------------------------------------------------------------
// kernel launchers
// -----------------------------------------------------------------------------------------
constexpr int kAttnStages = 6;   // 6 x 32 KB K|V stages + 2 Q tiles = 224 KB (dual tail items run two 3-deep streams)
long long* g_attn_timing = nullptr;   // debug: device buffer for the DSG_*_TIMING builds
int* g_heartbeat = nullptr;           // diagnostic: per-SM (kernel, stage) marks of the tcgen05 kernels (hb_mark), 1024 ints

// The weight tensor maps come in two flavours: full 128-row granules (plain kernel) and 64-row half granules (cluster
// kernel: each CTA of a cta_group::2 pair holds one half of the B operand).
cudaError_t launch_mlp_fused(const CUtensorMap& a, const CUtensorMap& w1, const CUtensorMap& w2, const CUtensorMap& x,
                             const MlpParams& p, int num_sms, bool pair, cudaStream_t s) {
  static bool attr[64][2] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr[dev & 63][pair]) {
    cudaError_t e = pair ? cudaFuncSetAttribute(mlp_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(MLP_SMEM))
                              : cudaFuncSetAttribute(mlp_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(MLP_SMEM));
    if (e != cudaSuccess) return e;
    attr[dev & 63][pair] = true;
  }
  MlpParams pp = p;
  pp.timing = g_attn_timing;
  pp.hb = g_heartbeat;
  const int m_blocks = (p.M + MLP_BM - 1) / MLP_BM;
  if (!pair) {
    const int grid = m_blocks < num_sms ? m_blocks : num_sms;
    mlp_fused_kernel<false><<<grid, MLP_THREADS, MLP_SMEM, s>>>(a, w1, w2, x, pp);
    return cudaGetLastError();
  }
  const int pairs = (m_blocks + 1) / 2;
  const int max_pairs = num_sms / 2;
  const int grid = 2 * (pairs < max_pairs ? pairs : max_pairs);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(MLP_THREADS);
  cfg.dynamicSmemBytes = MLP_SMEM;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, mlp_fused_kernel<true>, a, w1, w2, x, pp);
}

constexpr int kLinPitch = 16;    // row pitch (floats) of the 'linear' head's logits buffer (n_classes <= 16)
constexpr int kHeadPart = 256;   // width of each bf16x3 part of relu(layer_1) (head_h1 <= 256, zero padded)

// Single-CTA launch: persistent CTAs, A and W tiles streamed through the ring.
template <int EPI>
cudaError_t launch_gemm_t(const CUtensorMap& a, const CUtensorMap& w, const CUtensorMap& out, const CUtensorMap& add,
                          const GemmParams& p, int num_sms, cudaStream_t s) {
  auto kern = gemm_bf16_tn_kernel<EPI, false>;
  constexpr size_t smem = gemm_smem_bytes(EPI, false, false);
  static_assert(smem <= 227 * 1024, "shared memory budget");
  static bool attr[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    attr[dev & 63] = true;
  }
  const int n_tiles = (p.N + GEMM_BN - 1) / GEMM_BN;
  const int m_tiles = (p.rows_per_batch + GEMM_BM - 1) / GEMM_BM * p.batches;
  const long long total = (long long)n_tiles * m_tiles;
  if (total <= 0 || total > INT32_MAX || p.K % GEMM_BK != 0 || n_tiles * GEMM_BN > GEMM_MAX_N) return cudaErrorInvalidValue;
  const int grid = total < num_sms ? int(total) : num_sms;    // persistent: one CTA per SM
  GemmParams pp = p;
  pp.timing = g_attn_timing;
  pp.hb = g_heartbeat;
  kern<<<grid, GEMM_THREADS, smem, s>>>(a, w, out, add, pp);
  return cudaGetLastError();
}

// CTA-pair launch (cta_group::2, gemm.cuh): `w` must be a tensor map with 96-row boxes (half a W tile).
// RES_A: the A row block (K <= 384) stays in shared memory for all n-tiles of its row-block pair.
template <int EPI, bool RES_A>
cudaError_t launch_gemm_pair_t(const CUtensorMap& a, const CUtensorMap& w, const CUtensorMap& out, const CUtensorMap& add,
                               const GemmParams& p, int num_sms, cudaStream_t s) {
  auto kern = gemm_bf16_tn_kernel<EPI, RES_A, true>;
  constexpr size_t smem = gemm_smem_bytes(EPI, RES_A, true);
  static_assert(smem <= 227 * 1024, "shared memory budget");
  static bool attr[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    attr[dev & 63] = true;
  }
  const int n_tiles = (p.N + GEMM_BN - 1) / GEMM_BN;
  const int m_tiles = (p.rows_per_batch + GEMM_BM - 1) / GEMM_BM * p.batches;
  const long long units = RES_A ? (m_tiles + 1) / 2 : (long long)n_tiles * ((m_tiles + 1) / 2);
  if (units <= 0 || units > INT32_MAX || p.K % GEMM_BK != 0 || n_tiles * GEMM_BN > GEMM_MAX_N) return cudaErrorInvalidValue;
  const int max_pairs = num_sms / 2;
  GemmParams pp = p;
  pp.timing = g_attn_timing;
  pp.hb = g_heartbeat;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * unsigned(units < max_pairs ? units : max_pairs));
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, a, w, out, add, pp);
}

template <int EPI>
cudaError_t launch_gemm_pair(const CUtensorMap& a, const CUtensorMap& w, const CUtensorMap& out, const CUtensorMap& add,
                             const GemmParams& p, int num_sms, cudaStream_t s) {
  // resident A (K <= 384: ViT-S qkv) measured best inside the whole step (7.56-7.71 k frames/s against 7.51-7.58 k
  // for streaming pairs and 7.47-7.54 k for single-CTA tiles)
  const bool res_a = p.K <= GEMM_RES_KB * GEMM_BK && p.N > GEMM_BN && p.a_wrap == 0;
  return res_a ? launch_gemm_pair_t<EPI, true>(a, w, out, add, p, num_sms, s)
               : launch_gemm_pair_t<EPI, false>(a, w, out, add, p, num_sms, s);
}

cudaError_t launch_gemm(int epi, const CUtensorMap& a, const CUtensorMap& w, const CUtensorMap& out,
                        const CUtensorMap& add, const GemmParams& p, int num_sms, cudaStream_t s) {
  switch (epi) {
    case EPI_BF16: return launch_gemm_t<EPI_BF16>(a, w, out, add, p, num_sms, s);
    case EPI_GELU_BF16: return launch_gemm_t<EPI_GELU_BF16>(a, w, out, add, p, num_sms, s);
    case EPI_RESID_F32: return launch_gemm_t<EPI_RESID_F32>(a, w, out, add, p, num_sms, s);
    case EPI_PATCH_F32: return launch_gemm_t<EPI_PATCH_F32>(a, w, out, add, p, num_sms, s);
    case EPI_RELU_F32: return launch_gemm_t<EPI_RELU_F32>(a, w, out, add, p, num_sms, s);
    case EPI_RELU_SPLIT_BF16: return launch_gemm_t<EPI_RELU_SPLIT_BF16>(a, w, out, add, p, num_sms, s);
    case EPI_BIAS_F32: return launch_gemm_t<EPI_BIAS_F32>(a, w, out, add, p, num_sms, s);
  }
  return cudaErrorInvalidValue;
}


// work-item plan of the attention kernel (see att_decode): lone last query tiles are paired across heads
void attn_plan_items(AttnParams& p) {
  const int q_tiles = (p.N + ATT_BM - 1) / ATT_BM;
  p.full_pairs = q_tiles / 2;
  p.lone = q_tiles & 1;
  p.num_items = p.B * p.H * p.full_pairs + (p.lone ? (p.B * p.H + 1) / 2 : 0);
}

// One device word per attention launch (slot = launch id mod 256) through which the unshifted kernel tells the shifted
// one, enqueued right behind it, that it has to redo the launch (attention.cuh, att_softmax_unshifted).
int* attn_range_flags(int dev) {
  static int* flags[64] = {};
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  int*& f = flags[dev & 63];
  if (f == nullptr) {
    if (cudaMalloc(&f, 256 * sizeof(int)) != cudaSuccess) { f = nullptr; return nullptr; }
    cudaMemset(f, 0, 256 * sizeof(int));
  }
  return f;
}
std::atomic<int> g_attn_launch_id{0};
int* g_attn_last_flag = nullptr;
int g_attn_last_id = 0;

template <bool UNSHIFTED>
cudaError_t launch_attention_kernel(const CUtensorMap& qkv, const AttnParams& p, int num_sms, int dev, cudaStream_t s) {
  auto kern = attn_fwd_kernel<kAttnStages, UNSHIFTED>;
  constexpr size_t smem = attn_smem_bytes<kAttnStages>();
  static bool attr[64] = {};
  if (!attr[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    attr[dev & 63] = true;
  }
  const int grid = p.num_items < num_sms ? p.num_items : num_sms;  // persistent: one CTA per SM
  kern<<<grid, ATT_THREADS, smem, s>>>(qkv, p);
  return cudaGetLastError();
}

// unshifted = true: the kernel without row maxima, followed by the classic one as its (normally empty) redo
cudaError_t launch_attention(const CUtensorMap& qkv, AttnParams p, int num_sms, cudaStream_t s, bool unshifted = true) {
  p.timing = g_attn_timing;
  p.hb = g_heartbeat;
  attn_plan_items(p);
  int dev = 0;
  cudaGetDevice(&dev);
  p.range_flag = nullptr;
  p.launch_id = 0;
  if (!unshifted) return launch_attention_kernel<false>(qkv, p, num_sms, dev, s);
  int* flags = attn_range_flags(dev);
  if (flags == nullptr) return cudaErrorMemoryAllocation;
  int id = ++g_attn_launch_id;
  if (id <= 0) { g_attn_launch_id = 1; id = 1; }
  p.range_flag = flags + (id & 255);
  p.launch_id = id;
  g_attn_last_flag = p.range_flag;
  g_attn_last_id = id;
  cudaError_t e = launch_attention_kernel<true>(qkv, p, num_sms, dev, s);
  if (e != cudaSuccess) return e;
  return launch_attention_kernel<false>(qkv, p, num_sms, dev, s);
}

cudaError_t launch_layernorm(const float* x, const float* g, const float* b, __nv_bfloat16* y, int M, int D, float eps,
                             bool split, cudaStream_t s) {
  const int rows_per_block = 8;
  dim3 grid((M + rows_per_block - 1) / rows_per_block);
  if (D == 384 && !split) layernorm384_kernel<__nv_bfloat16><<<(M + 31) / 32, 256, 0, s>>>(x, g, b, y, M, eps);
  else if (D == 768 && !split) layernorm_kernel<768, false, __nv_bfloat16><<<grid, 256, 0, s>>>(x, g, b, y, M, eps);
  else if (D == 384 && split) layernorm_kernel<384, true, __nv_bfloat16><<<grid, 256, 0, s>>>(x, g, b, y, M, eps);
  else if (D == 768 && split) layernorm_kernel<768, true, __nv_bfloat16><<<grid, 256, 0, s>>>(x, g, b, y, M, eps);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}

// fp32 output (backbone features: dino.norm applied to the residual stream), same kernels as above
cudaError_t launch_layernorm_f32(const float* x, const float* g, const float* b, float* y, int M, int D, float eps,
                                 cudaStream_t s) {
  if (M <= 0) return cudaErrorInvalidValue;
  if (D == 384) layernorm384_kernel<float><<<(M + 31) / 32, 256, 0, s>>>(x, g, b, y, M, eps);
  else if (D == 768) layernorm_kernel<768, false, float><<<(M + 7) / 8, 256, 0, s>>>(x, g, b, y, M, eps);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}

// Embedding kernels (kernels.cuh): clusters of EMB_SPLIT CTAs along x
template <typename... KArgs, typename... Args>
cudaError_t launch_emb_cluster(void (*kern)(KArgs...), dim3 grid, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(EMB_THREADS);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = EMB_SPLIT; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// o [B, D] bf16 = attention output of the CLS query, xc [B, D] fp32 = CLS rows of x
cudaError_t launch_cls_attn_out(const __nv_bfloat16* qkv, const float* x, __nv_bfloat16* o, float* xc, int B, int N,
                                int D, int H, cudaStream_t s) {
  return launch_emb_cluster(cls_attn_out_kernel, dim3(EMB_SPLIT, H, B), s, qkv, x, o, xc, N, D);
}

// cls [B, D] (or null) = final norm of the CLS rows, mean [B, D] = final norm averaged over the patch tokens
cudaError_t launch_embed_pool(const float* x, const float* g, const float* b, float* cls, float* mean, int B, int Ntok,
                              int D, float eps, cudaStream_t s) {
  if (D == 384) return launch_emb_cluster(embed_pool_kernel<384>, dim3(EMB_SPLIT, B), s, x, g, b, cls, mean, Ntok, eps);
  if (D == 768) return launch_emb_cluster(embed_pool_kernel<768>, dim3(EMB_SPLIT, B), s, x, g, b, cls, mean, Ntok, eps);
  return cudaErrorInvalidValue;
}

// gh x gw patch grid (gh rows, gw columns)
cudaError_t launch_posembed(const float* pos_src, float* out, int G0, int gh, int gw, int D, cudaStream_t s) {
  if (gh == G0 && gw == G0) {
    // reference vision_transformer.py:205-206 (npatch == N and w == h): same grid -> table returned unchanged.  A
    // rectangle with gh*gw == G0*G0 (14 x 56) is resampled.
    return cudaMemcpyAsync(out, pos_src, size_t(G0 * G0 + 1) * D * sizeof(float), cudaMemcpyDeviceToDevice, s);
  }
  // reference :212-217 (python doubles): scale_factor = ((gh + 0.1) / G0, (gw + 0.1) / G0), the first for the rows
  // (its `w` is x.shape[2]); ATen compute_scales_value<float> per axis
  const float rscale_y = float(1.0 / ((double(gh) + 0.1) / double(G0)));
  const float rscale_x = float(1.0 / ((double(gw) + 0.1) / double(G0)));
  const size_t total = size_t(gh * gw + 1) * D;
  posembed_bicubic_kernel<<<unsigned((total + 255) / 256), 256, 0, s>>>(pos_src, out, G0, gh, gw, D, rscale_y, rscale_x);
  return cudaGetLastError();
}

cudaError_t launch_im2col(const float* frames, __nv_bfloat16* A, int B, int gh, int gw, cudaStream_t s) {
  const size_t total = size_t(B) * 3 * gh * 4 * gw;
  im2col_patch8_kernel<<<unsigned((total + 255) / 256), 256, 0, s>>>(frames, A, B, gh, gw);
  return cudaGetLastError();
}

cudaError_t launch_im2col_u8(const uint8_t* frames, __nv_bfloat16* A, int B, int gh, int gw, const PreprocParams& pp,
                             cudaStream_t s) {
  const size_t total = size_t(B) * 3 * (gh * 8) * gw;
  im2col_u8_kernel<<<unsigned((total + 255) / 256), 256, 0, s>>>(frames, A, B, gh, gw, pp);
  return cudaGetLastError();
}

cudaError_t launch_replicate(const uint8_t* lowres, int64_t* labels, int B, int g, int p, cudaStream_t s) {
  const int W = g * p;
  const size_t total = (W & 1) ? size_t(B) * W * W : size_t(B) * W * (W / 2);
  if (total == 0) return cudaSuccess;
  replicate_labels_kernel<<<unsigned((total + 255) / 256), 256, 0, s>>>(lowres, reinterpret_cast<long long*>(labels),
                                                                        B, g, p);
  return cudaGetLastError();
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct BlockW {
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  __nv_bfloat16 *qkv_w = nullptr, *proj_w = nullptr, *fc1_w = nullptr, *fc2_w = nullptr;
  float *qkv_b = nullptr, *proj_b = nullptr, *fc1_b = nullptr, *fc2_b = nullptr;
  // fc1 as loaded (fp32): fc1_w / fc1_b above are derived from these by finalize_weights - plain bf16 / copy, or with
  // LayerNorm2's gamma / beta folded in when the fused MLP kernel computes the LayerNorm itself
  float *fc1_w32 = nullptr, *fc1_b32 = nullptr;
  CUtensorMap tm_qkv, tm_proj, tm_fc1, tm_fc2;
  CUtensorMap tm_fc1_g, tm_fc2_g;   // 128-row granule views for the fused MLP kernel
  CUtensorMap tm_fc1_h, tm_fc2_h;   // 64-row half granules (CTA-pair variant)
  CUtensorMap tm_qkv_h, tm_fc1_p, tm_fc2_p;   // 96-row half W tiles (CTA-pair GEMMs)
};

struct WeightSlot {
  int kind;  // 0 = fp32 copy, 1 = bf16 convert, 3 = bf16x3 split [hi|hi|lo], 4 = same with K padded to kHeadPart
  void* dst;
  std::vector<int64_t> shape;
};

// One activation workspace carved into the buffers of a forward pass, with the tensor maps that
// describe them (valid for one (base pointer, batch, height, width) binding).
struct WorkBufs {
  void* base = nullptr;
  int batch = 0, res_h = 0, res_w = 0;
  float* x = nullptr;               // fp32 residual stream [B*N, D]
  __nv_bfloat16* abuf = nullptr;    // bf16 GEMM A operand [B*N, D] (LayerNorm / attention output)
  __nv_bfloat16* qkv = nullptr;     // bf16 [B*N, 3D]
  __nv_bfloat16* hid = nullptr;     // bf16 [B*N, hidden]; also im2col [B*P, 192] and head h1 fp32 [B*N, H1]
  uint8_t* lowres = nullptr;        // [B*P]
  CUtensorMap tm_im2col, tm_abuf, tm_hid, tm_qkv3d;                                  // A operands / attention
  CUtensorMap tm_x_out, tm_x_patch, tm_pos_add, tm_qkv_out, tm_hid_out;              // GEMM outputs / addends
  CUtensorMap tm_qkv_a, tm_h1s_out, tm_h1s_a, tm_h2_out, tm_lin_out;                 // segmentation head
  // CLS rows of the last block (embeddings), in regions that are dead by then: the attention / LayerNorm2 output
  // [B, D] bf16 at the start of abuf, the residual rows [B, D] fp32 (also the gather buffer of the earlier blocks'
  // CLS rows) and the fc1 output [B, hidden] bf16 in hid
  float* cls_x = nullptr;
  __nv_bfloat16* cls_hid = nullptr;
  CUtensorMap tm_cls_a, tm_cls_x, tm_cls_hid_out, tm_cls_hid_a;
};

// predict_host pipeline lane: own stream, device staging and workspace, so that the copies of one
// chunk of frames overlap the kernels of another
// Worker threads of the host entry points (label-map expansion, see predict_host_impl).
class HostPool {
 public:
  // `spawn` exists for the unit test (dinoseg_debug_host_pool): it lets a thread creation fail on purpose.
  explicit HostPool(int n, const std::function<void(int)>& spawn_hook = nullptr) {
    try {
      for (int i = 0; i < n; ++i) {
        if (spawn_hook) spawn_hook(i);
        threads_.emplace_back([this] { run(); });
      }
    } catch (...) {
      // std::thread could not be created (EAGAIN: pids / nproc limit).  A smaller pool still does the job; with no
      // thread at all the caller falls back to the DMA path.  Never unwind with joinable threads in threads_
      // (std::terminate) or with workers that hold a dangling `this`.
      if (threads_.empty()) throw;
    }
  }
  ~HostPool() {
    { std::lock_guard<std::mutex> g(m_); stop_ = true; }
    cv_.notify_all();
    for (std::thread& t : threads_) t.join();
  }
  void submit(std::function<void()> f) {
    { std::lock_guard<std::mutex> g(m_); q_.push_back(std::move(f)); ++pending_; }
    cv_.notify_one();
  }
  void wait_all() {
    std::unique_lock<std::mutex> g(m_);
    done_.wait(g, [this] { return pending_ == 0; });
  }
  int size() const { return int(threads_.size()); }

 private:
  void run() {
    for (;;) {
      std::function<void()> f;
      {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [this] { return stop_ || !q_.empty(); });
        if (q_.empty()) return;
        f = std::move(q_.front());
        q_.pop_front();
      }
      f();
      { std::lock_guard<std::mutex> g(m_); if (--pending_ == 0) done_.notify_all(); }
    }
  }
  std::vector<std::thread> threads_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  std::deque<std::function<void()>> q_;
  int pending_ = 0;
  bool stop_ = false;
};

// predict() tail on the host (reference pl_torch_modules.py:297-298: np.kron(low, ones((p, p)))): one frame's low-res
// map [g, g] u8 -> int64 [g*p, g*p].  One label row is built in a small buffer and written p times with streaming
// (non-temporal) stores: the maps are write-only here, and without the read-for-ownership traffic of ordinary
// stores the expansion costs half the memory bandwidth.
void expand_labels_host(const uint8_t* low, int64_t* out, int g, int p) {
  const size_t W = size_t(g) * p;                  // <= 480
  alignas(16) int64_t row[480];
  const bool nt = (reinterpret_cast<uintptr_t>(out) % 16 == 0) && (W % 2 == 0);
  for (int i = 0; i < g; ++i) {
    const uint8_t* lr = low + size_t(i) * g;
    for (int j = 0; j < g; ++j) {
      const int64_t v = lr[j];
      int64_t* d = row + size_t(j) * p;
      for (int k = 0; k < p; ++k) d[k] = v;
    }
    for (int r = 0; r < p; ++r) {
      int64_t* dst = out + (size_t(i) * p + r) * W;
      if (nt) {
        const __m128i* src = reinterpret_cast<const __m128i*>(row);
        __m128i* d = reinterpret_cast<__m128i*>(dst);
        for (size_t k = 0; k < W / 2; ++k) _mm_stream_si128(d + k, _mm_load_si128(src + k));
      } else {
        memcpy(dst, row, W * sizeof(int64_t));
      }
    }
  }
  if (nt) _mm_sfence();
}

// One slot of the host-path pipeline: device staging for a chunk of frames, a workspace and staging for its results.
// in_done: the chunk's frames have arrived; comp_done: its kernels have finished (the frames / workspace may be
// reused); out_done: its results have left (lowres / labels staging may be reused).
struct HostLane {
  cudaEvent_t in_done = nullptr, comp_done = nullptr, out_done = nullptr;
  float* frames = nullptr; size_t frames_cap = 0;
  void* ws = nullptr; size_t ws_cap = 0;
  uint8_t* lowres = nullptr; size_t lowres_cap = 0;
  int64_t* labels = nullptr; size_t labels_cap = 0;
  WorkBufs bufs;
};

}  // namespace

struct dinoseg {
  dinoseg_cfg cfg{};
  int device = 0;
  int num_sms = 148;
  std::string err;

  // parameters
  float* cls = nullptr;
  float* pos_src = nullptr;
  __nv_bfloat16* pe_w = nullptr;
  float* pe_b = nullptr;
  CUtensorMap tm_pe, tm_pe_p;       // (_p: 96-row half W tiles for the CTA-pair GEMM)
  std::vector<BlockW> blocks;
  float *norm_g = nullptr, *norm_b = nullptr;
  __nv_bfloat16* h1_w = nullptr;    // bf16x3 [H1, 3D]   = [hi | hi | lo]
  __nv_bfloat16* h2_w = nullptr;    // bf16x3 [H2, 3*256] = [hi | hi | lo], K zero padded 200 -> 256
  float *h1_b = nullptr, *b2 = nullptr, *w3 = nullptr, *b3 = nullptr;
  CUtensorMap tm_h1, tm_h2;
  // fused head (head.cuh): layer_1 as loaded (fp32), and with the final LayerNorm folded in: [H1, 2D] = [hi | lo], bias
  float* h1_w32 = nullptr;
  __nv_bfloat16* h1f_w = nullptr;
  float* h1f_b = nullptr;
  CUtensorMap tm_h1f_hi, tm_h1f_lo, tm_w2_hi, tm_w2_lo;
  bool fused_head = false;          // MLP head on D = 384: LayerNorm -> layer_1/2/3 -> argmax -> replication in ONE kernel
  std::map<std::string, WeightSlot> slots;
  std::set<std::string> have;
  std::vector<void*> allocs;

  // resolution state: res_h x res_w pixels, gh x gw patches (0 = not set).  Label maps (p_rep > 0) exist for square
  // grids only.
  int res_h = 0, res_w = 0, gh = 0, gw = 0, P = 0, Ntok = 0, p_rep = 0;
  float* pos = nullptr;
  size_t pos_cap = 0;

  WorkBufs user;                    // binding of the caller-provided workspace (dinoseg_forward)
  WorkBufs* last = nullptr;         // buffers of the most recent forward (dinoseg_copy_buffer)

  int debug_stop = 0;
  int launches = 0;
  bool fused_mlp = false;           // D = 384 / hidden = 1536: fused fc1 -> GELU -> fc2 kernel
  bool attn_unshifted = true;       // attention without row maxima + the classic kernel as its redo (attention.cuh)
  bool fuse_ln = true;              // the fused MLP kernel computes LayerNorm2 itself (no LN launch, no bf16 copy of the tokens)
  bool weights_dirty = true;        // fc1_w / fc1_b have to be (re)derived from the loaded parameters
  bool folded = false;              // ... and currently carry LayerNorm2's gamma / beta
  // CTA-pair (cta_group::2) kernels: on by default (dinoseg_set_pair_kernels / DINOSEG_PAIR=0 select the single-CTA
  // forms).  Bit-identical results; +2 % on the ViT-S step, +5 % on ViT-B.  A device / partition without 2-CTA
  // clusters makes the launch fail, in which case forward_impl switches to the single-CTA kernels for good.
  bool gemm_pair = true;            // qkv / patch-embed (ViT-B: fc1, fc2) GEMMs as CTA pairs
  bool mlp_pair = false;            // the fused MLP as CTA pairs (set in dinoseg_create when the fused kernel applies)

  // optional per-kernel-kind timing (cudaEvents around every launch of a forward)
  bool profile = false;
  uint32_t profile_mask = 0xffffffffu;  // bit k set = kind k gets its pair of events
  std::vector<cudaEvent_t> ev;       // 2 per launch slot
  std::vector<int> ev_kind;          // kind of each recorded launch
  int ev_used = 0;

  // predict_host pipeline (lazily created)
  // Three slots, THREE STREAMS with fixed roles: copy-in (H2D), compute (every kernel), copy-out (D2H).  All kernels
  // of the host path run on the ONE compute stream, in order: copies overlap kernels, kernels never overlap kernels.
  // (Round 1 gave every slot its own stream, so kernels of different chunks ran concurrently; a cluster of a
  // cta_group::2 kernel that starts while another stream's kernels are resident can block in tcgen05.alloc for ever -
  // DESIGN.md section 4.5 - and the overlap bought nothing: each kernel is persistent and fills the GPU by itself.)
  static constexpr int kLanes = 3;
  HostLane lanes[kLanes];
  cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
  unsigned slot_seq = 0;            // chunks enqueued so far (slot of a chunk = slot_seq % kLanes)
  cudaEvent_t host_start = nullptr;
  int host_chunk = 0;               // frames per pipeline chunk; 0 = automatic (see pick_host_chunk)
  // host label maps: 1 = copy the low-res maps (g*g bytes per frame) to the host and expand them to int64 there with
  // worker threads (what the reference does with np.kron); 0 = replicate on the GPU and copy 8*(g*p)^2 bytes per frame
  // -1 (default) = decide from the host cores this rank can use (see host_expand_on)
  int host_expand = -1;
  HostPool* pool = nullptr;
  bool pool_failed = false;         // no worker thread could be created: DMA path from now on
  // outstanding dinoseg_predict_host_submit calls (ring of slots; id 0 = free)
  static constexpr int kTickets = 4;
  struct Ticket {
    int64_t id = 0;
    cudaEvent_t done = nullptr;       // recorded on the copy-out stream after the submission's last copy
    bool expand = false;
    std::vector<int> plan;            // frames per chunk
    std::vector<cudaEvent_t> chunk_done;
    uint8_t* low_stage = nullptr;     // pinned [batch, g*g]: low-res maps of this submission (expand mode)
    size_t low_stage_cap = 0;
    uint8_t* host_lowres = nullptr;
    int64_t* host_labels = nullptr;
    int g = 0, p_rep = 0;
  };
  Ticket tickets[kTickets];
  int64_t next_ticket = 1;
};

namespace {

template <typename T>
int dev_alloc(dinoseg* h, T** p, size_t count) {
  void* q = nullptr;
  DSG_CUDA(h, cudaMalloc(&q, count * sizeof(T)));
  h->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return 0;
}

int add_slot(dinoseg* h, const std::string& key, int kind, void* dst, std::vector<int64_t> shape) {
  h->slots[key] = WeightSlot{kind, dst, std::move(shape)};
  return 0;
}

struct WsLayout {
  size_t x, abuf, qkv, hid, lowres, total;
};

WsLayout ws_layout(const dinoseg* h, int batch) {
  const size_t M = size_t(batch) * h->Ntok;
  const size_t D = h->cfg.embed_dim;
  WsLayout L{};
  size_t off = 0;
  L.x = off; off = align_up(off + M * D * 4, 1024);
  L.abuf = off; off = align_up(off + M * D * 2, 1024);
  L.qkv = off; off = align_up(off + M * 3 * D * 2, 1024);
  size_t hid_bytes = M * size_t(h->cfg.mlp_hidden) * 2;
  const size_t h1_bytes = M * size_t(2 * kHeadPart) * 2;   // relu(layer_1) as bf16x3 [M, hi | lo], kHeadPart columns each
  const size_t im2col_bytes = size_t(batch) * h->P * IM2COL_KA * 2;
  if (h1_bytes > hid_bytes) hid_bytes = h1_bytes;
  if (im2col_bytes > hid_bytes) hid_bytes = im2col_bytes;
  L.hid = off; off = align_up(off + hid_bytes, 1024);
  L.lowres = off; off = align_up(off + size_t(batch) * h->P, 1024);
  L.total = off;
  return L;
}

int bind_workspace(dinoseg* h, WorkBufs& w, void* ws, size_t ws_bytes, int batch) {
  const WsLayout L = ws_layout(h, batch);
  if (ws_bytes < L.total) DSG_FAIL(h, "workspace too small: %zu < %zu bytes", ws_bytes, L.total);
  if ((reinterpret_cast<uintptr_t>(ws) & 1023) != 0) DSG_FAIL(h, "workspace must be 1024-byte aligned");
  if (w.base == ws && w.batch == batch && w.res_h == h->res_h && w.res_w == h->res_w) return 0;
  uint8_t* base = static_cast<uint8_t*>(ws);
  w.x = reinterpret_cast<float*>(base + L.x);
  w.abuf = reinterpret_cast<__nv_bfloat16*>(base + L.abuf);
  w.qkv = reinterpret_cast<__nv_bfloat16*>(base + L.qkv);
  w.hid = reinterpret_cast<__nv_bfloat16*>(base + L.hid);
  w.lowres = base + L.lowres;
  const uint64_t M = uint64_t(batch) * h->Ntok;
  const uint64_t D = h->cfg.embed_dim;
  const uint64_t HID = h->cfg.mlp_hidden, H1 = h->cfg.head_h1;
  bool ok = true;
  ok &= make_tmap_gemm_a(&w.tm_im2col, w.hid, h->P, batch, IM2COL_KA);   // per frame: tiles never straddle frames
  ok &= make_tmap_gemm_a(&w.tm_abuf, w.abuf, M, 1, D);
  ok &= make_tmap_gemm_a(&w.tm_hid, w.hid, M, 1, HID);
  ok &= make_tmap_qkv(&w.tm_qkv3d, w.qkv, batch, h->Ntok, 3 * D);
  ok &= make_tmap_gemm_out(&w.tm_x_out, w.x, true, D, M, 1, D);
  ok &= make_tmap_gemm_out(&w.tm_x_patch, w.x, true, D, h->Ntok, batch, D);
  ok &= make_tmap_gemm_out(&w.tm_pos_add, h->pos, true, D, h->Ntok, 1, D);
  ok &= make_tmap_gemm_out(&w.tm_qkv_out, w.qkv, false, 3 * D, M, 1, 3 * D);
  ok &= make_tmap_gemm_out(&w.tm_hid_out, w.hid, false, HID, M, 1, HID);
  // head: final-norm tokens as bf16x3 [M, 3D] in the qkv buffer, relu(layer_1) as bf16x3 [M, 3*256] in
  // the hidden buffer, relu(layer_2) fp32 [M, H2] in the (then dead) residual-stream buffer
  ok &= make_tmap_gemm_a(&w.tm_qkv_a, w.qkv, M, 1, 2 * D);                 // final LN as [hi | lo]
  ok &= make_tmap_gemm_out(&w.tm_h1s_out, w.hid, false, 2 * kHeadPart, M, 1, 2 * kHeadPart);
  ok &= make_tmap_gemm_a(&w.tm_h1s_a, w.hid, M, 1, 2 * kHeadPart);
  ok &= make_tmap_gemm_out(&w.tm_h2_out, w.x, true, h->cfg.head_h2, M, 1, h->cfg.head_h2);
  ok &= make_tmap_gemm_out(&w.tm_lin_out, w.x, true, h->cfg.n_classes, M, 1, kLinPitch);   // 'linear' head logits
  w.cls_x = reinterpret_cast<float*>(w.hid);
  w.cls_hid = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<uint8_t*>(w.hid) + align_up(size_t(batch) * D * 4, 1024));
  ok &= make_tmap_gemm_a(&w.tm_cls_a, w.abuf, batch, 1, D);
  ok &= make_tmap_gemm_out(&w.tm_cls_x, w.cls_x, true, D, batch, 1, D);
  ok &= make_tmap_gemm_out(&w.tm_cls_hid_out, w.cls_hid, false, HID, batch, 1, HID);
  ok &= make_tmap_gemm_a(&w.tm_cls_hid_a, w.cls_hid, batch, 1, HID);
  (void)H1;
  if (!ok) DSG_FAIL(h, "cuTensorMapEncodeTiled failed for the workspace tensor maps");
  w.base = ws;
  w.batch = batch;
  w.res_h = h->res_h;
  w.res_w = h->res_w;
  return 0;
}

}  // namespace

namespace {
enum Kind { K_IM2COL = 0, K_CLS, K_GEMM_PATCH, K_LN, K_GEMM_QKV, K_ATTN, K_GEMM_PROJ, K_GEMM_FC1, K_GEMM_FC2,
            K_GEMM_HEAD, K_HEAD_TAIL, K_REPLICATE, K_MLP_FUSED, K_HEAD_FUSED, K_CLS_GATHER, K_CLS_ATTN_OUT, K_EMBED_POOL,
            K_COUNT };
const char* const kKindNames[K_COUNT] = {"im2col", "cls_row", "gemm_patch", "layernorm", "gemm_qkv", "attention",
                                         "gemm_proj", "gemm_fc1", "gemm_fc2", "gemm_head", "head_tail", "replicate",
                                         "mlp_fused", "head_fused", "cls_gather", "cls_attn_out", "embed_pool"};

// RAII pair of events around one launch (no-op unless profiling is on)
struct LaunchScope {
  dinoseg* h; cudaStream_t s; int slot;
  LaunchScope(dinoseg* h_, int kind, cudaStream_t s_) : h(h_), s(s_), slot(-1) {
    if (!h->profile || !((h->profile_mask >> kind) & 1u)) return;
    slot = h->ev_used++;
    while (int(h->ev.size()) < 2 * (slot + 1)) {
      cudaEvent_t e; cudaEventCreate(&e); h->ev.push_back(e);
    }
    if (int(h->ev_kind.size()) <= slot) h->ev_kind.resize(slot + 1);
    h->ev_kind[slot] = kind;
    cudaEventRecord(h->ev[2 * slot], s);
  }
  ~LaunchScope() { if (slot >= 0) cudaEventRecord(h->ev[2 * slot + 1], s); }
};
}  // namespace

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" {

const char* dinoseg_last_error(const dinoseg_t* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int dinoseg_create(const dinoseg_cfg* cfg, int device, dinoseg_t** out) {
  dinoseg* null_h = nullptr;
  if (!cfg || !out) DSG_FAIL(null_h, "dinoseg_create: null argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    DSG_FAIL(null_h, "dinoseg_create: no CUDA device available (this library has no CPU path)");
  if (device < 0 || device >= ndev) DSG_FAIL(null_h, "dinoseg_create: invalid device %d", device);
  cudaDeviceProp prop;
  DSG_CUDA(null_h, cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    DSG_FAIL(null_h, "dinoseg_create: device %d is sm_%d%d; this library contains sm_100a code only", device,
             prop.major, prop.minor);
  if (cfg->embed_dim != 384 && cfg->embed_dim != 768) DSG_FAIL(null_h, "embed_dim must be 384 or 768");
  if (cfg->num_heads * 64 != cfg->embed_dim) DSG_FAIL(null_h, "head_dim must be 64 (num_heads = embed_dim/64)");
  if (cfg->patch != 8) DSG_FAIL(null_h, "patch size must be 8");
  if (cfg->n_blocks < 0 || cfg->n_blocks > 12) DSG_FAIL(null_h, "n_blocks out of range");
  if (cfg->n_classes < 1 || cfg->n_classes > HEAD_MAX_C) DSG_FAIL(null_h, "n_classes must be in [1,%d]", HEAD_MAX_C);
  if (cfg->head_kind != 0 && cfg->head_kind != 1) DSG_FAIL(null_h, "head_kind must be 0 ('mlp') or 1 ('linear')");
  if (cfg->head_h1 % 8 != 0 || cfg->head_h1 < 8 || cfg->head_h1 > kHeadPart || cfg->head_h2 % 4 != 0 ||
      cfg->head_h2 > HT_MAX_H2 || cfg->head_h2 < 4)
    DSG_FAIL(null_h, "unsupported head widths %d/%d", cfg->head_h1, cfg->head_h2);
  if (cfg->mlp_hidden % 64 != 0) DSG_FAIL(null_h, "mlp_hidden must be a multiple of 64");
  if (!get_encode()) DSG_FAIL(null_h, "cuTensorMapEncodeTiled not available from the driver");
  DSG_CUDA(null_h, cudaSetDevice(device));

  if (!g_heartbeat) {                     // one array per process, never freed (diagnostics)
    if (cudaMalloc(&g_heartbeat, 1024 * sizeof(int)) == cudaSuccess) cudaMemset(g_heartbeat, 0, 1024 * sizeof(int));
    else { g_heartbeat = nullptr; (void)cudaGetLastError(); }
  }
  dinoseg* h = new dinoseg();
  h->cfg = *cfg;
  h->device = device;
  h->fused_mlp = cfg->embed_dim == MLP_D && cfg->mlp_hidden == MLP_HID;
  h->mlp_pair = h->fused_mlp;
  h->fused_head = cfg->head_kind == 0 && cfg->embed_dim == HEAD_D && cfg->head_h1 <= HEAD_N1 && cfg->head_h2 <= HEAD_W3_PITCH - 4 &&
                  kHeadPart == HEAD_K2;
  if (const char* mode = getenv("DINOSEG_FUSED_HEAD")) h->fused_head = h->fused_head && atoi(mode) != 0;   // measurement override
  if (const char* mode = getenv("DINOSEG_PAIR")) {   // CTA-pair kernels: 0.486 vs 0.494 ms (MLP), 0.188 vs 0.212 ms (qkv)
    h->gemm_pair = atoi(mode) != 0;
    h->mlp_pair = h->fused_mlp && atoi(mode) != 0;
  }
  if (const char* mode = getenv("DINOSEG_HOST_EXPAND")) h->host_expand = atoi(mode) != 0 ? 1 : 0;   // measurement override
  if (const char* mode = getenv("DINOSEG_FUSE_LN")) h->fuse_ln = atoi(mode) != 0;         // measurement override
  if (const char* mode = getenv("DINOSEG_ATTN_UNSHIFTED")) h->attn_unshifted = atoi(mode) != 0;   // measurement override
  if (const char* mode = getenv("DINOSEG_HOST_CHUNK")) h->host_chunk = atoi(mode) > 0 ? atoi(mode) : 0;   // measurement override
  if (const char* mode = getenv("DINOSEG_GEMM_PAIR")) h->gemm_pair = atoi(mode) != 0;   // measurement override
  if (const char* mode = getenv("DINOSEG_MLP_MODE")) {   // measurement override: 0 unfused, 1 fused, 2 fused as CTA pairs
    const int m = atoi(mode);
    h->fused_mlp = h->fused_mlp && m != 0;
    h->mlp_pair = h->fused_mlp && m == 2;
  }
  h->num_sms = prop.multiProcessorCount;
  const int D = cfg->embed_dim, HID = cfg->mlp_hidden, G0 = cfg->pos_grid, C = cfg->n_classes;
  const bool linear_head = cfg->head_kind == 1;          // reference pl_torch_modules.py:127-138: Linear(D, C)
  const int H1 = linear_head ? C : cfg->head_h1, H2 = cfg->head_h2;
  int rc = 0;
  rc |= dev_alloc(h, &h->cls, D);
  rc |= dev_alloc(h, &h->pos_src, size_t(G0 * G0 + 1) * D);
  rc |= dev_alloc(h, &h->pe_w, size_t(D) * IM2COL_K3);
  rc |= dev_alloc(h, &h->pe_b, D);
  rc |= dev_alloc(h, &h->norm_g, D);
  rc |= dev_alloc(h, &h->norm_b, D);
  rc |= dev_alloc(h, &h->h1_w, size_t(H1) * 3 * D);
  rc |= dev_alloc(h, &h->h2_w, size_t(H2) * 3 * kHeadPart);
  rc |= dev_alloc(h, &h->h1_b, H1);
  rc |= dev_alloc(h, &h->h1_w32, size_t(H1) * D);
  rc |= dev_alloc(h, &h->h1f_w, size_t(H1) * 2 * D);
  rc |= dev_alloc(h, &h->h1f_b, H1);
  rc |= dev_alloc(h, &h->b2, H2);
  rc |= dev_alloc(h, &h->w3, size_t(C) * H2);
  rc |= dev_alloc(h, &h->b3, C);
  add_slot(h, "dino.cls_token", 0, h->cls, {1, 1, D});
  add_slot(h, "dino.pos_embed", 0, h->pos_src, {1, G0 * G0 + 1, D});
  add_slot(h, "dino.patch_embed.proj.weight", 3, h->pe_w, {D, 3, 8, 8});   // bf16x3 [D, 3*192]
  add_slot(h, "dino.patch_embed.proj.bias", 0, h->pe_b, {D});
  add_slot(h, "dino.norm.weight", 0, h->norm_g, {D});
  add_slot(h, "dino.norm.bias", 0, h->norm_b, {D});
  add_slot(h, "clf.layer_1.weight", 3, h->h1_w, {H1, D});
  add_slot(h, "clf.layer_1.bias", 0, h->h1_b, {H1});
  if (!linear_head) {
    add_slot(h, "clf.layer_2.weight", 4, h->h2_w, {H2, H1});
    add_slot(h, "clf.layer_2.bias", 0, h->b2, {H2});
    add_slot(h, "clf.layer_3.weight", 0, h->w3, {C, H2});
    add_slot(h, "clf.layer_3.bias", 0, h->b3, {C});
  }
  h->blocks.resize(cfg->n_blocks);
  for (int i = 0; i < cfg->n_blocks && rc == 0; ++i) {
    BlockW& b = h->blocks[i];
    const std::string pre = "dino.blocks." + std::to_string(i) + ".";
    rc |= dev_alloc(h, &b.ln1_g, D); rc |= dev_alloc(h, &b.ln1_b, D);
    rc |= dev_alloc(h, &b.ln2_g, D); rc |= dev_alloc(h, &b.ln2_b, D);
    rc |= dev_alloc(h, &b.qkv_w, size_t(3) * D * D); rc |= dev_alloc(h, &b.qkv_b, 3 * D);
    rc |= dev_alloc(h, &b.proj_w, size_t(D) * D); rc |= dev_alloc(h, &b.proj_b, D);
    rc |= dev_alloc(h, &b.fc1_w, size_t(HID) * D); rc |= dev_alloc(h, &b.fc1_b, HID);
    rc |= dev_alloc(h, &b.fc1_w32, size_t(HID) * D); rc |= dev_alloc(h, &b.fc1_b32, HID);
    rc |= dev_alloc(h, &b.fc2_w, size_t(D) * HID); rc |= dev_alloc(h, &b.fc2_b, D);
    if (rc) break;
    add_slot(h, pre + "norm1.weight", 0, b.ln1_g, {D}); add_slot(h, pre + "norm1.bias", 0, b.ln1_b, {D});
    add_slot(h, pre + "norm2.weight", 0, b.ln2_g, {D}); add_slot(h, pre + "norm2.bias", 0, b.ln2_b, {D});
    add_slot(h, pre + "attn.qkv.weight", 1, b.qkv_w, {3 * D, D}); add_slot(h, pre + "attn.qkv.bias", 0, b.qkv_b, {3 * D});
    add_slot(h, pre + "attn.proj.weight", 1, b.proj_w, {D, D}); add_slot(h, pre + "attn.proj.bias", 0, b.proj_b, {D});
    add_slot(h, pre + "mlp.fc1.weight", 0, b.fc1_w32, {HID, D}); add_slot(h, pre + "mlp.fc1.bias", 0, b.fc1_b32, {HID});
    add_slot(h, pre + "mlp.fc2.weight", 1, b.fc2_w, {D, HID}); add_slot(h, pre + "mlp.fc2.bias", 0, b.fc2_b, {D});
    bool ok = true;
    ok &= make_tmap_2d(&b.tm_qkv, b.qkv_w, 3 * D, D, D, GEMM_BN);
    ok &= make_tmap_2d(&b.tm_qkv_h, b.qkv_w, 3 * D, D, D, GEMM_BN / 2);
    ok &= make_tmap_2d(&b.tm_fc1_p, b.fc1_w, HID, D, D, GEMM_BN / 2);
    ok &= make_tmap_2d(&b.tm_fc2_p, b.fc2_w, D, HID, HID, GEMM_BN / 2);
    ok &= make_tmap_2d(&b.tm_proj, b.proj_w, D, D, D, GEMM_BN);
    ok &= make_tmap_2d(&b.tm_fc1, b.fc1_w, HID, D, D, GEMM_BN);
    ok &= make_tmap_2d(&b.tm_fc2, b.fc2_w, D, HID, HID, GEMM_BN);
    ok &= make_tmap_2d(&b.tm_fc1_g, b.fc1_w, HID, D, D, 128);
    ok &= make_tmap_2d(&b.tm_fc2_g, b.fc2_w, D, HID, HID, 128);
    ok &= make_tmap_2d(&b.tm_fc1_h, b.fc1_w, HID, D, D, 64);
    ok &= make_tmap_2d(&b.tm_fc2_h, b.fc2_w, D, HID, HID, 64);
    if (!ok) { h->err = "cuTensorMapEncodeTiled failed for block weights"; rc = -1; }
  }
  if (rc == 0) {
    bool ok = make_tmap_2d(&h->tm_pe, h->pe_w, D, IM2COL_K3, IM2COL_K3, GEMM_BN);
    ok &= make_tmap_2d(&h->tm_pe_p, h->pe_w, D, IM2COL_K3, IM2COL_K3, GEMM_BN / 2);
    ok &= make_tmap_2d(&h->tm_h1, h->h1_w, H1, 3 * D, 3 * D, GEMM_BN);
    ok &= make_tmap_2d(&h->tm_h2, h->h2_w, H2, 3 * kHeadPart, 3 * kHeadPart, GEMM_BN);
    // fused head: layer_1 [hi | lo] halves as [208 x 64] boxes; layer_2's hi / lo parts of the [hi | hi | lo] packing
    ok &= make_tmap_2d(&h->tm_h1f_hi, h->h1f_w, H1, D, 2 * D, HEAD_N1);
    ok &= make_tmap_2d(&h->tm_h1f_lo, h->h1f_w + D, H1, D, 2 * D, HEAD_N1);
    ok &= make_tmap_2d(&h->tm_w2_hi, h->h2_w, H2, kHeadPart, 3 * kHeadPart, HEAD_N2);
    ok &= make_tmap_2d(&h->tm_w2_lo, h->h2_w + 2 * kHeadPart, H2, kHeadPart, 3 * kHeadPart, HEAD_N2);
    if (!ok) { h->err = "cuTensorMapEncodeTiled failed for patch/head weights"; rc = -1; }
  }
  if (rc != 0) {
    g_create_error = h->err;
    dinoseg_destroy(h);
    return -1;
  }
  *out = h;
  return 0;
}

void dinoseg_destroy(dinoseg_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (void* p : h->allocs) cudaFree(p);
  if (h->pos) cudaFree(h->pos);
  for (cudaStream_t st : {h->s_in, h->s_comp, h->s_out})
    if (st) cudaStreamSynchronize(st);
  for (HostLane& l : h->lanes) {
    if (l.frames) cudaFree(l.frames);
    if (l.ws) cudaFree(l.ws);
    if (l.lowres) cudaFree(l.lowres);
    if (l.labels) cudaFree(l.labels);
    for (cudaEvent_t e : {l.in_done, l.comp_done, l.out_done})
      if (e) cudaEventDestroy(e);
  }
  for (cudaStream_t st : {h->s_in, h->s_comp, h->s_out})
    if (st) cudaStreamDestroy(st);
  if (h->host_start) cudaEventDestroy(h->host_start);
  delete h->pool;
  for (dinoseg::Ticket& t : h->tickets) {
    if (t.low_stage) cudaFreeHost(t.low_stage);
    for (cudaEvent_t e : t.chunk_done) cudaEventDestroy(e);
    if (t.done) cudaEventDestroy(t.done);
  }
  for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
  delete h;
}

int dinoseg_set_weight(dinoseg_t* h, const char* key, const float* dev_ptr, const int64_t* shape, int ndim,
                       void* stream) {
  if (!h) return -1;
  if (!key || !dev_ptr || !shape) DSG_FAIL(h, "dinoseg_set_weight: null argument");
  auto it = h->slots.find(key);
  if (it == h->slots.end()) DSG_FAIL(h, "dinoseg_set_weight: unexpected key '%s'", key);
  const WeightSlot& sl = it->second;
  bool same = int(sl.shape.size()) == ndim;
  size_t n = 1;
  for (int i = 0; same && i < ndim; ++i) same = sl.shape[i] == shape[i];
  for (int64_t d : sl.shape) n *= size_t(d);
  if (!same) {
    std::string want, got;
    for (int64_t d : sl.shape) want += std::to_string(d) + ",";
    for (int i = 0; i < ndim; ++i) got += std::to_string(shape[i]) + ",";
    DSG_FAIL(h, "dinoseg_set_weight: size mismatch for %s: expected (%s) got (%s)", key, want.c_str(), got.c_str());
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DSG_CUDA(h, cudaSetDevice(h->device));
  if (sl.kind == 1) {
    const unsigned blocks = unsigned(std::min<size_t>((n + 255) / 256, 4096));
    f32_to_bf16_kernel<<<blocks, 256, 0, s>>>(dev_ptr, static_cast<__nv_bfloat16*>(sl.dst), n);
    DSG_CUDA(h, cudaGetLastError());
  } else if (sl.kind == 3 || sl.kind == 4) {
    const int N = int(sl.shape[0]), K = int(n / size_t(sl.shape[0]));
    const int Kp = sl.kind == 3 ? K : kHeadPart;
    split_weight_kernel<<<256, 256, 0, s>>>(dev_ptr, static_cast<__nv_bfloat16*>(sl.dst), N, K, Kp);
    DSG_CUDA(h, cudaGetLastError());
  } else {
    DSG_CUDA(h, cudaMemcpyAsync(sl.dst, dev_ptr, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  if (std::string(key) == "clf.layer_1.weight")     // the fused head folds the final LayerNorm into it (finalize_weights)
    DSG_CUDA(h, cudaMemcpyAsync(h->h1_w32, dev_ptr, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  h->have.insert(key);
  h->weights_dirty = true;          // derived operands (fc1 with or without the folded LayerNorm2) are rebuilt lazily
  return 0;
}

int dinoseg_missing_weights(const dinoseg_t* h) {
  if (!h) return -1;
  return int(h->slots.size()) - int(h->have.size());
}

int dinoseg_set_resolution(dinoseg_t* h, int resolution, void* stream) {
  return dinoseg_set_resolution_hw(h, resolution, resolution, stream);
}

int dinoseg_set_resolution_hw(dinoseg_t* h, int height, int width, void* stream) {
  if (!h) return -1;
  if (height <= 0 || width <= 0 || height % 8 != 0 || width % 8 != 0) DSG_FAIL(h, "Resolution should be a multiple of 8.");
  if (!h->have.count("dino.pos_embed")) DSG_FAIL(h, "dinoseg_set_resolution: dino.pos_embed has not been set");
  const int gh = height / 8, gw = width / 8;
  if (gh > 480 || gw > 480) DSG_FAIL(h, "resolution %dx%d too large (patch grid %dx%d, a side > 480)", height, width, gh, gw);
  const int D = h->cfg.embed_dim;
  const size_t need = size_t(gh * gw + 1) * D;
  DSG_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (need > h->pos_cap) {
    if (h->pos) {
      DSG_CUDA(h, cudaStreamSynchronize(s));
      DSG_CUDA(h, cudaFree(h->pos));
      h->pos = nullptr;
    }
    DSG_CUDA(h, cudaMalloc(&h->pos, need * sizeof(float)));
    h->pos_cap = need;
  }
  DSG_CUDA(h, launch_posembed(h->pos_src, h->pos, h->cfg.pos_grid, gh, gw, D, s));
  h->res_h = height;
  h->res_w = width;
  h->gh = gh;
  h->gw = gw;
  h->P = gh * gw;
  h->Ntok = gh * gw + 1;
  h->p_rep = gh == gw ? 480 / gh : 0;  // reference pl_torch_modules.py:297 (predict's np.kron assumes a square grid)
  h->user.base = nullptr;  // tensor maps depend on Ntok
  for (HostLane& l : h->lanes) l.bufs.base = nullptr;
  return 0;
}

size_t dinoseg_workspace_bytes(const dinoseg_t* h, int batch) {
  if (!h || h->res_h == 0 || batch <= 0) return 0;
  return ws_layout(h, batch).total;
}

int dinoseg_set_debug_stop(dinoseg_t* h, int stage) {
  if (!h) return -1;
  h->debug_stop = stage;
  return 0;
}

int dinoseg_last_launch_count(const dinoseg_t* h) { return h ? h->launches : -1; }

int dinoseg_profile_enable(dinoseg_t* h, int on) {
  if (!h) return -1;
  h->profile = on != 0;
  h->ev_used = 0;
  return 0;
}

int dinoseg_profile_set_mask(dinoseg_t* h, uint32_t kind_mask) {
  if (!h) return -1;
  h->profile_mask = kind_mask;
  return 0;
}

// Diagnostic for work that does not finish (callable from another host thread while the launching thread is blocked
// in a synchronise): the profiled launches whose start event has completed and whose end event has not - the kernels
// that are running (or stuck) right now, one per stream at most.  Returns how many were written to kinds[] / slots[]
// (up to max_out); -2 without profiling.  *not_started (optional): launches whose start event is pending as well.
int dinoseg_debug_pending_kinds(dinoseg_t* h, int* kinds, int* slots, int max_out, int* not_started) {
  if (!h || !kinds || !slots || max_out < 1) return -2;
  if (!h->profile || h->ev_used == 0) return -2;
  int n_out = 0, waiting = 0;
  for (int i = 0; i < h->ev_used && 2 * i + 1 < int(h->ev.size()); ++i) {
    if (cudaEventQuery(h->ev[2 * i + 1]) == cudaSuccess) continue;
    if (cudaEventQuery(h->ev[2 * i]) == cudaSuccess) {
      if (n_out < max_out) { kinds[n_out] = h->ev_kind[i]; slots[n_out] = i; ++n_out; }
    } else {
      ++waiting;
    }
  }
  (void)cudaGetLastError();
  if (not_started) *not_started = waiting;
  return n_out;
}

// Copies the heartbeat array (hb_mark: entry [sm] = kernel code * 10 + stage while a tcgen05 kernel's CTA sits on that
// SM, negative after it left) to the host on a stream of its own, so that it works while other streams are stuck.
// kernel codes: 100 + EPI*10 + 2*RES_A + PAIR = GEMM, 200 + PAIR = fused MLP, 300 + SMW = attention.
int dinoseg_debug_heartbeat(int* host_out, int n) {
  if (!host_out || n < 1 || !g_heartbeat) return -1;
  static cudaStream_t diag = nullptr;
  if (!diag && cudaStreamCreateWithFlags(&diag, cudaStreamNonBlocking) != cudaSuccess) return -2;
  if (n > 1024) n = 1024;
  if (cudaMemcpyAsync(host_out, g_heartbeat, size_t(n) * sizeof(int), cudaMemcpyDeviceToHost, diag) != cudaSuccess) return -3;
  return cudaStreamSynchronize(diag) == cudaSuccess ? n : -4;
}

int dinoseg_profile_num_kinds(void) { return K_COUNT; }
const char* dinoseg_profile_kind_name(int kind) { return (kind >= 0 && kind < K_COUNT) ? kKindNames[kind] : ""; }

// Before dinoseg_profile_read: time between the first launch's start event and the last launch's end event, and the
// part of it that lies BETWEEN launches (end event of one -> start event of the next; includes the event records).
int dinoseg_profile_gaps(dinoseg_t* h, float* span_ms, float* gap_ms) {
  if (!h || !span_ms || !gap_ms) return -1;
  *span_ms = 0.f; *gap_ms = 0.f;
  if (h->ev_used < 1) return 0;
  cudaError_t e = cudaEventSynchronize(h->ev[2 * (h->ev_used - 1) + 1]);
  if (e == cudaSuccess) e = cudaEventElapsedTime(span_ms, h->ev[0], h->ev[2 * (h->ev_used - 1) + 1]);
  for (int i = 0; e == cudaSuccess && i + 1 < h->ev_used; ++i) {
    float ms = 0.f;
    e = cudaEventElapsedTime(&ms, h->ev[2 * i + 1], h->ev[2 * (i + 1)]);
    *gap_ms += ms;
  }
  if (e != cudaSuccess) DSG_FAIL(h, "dinoseg_profile_gaps: %s", cudaGetErrorString(e));
  return 0;
}

int dinoseg_profile_read(dinoseg_t* h, float* ms_by_kind, int* launches_by_kind, int n_kinds) {
  if (!h || !ms_by_kind || !launches_by_kind || n_kinds < K_COUNT) return -1;
  for (int k = 0; k < K_COUNT; ++k) { ms_by_kind[k] = 0.f; launches_by_kind[k] = 0; }
  for (int i = 0; i < h->ev_used; ++i) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(h->ev[2 * i + 1]);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, h->ev[2 * i], h->ev[2 * i + 1]);
    if (e != cudaSuccess) DSG_FAIL(h, "dinoseg_profile_read: %s", cudaGetErrorString(e));
    ms_by_kind[h->ev_kind[i]] += ms;
    launches_by_kind[h->ev_kind[i]] += 1;
  }
  h->ev_used = 0;
  return 0;
}

// Derived operands: fc1 weight (bf16) and bias of every block, with LayerNorm2's affine transform folded in when the
// fused MLP kernel normalises the tokens itself (fold_ln_weight_kernel), plain otherwise.  Runs when a parameter or the
// mode changed; synchronises the stream so that forwards on other streams see the result.
static int finalize_weights(dinoseg_t* h, cudaStream_t s) {
  const bool fold = h->fused_mlp && h->fuse_ln;
  if (!h->weights_dirty && h->folded == fold) return 0;
  const int D = h->cfg.embed_dim, HID = h->cfg.mlp_hidden;
  for (BlockW& b : h->blocks) {
    if (fold) {
      fold_ln_weight_kernel<<<(HID * 32 + 255) / 256, 256, 0, s>>>(b.fc1_w32, b.fc1_b32, b.ln2_g, b.ln2_b, b.fc1_w, b.fc1_b,
                                                                   HID, D);
    } else {
      const size_t n = size_t(HID) * D;
      f32_to_bf16_kernel<<<unsigned(std::min<size_t>((n + 255) / 256, 4096)), 256, 0, s>>>(b.fc1_w32, b.fc1_w, n);
      DSG_CUDA(h, cudaMemcpyAsync(b.fc1_b, b.fc1_b32, size_t(HID) * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    DSG_CUDA(h, cudaGetLastError());
  }
  if (h->cfg.head_kind == 0 && h->cfg.embed_dim == HEAD_D) {   // fused head: final LayerNorm folded into layer_1, hi | lo
    const int H1 = h->cfg.head_h1;
    fold_split_ln_weight_kernel<<<(H1 * 32 + 255) / 256, 256, 0, s>>>(h->h1_w32, h->h1_b, h->norm_g, h->norm_b, h->h1f_w,
                                                                      h->h1f_b, H1, D);
    DSG_CUDA(h, cudaGetLastError());
  }
  DSG_CUDA(h, cudaStreamSynchronize(s));
  h->weights_dirty = false;
  h->folded = fold;
  return 0;
}

cudaError_t launch_head_fused(dinoseg_t* h, const float* x, int M, float* logprobs, uint8_t* lowres, long long* labels,
                              cudaStream_t s) {
  static bool attr[64][2] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  const int big = h->cfg.n_classes > 8 ? 1 : 0;
  if (!attr[dev & 63][big]) {
    cudaError_t e = big ? cudaFuncSetAttribute(head_fused_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(HEAD_SMEM))
                        : cudaFuncSetAttribute(head_fused_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(HEAD_SMEM));
    if (e != cudaSuccess) return e;
    attr[dev & 63][big] = true;
  }
  HeadParams p{};
  p.M = M; p.x = x; p.ln_eps = h->cfg.ln_eps;
  p.b1f = h->h1f_b; p.b2 = h->b2; p.w3 = h->w3; p.b3 = h->b3;
  p.H1 = h->cfg.head_h1; p.H2 = h->cfg.head_h2; p.C = h->cfg.n_classes;
  p.Ntok = h->Ntok; p.gh = h->gh; p.gw = h->gw; p.p = h->p_rep;
  p.logprobs = logprobs; p.lowres = lowres; p.labels = labels;
  p.hb = g_heartbeat;
  const int m_blocks = (M + HEAD_BM - 1) / HEAD_BM;
  const int grid = m_blocks < h->num_sms ? m_blocks : h->num_sms;
  if (big) head_fused_kernel<16><<<grid, HEAD_THREADS, HEAD_SMEM, s>>>(h->tm_h1f_hi, h->tm_h1f_lo, h->tm_w2_hi, h->tm_w2_lo, p);
  else head_fused_kernel<8><<<grid, HEAD_THREADS, HEAD_SMEM, s>>>(h->tm_h1f_hi, h->tm_h1f_lo, h->tm_w2_hi, h->tm_w2_lo, p);
  return cudaGetLastError();
}

// Backbone features requested from forward_impl: after every block i >= first, the final LayerNorm (dino.norm) of the
// residual stream goes to out[i - first] (fp32 [M, D] slices); backbone_only ends the pass before the head.
// cls_rows (embeddings): only the B CLS rows are normed, out is fp32 [n, B, D] (or null) and patch_mean fp32 [B, D]
// (or null).  Without patch_mean the last block runs for the CLS rows only after its qkv GEMM (see forward_impl).
struct FeatureReq {
  float* out = nullptr;
  int first = 0;
  bool backbone_only = false;
  bool cls_rows = false;
  float* patch_mean = nullptr;
};

// The last block for the CLS rows only (embeddings without the patch mean), after LayerNorm1 and the qkv GEMM have run
// over all rows (the CLS query attends to every key and value).  Everything after the attention reads and writes the
// CLS rows alone, so it runs at M = B on the compact buffers of `w`: the CLS query's attention output and the gathered
// residual rows (one kernel), the proj GEMM, the MLP as the full-size path selects it, and the fp32 final LayerNorm
// into `cls_out` ([B, D]).  The single row block of M = B <= 128 is fine for the CTA-pair forms: their second row block
// lies past the end, loads zeros and stores nothing.  x (all rows) is left as the qkv GEMM found it.
static int cls_only_tail(dinoseg_t* h, WorkBufs& w, BlockW& b, int batch, float* cls_out, cudaStream_t s, int& n) {
  const int D = h->cfg.embed_dim, HID = h->cfg.mlp_hidden;
  const float eps = h->cfg.ln_eps;
  const int sms = h->num_sms;
  auto gp = [&](int N, int K, const float* bias) {
    GemmParams p{};
    p.N = N; p.K = K; p.rows_per_batch = batch; p.batches = 1; p.row_off = 0; p.add_batched = 0; p.bias = bias;
    p.col_scale = 1.f; p.scale_cols = 0;
    return p;
  };
  {
    LaunchScope ls(h, K_CLS_ATTN_OUT, s);
    DSG_CUDA(h, launch_cls_attn_out(w.qkv, w.x, w.abuf, w.cls_x, batch, h->Ntok, D, h->cfg.num_heads, s));
    ++n;
  }
  {
    LaunchScope ls(h, K_GEMM_PROJ, s);
    DSG_CUDA(h, launch_gemm(EPI_RESID_F32, w.tm_cls_a, b.tm_proj, w.tm_cls_x, w.tm_cls_x, gp(D, D, b.proj_b), sms, s));
    ++n;
  }
  if (h->fused_mlp) {
    MlpParams p{};
    p.M = batch; p.x = w.cls_x; p.b1 = b.fc1_b; p.b2 = b.fc2_b;
    if (h->fuse_ln) {
      p.fuse_ln = 1; p.ln_eps = eps;
    } else {
      LaunchScope ls(h, K_LN, s); DSG_CUDA(h, launch_layernorm(w.cls_x, b.ln2_g, b.ln2_b, w.abuf, batch, D, eps, false, s)); ++n;
    }
    LaunchScope ls(h, K_MLP_FUSED, s);
    if (h->mlp_pair && launch_mlp_fused(w.tm_cls_a, b.tm_fc1_h, b.tm_fc2_h, w.tm_cls_x, p, sms, true, s) != cudaSuccess) {
      (void)cudaGetLastError();
      h->mlp_pair = false;
    }
    if (!h->mlp_pair) DSG_CUDA(h, launch_mlp_fused(w.tm_cls_a, b.tm_fc1_g, b.tm_fc2_g, w.tm_cls_x, p, sms, false, s));
    ++n;
  } else {
    { LaunchScope ls(h, K_LN, s); DSG_CUDA(h, launch_layernorm(w.cls_x, b.ln2_g, b.ln2_b, w.abuf, batch, D, eps, false, s)); ++n; }
    {
      LaunchScope ls(h, K_GEMM_FC1, s);
      const GemmParams p = gp(HID, D, b.fc1_b);
      if (h->gemm_pair &&
          launch_gemm_pair<EPI_GELU_BF16>(w.tm_cls_a, b.tm_fc1_p, w.tm_cls_hid_out, w.tm_cls_hid_out, p, sms, s) != cudaSuccess) {
        (void)cudaGetLastError();
        h->gemm_pair = false;
      }
      if (!h->gemm_pair) DSG_CUDA(h, launch_gemm(EPI_GELU_BF16, w.tm_cls_a, b.tm_fc1, w.tm_cls_hid_out, w.tm_cls_hid_out, p, sms, s));
      ++n;
    }
    {
      LaunchScope ls(h, K_GEMM_FC2, s);
      const GemmParams p = gp(D, HID, b.fc2_b);
      if (h->gemm_pair &&
          launch_gemm_pair<EPI_RESID_F32>(w.tm_cls_hid_a, b.tm_fc2_p, w.tm_cls_x, w.tm_cls_x, p, sms, s) != cudaSuccess) {
        (void)cudaGetLastError();
        h->gemm_pair = false;
      }
      if (!h->gemm_pair) DSG_CUDA(h, launch_gemm(EPI_RESID_F32, w.tm_cls_hid_a, b.tm_fc2, w.tm_cls_x, w.tm_cls_x, p, sms, s));
      ++n;
    }
  }
  LaunchScope ls(h, K_LN, s);
  DSG_CUDA(h, launch_layernorm_f32(w.cls_x, h->norm_g, h->norm_b, cls_out, batch, D, eps, s));
  ++n;
  return 0;
}

// Launch sequence of one forward pass over `batch` frames on the buffers of `w` (already bound).
// `frames` are normalised fp32 NCHW frames, or (frames == nullptr) `frames_u8` raw uint8 HWC frames that are resized
// and normalised on the fly (pp).  `feat` (optional): backbone features to emit on the way.
static int forward_impl(dinoseg_t* h, WorkBufs& w, const float* frames, const uint8_t* frames_u8, const PreprocParams* pp,
                        int batch, float* logprobs, uint8_t* lowres, int64_t* labels, cudaStream_t s,
                        const FeatureReq* feat = nullptr) {
  if (h->res_h == 0) DSG_FAIL(h, "dinoseg_forward: call dinoseg_set_resolution first");
  if (labels && h->gh != h->gw)
    DSG_FAIL(h, "dinoseg_forward: label maps exist for square patch grids only (resolution %dx%d); pass labels = NULL",
             h->res_h, h->res_w);
  if (dinoseg_missing_weights(h) != 0) {
    std::string miss;
    for (auto& kv : h->slots)
      if (!h->have.count(kv.first)) { miss = kv.first; break; }
    DSG_FAIL(h, "dinoseg_forward: %d parameters not set (first missing: %s)", dinoseg_missing_weights(h),
             miss.c_str());
  }
  if ((!frames && !(frames_u8 && pp)) || batch <= 0) DSG_FAIL(h, "dinoseg_forward: bad arguments");
  if (finalize_weights(h, s) != 0) return -1;
  if (size_t(batch) * h->Ntok > size_t(INT32_MAX) / 4) DSG_FAIL(h, "dinoseg_forward: batch too large");
  h->last = &w;
  const int D = h->cfg.embed_dim, HID = h->cfg.mlp_hidden, H = h->cfg.num_heads;
  const int M = batch * h->Ntok;
  const float eps = h->cfg.ln_eps;
  int n = 0;
  h->launches = 0;
  const int stop = h->debug_stop;
  if (!h->profile) h->ev_used = 0;

  // ---- prepare_tokens (vision_transformer.py:224-235) ----
  const int sms = h->num_sms;
  auto gp = [&](int N, int K, const float* bias) {
    GemmParams p{};
    p.N = N; p.K = K; p.rows_per_batch = M; p.batches = 1; p.row_off = 0; p.add_batched = 0; p.bias = bias;
    p.col_scale = 1.f; p.scale_cols = 0;
    return p;
  };
  {
    LaunchScope ls(h, K_IM2COL, s);
    if (frames) DSG_CUDA(h, launch_im2col(frames, w.hid, batch, h->gh, h->gw, s));
    else DSG_CUDA(h, launch_im2col_u8(frames_u8, w.hid, batch, h->gh, h->gw, *pp, s));
    ++n;
  }
  {
    LaunchScope ls(h, K_CLS, s);
    cls_row_kernel<<<(batch * D + 255) / 256, 256, 0, s>>>(h->cls, h->pos, w.x, batch, h->Ntok, D);
    DSG_CUDA(h, cudaGetLastError()); ++n;
  }
  {
    GemmParams p = gp(D, IM2COL_K3, h->pe_b);
    p.a_wrap = IM2COL_KA;
    p.rows_per_batch = h->P; p.batches = batch; p.row_off = 1;   // out row = b*Ntok + 1 + t, + pos[1 + t]
    LaunchScope ls(h, K_GEMM_PATCH, s);
    if (h->gemm_pair &&
        launch_gemm_pair<EPI_PATCH_F32>(w.tm_im2col, h->tm_pe_p, w.tm_x_patch, w.tm_pos_add, p, sms, s) != cudaSuccess) {
      (void)cudaGetLastError();
      h->gemm_pair = false;
    }
    if (!h->gemm_pair) DSG_CUDA(h, launch_gemm(EPI_PATCH_F32, w.tm_im2col, h->tm_pe, w.tm_x_patch, w.tm_pos_add, p, sms, s));
    ++n;
  }
  if (stop == 1) { h->launches = n; return 0; }

  // ---- transformer blocks (vision_transformer.py:122-140) ----
  for (int i = 0; i < h->cfg.n_blocks; ++i) {
    BlockW& b = h->blocks[i];
    { LaunchScope ls(h, K_LN, s); DSG_CUDA(h, launch_layernorm(w.x, b.ln1_g, b.ln1_b, w.abuf, M, D, eps, false, s)); ++n; }
    {
      GemmParams p = gp(3 * D, D, b.qkv_b);
      p.reverse = 1;                             // LN1 wrote abuf first-to-last
      p.col_scale = 0.125f * ATT_LOG2E; p.scale_cols = D;  // q * head_dim^-0.5 (vision_transformer.py:73,85), times log2(e): attention.cuh
      LaunchScope ls(h, K_GEMM_QKV, s);
      if (h->gemm_pair &&
          launch_gemm_pair<EPI_BF16>(w.tm_abuf, b.tm_qkv_h, w.tm_qkv_out, w.tm_qkv_out, p, sms, s) != cudaSuccess) {
        (void)cudaGetLastError();   // no 2-CTA clusters on this device / partition: one CTA per tile
        h->gemm_pair = false;
      }
      if (!h->gemm_pair) DSG_CUDA(h, launch_gemm(EPI_BF16, w.tm_abuf, b.tm_qkv, w.tm_qkv_out, w.tm_qkv_out, p, sms, s));
      ++n;
    }
    if (stop == 2 + 3 * i) { h->launches = n; return 0; }
    if (feat && feat->cls_rows && !feat->patch_mean && i == h->cfg.n_blocks - 1) {
      if (cls_only_tail(h, w, b, batch, feat->out + size_t(i - feat->first) * batch * D, s, n) != 0) return -1;
      break;
    }
    {
      AttnParams p{};
      p.B = batch; p.H = H; p.N = h->Ntok; p.D = D; p.out = w.abuf;
      LaunchScope ls(h, K_ATTN, s);
      DSG_CUDA(h, launch_attention(w.tm_qkv3d, p, h->num_sms, s, h->attn_unshifted)); n += h->attn_unshifted ? 2 : 1;
    }
    {
      GemmParams p = gp(D, D, b.proj_b);
      p.reverse = 1;                             // the attention kernel wrote abuf first-to-last
      LaunchScope ls(h, K_GEMM_PROJ, s);
      DSG_CUDA(h, launch_gemm(EPI_RESID_F32, w.tm_abuf, b.tm_proj, w.tm_x_out, w.tm_x_out, p, sms, s)); ++n;
    }
    if (stop == 3 + 3 * i) { h->launches = n; return 0; }
    if (h->fused_mlp) {
      // LayerNorm2 -> fc1 -> GELU -> fc2 -> +x in ONE kernel (ViT-S: D = 384, hidden = 1536); with fuse_ln off the
      // LayerNorm runs as its own kernel and the MLP kernel TMA-loads its bf16 output
      MlpParams p{};
      p.M = M; p.x = w.x; p.b1 = b.fc1_b; p.b2 = b.fc2_b;
      if (h->fuse_ln) {
        p.fuse_ln = 1; p.ln_eps = eps;             // gamma / beta are in fc1_w / fc1_b (finalize_weights)
      } else {
        LaunchScope ls(h, K_LN, s); DSG_CUDA(h, launch_layernorm(w.x, b.ln2_g, b.ln2_b, w.abuf, M, D, eps, false, s)); ++n;
      }
      // start with the rows the producer of x / A wrote last: LN2 writes first-to-last (-> walk backwards), the proj GEMM
      // walks backwards itself (-> walk forwards when the LayerNorm is fused and this kernel follows it directly)
      p.reverse = h->fuse_ln ? 0 : 1;
      LaunchScope ls(h, K_MLP_FUSED, s);
      if (h->mlp_pair && launch_mlp_fused(w.tm_abuf, b.tm_fc1_h, b.tm_fc2_h, w.tm_x_out, p, sms, true, s) != cudaSuccess) {
        (void)cudaGetLastError();   // no 2-CTA clusters on this device / partition: same kernel, one CTA per row block
        h->mlp_pair = false;
      }
      if (!h->mlp_pair) DSG_CUDA(h, launch_mlp_fused(w.tm_abuf, b.tm_fc1_g, b.tm_fc2_g, w.tm_x_out, p, sms, false, s));
      ++n;
    } else {
      { LaunchScope ls(h, K_LN, s); DSG_CUDA(h, launch_layernorm(w.x, b.ln2_g, b.ln2_b, w.abuf, M, D, eps, false, s)); ++n; }
      {
        GemmParams p = gp(HID, D, b.fc1_b);
        p.reverse = 1;                           // LN2 wrote abuf first-to-last; fc2 then reads hid first-to-last
        LaunchScope ls(h, K_GEMM_FC1, s);
        if (h->gemm_pair &&
            launch_gemm_pair<EPI_GELU_BF16>(w.tm_abuf, b.tm_fc1_p, w.tm_hid_out, w.tm_hid_out, p, sms, s) != cudaSuccess) {
          (void)cudaGetLastError();
          h->gemm_pair = false;
        }
        if (!h->gemm_pair) DSG_CUDA(h, launch_gemm(EPI_GELU_BF16, w.tm_abuf, b.tm_fc1, w.tm_hid_out, w.tm_hid_out, p, sms, s));
        ++n;
      }
      {
        GemmParams p = gp(D, HID, b.fc2_b);
        LaunchScope ls(h, K_GEMM_FC2, s);
        if (h->gemm_pair &&
            launch_gemm_pair<EPI_RESID_F32>(w.tm_hid, b.tm_fc2_p, w.tm_x_out, w.tm_x_out, p, sms, s) != cudaSuccess) {
          (void)cudaGetLastError();
          h->gemm_pair = false;
        }
        if (!h->gemm_pair) DSG_CUDA(h, launch_gemm(EPI_RESID_F32, w.tm_hid, b.tm_fc2, w.tm_x_out, w.tm_x_out, p, sms, s));
        ++n;
      }
    }
    if (feat && feat->cls_rows && i == h->cfg.n_blocks - 1 && feat->patch_mean) {
      LaunchScope ls(h, K_EMBED_POOL, s);
      float* cls = feat->out ? feat->out + size_t(i - feat->first) * batch * D : nullptr;
      DSG_CUDA(h, launch_embed_pool(w.x, h->norm_g, h->norm_b, cls, feat->patch_mean, batch, h->Ntok, D, eps, s));
      ++n;
    } else if (feat && feat->cls_rows && i >= feat->first && feat->out) {
      // the B CLS rows, gathered into [B, D] and normed by the same fp32 LayerNorm kernel as the features
      {
        LaunchScope ls(h, K_CLS_GATHER, s);
        DSG_CUDA(h, cudaMemcpy2DAsync(w.cls_x, size_t(D) * 4, w.x, size_t(h->Ntok) * D * 4, size_t(D) * 4, batch,
                                      cudaMemcpyDeviceToDevice, s));
        ++n;
      }
      LaunchScope ls(h, K_LN, s);
      DSG_CUDA(h, launch_layernorm_f32(w.cls_x, h->norm_g, h->norm_b, feat->out + size_t(i - feat->first) * batch * D,
                                       batch, D, eps, s));
      ++n;
    } else if (feat && !feat->cls_rows && i >= feat->first) {
      // before anything else touches x (the kernel-chain head reuses its buffer for relu(layer_2))
      LaunchScope ls(h, K_LN, s);
      DSG_CUDA(h, launch_layernorm_f32(w.x, h->norm_g, h->norm_b, feat->out + size_t(i - feat->first) * M * D, M, D, eps, s));
      ++n;
    }
    if (stop == 4 + 3 * i) { h->launches = n; return 0; }
  }
  if (feat && feat->backbone_only) { h->launches = n; return 0; }

  // ---- final norm + head (vision_transformer.py:243, pl_torch_modules.py:243-255) ----
  // The head runs in "bf16x3" precision (operands split into hi + lo bf16 parts, three-fold K): its plain
  // bf16 rounding would otherwise be the largest contribution to the log-prob error.
  uint8_t* lr = lowres ? lowres : w.lowres;
  if (h->fused_head) {
    // ONE kernel: LayerNorm -> layer_1 -> layer_2 -> layer_3 -> log_softmax -> argmax -> p x p replication (head.cuh)
    LaunchScope ls(h, K_HEAD_FUSED, s);
    DSG_CUDA(h, launch_head_fused(h, w.x, M, logprobs, lr, (labels && h->p_rep > 0) ? reinterpret_cast<long long*>(labels) : nullptr, s));
    h->launches = ++n;
    return 0;
  }
  { LaunchScope ls(h, K_LN, s); DSG_CUDA(h, launch_layernorm(w.x, h->norm_g, h->norm_b, w.qkv, M, D, eps, true, s)); ++n; }
  // tail kernel: eight lanes per patch, 32 patches per 256-thread block; it also writes the p x p blocks of the int64
  // label map (reference pl_torch_modules.py:297-298) when the caller wants one and the map is not empty (p = 480 // g)
  const int tail_grid = std::min((batch * h->P + 31) / 32, 16 * h->num_sms);
  long long* tail_labels = (labels && h->p_rep > 0) ? reinterpret_cast<long long*>(labels) : nullptr;
  if (h->cfg.head_kind == 1) {
    // 'linear' head (pl_torch_modules.py:127-138): one bf16x3 GEMM -> logits [M, C] (row pitch kLinPitch) -> log_softmax
    {
      GemmParams p = gp(h->cfg.n_classes, 3 * D, h->h1_b);
      p.a_wrap = 2 * D;
      LaunchScope ls(h, K_GEMM_HEAD, s);
      DSG_CUDA(h, launch_gemm(EPI_BIAS_F32, w.tm_qkv_a, h->tm_h1, w.tm_lin_out, w.tm_lin_out, p, sms, s)); ++n;
    }
    LaunchScope ls(h, K_HEAD_TAIL, s);
    if (h->cfg.n_classes <= 8)
      head_tail_kernel<true, 8><<<tail_grid, 256, 0, s>>>(w.x, kLinPitch, nullptr, nullptr, logprobs, lr, tail_labels, batch,
                                                          h->gh, h->gw, h->p_rep, h->Ntok, 0, h->cfg.n_classes);
    else
      head_tail_kernel<true, 16><<<tail_grid, 256, 0, s>>>(w.x, kLinPitch, nullptr, nullptr, logprobs, lr, tail_labels, batch,
                                                           h->gh, h->gw, h->p_rep, h->Ntok, 0, h->cfg.n_classes);
    DSG_CUDA(h, cudaGetLastError()); ++n;
  } else {
    {
      GemmParams p = gp(h->cfg.head_h1, 3 * D, h->h1_b);
      p.split_part = kHeadPart;
      p.a_wrap = 2 * D;
      LaunchScope ls(h, K_GEMM_HEAD, s);
      DSG_CUDA(h, launch_gemm(EPI_RELU_SPLIT_BF16, w.tm_qkv_a, h->tm_h1, w.tm_h1s_out, w.tm_h1s_out, p, sms, s)); ++n;
    }
    {
      GemmParams p = gp(h->cfg.head_h2, 3 * kHeadPart, h->b2);
      p.a_wrap = 2 * kHeadPart;
      LaunchScope ls(h, K_GEMM_HEAD, s);
      DSG_CUDA(h, launch_gemm(EPI_RELU_F32, w.tm_h1s_a, h->tm_h2, w.tm_h2_out, w.tm_h2_out, p, sms, s)); ++n;
    }
    LaunchScope ls(h, K_HEAD_TAIL, s);
    if (h->cfg.n_classes <= 8)
      head_tail_kernel<false, 8><<<tail_grid, 256, 0, s>>>(w.x, h->cfg.head_h2, h->w3, h->b3, logprobs, lr, tail_labels, batch,
                                                           h->gh, h->gw, h->p_rep, h->Ntok, h->cfg.head_h2, h->cfg.n_classes);
    else
      head_tail_kernel<false, 16><<<tail_grid, 256, 0, s>>>(w.x, h->cfg.head_h2, h->w3, h->b3, logprobs, lr, tail_labels, batch,
                                                            h->gh, h->gw, h->p_rep, h->Ntok, h->cfg.head_h2, h->cfg.n_classes);
    DSG_CUDA(h, cudaGetLastError()); ++n;
  }
  h->launches = n;
  return 0;
}

int dinoseg_forward(dinoseg_t* h, const float* frames, int batch, float* logprobs, uint8_t* lowres, int64_t* labels,
                    void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return -1;
  if (h->res_h == 0) DSG_FAIL(h, "dinoseg_forward: call dinoseg_set_resolution first");
  if (!frames || batch <= 0 || !workspace) DSG_FAIL(h, "dinoseg_forward: bad arguments");
  DSG_CUDA(h, cudaSetDevice(h->device));
  if (bind_workspace(h, h->user, workspace, workspace_bytes, batch) != 0) return -1;
  return forward_impl(h, h->user, frames, nullptr, nullptr, batch, logprobs, lowres, labels,
                      static_cast<cudaStream_t>(stream));
}

// Frames per pipeline chunk.
// streaming == false (the synchronous call, nothing else in flight): small enough to overlap the copies with the
// kernels inside ONE call (6..16 frames), and such that the 128-token row blocks of a chunk fill whole waves of the
// persistent kernels (one CTA per SM).  Swept on B200 at 480 px, batch 64: 5 -> 5474, 8 -> 6067, 10 -> 6163,
// 16 -> 5796, 21 -> 5885, 32 -> 5367 frames/s.
// streaming == true (dinoseg_predict_host_submit: the caller keeps several submissions in flight): the copies of one
// submission overlap the kernels of its neighbours, so chunks are as large as a 2 GB workspace allows (64 frames at
// 480 px, 16 at 960 px) - every kernel then runs at the efficiency of the device path instead of paying its tail
// wave once per ~10 frames.
static int pick_host_chunk(const dinoseg* h, int batch, bool streaming) {
  if (h->host_chunk > 0) return h->host_chunk < batch ? h->host_chunk : batch;
  if (streaming) {
    const long long max_rows = 262144;                       // ~2 GB of workspace for ViT-S
    long long c = max_rows / h->Ntok;
    if (c < 1) c = 1;
    if (c >= batch) return batch;
    const int parts = int((batch + c - 1) / c);              // equal parts rather than full chunks plus a remainder
    return (batch + parts - 1) / parts;
  }
  int best = batch < 6 ? batch : 6;
  double best_eff = -1.0;
  for (int c = 6; c <= 16 && c <= batch; ++c) {
    const long long blocks = ((long long)c * h->Ntok + 127) / 128;
    const long long waves = (blocks + h->num_sms - 1) / h->num_sms;
    const double eff = double(blocks) / double(waves * h->num_sms);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = c; }
  }
  return best;
}

// host cores this process may use, divided by the ranks that share the host (torchrun exports LOCAL_WORLD_SIZE)
static int host_cores_per_rank() {
  int cpus = 0;
  cpu_set_t set;
  if (sched_getaffinity(0, sizeof(set), &set) == 0) cpus = CPU_COUNT(&set);
  if (cpus <= 0) cpus = int(std::thread::hardware_concurrency());
  const char* lw = getenv("LOCAL_WORLD_SIZE");
  const int ranks = lw && atoi(lw) > 0 ? atoi(lw) : 1;
  return cpus / ranks;
}

// Label maps of the host entry points: expand on the host (low-res maps over PCIe, int64 maps written by worker
// threads) or replicate on the GPU and copy the int64 maps out.  Automatic choice: host expansion needs cores - with
// >= 8 per rank it measured +2.5 % end to end (one GPU, 16 cores), with 4 per rank (eight GPUs on a 32-vCPU host)
// the workers compete with the ranks' own threads and the DMA path is the safer one.
static bool host_expand_on(const dinoseg* h) {
  if (h->pool_failed) return false;
  if (h->host_expand >= 0) return h->host_expand != 0;
  static const bool enough = host_cores_per_rank() >= 8;
  return enough;
}

static dinoseg::Ticket* find_ticket(dinoseg_t* h, int64_t id) {
  for (dinoseg::Ticket& t : h->tickets)
    if (t.id == id) return &t;
  return nullptr;
}

// Completes one submission: host-side expansion of its label maps (expand mode), then its lanes' last copies.
static int ticket_wait(dinoseg_t* h, dinoseg::Ticket& t) {
  int rc = 0;
  if (t.expand) {
    // chunk by chunk, as the low-res maps arrive: one expansion task per frame
    const size_t P = size_t(t.g) * t.g, W = size_t(t.g) * t.p_rep;
    int f0 = 0;
    for (size_t c = 0; c < t.plan.size(); f0 += t.plan[c], ++c) {
      if (t.plan[c] <= 0) continue;
      if (cudaEventSynchronize(t.chunk_done[c]) != cudaSuccess) { rc = -1; break; }
      if (t.host_lowres) memcpy(t.host_lowres + size_t(f0) * P, t.low_stage + size_t(f0) * P, size_t(t.plan[c]) * P);
      for (int i = 0; i < t.plan[c]; ++i) {
        const uint8_t* low = t.low_stage + size_t(f0 + i) * P;
        int64_t* out = t.host_labels + size_t(f0 + i) * W * W;
        const int g = t.g, prep = t.p_rep;
        h->pool->submit([low, out, g, prep] { expand_labels_host(low, out, g, prep); });
      }
    }
    h->pool->wait_all();
  }
  if (cudaEventSynchronize(t.done) != cudaSuccess) rc = -1;
  t.id = 0;
  if (rc != 0) { h->err = "dinoseg_predict_host_wait: a CUDA operation of the submission failed"; }
  return rc;
}

// Shared implementation of the host entry points: `host_frames` are fp32 normalised frames (pp == nullptr) or raw
// uint8 HWC frames of src_h x src_w pixels (pp != nullptr).  Enqueues the whole submission and returns its ticket
// (> 0) without waiting for the GPU; < 0 on error (nothing is left in flight then).
static int64_t predict_host_submit_impl(dinoseg_t* h, const void* host_frames, const PreprocParams* pp, int batch,
                                        uint8_t* host_lowres, int64_t* host_labels, void* stream, const char* who,
                                        bool streaming) {
  if (!h) return -1;
  if (h->res_h == 0) DSG_FAIL(h, "%s: call dinoseg_set_resolution first", who);
  if (h->gh != h->gw)   // frame and label-map sizes below are those of a square grid (predict's semantics)
    DSG_FAIL(h, "%s: the host entry points take square resolutions only (resolution %dx%d)", who, h->res_h, h->res_w);
  if (!host_frames || batch <= 0) DSG_FAIL(h, "%s: bad arguments", who);
  dinoseg::Ticket* tk = find_ticket(h, 0);
  if (!tk) DSG_FAIL(h, "%s: %d submissions are outstanding; call dinoseg_predict_host_wait first", who, dinoseg::kTickets);
  DSG_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // The batch is cut into chunks that go round-robin through three slots (frame staging + workspace + result staging):
  // the H2D copy of chunk c+1 (copy-in stream) and the D2H copy of chunk c-1 (copy-out stream) overlap the kernels of
  // chunk c (compute stream).  Frames are independent, so chunking does not change any result bit.  Consecutive
  // submissions queue behind each other on the same three streams: the first H2D copy of submission k+1 overlaps the
  // last kernels and the last D2H copy of submission k.
  const int chunk = pick_host_chunk(h, batch, streaming);
  const size_t frame_bytes = pp ? size_t(pp->src_h) * pp->src_w * 3 : size_t(3) * h->res_h * h->res_h * sizeof(float);
  const size_t W = size_t(h->gh) * h->p_rep;
  const size_t label_elems = W * W;
  const size_t wbytes = dinoseg_workspace_bytes(h, chunk);
  if (!h->host_start) DSG_CUDA(h, cudaEventCreateWithFlags(&h->host_start, cudaEventDisableTiming));
  if (!h->s_in) DSG_CUDA(h, cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
  if (!h->s_comp) DSG_CUDA(h, cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking));
  if (!h->s_out) DSG_CUDA(h, cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
  if (!tk->done) DSG_CUDA(h, cudaEventCreateWithFlags(&tk->done, cudaEventDisableTiming));
  auto grow = [&](HostLane&, void** p, size_t* cap, size_t need) -> cudaError_t {
    if (need <= *cap) return cudaSuccess;
    if (*p) {                                  // a buffer of an earlier, smaller submission: nothing may still use it
      cudaStreamSynchronize(h->s_in); cudaStreamSynchronize(h->s_comp); cudaStreamSynchronize(h->s_out);
      cudaFree(*p); *p = nullptr; *cap = 0;
    }
    cudaError_t e = cudaMalloc(p, need);
    if (e == cudaSuccess) *cap = need;
    return e;
  };
  // chunk plan: a SHORT first chunk (its H2D copy is the pipeline fill that nothing overlaps) and a short last one
  // (its D2H copy is the drain), full chunks in between
  std::vector<int>& plan = tk->plan;
  plan.clear();
  if (batch <= chunk) {
    plan.push_back(batch);
  } else if (streaming) {
    for (int rest = batch; rest > 0; rest -= chunk) plan.push_back(rest < chunk ? rest : chunk);
  } else {
    int rest = batch;
    const int rem = batch % chunk;
    const int first = rem ? rem : chunk / 2;
    plan.push_back(first);
    rest -= first;
    while (rest > chunk) { plan.push_back(chunk); rest -= chunk; }
    plan.push_back(rest);           // = chunk, or the other half of a split chunk when chunk divides batch
  }
  const int nchunks = int(plan.size());
  // slots are taken round-robin ACROSS submissions (h->slot_seq), so that a one-chunk submission does not wait for the
  // buffers of the one before it
  const int nlanes = dinoseg::kLanes;
  const bool want_labels = host_labels && label_elems;
  // Label maps: the int64 [g*p, g*p] map is 512x the size of the low-res map it replicates.  With host expansion the
  // GPU ships the low-res maps (3.6 KB per frame at 480 px) and worker threads expand them into the caller's buffer
  // (in dinoseg_predict_host_wait, while later submissions are already computing), instead of 1.84 MB per frame over PCIe.
  bool expand = want_labels && host_expand_on(h);
  if (expand && !h->pool) {
    int n = host_cores_per_rank();
    if (const char* e = getenv("DINOSEG_HOST_THREADS")) n = atoi(e);
    n = n < 1 ? 1 : (n > 8 ? 8 : n);
    try {
      h->pool = new HostPool(n);
    } catch (...) {                              // no threads to be had: GPU replication + whole-map copies
      h->pool = nullptr;
      h->pool_failed = true;
      expand = false;
    }
  }
  if (expand) {
    const size_t need = size_t(batch) * h->P;
    if (need > tk->low_stage_cap) {
      if (tk->low_stage) { cudaFreeHost(tk->low_stage); tk->low_stage = nullptr; tk->low_stage_cap = 0; }
      DSG_CUDA(h, cudaHostAlloc(reinterpret_cast<void**>(&tk->low_stage), need, cudaHostAllocDefault));
      tk->low_stage_cap = need;
    }
    while (int(tk->chunk_done.size()) < nchunks) {
      cudaEvent_t e;
      DSG_CUDA(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      tk->chunk_done.push_back(e);
    }
  }
  // a slot's events and buffers are created / grown when a chunk first needs them
  auto prepare_slot = [&](HostLane& l) -> int {
    for (cudaEvent_t* e : {&l.in_done, &l.comp_done, &l.out_done})
      if (!*e) DSG_CUDA(h, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    const size_t ws_before = l.ws_cap;
    DSG_CUDA(h, grow(l, reinterpret_cast<void**>(&l.frames), &l.frames_cap, size_t(chunk) * frame_bytes));
    DSG_CUDA(h, grow(l, &l.ws, &l.ws_cap, wbytes));
    DSG_CUDA(h, grow(l, reinterpret_cast<void**>(&l.lowres), &l.lowres_cap, size_t(chunk) * h->P));
    if (want_labels && !expand)
      DSG_CUDA(h, grow(l, reinterpret_cast<void**>(&l.labels), &l.labels_cap, size_t(chunk) * label_elems * sizeof(int64_t)));
    if (l.ws_cap != ws_before) l.bufs.base = nullptr;
    return 0;
  };
  // From here on work is in flight: every error exit drains the lanes first, so that the caller may free its buffers.
  auto enqueue = [&]() -> int {
    // the pipeline starts after whatever the caller queued on its stream
    DSG_CUDA(h, cudaEventRecord(h->host_start, s));
    DSG_CUDA(h, cudaStreamWaitEvent(h->s_in, h->host_start, 0));
    int f0 = 0;
    for (int c = 0; c < nchunks; f0 += plan[c], ++c) {
      HostLane& l = h->lanes[(h->slot_seq++) % nlanes];
      const int nb = plan[c];
      if (nb <= 0) continue;
      if (prepare_slot(l) != 0) return -1;
      // copy-in: the slot's frame staging is free once the kernels of its previous chunk have finished
      // (waiting on an event that has never been recorded is a no-op: first use of the slot)
      DSG_CUDA(h, cudaStreamWaitEvent(h->s_in, l.comp_done, 0));
      DSG_CUDA(h, cudaMemcpyAsync(l.frames, static_cast<const uint8_t*>(host_frames) + size_t(f0) * frame_bytes,
                                  size_t(nb) * frame_bytes, cudaMemcpyHostToDevice, h->s_in));
      DSG_CUDA(h, cudaEventRecord(l.in_done, h->s_in));
      // compute: after the frames have arrived and the slot's previous results have left
      DSG_CUDA(h, cudaStreamWaitEvent(h->s_comp, l.in_done, 0));
      DSG_CUDA(h, cudaStreamWaitEvent(h->s_comp, l.out_done, 0));
      if (bind_workspace(h, l.bufs, l.ws, l.ws_cap, nb) != 0) return -1;
      if (forward_impl(h, l.bufs, pp ? nullptr : l.frames, pp ? reinterpret_cast<const uint8_t*>(l.frames) : nullptr, pp, nb,
                       nullptr, l.lowres, (want_labels && !expand) ? l.labels : nullptr, h->s_comp) != 0)
        return -1;
      DSG_CUDA(h, cudaEventRecord(l.comp_done, h->s_comp));
      // copy-out
      DSG_CUDA(h, cudaStreamWaitEvent(h->s_out, l.comp_done, 0));
      if (expand) {
        DSG_CUDA(h, cudaMemcpyAsync(tk->low_stage + size_t(f0) * h->P, l.lowres, size_t(nb) * h->P, cudaMemcpyDeviceToHost,
                                    h->s_out));
        DSG_CUDA(h, cudaEventRecord(tk->chunk_done[c], h->s_out));
      } else {
        if (host_lowres)
          DSG_CUDA(h, cudaMemcpyAsync(host_lowres + size_t(f0) * h->P, l.lowres, size_t(nb) * h->P, cudaMemcpyDeviceToHost,
                                      h->s_out));
        if (want_labels)
          DSG_CUDA(h, cudaMemcpyAsync(host_labels + size_t(f0) * label_elems, l.labels,
                                      size_t(nb) * label_elems * sizeof(int64_t), cudaMemcpyDeviceToHost, h->s_out));
      }
      DSG_CUDA(h, cudaEventRecord(l.out_done, h->s_out));
    }
    // (the caller's stream is NOT made to wait for the pipeline: the results are host buffers, complete when
    // dinoseg_predict_host_wait returns, and a wait here would serialise consecutive submissions)
    DSG_CUDA(h, cudaEventRecord(tk->done, h->s_out));      // the copy-out stream is in order: one event covers all chunks
    return 0;
  };
  if (enqueue() != 0) {
    const std::string why = h->err;
    for (cudaStream_t st : {h->s_in, h->s_comp, h->s_out})
      if (st) cudaStreamSynchronize(st);
    if (h->pool) h->pool->wait_all();
    (void)cudaGetLastError();
    h->err = why;
    return -1;
  }
  tk->expand = expand;
  tk->host_lowres = host_lowres;
  tk->host_labels = host_labels;
  tk->g = h->gh;
  tk->p_rep = h->p_rep;
  tk->id = h->next_ticket++;
  return tk->id;
}

static int predict_host_wait_impl(dinoseg_t* h, int64_t ticket) {
  if (!h) return -1;
  DSG_CUDA(h, cudaSetDevice(h->device));
  if (ticket == 0) {                     // everything outstanding, oldest first
    int rc = 0;
    for (;;) {
      dinoseg::Ticket* oldest = nullptr;
      for (dinoseg::Ticket& t : h->tickets)
        if (t.id != 0 && (!oldest || t.id < oldest->id)) oldest = &t;
      if (!oldest) return rc;
      if (ticket_wait(h, *oldest) != 0) rc = -1;
    }
  }
  dinoseg::Ticket* t = ticket > 0 ? find_ticket(h, ticket) : nullptr;
  if (!t) DSG_FAIL(h, "dinoseg_predict_host_wait: unknown ticket %lld (already waited for?)", (long long)ticket);
  return ticket_wait(h, *t);
}

static int predict_host_impl(dinoseg_t* h, const void* host_frames, const PreprocParams* pp, int batch,
                             uint8_t* host_lowres, int64_t* host_labels, void* stream, const char* who) {
  const int64_t t = predict_host_submit_impl(h, host_frames, pp, batch, host_lowres, host_labels, stream, who, false);
  return t < 0 ? -1 : predict_host_wait_impl(h, t);
}

static int make_preproc(dinoseg_t* h, int src_h, int src_w, const float* mean, const float* std_, PreprocParams* pp) {
  if (src_h < 1 || src_w < 1 || src_h > 16384 || src_w > 16384 || !mean || !std_) DSG_FAIL(h, "bad preprocessing arguments");
  pp->src_h = src_h; pp->src_w = src_w;
  for (int c = 0; c < 3; ++c) {
    // albumentations Normalize: mean * 255 and 1 / (std * 255), both in float32
    pp->mean255[c] = mean[c] * 255.0f;
    pp->denom[c] = 1.0f / (std_[c] * 255.0f);
  }
  return 0;
}

int dinoseg_predict_host(dinoseg_t* h, const float* host_frames, int batch, uint8_t* host_lowres,
                         int64_t* host_labels, void* stream) {
  return predict_host_impl(h, host_frames, nullptr, batch, host_lowres, host_labels, stream, "dinoseg_predict_host");
}

int dinoseg_predict_host_u8(dinoseg_t* h, const uint8_t* host_frames, int batch, int src_h, int src_w, const float* mean,
                            const float* std_, uint8_t* host_lowres, int64_t* host_labels, void* stream) {
  if (!h) return -1;
  PreprocParams pp;
  if (make_preproc(h, src_h, src_w, mean, std_, &pp) != 0) return -1;
  return predict_host_impl(h, host_frames, &pp, batch, host_lowres, host_labels, stream, "dinoseg_predict_host_u8");
}

int64_t dinoseg_predict_host_submit(dinoseg_t* h, const float* host_frames, int batch, uint8_t* host_lowres,
                                    int64_t* host_labels, void* stream) {
  return predict_host_submit_impl(h, host_frames, nullptr, batch, host_lowres, host_labels, stream,
                                  "dinoseg_predict_host_submit", true);
}

int64_t dinoseg_predict_host_submit_u8(dinoseg_t* h, const uint8_t* host_frames, int batch, int src_h, int src_w,
                                       const float* mean, const float* std_, uint8_t* host_lowres, int64_t* host_labels,
                                       void* stream) {
  if (!h) return -1;
  PreprocParams pp;
  if (make_preproc(h, src_h, src_w, mean, std_, &pp) != 0) return -1;
  return predict_host_submit_impl(h, host_frames, &pp, batch, host_lowres, host_labels, stream,
                                  "dinoseg_predict_host_submit_u8", true);
}

int dinoseg_predict_host_wait(dinoseg_t* h, int64_t ticket) { return predict_host_wait_impl(h, ticket); }

int dinoseg_forward_u8(dinoseg_t* h, const uint8_t* frames, int batch, int src_h, int src_w, const float* mean,
                       const float* std_, float* logprobs, uint8_t* lowres, int64_t* labels, void* workspace,
                       size_t workspace_bytes, void* stream) {
  if (!h) return -1;
  if (h->res_h == 0) DSG_FAIL(h, "dinoseg_forward_u8: call dinoseg_set_resolution first");
  if (!frames || batch <= 0 || !workspace) DSG_FAIL(h, "dinoseg_forward_u8: bad arguments");
  PreprocParams pp;
  if (make_preproc(h, src_h, src_w, mean, std_, &pp) != 0) return -1;
  DSG_CUDA(h, cudaSetDevice(h->device));
  if (bind_workspace(h, h->user, workspace, workspace_bytes, batch) != 0) return -1;
  return forward_impl(h, h->user, nullptr, frames, &pp, batch, logprobs, lowres, labels, static_cast<cudaStream_t>(stream));
}

int dinoseg_set_pair_kernels(dinoseg_t* h, int on) {
  if (!h || on < 0 || on > 1) return -1;
  h->gemm_pair = on != 0;
  h->mlp_pair = h->fused_mlp && on != 0;
  return 0;
}

int dinoseg_expand_labels_host(const uint8_t* lowres, int batch, int g, int p, int64_t* labels) {
  if (!lowres || !labels || batch <= 0 || g <= 0 || p <= 0 || size_t(g) * p > 480) return -1;
  const size_t W = size_t(g) * p;
  for (int b = 0; b < batch; ++b) expand_labels_host(lowres + size_t(b) * g * g, labels + size_t(b) * W * W, g, p);
  return 0;
}

int dinoseg_get_pair_kernels(const dinoseg_t* h) { return h ? (h->gemm_pair ? 1 : 0) | (h->mlp_pair ? 2 : 0) : -1; }

int dinoseg_set_host_expand(dinoseg_t* h, int on) {
  if (!h || on < -1 || on > 1) return -1;
  h->host_expand = on;              // -1 = automatic (cores per rank), 0 = GPU replication + DMA, 1 = host expansion
  return 0;
}

int dinoseg_get_host_expand(const dinoseg_t* h) { return h ? (host_expand_on(h) ? 1 : 0) : -1; }

int dinoseg_set_host_chunk(dinoseg_t* h, int frames_per_chunk) {
  if (!h || frames_per_chunk < 0) return -1;
  h->host_chunk = frames_per_chunk;   // 0 = automatic
  return 0;
}

int dinoseg_argmax_replicate(const float* logprobs, int batch, int g, int n_classes, int p, uint8_t* lowres,
                             int64_t* labels, void* stream) {
  if (!logprobs || !lowres || batch <= 0 || g <= 0 || n_classes < 1 || n_classes > HEAD_MAX_C || p < 0) return -1;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int rows = batch * g * g;
  argmax_rows_kernel<<<(rows + 255) / 256, 256, 0, s>>>(logprobs, lowres, rows, n_classes);
  if (cudaGetLastError() != cudaSuccess) return -2;
  if (labels && p > 0 && launch_replicate(lowres, labels, batch, g, p, s) != cudaSuccess) return -3;
  return 0;
}

int dinoseg_half_counts(const uint8_t* lowres, int batch, int g, int p, int n_classes, int32_t* counts, void* stream) {
  if (!lowres || !counts || batch <= 0 || g <= 0 || p <= 0 || n_classes < 1 || n_classes > 256) return -1;
  half_counts_kernel<<<batch, 256, 0, static_cast<cudaStream_t>(stream)>>>(lowres, counts, g, p, n_classes);
  return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int64_t dinoseg_copy_buffer(dinoseg_t* h, const char* name, void* dst, size_t dst_bytes, void* stream) {
  if (!h || !name || !dst) return -1;
  const void* src = nullptr;
  size_t bytes = 0;
  const WorkBufs* w = h->last;
  const size_t M = size_t(w ? w->batch : 0) * h->Ntok, D = h->cfg.embed_dim;
  const std::string nm(name);
  if (nm == "pos") { src = h->pos; bytes = size_t(h->Ntok) * D * 4; }
  else if (nm == "x") { src = w ? w->x : nullptr; bytes = M * D * 4; }
  else if (nm == "abuf") { src = w ? w->abuf : nullptr; bytes = M * D * 2; }
  else if (nm == "qkv") { src = w ? w->qkv : nullptr; bytes = M * 3 * D * 2; }
  else DSG_FAIL(h, "dinoseg_copy_buffer: unknown buffer '%s'", name);
  if (!src || bytes == 0) DSG_FAIL(h, "dinoseg_copy_buffer: buffer '%s' not available yet", name);
  if (bytes > dst_bytes) DSG_FAIL(h, "dinoseg_copy_buffer: destination too small (%zu < %zu)", dst_bytes, bytes);
  DSG_CUDA(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return int64_t(bytes);
}

// ---- kernel-level entry points ------------------------------------------------------------
int dinoseg_op_gemm(const void* A, const void* W, const float* bias, void* out, int M, int N, int K, int ldo, int epi,
                    float col_scale, int scale_cols, const float* pos, int P, int Ntok, void* stream) {
  if (!A || !W || !out || M <= 0 || N <= 0 || K <= 0 || (K % GEMM_BK) != 0 || epi < 0 || epi > EPI_RELU_F32) return -1;  // (the split epilogue is exercised end to end)
  const bool f32 = gemm_out_is_f32(epi);
  if (f32 ? (N % 4 != 0) : (N % 8 != 0)) return -1;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  CUtensorMap ta, tw, to, tadd;
  GemmParams p{};
  p.N = N; p.K = K; p.bias = bias; p.col_scale = col_scale; p.scale_cols = scale_cols;
  bool ok = make_tmap_2d(&tw, W, N, K, K, GEMM_BN);
  if (epi == EPI_PATCH_F32) {
    // A [B*P, K] -> out [B*Ntok, N]: row b*Ntok + 1 + t = acc + bias + pos[1 + t]
    if (!pos || P <= 0 || Ntok != P + 1 || M % P != 0) return -1;
    const int B = M / P;
    p.rows_per_batch = P; p.batches = B; p.row_off = 1; p.add_batched = 0;
    ok &= make_tmap_gemm_a(&ta, A, P, B, K);
    ok &= make_tmap_gemm_out(&to, out, true, N, Ntok, B, ldo);
    ok &= make_tmap_gemm_out(&tadd, pos, true, N, Ntok, 1, N);
  } else {
    p.rows_per_batch = M; p.batches = 1; p.row_off = 0; p.add_batched = 0;
    ok &= make_tmap_gemm_a(&ta, A, M, 1, K);
    ok &= make_tmap_gemm_out(&to, out, f32, N, M, 1, ldo);
    tadd = to;
  }
  if (!ok) return -2;
  return launch_gemm(epi, ta, tw, to, tadd, p, sms, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : -3;
}

int dinoseg_op_gemm_pair(const void* A, const void* W, const float* bias, void* out, int M, int N, int K, int ldo, int epi,
                         float col_scale, int scale_cols, void* stream) {
  if (!A || !W || !out || M <= 0 || N <= 0 || K <= 0 || (K % GEMM_BK) != 0 || N % 8 != 0) return -1;
  if (epi != EPI_BF16 && epi != EPI_GELU_BF16 && epi != EPI_RESID_F32) return -1;
  const bool f32 = gemm_out_is_f32(epi);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  CUtensorMap ta, tw, to;
  GemmParams p{};
  p.N = N; p.K = K; p.bias = bias; p.col_scale = col_scale; p.scale_cols = scale_cols;
  p.rows_per_batch = M; p.batches = 1;
  bool ok = make_tmap_2d(&tw, W, N, K, K, GEMM_BN / 2);
  ok &= make_tmap_gemm_a(&ta, A, M, 1, K);
  ok &= make_tmap_gemm_out(&to, out, f32, N, M, 1, ldo);
  if (!ok) return -2;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const cudaError_t e = epi == EPI_BF16        ? launch_gemm_pair<EPI_BF16>(ta, tw, to, to, p, sms, s)
                        : epi == EPI_GELU_BF16 ? launch_gemm_pair<EPI_GELU_BF16>(ta, tw, to, to, p, sms, s)
                                               : launch_gemm_pair<EPI_RESID_F32>(ta, tw, to, to, p, sms, s);
  return e == cudaSuccess ? 0 : -3;
}

// Test hook for the worker pool of the host entry points: create a pool of n threads where the creation of thread number
// fail_at throws (fail_at < 0: none does), run one task per requested thread, destroy the pool.  Returns the number of
// threads the pool ended up with (0 when not even the first could be created: the caller's DMA fallback), or -1 if the
// tasks did not all run.  A partial failure must neither terminate the process nor leak a worker.
int dinoseg_debug_host_pool(int n, int fail_at) {
  if (n < 1 || n > 64) return -1;
  int size = 0;
  std::atomic<int> ran{0};
  try {
    HostPool pool(n, [fail_at](int i) { if (i == fail_at) throw std::system_error(std::make_error_code(std::errc::resource_unavailable_try_again)); });
    size = pool.size();
    for (int i = 0; i < n; ++i) pool.submit([&ran] { ran.fetch_add(1); });
    pool.wait_all();
  } catch (...) {
    return 0;
  }
  return ran.load() == n ? size : -1;
}

int dinoseg_debug_attn_items(int B, int H, int N, int32_t* items, int max_items) {
  if (B <= 0 || H <= 0 || N <= 0) return -1;
  AttnParams p{};
  p.B = B; p.H = H; p.N = N; p.D = H * ATT_DH;
  attn_plan_items(p);
  if (!items) return p.num_items;
  if (max_items < p.num_items) return -1;
  for (int i = 0; i < p.num_items; ++i) {
    const AttItem I = att_decode(p, i);
    int32_t* o = items + size_t(i) * 6;
    o[0] = I.bh[0]; o[1] = I.q0[0]; o[2] = I.bh[1]; o[3] = I.q0[1]; o[4] = I.act1 ? 1 : 0; o[5] = I.dual ? 1 : 0;
  }
  return p.num_items;
}

int dinoseg_debug_set_attn_timing(long long* dev_ptr) {
#if defined(DSG_ATTN_TIMING) || defined(DSG_GEMM_TIMING) || defined(DSG_MLP_TIMING)
  g_attn_timing = dev_ptr;
  return 0;
#else
  (void)dev_ptr;
  return -1;   // the library was not built with -DDSG_ATTN_TIMING
#endif
}

int dinoseg_cls_attention(dinoseg_t* h, const float* frames, int batch, float* attn, void* workspace,
                          size_t workspace_bytes, void* stream) {
  if (!h) return -1;
  if (h->res_h == 0) DSG_FAIL(h, "dinoseg_cls_attention: call dinoseg_set_resolution first");
  if (!frames || !attn || batch <= 0 || !workspace) DSG_FAIL(h, "dinoseg_cls_attention: bad arguments");
  if (h->cfg.n_blocks < 1) DSG_FAIL(h, "dinoseg_cls_attention: the model has no transformer block");
  DSG_CUDA(h, cudaSetDevice(h->device));
  if (bind_workspace(h, h->user, workspace, workspace_bytes, batch) != 0) return -1;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // run the path up to the qkv GEMM of the last kept block, then softmax(q_cls k^T) per head
  const int saved = h->debug_stop;
  h->debug_stop = 2 + 3 * (h->cfg.n_blocks - 1);
  const int rc = forward_impl(h, h->user, frames, nullptr, nullptr, batch, nullptr, nullptr, nullptr, s);
  h->debug_stop = saved;
  if (rc != 0) return rc;
  dim3 grid(h->cfg.num_heads, batch);
  cls_attention_kernel<<<grid, 256, 0, s>>>(h->user.qkv, attn, h->Ntok, h->cfg.embed_dim, h->cfg.num_heads);
  DSG_CUDA(h, cudaGetLastError());
  return 0;
}

// Backbone features of the last min(n_last, n_blocks) blocks in ONE pass over the blocks (no head).
static int features_impl(dinoseg_t* h, const float* frames, const uint8_t* frames_u8, const PreprocParams* pp, int batch,
                         int n_last, float* out, void* workspace, size_t workspace_bytes, void* stream, const char* what) {
  if (h->res_h == 0) DSG_FAIL(h, "%s: call dinoseg_set_resolution first", what);
  if ((!frames && !frames_u8) || batch <= 0 || !workspace) DSG_FAIL(h, "%s: bad arguments", what);
  if (!out) DSG_FAIL(h, "%s: out is NULL", what);
  if (n_last < 1) DSG_FAIL(h, "%s: n_last must be >= 1 (got %d)", what, n_last);
  if (h->cfg.n_blocks < 1) DSG_FAIL(h, "%s: the model has no transformer block", what);
  DSG_CUDA(h, cudaSetDevice(h->device));
  if (bind_workspace(h, h->user, workspace, workspace_bytes, batch) != 0) return -1;
  FeatureReq req;
  req.out = out;
  req.first = h->cfg.n_blocks - std::min(n_last, h->cfg.n_blocks);
  req.backbone_only = true;
  const int saved = h->debug_stop;   // a debug stop would leave slices of `out` unwritten
  h->debug_stop = 0;
  const int rc = forward_impl(h, h->user, frames, frames_u8, pp, batch, nullptr, nullptr, nullptr,
                              static_cast<cudaStream_t>(stream), &req);
  h->debug_stop = saved;
  return rc;
}

int dinoseg_features(dinoseg_t* h, const float* frames, int batch, int n_last, float* out, void* workspace,
                     size_t workspace_bytes, void* stream) {
  if (!h) return -1;
  return features_impl(h, frames, nullptr, nullptr, batch, n_last, out, workspace, workspace_bytes, stream,
                       "dinoseg_features");
}

int dinoseg_features_u8(dinoseg_t* h, const uint8_t* frames, int batch, int src_h, int src_w, const float* mean,
                        const float* std_, int n_last, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return -1;
  PreprocParams pp;
  if (make_preproc(h, src_h, src_w, mean, std_, &pp) != 0) return -1;
  return features_impl(h, nullptr, frames, &pp, batch, n_last, out, workspace, workspace_bytes, stream,
                       "dinoseg_features_u8");
}

// Image embeddings: CLS rows of the last min(n_last, n_blocks) blocks and / or the patch-token mean of the last one, in
// one pass over the blocks (no head).
static int embeddings_impl(dinoseg_t* h, const float* frames, const uint8_t* frames_u8, const PreprocParams* pp, int batch,
                           int n_last, float* cls_out, float* patch_mean, void* workspace, size_t workspace_bytes,
                           void* stream, const char* what) {
  if (h->res_h == 0) DSG_FAIL(h, "%s: call dinoseg_set_resolution first", what);
  if ((!frames && !frames_u8) || batch <= 0 || !workspace) DSG_FAIL(h, "%s: bad arguments", what);
  if (!cls_out && !patch_mean) DSG_FAIL(h, "%s: cls_out and patch_mean are both NULL", what);
  if (n_last < 1) DSG_FAIL(h, "%s: n_last must be >= 1 (got %d)", what, n_last);
  if (h->cfg.n_blocks < 1) DSG_FAIL(h, "%s: the model has no transformer block", what);
  DSG_CUDA(h, cudaSetDevice(h->device));
  if (bind_workspace(h, h->user, workspace, workspace_bytes, batch) != 0) return -1;
  FeatureReq req;
  req.out = cls_out;
  req.first = h->cfg.n_blocks - std::min(n_last, h->cfg.n_blocks);
  req.backbone_only = true;
  req.cls_rows = true;
  req.patch_mean = patch_mean;
  const int saved = h->debug_stop;   // a debug stop would leave the outputs unwritten
  h->debug_stop = 0;
  const int rc = forward_impl(h, h->user, frames, frames_u8, pp, batch, nullptr, nullptr, nullptr,
                              static_cast<cudaStream_t>(stream), &req);
  h->debug_stop = saved;
  return rc;
}

int dinoseg_embeddings(dinoseg_t* h, const float* frames, int batch, int n_last, float* cls_out, float* patch_mean,
                       void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return -1;
  return embeddings_impl(h, frames, nullptr, nullptr, batch, n_last, cls_out, patch_mean, workspace, workspace_bytes,
                         stream, "dinoseg_embeddings");
}

int dinoseg_embeddings_u8(dinoseg_t* h, const uint8_t* frames, int batch, int src_h, int src_w, const float* mean,
                          const float* std_, int n_last, float* cls_out, float* patch_mean, void* workspace,
                          size_t workspace_bytes, void* stream) {
  if (!h) return -1;
  PreprocParams pp;
  if (make_preproc(h, src_h, src_w, mean, std_, &pp) != 0) return -1;
  return embeddings_impl(h, nullptr, frames, &pp, batch, n_last, cls_out, patch_mean, workspace, workspace_bytes, stream,
                         "dinoseg_embeddings_u8");
}

int dinoseg_set_fused_mlp(dinoseg_t* h, int on) {
  if (!h) return -1;
  if (on && !(h->cfg.embed_dim == MLP_D && h->cfg.mlp_hidden == MLP_HID))
    DSG_FAIL(h, "the fused MLP kernel needs embed_dim 384 and mlp_hidden 1536");
  h->fused_mlp = on != 0;
  h->mlp_pair = on == 2;
  h->weights_dirty = true;          // fc1 with / without the folded LayerNorm2
  return 0;
}

int dinoseg_set_fused_head(dinoseg_t* h, int on) {
  if (!h) return -1;
  if (on && !(h->cfg.head_kind == 0 && h->cfg.embed_dim == HEAD_D && h->cfg.head_h1 <= HEAD_N1 && h->cfg.head_h2 <= HEAD_W3_PITCH - 4))
    DSG_FAIL(h, "the fused head kernel needs the 'mlp' head on embed_dim 384 with head widths <= 208 / 100");
  h->fused_head = on != 0;
  return 0;
}

int dinoseg_op_mlp(float* x, const void* A_bf16, const void* W1_bf16, const float* b1, const void* W2_bf16,
                   const float* b2, int M, void* stream) {
  return dinoseg_op_mlp_ex(x, A_bf16, W1_bf16, b1, W2_bf16, b2, M, 0, stream);
}

int dinoseg_op_mlp_ex(float* x, const void* A_bf16, const void* W1_bf16, const float* b1, const void* W2_bf16,
                      const float* b2, int M, int pair, void* stream) {
  if (!x || !A_bf16 || !W1_bf16 || !b1 || !W2_bf16 || !b2 || M <= 0) return -1;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  CUtensorMap ta, t1, t2, tx;
  const uint32_t wrows = pair ? 64 : 128;
  bool ok = make_tmap_gemm_a(&ta, A_bf16, M, 1, MLP_D);
  ok &= make_tmap_2d(&t1, W1_bf16, MLP_HID, MLP_D, MLP_D, wrows);
  ok &= make_tmap_2d(&t2, W2_bf16, MLP_D, MLP_HID, MLP_HID, wrows);
  ok &= make_tmap_gemm_out(&tx, x, true, MLP_D, M, 1, MLP_D);
  if (!ok) return -2;
  MlpParams p{};
  p.M = M; p.x = x; p.b1 = b1; p.b2 = b2;
  return launch_mlp_fused(ta, t1, t2, tx, p, sms, pair != 0, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : -3;
}

int dinoseg_op_fold_ln(const float* W, const float* bias, const float* gamma, const float* beta, int N, int K,
                       void* W_out_bf16, float* bias_out, void* stream) {
  if (!W || !bias || !gamma || !beta || !W_out_bf16 || !bias_out || N <= 0 || K <= 0) return -1;
  fold_ln_weight_kernel<<<(N * 32 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      W, bias, gamma, beta, static_cast<__nv_bfloat16*>(W_out_bf16), bias_out, N, K);
  return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int dinoseg_op_mlp_ln(float* x, float eps, const void* W1f_bf16, const float* b1f, const void* W2_bf16, const float* b2,
                      int M, int pair, void* stream) {
  if (!x || !W1f_bf16 || !b1f || !W2_bf16 || !b2 || M <= 0) return -1;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  CUtensorMap t1, t2, tx;
  const uint32_t wrows = pair ? 64 : 128;
  bool ok = make_tmap_2d(&t1, W1f_bf16, MLP_HID, MLP_D, MLP_D, wrows);
  ok &= make_tmap_2d(&t2, W2_bf16, MLP_D, MLP_HID, MLP_HID, wrows);
  ok &= make_tmap_gemm_out(&tx, x, true, MLP_D, M, 1, MLP_D);
  if (!ok) return -2;
  MlpParams p{};
  p.M = M; p.x = x; p.b1 = b1f; p.b2 = b2;
  p.fuse_ln = 1; p.ln_eps = eps;
  // (the A tensor map is not used by the fused-LayerNorm form; tx stands in for it)
  return launch_mlp_fused(tx, t1, t2, tx, p, sms, pair != 0, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : -3;
}

int dinoseg_op_attention(const void* qkv, void* out, int B, int N, int H, void* stream) {
  if (!qkv || !out || B <= 0 || N <= 0 || H <= 0) return -1;
  CUtensorMap tq;
  if (!make_tmap_qkv(&tq, qkv, B, N, uint64_t(3) * H * 64)) return -2;
  AttnParams p{};
  p.B = B; p.H = H; p.N = N; p.D = H * 64; p.out = static_cast<__nv_bfloat16*>(out);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const char* mode = getenv("DINOSEG_ATTN_UNSHIFTED");
  return launch_attention(tq, p, sms, static_cast<cudaStream_t>(stream), mode == nullptr || atoi(mode) != 0) == cudaSuccess ? 0 : -3;
}

int dinoseg_debug_attn_redone(void) {
  if (g_attn_last_flag == nullptr) return 0;
  int v = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  if (cudaMemcpy(&v, g_attn_last_flag, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return v == g_attn_last_id ? 1 : 0;
}

int dinoseg_op_layernorm(const float* x, const float* gamma, const float* beta, void* y, int M, int D, float eps,
                         void* stream) {
  return launch_layernorm(x, gamma, beta, static_cast<__nv_bfloat16*>(y), M, D, eps, false,
                          static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : -1;
}

int dinoseg_op_layernorm_f32(const float* x, const float* gamma, const float* beta, float* y, int M, int D, float eps,
                             void* stream) {
  if (!x || !gamma || !beta || !y) return -1;
  return launch_layernorm_f32(x, gamma, beta, y, M, D, eps, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : -1;
}

int dinoseg_op_posembed(const float* pos_src, float* out, int G0, int g, int D, void* stream) {
  return launch_posembed(pos_src, out, G0, g, g, D, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : -1;
}

int dinoseg_op_im2col(const float* frames, void* A, int B, int g, void* stream) {
  return launch_im2col(frames, static_cast<__nv_bfloat16*>(A), B, g, g, static_cast<cudaStream_t>(stream)) == cudaSuccess
             ? 0 : -1;
}

int dinoseg_op_f32_to_bf16(const float* in, void* out, size_t n, void* stream) {
  const unsigned blocks = unsigned(std::min<size_t>((n + 255) / 256, 4096));
  f32_to_bf16_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(in, static_cast<__nv_bfloat16*>(out), n);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // extern "C"
