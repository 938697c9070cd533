// Memory-bound kernels of the DINOSeg hot path (HBM-bound: coalesced 16-byte accesses,
// warp-shuffle reductions, no tensor cores).
#pragma once
#include <type_traits>

#include "ptx.cuh"

namespace dsg {

// ---------------------------------------------------------------------------------------
// fp32 -> bf16 conversion (weight packing at load time)
// ---------------------------------------------------------------------------------------
__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n) {
  size_t i = (size_t(blockIdx.x) * blockDim.x + threadIdx.x);
  const size_t stride = size_t(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) out[i] = __float2bfloat16_rn(in[i]);
}

// "bf16x3" operand split.  A product x*w with both operands rounded to bf16 carries a 2^-9 relative
// error; writing x = hi + lo (hi = bf16(x), lo = bf16(x - hi)) and using
//     x*w ~= x_hi*w_hi + x_lo*w_hi + x_hi*w_lo
// brings it to ~2^-16 while staying on the bf16 tensor cores: the three products are obtained from ONE
// GEMM of three-fold K over the operands A' = [hi | lo | hi], W' = [hi | hi | lo].  A' is stored as [hi | lo] only:
// the GEMM producer wraps its A column at 2*K (GemmParams::a_wrap), so the third segment re-reads hi (from L2).
//  Used for the
// segmentation head (0.7 % of the FLOPs), whose bf16 rounding otherwise dominates the log-prob error.
// W [N, K] fp32 -> W' [N, 3*Kp] bf16 (each part zero padded from K to Kp columns)
__global__ void split_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int N, int K, int Kp) {
  const size_t total = size_t(N) * Kp;
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
    const int n = int(i / Kp), k = int(i - size_t(n) * Kp);
    float v = k < K ? w[size_t(n) * K + k] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    __nv_bfloat16* o = out + size_t(n) * 3 * Kp + k;
    o[0] = hi; o[Kp] = hi; o[2 * Kp] = lo;
  }
}

// ---------------------------------------------------------------------------------------
// Positional-embedding table for a gh x gw patch grid (reference vision_transformer.py:202-222):
// row 0 = pos[0] (cls); rows 1 + i*gw + j = bicubic resample of the G0 x G0 source grid with torch's
// F.interpolate(scale_factor=((gh+0.1)/G0, (gw+0.1)/G0), mode='bicubic', align_corners=False) semantics, per axis:
//   src = rscale*(dst+0.5)-0.5 with rscale = float(1/scale_factor); taps floor(src)-1..+2 clamped
//   to [0,G0-1]; cubic-convolution weights with A = -0.75; inner sum over x, outer over y.
// Runs once per set_resolution(); the reference recomputes it every forward.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void cubic_coeffs(float t, float (&w)[4]) {
  const float A = -0.75f;
  const float x0 = t + 1.0f;
  w[0] = ((A * x0 - 5.0f * A) * x0 + 8.0f * A) * x0 - 4.0f * A;
  w[1] = ((A + 2.0f) * t - (A + 3.0f)) * t * t + 1.0f;
  const float t1 = 1.0f - t;
  w[2] = ((A + 2.0f) * t1 - (A + 3.0f)) * t1 * t1 + 1.0f;
  const float x3 = 2.0f - t;
  w[3] = ((A * x3 - 5.0f * A) * x3 + 8.0f * A) * x3 - 4.0f * A;
}

__global__ void posembed_bicubic_kernel(const float* __restrict__ pos_src /*[G0*G0+1, D]*/,
                                        float* __restrict__ out /*[gh*gw+1, D]*/, int G0, int gh, int gw, int D,
                                        float rscale_y, float rscale_x) {
  const size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t total = size_t(gh * gw + 1) * D;
  if (idx >= total) return;
  const int t = int(idx / D);
  const int d = int(idx - size_t(t) * D);
  if (t == 0) { out[idx] = pos_src[d]; return; }
  const int oy = (t - 1) / gw, ox = (t - 1) - oy * gw;
  const float sy = rscale_y * (float(oy) + 0.5f) - 0.5f;
  const float sx = rscale_x * (float(ox) + 0.5f) - 0.5f;
  int iy = min(int(floorf(sy)), G0 - 1);
  int ix = min(int(floorf(sx)), G0 - 1);
  const float ty = fminf(fmaxf(sy - float(iy), 0.f), 1.f);
  const float tx = fminf(fmaxf(sx - float(ix), 0.f), 1.f);
  float wy[4], wx[4];
  cubic_coeffs(ty, wy);
  cubic_coeffs(tx, wx);
  float acc = 0.f;
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int yy = min(max(iy - 1 + a, 0), G0 - 1);
    float rowacc = 0.f;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int xx = min(max(ix - 1 + b, 0), G0 - 1);
      rowacc += wx[b] * pos_src[size_t(1 + yy * G0 + xx) * D + d];
    }
    acc += wy[a] * rowacc;
  }
  out[idx] = acc;
}

// ---------------------------------------------------------------------------------------
// im2col for the 8x8/stride-8 patch-embed conv (reference vision_transformer.py:153,157):
//   A[b*P + i*gw + j][c*64 + ky*8 + kx] = frame[b][c][i*8+ky][j*8+kx],   P = gh*gw, frames [B, 3, 8*gh, 8*gw]
// written as the bf16x3 operand [hi | lo] (2 x 192 columns, see split_weight_kernel): the rounding of
// the pixels / conv weights to plain bf16 is the largest single contribution to the final log-prob error.
// One thread moves two image rows of one patch (2 x 32 B in, 2 x 32 B out).
// ---------------------------------------------------------------------------------------
constexpr int IM2COL_K = 192;
constexpr int IM2COL_K3 = 3 * IM2COL_K;   // reduction length of the patch-embed GEMM
constexpr int IM2COL_KA = 2 * IM2COL_K;   // stored columns of its A operand [hi | lo]

__device__ __forceinline__ void split_pack8(const float4& a0, const float4& a1, uint4& hi, uint4& lo) {
  hi.x = pack_bf16x2(a0.x, a0.y); hi.y = pack_bf16x2(a0.z, a0.w);
  hi.z = pack_bf16x2(a1.x, a1.y); hi.w = pack_bf16x2(a1.z, a1.w);
  lo.x = pack_bf16x2(a0.x - __uint_as_float(hi.x << 16), a0.y - __uint_as_float(hi.x & 0xffff0000u));
  lo.y = pack_bf16x2(a0.z - __uint_as_float(hi.y << 16), a0.w - __uint_as_float(hi.y & 0xffff0000u));
  lo.z = pack_bf16x2(a1.x - __uint_as_float(hi.z << 16), a1.y - __uint_as_float(hi.z & 0xffff0000u));
  lo.w = pack_bf16x2(a1.z - __uint_as_float(hi.w << 16), a1.w - __uint_as_float(hi.w & 0xffff0000u));
}

__global__ void im2col_patch8_kernel(const float* __restrict__ frames, __nv_bfloat16* __restrict__ A, int B,
                                     int gh, int gw) {
  const int H = gh * 8, W = gw * 8;
  const size_t total = size_t(B) * 3 * gh * 4 * gw;  // (b, c, i, kyp, j)
  size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int j = int(idx % gw); idx /= gw;
  const int kyp = int(idx % 4); idx /= 4;
  const int i = int(idx % gh); idx /= gh;
  const int c = int(idx % 3);
  const int b = int(idx / 3);
  const float* src = frames + ((size_t(b) * 3 + c) * H + (i * 8 + kyp * 2)) * W + j * 8;
  const float4 a0 = __ldg(reinterpret_cast<const float4*>(src));
  const float4 a1 = __ldg(reinterpret_cast<const float4*>(src + 4));
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(src + W));
  const float4 b1 = __ldg(reinterpret_cast<const float4*>(src + W + 4));
  uint4 h0, l0, h1, l1;
  split_pack8(a0, a1, h0, l0);
  split_pack8(b0, b1, h1, l1);
  __nv_bfloat16* dst = A + (size_t(b) * gh * gw + size_t(i) * gw + j) * IM2COL_KA + c * 64 + kyp * 16;
  *reinterpret_cast<uint4*>(dst) = h0;
  *reinterpret_cast<uint4*>(dst + 8) = h1;
  *reinterpret_cast<uint4*>(dst + IM2COL_K) = l0;
  *reinterpret_cast<uint4*>(dst + IM2COL_K + 8) = l1;
}

// ---------------------------------------------------------------------------------------
// Preprocessing of DINOSeg.predict fused into the im2col (reference pl_torch_modules.py:33-41, :291):
//   uint8 HWC RGB frame [Hs, Ws, 3] -> albumentations Resize(H, W) = cv2.resize(INTER_LINEAR) ->
//   Normalize: (pix - mean*255) * (1 / (std*255)) in fp32 -> CHW -> 8x8 patches (bf16x3 operand as above).
// The resize reproduces OpenCV's 8-bit bilinear path in integer arithmetic: source coordinate
// (d + 0.5) * src/dst - 0.5, taps clamped at the borders, 11-bit fixed-point weights
// (INTER_RESIZE_COEF_BITS), horizontal pass in int32, vertical pass
// ((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2, i.e. the uint8 image cv2 would hand to
// Normalize.  Each axis has its own scale src/dst; same-size frames (Hs = H, Ws = W) pass through exactly.
// H = 8*gh, W = 8*gw.  One thread = 8 output pixels of one row.
// ---------------------------------------------------------------------------------------
struct PreprocParams {
  int src_h, src_w;
  float mean255[3];     // float32(mean) * 255
  float denom[3];       // 1 / (float32(std) * 255)
};

// cv::resize INTER_LINEAR coefficients for destination index d: f = (d + 0.5) * scale - 0.5 (in fp32), s = floor(f),
// weights saturate_cast<short>(w * 2048) (round half to even).  Horizontally OpenCV zeroes the fraction at the
// borders, vertically it only clamps the two rows.
__device__ __forceinline__ void cv_linear_coef(int d, double scale, int src_size, bool horizontal, int& s0, int& s1,
                                               int& a0, int& a1) {
  float f = float((double(d) + 0.5) * scale - 0.5);
  int sx = int(floorf(f));
  f -= float(sx);
  if (horizontal) {
    if (sx < 0) { f = 0.f; sx = 0; }
    if (sx >= src_size - 1) { f = 0.f; sx = src_size - 1; }
  }
  s0 = min(max(sx, 0), src_size - 1);
  s1 = min(max(sx + 1, 0), src_size - 1);
  a0 = __float2int_rn((1.f - f) * 2048.f);
  a1 = __float2int_rn(f * 2048.f);
}

__global__ void im2col_u8_kernel(const uint8_t* __restrict__ frames /*[B, H, W, 3]*/, __nv_bfloat16* __restrict__ A,
                                 int B, int gh, int gw, PreprocParams pp) {
  const int H = gh * 8, W = gw * 8;
  const size_t total = size_t(B) * 3 * H * gw;     // (b, c, y, j): 8 pixels each
  size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int j = int(idx % gw); idx /= gw;
  const int y = int(idx % H); idx /= H;
  const int c = int(idx % 3);
  const int b = int(idx / 3);
  const uint8_t* src = frames + size_t(b) * pp.src_h * pp.src_w * 3;
  const bool same = pp.src_h == H && pp.src_w == W;
  const double sy = double(pp.src_h) / double(H), sx = double(pp.src_w) / double(W);
  int y0, y1, b0, b1;
  cv_linear_coef(y, sy, pp.src_h, false, y0, y1, b0, b1);
  float v[8];
#pragma unroll
  for (int kx = 0; kx < 8; ++kx) {
    const int x = j * 8 + kx;
    int pix;
    if (same) {
      pix = src[(size_t(y) * pp.src_w + x) * 3 + c];
    } else {
      int x0, x1, a0, a1;
      cv_linear_coef(x, sx, pp.src_w, true, x0, x1, a0, a1);
      const int r0 = int(src[(size_t(y0) * pp.src_w + x0) * 3 + c]) * a0 + int(src[(size_t(y0) * pp.src_w + x1) * 3 + c]) * a1;
      const int r1 = int(src[(size_t(y1) * pp.src_w + x0) * 3 + c]) * a0 + int(src[(size_t(y1) * pp.src_w + x1) * 3 + c]) * a1;
      pix = (((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2;
      pix = pix < 0 ? 0 : (pix > 255 ? 255 : pix);
    }
    v[kx] = (float(pix) - pp.mean255[c]) * pp.denom[c];
  }
  uint4 hi, lo;
  split_pack8(make_float4(v[0], v[1], v[2], v[3]), make_float4(v[4], v[5], v[6], v[7]), hi, lo);
  const int i = y >> 3, ky = y & 7;
  __nv_bfloat16* dst = A + (size_t(b) * gh * gw + size_t(i) * gw + j) * IM2COL_KA + c * 64 + ky * 8;
  *reinterpret_cast<uint4*>(dst) = hi;
  *reinterpret_cast<uint4*>(dst + IM2COL_K) = lo;
}

// x[b*Ntok + 0, :] = cls + pos[0]      (reference vision_transformer.py:229-233)
__global__ void cls_row_kernel(const float* __restrict__ cls, const float* __restrict__ pos, float* __restrict__ x,
                               int B, int Ntok, int D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * D) return;
  const int b = i / D, d = i - b * D;
  x[size_t(b) * Ntok * D + d] = cls[d] + pos[d];
}

// ---------------------------------------------------------------------------------------
// LayerNorm (eps inside the sqrt, biased variance; reference :114,:118,:183 with eps=1e-6 :303)
// fp32 in -> bf16 out (the bf16 copy is the A operand of the following GEMM).  One warp per row.
// ---------------------------------------------------------------------------------------
// Row statistics for D = 384 with EIGHT LANES PER ROW (a warp works on four rows at once): lane `sub` of a row's group
// holds the row's float4 number i*8 + sub, i = 0..11.  Two-pass statistics in registers, sums over the group with three
// xor-shuffles - one shuffle instruction serves four rows, so the dependent shuffle chain per row is 6 long instead of
// the 10 of a warp-per-row reduction (what bounds a single warp that has to normalise many rows in a row: the fused
// LayerNorm fill of mlp.cuh, which shares this function with the LayerNorm kernel so that both produce the same bits).
constexpr int LN384_V = 12;
__device__ __forceinline__ void ln384_stats(const float4 (&v)[LN384_V], float eps, float& mean, float& rstd) {
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < LN384_V; ++i) sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  sum += __shfl_xor_sync(0xffffffffu, sum, 1);
  sum += __shfl_xor_sync(0xffffffffu, sum, 2);
  sum += __shfl_xor_sync(0xffffffffu, sum, 4);
  mean = sum * (1.0f / 384.0f);
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < LN384_V; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    sq += (a * a + b * b) + (c * c + d * d);
  }
  sq += __shfl_xor_sync(0xffffffffu, sq, 1);
  sq += __shfl_xor_sync(0xffffffffu, sq, 2);
  sq += __shfl_xor_sync(0xffffffffu, sq, 4);
  rstd = rsqrtf(sq * (1.0f / 384.0f) + eps);
}
// normalised, affine-transformed float4 number i of the row -> four outputs at float4 position i of the output row:
// bf16 (two packed words, one 8-byte store) or fp32 (one 16-byte store)
__device__ __forceinline__ void ln_out4(__nv_bfloat16* yr, int i, const float4& v, float mean, float rstd,
                                        const float4& gm, const float4& bt) {
  const float a = (v.x - mean) * rstd * gm.x + bt.x, b = (v.y - mean) * rstd * gm.y + bt.y;
  const float c = (v.z - mean) * rstd * gm.z + bt.z, d = (v.w - mean) * rstd * gm.w + bt.w;
  uint2 o;
  o.x = pack_bf16x2(a, b);
  o.y = pack_bf16x2(c, d);
  reinterpret_cast<uint2*>(yr)[i] = o;
}
__device__ __forceinline__ void ln_out4(float* yr, int i, const float4& v, float mean, float rstd, const float4& gm,
                                        const float4& bt) {
  reinterpret_cast<float4*>(yr)[i] = make_float4((v.x - mean) * rstd * gm.x + bt.x, (v.y - mean) * rstd * gm.y + bt.y,
                                                 (v.z - mean) * rstd * gm.z + bt.z, (v.w - mean) * rstd * gm.w + bt.w);
}

// normalised float4 WITHOUT the affine transform (the consumer's weights carry gamma and beta: fold_ln_weight_kernel)
__device__ __forceinline__ uint2 ln384_out_plain(const float4& v, float mean, float rstd) {
  uint2 o;
  o.x = pack_bf16x2((v.x - mean) * rstd, (v.y - mean) * rstd);
  o.y = pack_bf16x2((v.z - mean) * rstd, (v.w - mean) * rstd);
  return o;
}

// LayerNorm folded into the Linear layer that consumes it (weight-load time):
//   Linear(LN(x)) = W (xhat * gamma + beta) + b = (W diag(gamma)) xhat + (b + W beta),   xhat = (x - mean) * rstd
// W [N, K] fp32 -> Wf [N, K] bf16 = W * gamma (per input column), bf [N] fp32 = b + W . beta (fp32 dot).  One warp per
// output row.  The kernel that consumes Wf then only has to produce xhat (mlp.cuh: fused LayerNorm2 -> fc1).
__global__ void __launch_bounds__(256)
fold_ln_weight_kernel(const float* __restrict__ W, const float* __restrict__ b, const float* __restrict__ gamma,
                      const float* __restrict__ beta, __nv_bfloat16* __restrict__ Wf, float* __restrict__ bf, int N, int K) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  const float* w = W + size_t(warp) * K;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float v = w[k];
    Wf[size_t(warp) * K + k] = __float2bfloat16_rn(v * gamma[k]);
    acc = fmaf(v, beta[k], acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) bf[warp] = b[warp] + acc;
}

// The same for a bf16x3 consumer: Wf = W * gamma split into hi + lo, stored as [N, 2K] = [hi | lo] (head.cuh).
__global__ void __launch_bounds__(256)
fold_split_ln_weight_kernel(const float* __restrict__ W, const float* __restrict__ b, const float* __restrict__ gamma,
                            const float* __restrict__ beta, __nv_bfloat16* __restrict__ Wf, float* __restrict__ bf, int N, int K) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  const float* w = W + size_t(warp) * K;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float v = w[k];
    const float f = v * gamma[k];
    const __nv_bfloat16 hi = __float2bfloat16_rn(f);
    Wf[size_t(warp) * 2 * K + k] = hi;
    Wf[size_t(warp) * 2 * K + K + k] = __float2bfloat16_rn(f - __bfloat162float(hi));
    acc = fmaf(v, beta[k], acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) bf[warp] = b[warp] + acc;
}

// D = 384, plain output (OutT = bf16: GEMM operand; fp32: backbone features): four rows per warp (eight lanes per row),
// 32 rows per 256-thread block
template <typename OutT>
__global__ void __launch_bounds__(256)
layernorm384_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                    OutT* __restrict__ y, int M, float eps) {
  const int sub = threadIdx.x & 7;
  const int row = blockIdx.x * 32 + (threadIdx.x >> 3);
  const bool live = row < M;
  const float4* xr = reinterpret_cast<const float4*>(x + size_t(live ? row : M - 1) * 384);
  float4 v[LN384_V];
#pragma unroll
  for (int i = 0; i < LN384_V; ++i) v[i] = xr[i * 8 + sub];
  float mean, rstd;
  ln384_stats(v, eps, mean, rstd);
  if (!live) return;
  OutT* yr = y + size_t(row) * 384;
#pragma unroll
  for (int i = 0; i < LN384_V; ++i)
    ln_out4(yr, i * 8 + sub, v[i], mean, rstd, __ldg(reinterpret_cast<const float4*>(gamma) + i * 8 + sub),
            __ldg(reinterpret_cast<const float4*>(beta) + i * 8 + sub));
}

// One warp per row.  SPLIT (bf16 only): y is [M, 2*D] = [hi | lo] (bf16x3 operand of the head GEMM, see
// split_weight_kernel).
template <int D, bool SPLIT, typename OutT>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                 OutT* __restrict__ y, int M, float eps) {
  static_assert(D % 128 == 0, "D must be a multiple of 128");
  static_assert(!SPLIT || std::is_same<OutT, __nv_bfloat16>::value, "the split output is bf16");
  constexpr int V = D / 128;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  if (row >= M) return;
  const float4* xr = reinterpret_cast<const float4*>(x + size_t(row) * D);
  float4 v[V];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    v[i] = xr[i * 32 + lane];
    sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum * (1.0f / D);
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    sq += (a * a + b * b) + (c * c + d * d);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq * (1.0f / D) + eps);
  OutT* yr = y + size_t(row) * (SPLIT ? 2 * D : D);
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + i * 32 + lane);
    const float4 bt = __ldg(reinterpret_cast<const float4*>(beta) + i * 32 + lane);
    if constexpr (SPLIT) {
      const float a = (v[i].x - mean) * rstd * gm.x + bt.x, b = (v[i].y - mean) * rstd * gm.y + bt.y;
      const float c = (v[i].z - mean) * rstd * gm.z + bt.z, d = (v[i].w - mean) * rstd * gm.w + bt.w;
      uint2 o;
      o.x = pack_bf16x2(a, b);
      o.y = pack_bf16x2(c, d);
      uint2* yw = reinterpret_cast<uint2*>(yr);
      yw[i * 32 + lane] = o;
      uint2 l;
      l.x = pack_bf16x2(a - __uint_as_float(o.x << 16), b - __uint_as_float(o.x & 0xffff0000u));
      l.y = pack_bf16x2(c - __uint_as_float(o.y << 16), d - __uint_as_float(o.y & 0xffff0000u));
      yw[D / 4 + i * 32 + lane] = l;
    } else {
      ln_out4(yr, i * 32 + lane, v[i], mean, rstd, gm, bt);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Controller-side reduction on the label map (SURVEY.md section 8(f)-4; reference docs/index.html "Controller": the
// potential-field controller steers away from the image half with the most obstacle patches).  Per frame, the number
// of OUTPUT-MAP pixels of every class left (x < W/2) and right (x >= W/2) of the centre line, W = g*p, computed from
// the low-res map (patch (i, j) covers p rows and the columns [j*p, (j+1)*p)): counts[b][side][c], int32.
// One CTA per frame; integer work, exact.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
half_counts_kernel(const uint8_t* __restrict__ lowres, int32_t* __restrict__ counts, int g, int p, int C) {
  __shared__ int hist[2 * 256];
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  const int b = blockIdx.x;
  const int half = (g * p) / 2;
  const uint8_t* low = lowres + size_t(b) * g * g;
  for (int idx = threadIdx.x; idx < g * g; idx += blockDim.x) {
    const int j = idx % g;
    const int c = low[idx];
    if (c >= C) continue;
    int left = half - j * p;
    left = left < 0 ? 0 : (left > p ? p : left);
    if (left) atomicAdd(&hist[c], left * p);
    if (p - left) atomicAdd(&hist[C + c], (p - left) * p);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) counts[size_t(b) * 2 * C + i] = hist[i];
}

// ---------------------------------------------------------------------------------------
// argmax with torch semantics: first maximum wins, NaN counts as the maximum
// (reference pl_torch_modules.py:295 torch.argmax)
// ---------------------------------------------------------------------------------------
constexpr int HEAD_MAX_C = 16;

// v has HEAD_MAX_C entries (C <= MAXC valid); fully unrolled so that v stays in registers
template <int MAXC = HEAD_MAX_C>
__device__ __forceinline__ int argmax_first(const float (&v)[HEAD_MAX_C], int C) {
  float best = v[0];
  int idx = 0;
#pragma unroll
  for (int c = 1; c < MAXC; ++c) {
    const float x = v[c];
    if (c < C && ((x > best) || (x != x && best == best))) { best = x; idx = c; }
  }
  return idx;
}


// ---------------------------------------------------------------------------------------
// Head tail: layer_3 -> log_softmax -> argmax -> p x p replication   (reference pl_torch_modules.py:121-123 / :135-138,
// :295, :297-298 np.kron), fp32 CUDA cores, HBM-bound (reads 400 B per patch, writes 8*p*p B per patch).
//   LINEAR = false: in = h2 = relu(layer_2(relu(layer_1))) [B*Ntok, ld] fp32 (produced by the two tensor-core GEMMs),
//                   z = in . W3^T + b3;   LINEAR = true: in = the 'linear' head's logits [B*Ntok, ld], z = in[:C].
// Input rows are tokens INCLUDING the cls row of every frame; output rows drop it (reference :243).  The patch grid is
// gh x gw (P = gh*gw patches per frame, row-major); the label map exists for square grids only (labels == nullptr
// otherwise).
// Eight lanes per patch row (four rows per warp per step): the lanes read the row as consecutive float4 (coalesced),
// keep partial dot products for all classes, all-reduce them with three xor-shuffles, and then every lane holds the
// row's logits.  The label is written to the low-res map and - fused, labels != nullptr - replicated into its p x p
// block of the int64 map: the eight lanes take the block's rows, 16-byte stores when p is even (the four patches of
// a warp are neighbours, so every output row receives 4*p*8 contiguous bytes per step).
// ---------------------------------------------------------------------------------------
constexpr int HT_MAX_H2 = 104;

// MAXC: compile-time bound of the class loops (8 or 16): every class slot costs instructions whether it is used or not
// (with MAXC = 16 and the reference's 7 classes the kernel was bound by instruction issue, not by HBM).
template <bool LINEAR, int MAXC>
__global__ void __launch_bounds__(256)
head_tail_kernel(const float* __restrict__ in /*[B*Ntok, ld]*/, int ld, const float* __restrict__ w3 /*[C, H2]*/,
                 const float* __restrict__ b3 /*[C]*/, float* __restrict__ logprobs /*[B*P, C] or null*/,
                 uint8_t* __restrict__ lowres /*[B*P] or null*/, long long* __restrict__ labels /*[B, g*p, g*p] or null*/,
                 int B, int gh, int gw, int p, int Ntok, int H2, int C) {
  __shared__ float sW3[LINEAR ? 1 : MAXC * HT_MAX_H2];
  __shared__ float sB3[HEAD_MAX_C];
  if constexpr (!LINEAR) {
    for (int i = threadIdx.x; i < MAXC * HT_MAX_H2; i += blockDim.x) {
      const int c = i / HT_MAX_H2, k = i - c * HT_MAX_H2;
      sW3[i] = (c < C && k < H2) ? w3[c * H2 + k] : 0.f;
    }
    if (threadIdx.x < HEAD_MAX_C) sB3[threadIdx.x] = threadIdx.x < C ? b3[threadIdx.x] : 0.f;
    __syncthreads();
  }
  const int P = gh * gw;
  const int total_rows = B * P;
  const int sub = threadIdx.x & 7;                           // lane within the row's group of eight
  const int grp = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int ngrp = (gridDim.x * blockDim.x) >> 3;
  const int W = gw * p;
  for (int r0 = 0; r0 < total_rows; r0 += ngrp) {            // uniform trip count: the shuffles below need full warps
    const int r = r0 + grp;
    const bool live = r < total_rows;
    const int rr = live ? r : total_rows - 1;
    const int b = rr / P, t = rr - b * P;
    const float* src = in + (size_t(b) * Ntok + 1 + t) * ld;
    float z[HEAD_MAX_C];
#pragma unroll
    for (int c = 0; c < HEAD_MAX_C; ++c) z[c] = 0.f;
    if constexpr (LINEAR) {
#pragma unroll
      for (int c = 0; c < MAXC; ++c)
        if (c < C) z[c] = __ldg(src + c);
    } else {
      for (int k4 = sub; k4 < H2 / 4; k4 += 8) {
        const float4 hv = __ldg(reinterpret_cast<const float4*>(src) + k4);
#pragma unroll
        for (int c = 0; c < MAXC; ++c) {
          if (c < C) {
            const float* wr = sW3 + c * HT_MAX_H2 + 4 * k4;
            z[c] = fmaf(hv.x, wr[0], z[c]); z[c] = fmaf(hv.y, wr[1], z[c]);
            z[c] = fmaf(hv.z, wr[2], z[c]); z[c] = fmaf(hv.w, wr[3], z[c]);
          }
        }
      }
#pragma unroll
      for (int c = 0; c < MAXC; ++c) {
        if (c < C) {
          z[c] += __shfl_xor_sync(0xffffffffu, z[c], 1);
          z[c] += __shfl_xor_sync(0xffffffffu, z[c], 2);
          z[c] += __shfl_xor_sync(0xffffffffu, z[c], 4);
          z[c] += sB3[c];
        }
      }
    }
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < MAXC; ++c)
      if (c < C) mx = fmaxf(mx, z[c]);
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c)
      if (c < C) se += expf(z[c] - mx);
    const float lse = logf(se);
#pragma unroll
    for (int c = 0; c < MAXC; ++c)
      if (c < C) z[c] = (z[c] - mx) - lse;
    if (!live) continue;
    if (logprobs != nullptr) {
#pragma unroll
      for (int c = 0; c < MAXC; ++c)
        if (c < C && (c & 7) == sub) logprobs[size_t(r) * C + c] = z[c];
    }
    const int label = argmax_first<MAXC>(z, C);
    if (lowres != nullptr && sub == 0) lowres[r] = uint8_t(label);
    if (labels != nullptr) {
      const int i = t / gw, j = t - i * gw;
      long long* blk = labels + (size_t(b) * W + size_t(i) * p) * W + size_t(j) * p;
      if ((p & 1) == 0) {
        const longlong2 v = make_longlong2(label, label);
        for (int yy = sub; yy < p; yy += 8) {
          longlong2* row = reinterpret_cast<longlong2*>(blk + size_t(yy) * W);
          for (int x2 = 0; x2 < (p >> 1); ++x2) row[x2] = v;
        }
      } else {
        for (int yy = sub; yy < p; yy += 8) {
          long long* row = blk + size_t(yy) * W;
          for (int x = 0; x < p; ++x) row[x] = label;
        }
      }
    }
  }
}

// log-probs [rows, C] -> label per row (torch.argmax semantics)
__global__ void argmax_rows_kernel(const float* __restrict__ logprobs, uint8_t* __restrict__ lowres, int rows,
                                   int C) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float z[HEAD_MAX_C];
#pragma unroll
  for (int c = 0; c < HEAD_MAX_C; ++c) z[c] = c < C ? logprobs[size_t(r) * C + c] : 0.f;
  lowres[r] = uint8_t(argmax_first(z, C));
}

// ---------------------------------------------------------------------------------------
// CLS-query attention of one block: out[b, h, j] = softmax_j( q_cls(b,h) . k_j(b,h) )
// (q as the qkv GEMM wrote it, pre-scaled by dh^-0.5 * log2(e): the scores are in log2 units, attention.cuh)
// = row 0 of the attention matrix VisionTransformer.get_last_selfattention returns (reference
// vision_transformer.py:273-280, :85-101), the only row its caller uses (visualize_attention.py:46-54).
// qkv: [B, N, 3D] bf16 as written by the qkv GEMM.  One CTA per (b, h); N x 64 dot products are nothing next to
// the hot path, so this is a plain block-reduction kernel.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
cls_attention_kernel(const __nv_bfloat16* __restrict__ qkv, float* __restrict__ out, int N, int D, int H) {
  const int h = blockIdx.x, b = blockIdx.y;
  const __nv_bfloat16* base = qkv + size_t(b) * N * 3 * D;
  __shared__ float sq[64];
  __shared__ float red[8];
  __shared__ float bcast;
  if (threadIdx.x < 64) sq[threadIdx.x] = __bfloat162float(base[h * 64 + threadIdx.x]);   // token 0 = cls, q part
  __syncthreads();
  float* o = out + (size_t(b) * H + h) * N;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const uint4* kp = reinterpret_cast<const uint4*>(base + size_t(j) * 3 * D + D + h * 64);
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint4 v = __ldg(kp + c);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        acc = fmaf(sq[c * 8 + 2 * e], __uint_as_float(w[e] << 16), acc);
        acc = fmaf(sq[c * 8 + 2 * e + 1], __uint_as_float(w[e] & 0xffff0000u), acc);
      }
    }
    o[j] = acc;
    mx = fmaxf(mx, acc);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
    bcast = m;
  }
  __syncthreads();
  mx = bcast;
  float sum = 0.f;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const float e = exp2f(o[j] - mx);
    o[j] = e;
    sum += e;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s);
  __syncthreads();
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    bcast = 1.0f / t;
  }
  __syncthreads();
  const float inv = bcast;
  for (int j = threadIdx.x; j < N; j += blockDim.x) o[j] *= inv;
}

// ---------------------------------------------------------------------------------------
// Image embeddings (DINOSeg.embeddings).  Both kernels split the tokens of a frame over a cluster of EMB_SPLIT CTAs
// and merge the per-CTA partials in rank order through distributed shared memory: one launch, no scratch buffer, no
// atomics.  The split does not depend on the batch size, so a frame's result is the same bits in any batch.
// ---------------------------------------------------------------------------------------
constexpr int EMB_SPLIT = 8;
constexpr int EMB_THREADS = 256;

__device__ __forceinline__ float ld_shared_cluster_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}

// online-softmax state (running maximum m in log2 units, sum l, unnormalised output o) of one CLS-query head
struct ClsSoftmax {
  float m, l, o[64];
};
// weight of a partial with maximum pm in a merge with maximum m; a partial that has seen no key (pm = -inf) has none
__device__ __forceinline__ float cls_softmax_scale(float pm, float m) { return pm == -INFINITY ? 0.f : exp2f(pm - m); }

// Attention output of the CLS query of the last block (what the CLS row of the proj GEMM's input is):
//   o[b, h*64 + c] = sum_j softmax_j(q_cls . k_j) v_j[c]   -> bf16 [B, D], the A operand of the proj GEMM at M = B,
// and xc[b] = x[b*Ntok] (the CLS rows of the residual stream, fp32 [B, D]), which that GEMM adds to.
// qkv: [B, N, 3D] bf16 as the qkv GEMM wrote it (q pre-scaled by dh^-0.5 * log2(e): scores in log2 units, as in
// cls_attention_kernel).  Grid (EMB_SPLIT, H, B), clusters of EMB_SPLIT along x: CTA s takes the s-th contiguous chunk
// of the keys.  Every thread keeps an online softmax over its keys: each exponent is taken against a running maximum
// that is >= the score, so scores of any range stay finite and the result is softmax with the exact row maximum.
// V is read as bf16 and accumulated in fp32.  Partials merge in a fixed tree: xor-butterfly in the warp, the warps in
// order, then the CTAs in rank order.
__global__ void __launch_bounds__(EMB_THREADS)
cls_attn_out_kernel(const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ x, __nv_bfloat16* __restrict__ o,
                    float* __restrict__ xc, int N, int D) {
  const int s = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const __nv_bfloat16* base = qkv + size_t(b) * N * 3 * D;
  __shared__ float sq[64];
  __shared__ float wm[EMB_THREADS / 32], wl[EMB_THREADS / 32], wo[EMB_THREADS / 32][64];
  __shared__ float res[66];                                   // this CTA's (m, l, o[64])
  if (threadIdx.x < 64) sq[threadIdx.x] = __bfloat162float(base[h * 64 + threadIdx.x]);   // token 0 = cls, q part
  if (s == 0 && h == 0)
    for (int d = threadIdx.x; d < D; d += EMB_THREADS) xc[size_t(b) * D + d] = x[size_t(b) * N * D + d];
  __syncthreads();

  const int chunk = (N + EMB_SPLIT - 1) / EMB_SPLIT;
  const int j0 = s * chunk, j1 = min(N, j0 + chunk);
  ClsSoftmax st;
  st.m = -INFINITY; st.l = 0.f;
#pragma unroll
  for (int c = 0; c < 64; ++c) st.o[c] = 0.f;
  for (int j = j0 + int(threadIdx.x); j < j1; j += EMB_THREADS) {
    const uint4* kp = reinterpret_cast<const uint4*>(base + size_t(j) * 3 * D + D + h * 64);
    const uint4* vp = reinterpret_cast<const uint4*>(base + size_t(j) * 3 * D + 2 * D + h * 64);
    float sc = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint4 v = __ldg(kp + c);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        sc = fmaf(sq[c * 8 + 2 * e], __uint_as_float(w[e] << 16), sc);
        sc = fmaf(sq[c * 8 + 2 * e + 1], __uint_as_float(w[e] & 0xffff0000u), sc);
      }
    }
    if (sc > st.m) {
      const float a = cls_softmax_scale(st.m, sc);
      st.l *= a;
#pragma unroll
      for (int c = 0; c < 64; ++c) st.o[c] *= a;
      st.m = sc;
    }
    const float p = exp2f(sc - st.m);
    st.l += p;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint4 v = __ldg(vp + c);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        st.o[c * 8 + 2 * e] = fmaf(p, __uint_as_float(w[e] << 16), st.o[c * 8 + 2 * e]);
        st.o[c * 8 + 2 * e + 1] = fmaf(p, __uint_as_float(w[e] & 0xffff0000u), st.o[c * 8 + 2 * e + 1]);
      }
    }
  }
  // warp: xor-butterfly (every lane ends with a deterministic function of the warp's 32 states; lane 0's is kept)
#pragma unroll
  for (int sh = 16; sh > 0; sh >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, st.m, sh), l2 = __shfl_xor_sync(0xffffffffu, st.l, sh);
    const float m = fmaxf(st.m, m2);
    const float sa = cls_softmax_scale(st.m, m), sb = cls_softmax_scale(m2, m);
    st.m = m;
    st.l = st.l * sa + l2 * sb;
#pragma unroll
    for (int c = 0; c < 64; ++c) st.o[c] = st.o[c] * sa + __shfl_xor_sync(0xffffffffu, st.o[c], sh) * sb;
  }
  if (lane == 0) {
    wm[warp] = st.m; wl[warp] = st.l;
#pragma unroll
    for (int c = 0; c < 64; ++c) wo[warp][c] = st.o[c];
  }
  __syncthreads();
  // CTA: the warps in order; thread c < 64 owns output column c
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    float m = -INFINITY;
    for (int w = 0; w < EMB_THREADS / 32; ++w) m = fmaxf(m, wm[w]);
    float l = 0.f, acc = 0.f;
    for (int w = 0; w < EMB_THREADS / 32; ++w) {
      const float a = cls_softmax_scale(wm[w], m);
      l = l + wl[w] * a;
      acc = acc + wo[w][c] * a;
    }
    res[2 + c] = acc;
    if (c == 0) { res[0] = m; res[1] = l; }
  }
  // cluster: rank 0 merges the CTAs in rank order
  cluster_sync_all();
  if (s == 0 && threadIdx.x < 64) {
    const int c = threadIdx.x;
    float m = -INFINITY;
    for (int r = 0; r < EMB_SPLIT; ++r) m = fmaxf(m, ld_shared_cluster_f32(mapa_rank(&res[0], r)));
    float l = 0.f, acc = 0.f;
    for (int r = 0; r < EMB_SPLIT; ++r) {
      const float mr = ld_shared_cluster_f32(mapa_rank(&res[0], r));
      const float a = cls_softmax_scale(mr, m);
      l = l + ld_shared_cluster_f32(mapa_rank(&res[1], r)) * a;
      acc = acc + ld_shared_cluster_f32(mapa_rank(&res[2 + c], r)) * a;
    }
    o[size_t(b) * D + h * 64 + c] = __float2bfloat16_rn(acc / l);
  }
  cluster_sync_all();                                         // the peers' shared memory stays until rank 0 has read it
}

// After the full last block: per frame, the final norm of the CLS row (cls_out [B, D], or null) and the mean of the
// final norm over the patch tokens, patch_mean[b] = gamma * mean_t(xhat_t) + beta (xhat = (x - mean) * rstd).  The row
// statistics and the CLS row's output use the LayerNorm kernels' arithmetic (ln384_stats / ln_out4 for D = 384, the
// warp-per-row sums of layernorm_kernel for D = 768), so cls_out equals dino.norm's CLS row bit for bit.  x is read
// once.  Grid (EMB_SPLIT, B), clusters of EMB_SPLIT: CTA s sums the s-th chunk of the patch tokens; per-lane sums, the
// row groups of a warp by xor-shuffles, the warps in order, the CTAs in rank order.
template <int D>
__global__ void __launch_bounds__(EMB_THREADS)
embed_pool_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                  float* __restrict__ cls_out, float* __restrict__ patch_mean, int Ntok, float eps) {
  static_assert(D == 384 || D == 768, "embed_pool_kernel: D = 384 or 768");
  constexpr int NW = EMB_THREADS / 32;
  // D = 384: eight lanes per row (four rows per warp), 12 float4 per lane; D = 768: one warp per row, 6 float4 per lane
  constexpr int V = D == 384 ? LN384_V : D / 128;
  constexpr int ROWS_PER_WARP = D == 384 ? 4 : 1;
  const int s = blockIdx.x, b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = D == 384 ? lane >> 3 : 0, sub = D == 384 ? (lane & 7) : lane;
  constexpr int STEP = D == 384 ? 8 : 32;                     // float4 stride of a lane inside its row
  __shared__ __align__(16) float red[NW][D];
  __shared__ float part[D];
  const float* xf = x + size_t(b) * Ntok * D;

  auto stats = [&](const float4 (&v)[V], float& mean, float& rstd) {
    if constexpr (D == 384) {
      ln384_stats(v, eps, mean, rstd);
    } else {
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < V; ++i) sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      mean = sum * (1.0f / D);
      float sq = 0.f;
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const float a = v[i].x - mean, bb = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
        sq += (a * a + bb * bb) + (c * c + d * d);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
      rstd = rsqrtf(sq * (1.0f / D) + eps);
    }
  };

  if (s == 0 && warp == 0 && cls_out != nullptr) {
    const float4* xr = reinterpret_cast<const float4*>(xf);
    float4 v[V];
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = xr[i * STEP + sub];
    float mean, rstd;
    stats(v, mean, rstd);
    if (grp == 0) {
      float* yr = cls_out + size_t(b) * D;
#pragma unroll
      for (int i = 0; i < V; ++i)
        ln_out4(yr, i * STEP + sub, v[i], mean, rstd, __ldg(reinterpret_cast<const float4*>(gamma) + i * STEP + sub),
                __ldg(reinterpret_cast<const float4*>(beta) + i * STEP + sub));
    }
  }

  const int P = Ntok - 1;
  const int chunk = (P + EMB_SPLIT - 1) / EMB_SPLIT;
  const int t0 = 1 + s * chunk, t1 = 1 + min(P, s * chunk + chunk);
  float4 acc[V];
#pragma unroll
  for (int i = 0; i < V; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int r0 = t0; r0 < t1; r0 += NW * ROWS_PER_WARP) {      // uniform trip count: the shuffles need full warps
    const int r = r0 + warp * ROWS_PER_WARP + grp;
    const bool live = r < t1;
    const float4* xr = reinterpret_cast<const float4*>(xf + size_t(live ? r : t0) * D);
    float4 v[V];
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = xr[i * STEP + sub];
    float mean, rstd;
    stats(v, mean, rstd);
    if (live) {
#pragma unroll
      for (int i = 0; i < V; ++i) {
        acc[i].x += (v[i].x - mean) * rstd; acc[i].y += (v[i].y - mean) * rstd;
        acc[i].z += (v[i].z - mean) * rstd; acc[i].w += (v[i].w - mean) * rstd;
      }
    }
  }
  if constexpr (D == 384) {
#pragma unroll
    for (int sh = 8; sh <= 16; sh <<= 1) {
#pragma unroll
      for (int i = 0; i < V; ++i) {
        acc[i].x += __shfl_xor_sync(0xffffffffu, acc[i].x, sh); acc[i].y += __shfl_xor_sync(0xffffffffu, acc[i].y, sh);
        acc[i].z += __shfl_xor_sync(0xffffffffu, acc[i].z, sh); acc[i].w += __shfl_xor_sync(0xffffffffu, acc[i].w, sh);
      }
    }
  }
  if (grp == 0) {
#pragma unroll
    for (int i = 0; i < V; ++i) reinterpret_cast<float4*>(red[warp])[i * STEP + sub] = acc[i];
  }
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += EMB_THREADS) {
    float t = 0.f;
    for (int w = 0; w < NW; ++w) t += red[w][d];
    part[d] = t;
  }
  cluster_sync_all();
  if (s == 0) {
    for (int d = threadIdx.x; d < D; d += EMB_THREADS) {
      float t = 0.f;
      for (int r = 0; r < EMB_SPLIT; ++r) t += ld_shared_cluster_f32(mapa_rank(&part[d], r));
      patch_mean[size_t(b) * D + d] = gamma[d] * (t / float(P)) + beta[d];
    }
  }
  cluster_sync_all();
}

// ---------------------------------------------------------------------------------------
// Nearest-neighbour block replication == np.kron(low_res, ones((p,p), int))
// (reference pl_torch_modules.py:297-298): out[b][y][x] = low[b][y/p][x/p], int64.
// ---------------------------------------------------------------------------------------
__global__ void replicate_labels_kernel(const uint8_t* __restrict__ lowres /*[B,g,g]*/,
                                        long long* __restrict__ out /*[B,g*p,g*p]*/, int B, int g, int p) {
  const int W = g * p;
  if ((W & 1) == 0) {
    const int W2 = W >> 1;
    const size_t total = size_t(B) * W * W2;
    size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x2 = int(idx % W2);
    const size_t t = idx / W2;
    const int y = int(t % W);
    const int b = int(t / W);
    const uint8_t* lr = lowres + (size_t(b) * g + y / p) * g;
    longlong2 v;
    v.x = lr[(2 * x2) / p];
    v.y = lr[(2 * x2 + 1) / p];
    reinterpret_cast<longlong2*>(out)[idx] = v;
  } else {
    const size_t total = size_t(B) * W * W;
    size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = int(idx % W);
    const size_t t = idx / W;
    const int y = int(t % W);
    const int b = int(t / W);
    out[idx] = lowres[(size_t(b) * g + y / p) * g + x / p];
  }
}

}  // namespace dsg
