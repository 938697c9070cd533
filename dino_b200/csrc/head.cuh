// Fused segmentation head for D = 384 (ViT-S):  one kernel from the residual stream to the label map.
//
//   x [M, 384] fp32 (tokens incl. the cls row of every frame)
//     -> final LayerNorm (reference vision_transformer.py:243)           statistics + xhat = (x - mean) * rstd
//     -> layer_1 + ReLU (pl_torch_modules.py:113, :118)                  bf16x3 tensor-core GEMM, N = 200 (208)
//     -> layer_2 + ReLU (:114, :120)                                     bf16x3 tensor-core GEMM, N = 100 (112)
//     -> layer_3 (:115, :122) -> log_softmax (:123) -> argmax (:295)     fp32 CUDA cores, one thread per token
//     -> drop cls (:243), p x p replication into the int64 map (:297-298 np.kron)
//
// Round 1 ran this as LayerNorm(split) -> GEMM -> GEMM -> tail kernel -> replicate: 354 MB read + 708 MB written by the
// LayerNorm (bf16x3 operand [hi | lo]), 708 + 236 MB through the first GEMM, 236 + 92 MB through the second, 92 MB into
// the tail: 2.4 GB of HBM traffic for 0.7 % of the FLOPs.  Here a persistent CTA walks 128-token row blocks and nothing
// but x (354 MB, read twice: once from HBM, once from L2) and the outputs touch memory.
//
// bf16x3 (see split_weight_kernel): x*w ~= x_hi*w_hi + x_lo*w_hi + x_hi*w_lo with x = hi + lo split into two bf16.
// The LayerNorm's gamma / beta are folded into layer_1 at weight-load time (W1 diag(gamma), b1 + W1 beta), so the
// kernel only normalises.
//
// Warp roles (576 threads, 1 CTA / SM):
//   warp 0       TMA producer: W1 (hi, lo) k-blocks [208 x 64] into the phase-1 ring, W2 (hi, lo) k-blocks [112 x 64]
//   warp 1       TMEM allocation + single-thread tcgen05.mma issuer
//   warps 2..5   LayerNorm: row statistics of the NEXT row block while the current one is in the tensor pipe, then per
//                k-block (64 columns) the A operand tiles xhat_hi / xhat_lo [128 x 64] bf16 in the UMMA layout
//   warps 6..13  epilogue 1 (two warps per TMEM lane quarter, alternate 32-column chunks): acc1 (+ b1, ReLU) -> h1_hi /
//                h1_lo as the A operand of layer 2 in shared memory - it sits between the two GEMMs of a row block
//   warps 14..17 epilogue 2: acc2 (+ b2, ReLU) -> layer_3 -> log_softmax -> argmax -> log-probs / low-res map / labels
//
// Shared memory (184 KB + tables): phase 1 uses two stages of [xhat_hi 16 | xhat_lo 16 | W1_hi 26 | W1_lo 26] KB;
// phase 2 overlays the same bytes with h1 (4 k-blocks x [hi 16 | lo 16] KB) and a two-stage W2 ring (2 x 28 KB): layer 2
// of a row block starts after its layer-1 MMAs have retired, the next row block's layer 1 after this one's layer-2 MMAs.
// TMEM: acc1 = 208 fp32 columns at 0, acc2 = 112 columns at 256; epilogue 2 of row block r overlaps layer 1 of r+1.
#pragma once
#include "kernels.cuh"

namespace dsg {

struct HeadParams {
  int M;                  // token rows (frames * Ntok)
  const float* x;         // [M, 384] fp32
  float ln_eps;
  const float* b1f;       // [H1] layer_1 bias with the LayerNorm's beta folded in
  const float* b2;        // [H2]
  const float* w3;        // [C, H2]
  const float* b3;        // [C]
  int H1, H2, C;          // 200, 100, n_classes
  int Ntok, gh, gw, p;    // tokens per frame (gh*gw + 1), patch grid (rows, columns), replication factor (480 / gh)
  float* logprobs;        // [B*P, C] or null
  uint8_t* lowres;        // [B*P] or null
  long long* labels;      // [B, g*p, g*p] or null (square grids only: gh == gw == g)
  int* hb;                // diagnostic heartbeat (see hb_mark), may be null
};

constexpr int HEAD_D = 384;
constexpr int HEAD_BM = 128;
constexpr int HEAD_N1 = 208;                          // layer_1 outputs padded to a multiple of 16
constexpr int HEAD_N2 = 112;                          // layer_2 outputs padded to a multiple of 16
constexpr int HEAD_K2 = 256;                          // layer_2 reduction length (200 padded to 4 k-blocks)
constexpr int HEAD_KB1 = HEAD_D / 64;                 // 6 k-blocks of layer 1
constexpr int HEAD_KB2 = HEAD_K2 / 64;                // 4 k-blocks of layer 2
constexpr int HEAD_A_TILE = 128 * 64 * 2;             // 16 KB: [128 x 64] bf16
constexpr int HEAD_W1_TILE = HEAD_N1 * 64 * 2;        // 26 KB
constexpr int HEAD_W2_TILE = HEAD_N2 * 64 * 2;        // 14 KB
constexpr int HEAD_STAGE1 = 2 * HEAD_A_TILE + 2 * HEAD_W1_TILE;   // 84 KB
constexpr int HEAD_H1_BYTES = HEAD_KB2 * 2 * HEAD_A_TILE;         // 128 KB
constexpr int HEAD_STAGE2 = 2 * HEAD_W2_TILE;                     // 28 KB
constexpr int HEAD_REGION = HEAD_H1_BYTES + 2 * HEAD_STAGE2;      // 184 KB (>= 2 * HEAD_STAGE1 = 168 KB)
static_assert(HEAD_REGION >= 2 * HEAD_STAGE1, "phase-2 layout must cover the phase-1 ring");
constexpr int HEAD_W3_PITCH = 104;
constexpr int HEAD_TABLE_FLOATS = HEAD_N1 + HEAD_N2 + HEAD_MAX_C * HEAD_W3_PITCH + HEAD_MAX_C;   // b1f, b2, W3, b3
constexpr int HEAD_THREADS = 64 + 128 + 256 + 128;    // 576
constexpr size_t HEAD_SMEM = size_t(HEAD_REGION) + HEAD_TABLE_FLOATS * sizeof(float) + HEAD_BM * sizeof(float2) + 256 +
                             1024;                    // + statistics + barriers + alignment slack

// -DDSG_HEAD_TIMING: the MMA issuer of CTA 0 accumulates the cycles it spends waiting per barrier and in total; the
// totals land in the heartbeat array at [900 + 2*i] (64-bit each), read with dinoseg_debug_heartbeat (tools/head_timing.py)
#ifdef DSG_HEAD_TIMING
#define HEAD_T(i) do { const long long _t = clock64(); tacc[i] += _t - tprev; tprev = _t; } while (0)
#else
#define HEAD_T(i) do { } while (0)
#endif

template <int MAXC>
__global__ void __launch_bounds__(HEAD_THREADS, 1)
head_fused_kernel(const __grid_constant__ CUtensorMap tmW1hi, const __grid_constant__ CUtensorMap tmW1lo,
                  const __grid_constant__ CUtensorMap tmW2hi, const __grid_constant__ CUtensorMap tmW2lo,
                  const HeadParams p) {
  constexpr uint32_t TMEM_COLS = 512, ACC1_COL = 0, ACC2_COL = 256;
  constexpr int HB_CODE = 400;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  uint8_t* region = smem;                                        // phase-1 ring / phase-2 h1 + W2 ring
  float* sB1 = reinterpret_cast<float*>(smem + HEAD_REGION);     // [208]
  float* sB2 = sB1 + HEAD_N1;                                    // [112]
  float* sW3 = sB2 + HEAD_N2;                                    // [HEAD_MAX_C][104]
  float* sB3 = sW3 + HEAD_MAX_C * HEAD_W3_PITCH;                 // [HEAD_MAX_C]
  float2* sStats = reinterpret_cast<float2*>(sB3 + HEAD_MAX_C);  // [128] (mean, rstd) of the row block being filled
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStats + HEAD_BM);
  uint64_t* full = bars;              // 2: stage filled (4 LayerNorm warps + producer's expect_tx / TMA bytes)
  uint64_t* empty = bars + 2;         // 2: the MMAs reading the stage have retired
  uint64_t* w2_full = bars + 4;       // 2
  uint64_t* w2_empty = bars + 6;      // 2
  uint64_t* mma1_done = bars + 8;     // acc1 complete; the phase-1 ring is dead (h1 / W2 may overlay it)
  uint64_t* mma2_done = bars + 9;     // acc2 complete; h1 / W2 are dead (the next row block's phase 1 may start)
  uint64_t* h1_ready = bars + 10;     // 8 arrivals: epilogue 1 has written h1
  uint64_t* acc1_empty = bars + 11;   // 8 arrivals: epilogue 1 has read acc1
  uint64_t* acc2_empty = bars + 12;   // 4 arrivals: epilogue 2 has read acc2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int m_blocks = (p.M + HEAD_BM - 1) / HEAD_BM;
  const int my_blocks = int(blockIdx.x) < m_blocks ? (m_blocks - 1 - int(blockIdx.x)) / int(gridDim.x) + 1 : 0;
  auto block_row0 = [&](int bi) { return (int(blockIdx.x) + bi * int(gridDim.x)) * HEAD_BM; };
  auto stage1 = [&](uint32_t u) { return region + size_t(u & 1u) * HEAD_STAGE1; };           // [A_hi | A_lo | W1_hi | W1_lo]
  auto h1_tile = [&](int kb, int lo) { return region + size_t(kb) * 2 * HEAD_A_TILE + size_t(lo) * HEAD_A_TILE; };
  auto stage2 = [&](uint32_t v) { return region + HEAD_H1_BYTES + size_t(v & 1u) * HEAD_STAGE2; };   // [W2_hi | W2_lo]

  hb_mark(p.hb, HB_CODE, 1);
  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmW1hi); tma_prefetch_desc(&tmW1lo); tma_prefetch_desc(&tmW2hi); tma_prefetch_desc(&tmW2lo);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&full[s], 5);
      mbar_init(&empty[s], 1);
      mbar_init(&w2_full[s], 1);
      mbar_init(&w2_empty[s], 1);
    }
    mbar_init(mma1_done, 1);
    mbar_init(mma2_done, 1);
    mbar_init(h1_ready, 8);
    mbar_init(acc1_empty, 8);
    mbar_init(acc2_empty, 4);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  for (int i = threadIdx.x; i < HEAD_TABLE_FLOATS; i += HEAD_THREADS) {     // biases / layer_3, zero padded
    float v = 0.f;
    if (i < HEAD_N1) v = i < p.H1 ? p.b1f[i] : 0.f;
    else if (i < HEAD_N1 + HEAD_N2) { const int c = i - HEAD_N1; v = c < p.H2 ? p.b2[c] : 0.f; }
    else if (i < HEAD_N1 + HEAD_N2 + HEAD_MAX_C * HEAD_W3_PITCH) {
      const int j = i - HEAD_N1 - HEAD_N2, k = j / HEAD_W3_PITCH, c = j - k * HEAD_W3_PITCH;
      v = (k < p.C && c < p.H2) ? p.w3[k * p.H2 + c] : 0.f;
    } else { const int k = i - HEAD_N1 - HEAD_N2 - HEAD_MAX_C * HEAD_W3_PITCH; v = k < p.C ? p.b3[k] : 0.f; }
    sB1[i] = v;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  hb_mark(p.hb, HB_CODE, 2);

  if (warp == 0) {
    if (elect_one()) {
      // ---------------- TMA producer: weights only (the A operands are produced by the LayerNorm / epilogue-1 warps) ----
      uint32_t u = 0, v = 0;
      for (int bi = 0; bi < my_blocks; ++bi) {
        for (int kb = 0; kb < HEAD_KB1; ++kb, ++u) {
          if (u >= 2) mbar_wait(&empty[u & 1], ((u >> 1) - 1) & 1);
          if (kb < 2 && bi > 0) mbar_wait(mma2_done, (bi - 1) & 1);       // h1 / W2 of the previous block are dead
          uint8_t* st = stage1(u);
          mbar_expect_tx(&full[u & 1], 2 * HEAD_W1_TILE);
          tma_load_2d(st + 2 * HEAD_A_TILE, &tmW1hi, &full[u & 1], kb * 64, 0);
          tma_load_2d(st + 2 * HEAD_A_TILE + HEAD_W1_TILE, &tmW1lo, &full[u & 1], kb * 64, 0);
        }
        mbar_wait(mma1_done, bi & 1);                                      // the phase-1 ring is dead
        for (int kb = 0; kb < HEAD_KB2; ++kb, ++v) {
          if (kb >= 2) mbar_wait(&w2_empty[v & 1], ((v >> 1) - 1) & 1);    // (the first two of a block: ring dead anyway)
          uint8_t* st = stage2(v);
          mbar_expect_tx(&w2_full[v & 1], 2 * HEAD_W2_TILE);
          tma_load_2d(st, &tmW2hi, &w2_full[v & 1], kb * 64, 0);
          tma_load_2d(st + HEAD_W2_TILE, &tmW2lo, &w2_full[v & 1], kb * 64, 0);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      // ---------------- MMA issuer ----------------
      constexpr uint32_t idesc1 = umma_idesc_bf16(HEAD_BM, HEAD_N1, 0);
      constexpr uint32_t idesc2 = umma_idesc_bf16(HEAD_BM, HEAD_N2, 0);
      uint32_t u = 0, v = 0;
#ifdef DSG_HEAD_TIMING
      long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      long long tprev = clock64();
#endif
      for (int bi = 0; bi < my_blocks; ++bi) {
        HEAD_T(7);
        if (bi > 0) { mbar_wait(acc1_empty, (bi - 1) & 1); tc_fence_after(); }
        HEAD_T(0);
        for (int kb = 0; kb < HEAD_KB1; ++kb, ++u) {
          HEAD_T(7);
          mbar_wait(&full[u & 1], (u >> 1) & 1);
          HEAD_T(kb == 0 ? 1 : 2);
          tc_fence_after();
          const uint32_t st = smem_u32(stage1(u));
          const uint64_t a_hi = umma_desc_sw128(st), a_lo = umma_desc_sw128(st + HEAD_A_TILE);
          const uint64_t w_hi = umma_desc_sw128(st + 2 * HEAD_A_TILE), w_lo = umma_desc_sw128(st + 2 * HEAD_A_TILE + HEAD_W1_TILE);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tmem_base + ACC1_COL, a_hi + uint64_t(k * 2), w_hi + uint64_t(k * 2), idesc1, (kb | k) != 0);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tmem_base + ACC1_COL, a_lo + uint64_t(k * 2), w_hi + uint64_t(k * 2), idesc1, 1u);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tmem_base + ACC1_COL, a_hi + uint64_t(k * 2), w_lo + uint64_t(k * 2), idesc1, 1u);
          tc_commit(&empty[u & 1]);
        }
        tc_commit(mma1_done);
        HEAD_T(7);
        mbar_wait(h1_ready, bi & 1);
        HEAD_T(3);
        if (bi > 0) mbar_wait(acc2_empty, (bi - 1) & 1);
        HEAD_T(4);
        tc_fence_after();
        for (int kb = 0; kb < HEAD_KB2; ++kb, ++v) {
          HEAD_T(7);
          mbar_wait(&w2_full[v & 1], (v >> 1) & 1);
          HEAD_T(5);
          tc_fence_after();
          const uint32_t st = smem_u32(stage2(v));
          const uint64_t a_hi = umma_desc_sw128(smem_u32(h1_tile(kb, 0))), a_lo = umma_desc_sw128(smem_u32(h1_tile(kb, 1)));
          const uint64_t w_hi = umma_desc_sw128(st), w_lo = umma_desc_sw128(st + HEAD_W2_TILE);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tmem_base + ACC2_COL, a_hi + uint64_t(k * 2), w_hi + uint64_t(k * 2), idesc2, (kb | k) != 0);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tmem_base + ACC2_COL, a_lo + uint64_t(k * 2), w_hi + uint64_t(k * 2), idesc2, 1u);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tmem_base + ACC2_COL, a_hi + uint64_t(k * 2), w_lo + uint64_t(k * 2), idesc2, 1u);
          tc_commit(&w2_empty[v & 1]);
        }
        tc_commit(mma2_done);
      }
#ifdef DSG_HEAD_TIMING
      HEAD_T(7);
      if (p.hb != nullptr && blockIdx.x == 0) {
        tacc[6] = my_blocks;
        for (int i = 0; i < 8; ++i) reinterpret_cast<long long*>(p.hb + 900)[i] = tacc[i];
      }
#endif
    }
  } else if (warp < 6) {
    // ---------------- LayerNorm warps: statistics, then the A operand k-block by k-block ----------------
    // Eight lanes per row, four rows per pass (ln384_stats).  Warp w takes rows w*32 .. w*32+31 of the row block.
    const int lw = warp - 2, sub = lane & 7, grp = lane >> 3;
    uint32_t u = 0;
    for (int bi = 0; bi < my_blocks; ++bi) {
      const int r0 = block_row0(bi);
      // the NEXT block's rows -> L2 now (192 KB: 12 lines per thread), so that its statistics pass finds them there
      if (bi + 1 < my_blocks) {
        const int rn = block_row0(bi + 1);
        const char* base = reinterpret_cast<const char*>(p.x + size_t(rn) * HEAD_D);
        const size_t bytes = size_t(max(0, min(HEAD_BM, p.M - rn))) * HEAD_D * sizeof(float);
        for (size_t off = size_t(threadIdx.x - 64) * 128; off < bytes; off += 128 * 128)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
      }
      // statistics of this block's rows (first read of x; L2 hits except for the first block); overlaps the tensor-pipe
      // work of block bi-1
      for (int pass = 0; pass < 8; ++pass) {
        const int r = lw * 32 + pass * 4 + grp;
        const int row = r0 + r;
        const float4* xr = reinterpret_cast<const float4*>(p.x + size_t(row < p.M ? row : 0) * HEAD_D);
        float4 v[LN384_V];
#pragma unroll
        for (int i = 0; i < LN384_V; ++i) v[i] = row < p.M ? __ldg(xr + i * 8 + sub) : make_float4(0.f, 0.f, 0.f, 0.f);
        float mean, rstd;
        ln384_stats(v, p.ln_eps, mean, rstd);
        if (sub == 0) sStats[r] = make_float2(mean, rstd);
      }
      __syncwarp();                               // statistics are written and read by the lanes of one warp
      for (int kb = 0; kb < HEAD_KB1; ++kb, ++u) {
        // columns kb*64 + sub*4 + {0, 32}: float4 numbers kb*16 + sub + {0, 8} of the row (second read of x: L2).  All 16
        // loads of the warp's 32 rows are issued before the first wait: the latency is paid once per k-block.
        float4 v0[8], v1[8];
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
          const int row = r0 + lw * 32 + pass * 4 + grp;
          const bool live = row < p.M;
          const float4* xr = reinterpret_cast<const float4*>(p.x + size_t(live ? row : 0) * HEAD_D) + kb * 16 + sub;
          v0[pass] = live ? __ldg(xr) : make_float4(0.f, 0.f, 0.f, 0.f);
          v1[pass] = live ? __ldg(xr + 8) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (u >= 2) mbar_wait(&empty[u & 1], ((u >> 1) - 1) & 1);
        if (kb < 2 && bi > 0) mbar_wait(mma2_done, (bi - 1) & 1);
        uint8_t* a_hi = stage1(u);
        uint8_t* a_lo = a_hi + HEAD_A_TILE;
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
          const int r = lw * 32 + pass * 4 + grp;
          const bool live = r0 + r < p.M;
          const float2 st = sStats[r];
          const float mean = live ? st.x : 0.f, rstd = live ? st.y : 0.f;
          uint4 hi, lo;
          split_pack8(make_float4((v0[pass].x - mean) * rstd, (v0[pass].y - mean) * rstd, (v0[pass].z - mean) * rstd,
                                  (v0[pass].w - mean) * rstd),
                      make_float4((v1[pass].x - mean) * rstd, (v1[pass].y - mean) * rstd, (v1[pass].z - mean) * rstd,
                                  (v1[pass].w - mean) * rstd), hi, lo);
          // v0 -> 8-byte half sub&1 of 16-byte chunk sub/2; v1 -> the same half of chunk sub/2 + 4
          const uint32_t off0 = uint32_t(r) * 128u + (uint32_t((sub >> 1) ^ (r & 7)) << 4) + uint32_t(sub & 1) * 8u;
          const uint32_t off1 = uint32_t(r) * 128u + (uint32_t(((sub >> 1) + 4) ^ (r & 7)) << 4) + uint32_t(sub & 1) * 8u;
          *reinterpret_cast<uint2*>(a_hi + off0) = make_uint2(hi.x, hi.y);
          *reinterpret_cast<uint2*>(a_hi + off1) = make_uint2(hi.z, hi.w);
          *reinterpret_cast<uint2*>(a_lo + off0) = make_uint2(lo.x, lo.y);
          *reinterpret_cast<uint2*>(a_lo + off1) = make_uint2(lo.z, lo.w);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[u & 1]);
      }
    }
  } else if (warp < 14) {
    // ---------------- epilogue 1: acc1 -> relu(acc1 + b1) -> h1_hi / h1_lo (A operand of layer 2) ----------------
    const int row = (warp & 3) * 32 + lane;        // TMEM lane = row of the block
    const int half = (warp - 6) >> 2;              // this warp takes the 32-column chunks half, half + 2, half + 4, half + 6
    const uint32_t acc = tmem_base + (uint32_t((warp & 3) * 32) << 16) + ACC1_COL;
    for (int bi = 0; bi < my_blocks; ++bi) {
      mbar_wait(mma1_done, bi & 1);
      __syncwarp();
      tc_fence_after();
#pragma unroll 1
      for (int c = half; c < 8; c += 2) {          // columns 0..207 hold data, 208..255 are zero padding
        float v[32];
        if (c < 6) {
          uint32_t r[32];
          tmem_ld_x32(acc + uint32_t(c * 32), r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(__uint_as_float(r[i]) + sB1[c * 32 + i], 0.f);
        } else if (c == 6) {
          uint32_t r[16];
          tmem_ld_x16(acc + 192u, r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaxf(__uint_as_float(r[i]) + sB1[192 + i], 0.f);
#pragma unroll
          for (int i = 16; i < 32; ++i) v[i] = 0.f;
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
        if (c >= 6) {                              // this warp's last chunk: its part of acc1 is in registers
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(acc1_empty);
        }
        uint8_t* t_hi = h1_tile(c >> 1, 0) + row * 128;
        uint8_t* t_lo = h1_tile(c >> 1, 1) + row * 128;
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
          uint4 hi, lo;
          split_pack8(make_float4(v[g8 * 8], v[g8 * 8 + 1], v[g8 * 8 + 2], v[g8 * 8 + 3]),
                      make_float4(v[g8 * 8 + 4], v[g8 * 8 + 5], v[g8 * 8 + 6], v[g8 * 8 + 7]), hi, lo);
          const uint32_t off = uint32_t((((c & 1) * 4 + g8) ^ (row & 7)) << 4);
          *reinterpret_cast<uint4*>(t_hi + off) = hi;
          *reinterpret_cast<uint4*>(t_lo + off) = lo;
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(h1_ready);
    }
  } else {
    // ---------------- epilogue 2: acc2 -> relu(acc2 + b2) -> layer_3 -> log_softmax -> argmax -> outputs ----------------
    const int row = (warp & 3) * 32 + lane;
    const uint32_t acc = tmem_base + (uint32_t((warp & 3) * 32) << 16) + ACC2_COL;
    const int P = p.gh * p.gw, W = p.gw * p.p;
    for (int bi = 0; bi < my_blocks; ++bi) {
      mbar_wait(mma2_done, bi & 1);
      __syncwarp();                                // (rows that skip the output part below rejoin here)
      tc_fence_after();
      float z[HEAD_MAX_C];
#pragma unroll
      for (int k = 0; k < HEAD_MAX_C; ++k) z[k] = 0.f;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {                // columns >= H2 carry relu(0 + 0) = 0 and W3 is zero padded there
        uint32_t r[32];
        tmem_ld_x32(acc + uint32_t(c * 32), r);
        tmem_ld_wait();
        if (c == 3) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(acc2_empty);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int col = c * 32 + i;
          if (col < HEAD_W3_PITCH) {
            const float h = fmaxf(__uint_as_float(r[i]) + (col < HEAD_N2 ? sB2[col] : 0.f), 0.f);
#pragma unroll
            for (int k = 0; k < MAXC; ++k) z[k] = fmaf(h, sW3[k * HEAD_W3_PITCH + col], z[k]);
          }
        }
      }
      const int m = block_row0(bi) + row;
      const int b = m / p.Ntok, tok = m - b * p.Ntok;
      if (m >= p.M || tok == 0) continue;          // past the end, or a cls row (reference :243 drops it)
      float mx = -INFINITY;
#pragma unroll
      for (int k = 0; k < MAXC; ++k)
        if (k < p.C) { z[k] += sB3[k]; mx = fmaxf(mx, z[k]); }
      float se = 0.f;
#pragma unroll
      for (int k = 0; k < MAXC; ++k)
        if (k < p.C) se += expf(z[k] - mx);
      const float lse = logf(se);
#pragma unroll
      for (int k = 0; k < MAXC; ++k)
        if (k < p.C) z[k] = (z[k] - mx) - lse;
      const int t = tok - 1;
      const size_t r_out = size_t(b) * P + t;
      if (p.logprobs != nullptr) {
#pragma unroll
        for (int k = 0; k < MAXC; ++k)
          if (k < p.C) p.logprobs[r_out * p.C + k] = z[k];
      }
      const int label = argmax_first<MAXC>(z, p.C);
      if (p.lowres != nullptr) p.lowres[r_out] = uint8_t(label);
      if (p.labels != nullptr) {
        const int i = t / p.gw, j = t - i * p.gw;
        long long* blk = p.labels + (size_t(b) * W + size_t(i) * p.p) * W + size_t(j) * p.p;
        if ((p.p & 1) == 0) {
          const longlong2 v2 = make_longlong2(label, label);
          for (int yy = 0; yy < p.p; ++yy) {
            longlong2* rowp = reinterpret_cast<longlong2*>(blk + size_t(yy) * W);
            for (int x2 = 0; x2 < (p.p >> 1); ++x2) rowp[x2] = v2;
          }
        } else {
          for (int yy = 0; yy < p.p; ++yy)
            for (int xx = 0; xx < p.p; ++xx) blk[size_t(yy) * W + xx] = label;
        }
      }
    }
  }

  hb_mark(p.hb, HB_CODE, 3);
  tc_fence_before();
  __syncthreads();
  hb_mark(p.hb, HB_CODE, 4);
  if (warp == 1) {
    tmem_dealloc(tmem_base, TMEM_COLS);
    hb_mark_left(p.hb, HB_CODE);
  }
}

}  // namespace dsg
