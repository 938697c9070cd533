// Dense "TN" GEMM on tcgen05/TMEM fed by TMA:   C[M,N] = A[M,K] * W[N,K]^T  (+ fused epilogue)
//
// A is a row-major bf16 activation matrix, W is an nn.Linear weight in its native [out,in]
// layout (both K-major UMMA operands, so no transposes anywhere).  This one kernel, with
// different epilogues, carries every linear layer of the DINOSeg hot path:
//   patch-embed (reference vision_transformer.py:153-157 as an im2col GEMM), qkv (:75,:82),
//   proj (:77,:105), fc1/GELU (:54-55,:60-61), fc2 (:56,:63), head layer_1 (pl_torch_modules.py:113,118).
//
// Persistent, warp-specialised (320 threads, 1 CTA per SM, tile = 128 x 192, n-tiles fastest so the
// CTAs that run concurrently share their A rows through L2):
//   warp 0      : TMA producer  (A tile 128x64, W tile 192x64 per k-block, SWIZZLE_128B, ring of STAGES)
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer; TWO accumulator stages
//                 (2 x 192 fp32 columns) so the epilogue of tile i overlaps the MMAs of tile i+1
//   warps 2..9  : epilogue (two warps per TMEM lane quarter, each taking half of a chunk's columns):
//                 tcgen05.ld (one accumulator row segment per thread) -> bias / activation / addend
//                 -> swizzled shared-memory staging -> TMA store (fully coalesced, tails clipped by
//                 the tensor map).  Addends (residual stream, positional table) are TMA-loaded into
//                 the same staging buffers two chunks ahead.
// RES_A variant (CTA pairs only, K <= 384): the CTA walks whole 128-row blocks; the A block (all k-blocks, 96 KB)
// stays resident in shared memory while the pair sweeps every n-tile of its row blocks, and is refilled k-block
// by k-block during the last n-tile.  Only the W tiles stream through the ring: the plain variant re-reads
// A and W for every tile and is bound by the L2 -> SM bandwidth (~11-13 TB/s measured), not by the MMAs.
// All global tensors are described by 3-D tensor maps {cols, rows_per_batch, batches}; plain
// matrices use batches = 1.  The patch-embed GEMM uses batches = frames so that a tile never
// straddles two frames and its output can skip each frame's cls row (row offset 1).
#pragma once
#include "kernels.cuh"
#include "ptx.cuh"

namespace dsg {

enum : int {
  EPI_BF16 = 0,       // out bf16 = (acc + bias) * (col < scale_cols ? col_scale : 1)
  EPI_GELU_BF16 = 1,  // out bf16 = gelu_erf(acc + bias)
  EPI_RESID_F32 = 2,  // out f32 = addend + acc + bias      (addend = out: in-place residual add)
  EPI_PATCH_F32 = 3,  // out f32[b, 1 + t] = acc + bias + pos[1 + t]   (addend = positional table)
  EPI_RELU_F32 = 4,   // out f32 = relu(acc + bias)
  EPI_RELU_SPLIT_BF16 = 5,  // v = relu(acc + bias); out bf16 [rows, 2*split_part] = [hi(v) | lo(v)] (bf16x3 operand)
  EPI_BIAS_F32 = 6,   // out f32 = acc + bias
};

struct GemmParams {
  int N, K;             // output columns, reduction length (K % 64 == 0)
  int rows_per_batch;   // rows of A / out per batch
  int batches;
  int row_off;          // output (and addend) row offset inside a batch (1 for the patch embed: cls row)
  int add_batched;      // 1: addend indexed by batch, 0: addend shared by all batches
  const float* bias;    // [N] (may be null)
  float col_scale;
  int scale_cols;
  int split_part;       // EPI_RELU_SPLIT_BF16: width of each of the two output parts (multiple of 64)
  int reverse;          // 1: row blocks are processed last to first (L2 reuse between consecutive kernels)
  int a_wrap;           // > 0: A has only a_wrap columns and the k index wraps (bf16x3 operand stored as [hi | lo])
  long long* timing;    // debug (DSG_GEMM_TIMING builds): [grid][3 roles][8] cycle totals
  int* hb;              // diagnostic heartbeat (see hb_mark), may be null
};

#ifdef DSG_GEMM_TIMING
#define GEMM_T(i) do { const long long _t = clock64(); tacc[i] += _t - tprev; tprev = _t; } while (0)
#define GEMM_T_DECL long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long tprev = clock64()
#define GEMM_T_DUMP(role) do { if (p.timing) for (int _i = 0; _i < 8; ++_i) \
    p.timing[(size_t(blockIdx.x) * 3 + (role)) * 8 + _i] = tacc[_i]; } while (0)
#else
#define GEMM_T(i) do { } while (0)
#define GEMM_T_DECL do { } while (0)
#define GEMM_T_DUMP(role) do { } while (0)
#endif

constexpr int GEMM_BM = 128;
constexpr int GEMM_BN = 192;
constexpr int GEMM_BK = 64;
constexpr int GEMM_EPI_THREADS = 256;                 // 8 epilogue warps: two per TMEM lane quarter
constexpr int GEMM_THREADS = 64 + GEMM_EPI_THREADS;
constexpr int GEMM_A_BYTES = GEMM_BM * GEMM_BK * 2;   // 16 KB
constexpr int GEMM_B_BYTES = GEMM_BN * GEMM_BK * 2;   // 24 KB
constexpr int GEMM_STAGE_BYTES = GEMM_A_BYTES + GEMM_B_BYTES;
constexpr int GEMM_STG_BYTES = 128 * 128;             // one staging buffer: 128 rows x 128 bytes

__host__ __device__ constexpr bool gemm_out_is_f32(int epi) {
  return epi == EPI_RESID_F32 || epi == EPI_PATCH_F32 || epi == EPI_RELU_F32 || epi == EPI_BIAS_F32;
}
__host__ __device__ constexpr bool gemm_has_addend(int epi) { return epi == EPI_RESID_F32 || epi == EPI_PATCH_F32; }
__host__ __device__ constexpr int gemm_nbuf(int epi) {
  return (gemm_out_is_f32(epi) || epi == EPI_RELU_SPLIT_BF16) ? 4 : 2;
}
__host__ __device__ constexpr int gemm_stages(int epi) { return gemm_nbuf(epi) == 4 ? 3 : 4; }
constexpr int GEMM_MAX_N = 3072;                      // bias vector staged in shared memory
constexpr int GEMM_BIAS_BYTES = GEMM_MAX_N * 4;
constexpr int GEMM_RES_KB = 6;                        // resident-A variant: up to 6 k-blocks (K <= 384)
// CTA-pair variant (cta_group::2): a stage holds this CTA's A tile and HALF of the W tile (96 rows)
constexpr int GEMM_PAIR_STAGE_BYTES = GEMM_A_BYTES + GEMM_B_BYTES / 2;   // 28 KB
__host__ __device__ constexpr int gemm_pair_stages(int epi) { return gemm_stages(epi) + 1; }
// ... or, with the A row block resident (K <= 384), only the half W tile (12 KB)
__host__ __device__ constexpr int gemm_pair_res_wstages(int epi) { return gemm_nbuf(epi) == 4 ? 3 : 6; }
__host__ __device__ constexpr size_t gemm_smem_bytes(int epi, bool res_a, bool pair) {
  return (pair ? (res_a ? size_t(GEMM_RES_KB) * GEMM_A_BYTES + size_t(gemm_pair_res_wstages(epi)) * (GEMM_B_BYTES / 2)
                        : size_t(gemm_pair_stages(epi)) * GEMM_PAIR_STAGE_BYTES)
               : size_t(gemm_stages(epi)) * GEMM_STAGE_BYTES) +
         size_t(gemm_nbuf(epi)) * GEMM_STG_BYTES + GEMM_BIAS_BYTES + 1024 /*align*/ + 256;
}

// GELU with the exact-erf definition (nn.GELU() default, reference vision_transformer.py:50):
//   gelu(x) = x * Phi(x),  Phi(-|x|) = 0.5 * erfc(|x|/sqrt2) = 0.5 * 2^-q(|x|)
// q = -log2(erfc(|x|/sqrt2)) is smooth; a degree-6 polynomial on [0, 4.95] (Chebyshev fit) gives
// |gelu - exact| <= 3e-6 in fp32 (tools/fit_gelu.py), 1000x below the bf16 rounding of the result,
// for 6 FMA + 1 MUFU.EX2 instead of erff()'s ~30 instructions.
__device__ __forceinline__ float gelu_erf(float x) {
  const float ax = fminf(fabsf(x), 4.949747468f);
  float q = -3.0103274184511974e-05f;
  q = fmaf(q, ax, 0.0007183064590208232f);
  q = fmaf(q, ax, -0.007799314800649881f);
  q = fmaf(q, ax, 0.05274621397256851f);
  q = fmaf(q, ax, 0.45945441722869873f);
  q = fmaf(q, ax, 1.150948166847229f);
  q = fmaf(q, ax, 1.0440264304634184e-05f);
  const float w = 0.5f * fast_exp2(-q);          // Phi(-|x|)
  return x >= 0.f ? fmaf(-x, w, x) : x * w;
}

// PAIR = true: the kernel runs as CTA pairs (clusters of two, tcgen05 cta_group::2).  A pair computes a 256 x 192
// tile: one M = 256 instruction per K step, issued by the leader CTA (cluster rank 0) and executed by both SMs, each
// on its own 128 rows of A and its own accumulator, with the 192 W rows split 96 / 96 between the two CTAs' shared
// memories.  The plain kernel is bound by the L2 -> SM delivery of its operands (40 KB per k-block per SM at
// ~42 B/clk/SM against 512 clk of MMA work); the pair loads 28 KB per k-block per SM.  Barriers as in mlp.cuh: what
// the issuer waits on lives in the leader CTA and collects both CTAs' arrivals, what it signals is multicast.
template <int EPI, bool RES_A, bool PAIR = false>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                    const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmAdd,
                    const GemmParams p) {
  // single-CTA resident A measured slower than streaming (qkv 0.235 vs 0.200 ms: with full 24 KB W tiles in the ring
  // the one A buffer cannot be refilled early enough); the half W tiles of a pair leave room for it
  static_assert(!RES_A || PAIR, "resident A is a CTA-pair form");
  constexpr bool OUT_F32 = gemm_out_is_f32(EPI);
  constexpr bool HAS_ADD = gemm_has_addend(EPI);
  constexpr bool SPLIT = EPI == EPI_RELU_SPLIT_BF16;
  constexpr int BPC = SPLIT ? 2 : 1;             // staging buffers per chunk
  constexpr int STAGES = PAIR ? (RES_A ? gemm_pair_res_wstages(EPI) : gemm_pair_stages(EPI)) : gemm_stages(EPI);
  constexpr int RING_BYTES = PAIR ? (RES_A ? GEMM_B_BYTES / 2 : GEMM_PAIR_STAGE_BYTES) : GEMM_STAGE_BYTES;
  constexpr uint32_t NCTA = PAIR ? 2 : 1;
  constexpr int A_RES_BYTES = RES_A ? GEMM_RES_KB * GEMM_A_BYTES : 0;
  constexpr int NBUF = gemm_nbuf(EPI);
  constexpr int CH = OUT_F32 ? 32 : 64;          // output columns per staging chunk (128 bytes per row)
  constexpr int NCH = GEMM_BN / CH;
  constexpr int PD = HAS_ADD ? 2 : 0;            // addend prefetch distance in chunks
  constexpr uint32_t TMEM_COLS = 512;
  constexpr uint32_t ACC_STRIDE = 256;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t pad = (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  uint8_t* ring = smem + A_RES_BYTES;            // [A slots (RES_A)] [ring] [staging] [barriers]
  uint8_t* stg = ring + size_t(STAGES) * RING_BYTES;
  float* sbias = reinterpret_cast<float*>(stg + size_t(NBUF) * GEMM_STG_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stg + size_t(NBUF) * GEMM_STG_BYTES + GEMM_BIAS_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* a_full = empty_bar + STAGES;         // GEMM_RES_KB (RES_A): A k-block landed
  uint64_t* a_empty = a_full + GEMM_RES_KB;      // GEMM_RES_KB (RES_A): last MMA reading the k-block retired
  uint64_t* acc_full = a_empty + GEMM_RES_KB;    // 2
  uint64_t* acc_empty = acc_full + 2;            // 2 (8 arrivals: one per epilogue warp)
  uint64_t* add_bar = acc_empty + 2;             // NBUF
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(add_bar + NBUF);

  // warp-uniform role index (the shuffle tells the compiler so) + elect.sync for the single issuing thread:
  // with a threadIdx-derived predicate every tcgen05.mma / TMA instruction gets wrapped in a divergence
  // 'waterfall' loop that costs ~100 clk per MMA (measured: tools/ubench/mma_bench.cu)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int num_kb = p.K / GEMM_BK;
  const int n_tiles = (p.N + GEMM_BN - 1) / GEMM_BN;
  const int m_tiles_pb = (p.rows_per_batch + GEMM_BM - 1) / GEMM_BM;
  const int m_total = m_tiles_pb * p.batches;
  // PAIR: the unit is a pair of neighbouring row blocks; cluster c takes the pair tiles c, c + G/2, ... and rank r the
  // r-th row block of the pair (a row block past the end loads zeros and stores nothing)
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0;
  const int m_units = PAIR ? (m_total + 1) / 2 : m_total;
  const int total_tiles = n_tiles * m_units;
  const int unit0 = PAIR ? int(blockIdx.x) / 2 : int(blockIdx.x);
  const int ustride = PAIR ? int(gridDim.x) / 2 : int(gridDim.x);
  // tiles of this CTA: plain = tile ids bid, bid+G, ... (n fastest); RES_A = every n-tile of row blocks bid, bid+G, ...
  const int my_tiles = RES_A ? (unit0 < m_units ? ((m_units - 1 - unit0) / ustride + 1) * n_tiles : 0)
                             : (unit0 < total_tiles ? (total_tiles - 1 - unit0) / ustride + 1 : 0);
  auto arrive_leader = [&](uint64_t* bar) {
    if constexpr (PAIR) mbar_arrive_cluster(mapa_rank(bar, 0));
    else mbar_arrive(bar);
  };
  // p.reverse: walk the row blocks from the last to the first.  The kernels of a layer alternate direction so that
  // each one starts with the rows its producer wrote last, which are still in L2 (the tensors are 2-4x the L2).
  auto tile_coords = [&](int t, int& mt, int& nt) {
    int unit;                                      // row block (or row-block pair)
    if constexpr (RES_A) {
      unit = unit0 + (t / n_tiles) * ustride;
      nt = t % n_tiles;
    } else {
      const int tile = unit0 + t * ustride;
      nt = tile % n_tiles;
      unit = tile / n_tiles;
    }
    if (p.reverse) unit = m_units - 1 - unit;
    mt = PAIR ? unit * 2 + int(cta_rank) : unit;
  };

  constexpr int HB_CODE = 100 + EPI * 10 + (RES_A ? 2 : 0) + (PAIR ? 1 : 0);
  hb_mark(p.hb, HB_CODE, 1);
  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmOut);
    if (HAS_ADD) tma_prefetch_desc(&tmAdd);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < GEMM_RES_KB; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&acc_full[s], 1);
      mbar_init(&acc_empty[s], GEMM_EPI_THREADS / 32 * NCTA);
    }
    for (int s = 0; s < NBUF; ++s) mbar_init(&add_bar[s], 1);
    fence_mbar_init();
  }
  // CTA pairs: BOTH CTAs must be running before either issues tcgen05.alloc.cta_group::2.  The two CTAs of a cluster
  // do not necessarily start at the same time: when kernels of other streams occupy the GPU, one SM of the pair can
  // drain much later than the other.  An allocation issued while the peer CTA is not resident yet returns, but the
  // peer's own allocation then blocks for ever (observed: rank 0 past the allocation, rank 1 stuck inside it; never
  // with one stream, where the two CTAs start together).  Hence a cluster barrier first - as CUTLASS' 2-SM kernels do
  // (cluster-wide pipeline-init barrier before the TMEM allocation) - which also publishes the barrier initialisation.
  if constexpr (PAIR) cluster_sync_all();
  if (warp == 1) {
    if constexpr (PAIR) tmem_alloc_pair(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  // bias (zero padded to a multiple of the tile width) once per persistent CTA
  for (int i = threadIdx.x; i < n_tiles * GEMM_BN; i += int(blockDim.x))
    sbias[i] = (p.bias != nullptr && i < p.N) ? __ldg(p.bias + i) : 0.f;
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();          // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  hb_mark(p.hb, HB_CODE, 2);

  if (warp == 0) {
    if (elect_one()) {
      uint32_t kc = 0;
      GEMM_T_DECL;
      for (int t = 0; t < my_tiles; ++t) {
        int mt, nt;
        tile_coords(t, mt, nt);
        const int bt = mt / m_tiles_pb;
        const int r0 = (mt - bt * m_tiles_pb) * GEMM_BM;
        const int mi = RES_A ? t / n_tiles : 0;    // index of the row block among this CTA's
        for (int kb = 0; kb < num_kb; ++kb, ++kc) {
          GEMM_T(7);
          if constexpr (RES_A) {
            if (nt == 0) {                         // (re)fill the resident A block, k-block by k-block
              mbar_wait(&a_empty[kb], (mi & 1) ^ 1);
              if (cta_rank == 0) mbar_expect_tx(&a_full[kb], 2 * GEMM_A_BYTES);
              tma_load_3d_pair(smem + size_t(kb) * GEMM_A_BYTES, &tmA, mapa_rank(&a_full[kb], 0), kb * GEMM_BK, r0, bt);
            }
          }
          const int s = kc % STAGES;
          GEMM_T(0);
          mbar_wait(&empty_bar[s], ((kc / STAGES) & 1) ^ 1);
          GEMM_T(1);
          uint8_t* sr = ring + size_t(s) * RING_BYTES;
          if constexpr (PAIR) {
            // my A tile and my 96 rows of the W tile; both CTAs' bytes complete on the leader's barrier
            if (cta_rank == 0) mbar_expect_tx(&full_bar[s], 2 * RING_BYTES);
            const uint32_t bar = mapa_rank(&full_bar[s], 0);
            if constexpr (!RES_A) {
              const int ak = kb * GEMM_BK;
              tma_load_3d_pair(sr, &tmA, bar, (p.a_wrap > 0 && ak >= p.a_wrap) ? ak - p.a_wrap : ak, r0, bt);
            }
            tma_load_2d_pair(sr + (RES_A ? 0 : GEMM_A_BYTES), &tmW, bar, kb * GEMM_BK,
                             nt * GEMM_BN + int(cta_rank) * (GEMM_BN / 2));
          } else {
            mbar_expect_tx(&full_bar[s], RING_BYTES);
            const int ak = kb * GEMM_BK;
            tma_load_3d(sr, &tmA, &full_bar[s], (p.a_wrap > 0 && ak >= p.a_wrap) ? ak - p.a_wrap : ak, r0, bt);
            tma_load_2d(sr + GEMM_A_BYTES, &tmW, &full_bar[s], kb * GEMM_BK, nt * GEMM_BN);
          }
          GEMM_T(2);
        }
      }
      // Producer tail: the leader's last multicast commits on this CTA's stage-empty barriers are otherwise never waited
      // for, and a CTA must not exit while an arrival may still be in flight towards its shared memory (it would land
      // in whatever the next CTA on this SM keeps there).
      if constexpr (PAIR) {
        for (uint32_t i = 0; i < uint32_t(STAGES) && i < kc; ++i) {
          const uint32_t idx = kc - 1 - i;
          mbar_wait(&empty_bar[idx % STAGES], (idx / STAGES) & 1);
        }
        if constexpr (RES_A) {
          if (my_tiles > 0) {
            const int last_mi = my_tiles / n_tiles - 1;
            for (int kb = 0; kb < num_kb; ++kb) mbar_wait(&a_empty[kb], last_mi & 1);
          }
        }
      }
      GEMM_T_DUMP(0);
    }
  } else if (warp == 1) {
    if (cta_rank == 0 && elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(PAIR ? 2 * GEMM_BM : GEMM_BM, GEMM_BN, 0);
      auto wait = [&](uint64_t* bar, uint32_t parity) {
        if constexpr (PAIR) mbar_wait_cluster(bar, parity);
        else mbar_wait(bar, parity);
      };
      auto commit = [&](uint64_t* bar) {
        if constexpr (PAIR) tc_commit_pair(bar, uint16_t(3));
        else tc_commit(bar);
      };
      uint32_t kc = 0;
      GEMM_T_DECL;
      for (int ti = 0; ti < my_tiles; ++ti) {
        int mt, nt;
        tile_coords(ti, mt, nt);
        const int as = ti & 1;
        GEMM_T(7);
        wait(&acc_empty[as], ((ti >> 1) & 1) ^ 1);        // epilogue has drained this accumulator stage
        GEMM_T(0);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(as) * ACC_STRIDE;
        const int mi = RES_A ? ti / n_tiles : 0;
        for (int kb = 0; kb < num_kb; ++kb, ++kc) {
          const int s = kc % STAGES;
          if constexpr (RES_A) {
            if (nt == 0) wait(&a_full[kb], mi & 1);
          }
          GEMM_T(7);
          wait(&full_bar[s], (kc / STAGES) & 1);
          GEMM_T(1);
          tc_fence_after();
          const uint32_t sr = smem_u32(ring + size_t(s) * RING_BYTES);
          const uint64_t adesc = umma_desc_sw128(RES_A ? smem_u32(smem + size_t(kb) * GEMM_A_BYTES) : sr);
          const uint64_t bdesc = umma_desc_sw128(RES_A ? sr : sr + GEMM_A_BYTES);
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) {
            // +32 bytes per K=16 step inside the 128-byte swizzle row (encoded >>4 -> +2)
            if constexpr (PAIR) umma_ss_pair(d_tmem, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), idesc, (kb | k) != 0);
            else umma_ss(d_tmem, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), idesc, (kb | k) != 0);
          }
          commit(&empty_bar[s]);
          if constexpr (RES_A) {
            if (nt == n_tiles - 1) commit(&a_empty[kb]);      // the next row block may overwrite this k-block
          }
          GEMM_T(2);
        }
        commit(&acc_full[as]);
      }
      GEMM_T_DUMP(1);
    }
  } else {
    // ---------------- epilogue: thread <-> accumulator row ----------------
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;              // which half of every chunk's columns this warp handles
    const int row = quarter * 32 + lane;
    const bool leader = threadIdx.x == 64;
    constexpr int HC = CH / 2;                     // columns per thread per chunk (32 bf16 / 16 fp32 = 64 bytes)
    const uint32_t lane_base = tmem_base + (uint32_t(quarter * 32) << 16);
    const int total_chunks = my_tiles * NCH;

    // coordinates of this CTA's current and next tile (one division per tile, none per chunk)
    struct TileXY { int col, r0, bt; };
    auto tile_xy = [&](int t) {
      int mt, nt;
      tile_coords(t, mt, nt);
      TileXY o;
      o.bt = mt / m_tiles_pb;
      o.r0 = (mt - o.bt * m_tiles_pb) * GEMM_BM;
      o.col = nt * GEMM_BN;
      return o;
    };
    TileXY cur = tile_xy(0), nxt = tile_xy(1);
    // addend prefetch for chunk q (= tile q / NCH, chunk q % NCH); q lies in the current or the next tile
    auto issue_add = [&](int q, int ti_cur) {
      const int tq = q / NCH;
      const TileXY& xy = tq == ti_cur ? cur : nxt;
      const int b = q % NBUF;
      mbar_expect_tx(&add_bar[b], GEMM_STG_BYTES);
      tma_load_3d(stg + size_t(b) * GEMM_STG_BYTES, &tmAdd, &add_bar[b], xy.col + (q - tq * NCH) * CH, p.row_off + xy.r0,
                  p.add_batched ? xy.bt : 0);
    };
    if (HAS_ADD && leader) {
      for (int q = 0; q < PD && q < total_chunks; ++q) issue_add(q, 0);
    }

    int g = 0;                                     // chunk counter of this CTA
    GEMM_T_DECL;
    for (int ti = 0; ti < my_tiles; ++ti) {
      const int as = ti & 1;
      if (ti > 0) { cur = nxt; nxt = tile_xy(ti + 1); }
      GEMM_T(7);
      mbar_wait(&acc_full[as], (ti >> 1) & 1);
      GEMM_T(0);
      tc_fence_after();
      const uint32_t acc = lane_base + uint32_t(as) * ACC_STRIDE;
#pragma unroll 1
      for (int c = 0; c < NCH; ++c, ++g) {
        const int col0 = cur.col + c * CH, r0 = cur.r0, bt = cur.bt;
        const int b = (g * BPC) % NBUF;
        uint8_t* sb = stg + size_t(b) * GEMM_STG_BYTES;
        const int colh = col0 + half * HC;         // first global column of this thread's segment
        // accumulator segment -> registers
        float v[HC];
        __syncwarp();
        if constexpr (HC == 32) {
          uint32_t r[32];
          tmem_ld_x32(acc + uint32_t(c * CH + half * HC), r);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
        } else {
          uint32_t r[16];
          tmem_ld_x16(acc + uint32_t(c * CH + half * HC), r);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
        }
        tmem_ld_wait();
        GEMM_T(1);
        if (c == NCH - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) arrive_leader(&acc_empty[as]); // the MMA warp may start tile ti+2 in this stage
        }
#pragma unroll
        for (int i = 0; i < HC; i += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(sbias + colh + i);   // smem broadcast
          v[i] += b4.x; v[i + 1] += b4.y; v[i + 2] += b4.z; v[i + 3] += b4.w;
        }
        // staging buffer b: the TMA store that last read it (chunk g - NBUF) must be done, and for
        // addend epilogues the prefetch of chunk g + PD goes into the buffer of chunk g + PD - NBUF
        GEMM_T(2);
        if (leader) {
          tma_store_wait_read<NBUF / BPC - PD - 1>();
          if (HAS_ADD && g + PD < total_chunks) issue_add(g + PD, ti);
        }
        GEMM_T(3);
        if constexpr (HAS_ADD) {
          mbar_wait(&add_bar[b], (g / NBUF) & 1);
        } else {
          named_bar_sync(1, GEMM_EPI_THREADS);
        }
        GEMM_T(4);
        // 128-byte staging row = 8 x 16-byte segments, XOR-swizzled with the row index (SWIZZLE_128B);
        // this thread owns segments half*4 .. half*4+3
        uint8_t* srow = sb + row * 128;
        if constexpr (OUT_F32) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float4* ptr = reinterpret_cast<float4*>(srow + (((half * 4 + k) ^ (row & 7)) << 4));
            float4 q = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
            if constexpr (HAS_ADD) {
              const float4 a = *ptr;
              q.x += a.x; q.y += a.y; q.z += a.z; q.w += a.w;
            } else if constexpr (EPI == EPI_RELU_F32) {
              q.x = fmaxf(q.x, 0.f); q.y = fmaxf(q.y, 0.f); q.z = fmaxf(q.z, 0.f); q.w = fmaxf(q.w, 0.f);
            }
            *ptr = q;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float w[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float x = v[8 * k + j];
              if constexpr (EPI == EPI_GELU_BF16) x = gelu_erf(x);
              else if constexpr (SPLIT) x = fmaxf(x, 0.f);
              else if (colh + 8 * k + j < p.scale_cols) x *= p.col_scale;
              w[j] = x;
            }
            const int seg = ((half * 4 + k) ^ (row & 7)) << 4;
            uint4 q;
            q.x = pack_bf16x2(w[0], w[1]); q.y = pack_bf16x2(w[2], w[3]);
            q.z = pack_bf16x2(w[4], w[5]); q.w = pack_bf16x2(w[6], w[7]);
            *reinterpret_cast<uint4*>(srow + seg) = q;
            if constexpr (SPLIT) {
              uint4 l;   // lo = bf16(v - hi)
              l.x = pack_bf16x2(w[0] - __uint_as_float(q.x << 16), w[1] - __uint_as_float(q.x & 0xffff0000u));
              l.y = pack_bf16x2(w[2] - __uint_as_float(q.y << 16), w[3] - __uint_as_float(q.y & 0xffff0000u));
              l.z = pack_bf16x2(w[4] - __uint_as_float(q.z << 16), w[5] - __uint_as_float(q.z & 0xffff0000u));
              l.w = pack_bf16x2(w[6] - __uint_as_float(q.w << 16), w[7] - __uint_as_float(q.w & 0xffff0000u));
              *reinterpret_cast<uint4*>(srow + GEMM_STG_BYTES + seg) = l;
            }
          }
        }
        GEMM_T(5);
        fence_proxy_async_smem();
        named_bar_sync(2, GEMM_EPI_THREADS);
        GEMM_T(6);
        if (leader) {
          if constexpr (SPLIT) {
            if (col0 < p.split_part) {
              tma_store_3d(&tmOut, sb, col0, p.row_off + r0, bt);
              tma_store_3d(&tmOut, sb + GEMM_STG_BYTES, p.split_part + col0, p.row_off + r0, bt);
            }
          } else {
            if (col0 < p.N) tma_store_3d(&tmOut, sb, col0, p.row_off + r0, bt);
          }
          tma_store_commit();
        }
      }
    }
    if (leader) { GEMM_T_DUMP(2); }
    if (leader) tma_store_wait<0>();               // all output bytes are globally visible before exit
  }

  hb_mark(p.hb, HB_CODE, 3);
  tc_fence_before();
  __syncthreads();
  hb_mark(p.hb, HB_CODE, 4);
  if constexpr (PAIR) cluster_sync_all();          // both CTAs are done with each other's barriers and TMEM
  hb_mark(p.hb, HB_CODE, 5);
  if (warp == 1) {
    if constexpr (PAIR) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
    hb_mark_left(p.hb, HB_CODE);                     // by the deallocating warp: a CTA stuck in dealloc stays visible
  }
}

}  // namespace dsg
