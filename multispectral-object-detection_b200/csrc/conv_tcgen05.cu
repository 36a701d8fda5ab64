// Implicit-GEMM convolution / GEMM on the 5th-gen tensor cores (sm_100a):
//   D[128 pixels, block_n couts] (fp32, TMEM) += A[128 pixels, 64 cin] * W[block_n couts, 64 cin]^T
//
//  * A tiles come straight from the NHWC activation tensor through a 4-D TMA tensor map
//    (C, W, H, B) with box (64, TW, TH, 1): one box per filter tap, shifted by the tap's
//    (dx, dy); out-of-bounds rows/cols/channels are zero-filled by TMA == conv zero padding
//    and K-tail padding.  Stride-2 convs use four "parity" maps (base pointer offset by
//    (py, px), W/H strides doubled) so every tap is again a dense box.
//    1x1 convs and nn.Linear are the same kernel with taps = 1, H = B = 1, W = M.
//  * W tiles come from a 3-D map (Cin, taps, Cout) over the packed [Cout][taps][Cin_p] weights.
//  * 128B / 64B / 32B-swizzled K-major smem tiles feed tcgen05.mma (UMMA 128 x block_n x 16, or 256 x block_n x 16 for a
//    CTA pair with cta_group::2; bf16 -> fp32); accumulators live in TMEM as a ring of 4 x 128 or 2 x 256 columns.
//  * Warp roles (640 threads, persistent CTAs, static round-robin tile schedule):
//      warp 0 TMA producer | warp 1 MMA issuer (one elected lane) | warp 2 TMEM alloc | warps 4-19 epilogue
//    Epilogue (2 teams x 2 column groups x 4 warps): tcgen05.ld -> +bias -> SiLU / GELU -> +residual (TMA-loaded tile)
//    -> bf16 / f32 -> swizzled smem staging -> TMA store into the NHWC channel slice.
//  * 3x3 stride-1 'row-reuse' mode: one (TH + 2) x TW pixel box per filter column serves the three vertical taps;
//    small weight matrices stay resident in smem; 1x1 convs walk a flat [B*H*W, C] matrix.  DESIGN.md section 3.1.
//
// Replaces the cuDNN/cuBLAS calls the reference reaches through nn.Conv2d / nn.Linear
// (models/common.py:41-50,450-453,533-536; models/yolo_test.py:46).
#include <stdlib.h>

#include "cft_common.cuh"
#include "tcgen05_ptx.cuh"

namespace {

using namespace cft;
using namespace cft::ptx;

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;            // bf16 elements = one 128B swizzle row
constexpr int kEpiGroups = 4;          // epilogue groups of 4 warps (one warp per TMEM lane quarter) each:
                                       // 2 teams (alternate tiles) x 2 column groups
constexpr int kEpiTeams = 2;
constexpr int kEpiColGroups = kEpiGroups / kEpiTeams;
constexpr int kEpilogueWarps = 4 * kEpiGroups;
constexpr int kThreads = 128 + 32 * kEpilogueWarps;   // TMA, MMA, TMEM-alloc, idle + epilogue warps
constexpr int kATileBytes = kBlockM * kBlockK * 2;  // 16 KiB
constexpr int kMaxStages = 8;
constexpr int kMaxAccStages = 4;       // TMEM accumulator ring: 2 x 256 columns, or 4 x 128 when block_n <= 128
constexpr int kTmemCols = 512;
constexpr int kSmemTotal = 227 * 1024;    // dynamic smem per CTA on sm_100
constexpr int kStageCBytes = 16 * 1024;   // one epilogue staging buffer (128 rows x 128 B)

constexpr int kTailBytes = 256 + 2048 + 64 + 1024;   // barriers + TMEM slot | bias staging (one copy per epilogue team) |
                                                     // chain-mode barriers | bias of the chained 1x1 (one copy per team)

struct __align__(64) TensorMaps {
  CUtensorMap a[4];
  CUtensorMap b;
  CUtensorMap c;   // output (TMA store), box (32 channels, TW, TH, 1); chain mode: 64-channel SWIZZLE_128B boxes
  CUtensorMap r;   // residual (TMA load), same geometry as c
  CUtensorMap b2;  // chain mode: weights of the chained 1x1, box (64, 1, Cout / ctas)
  CUtensorMap c2;  // chain mode: output of the chained 1x1, same geometry as c
};

struct ConvParams {
  int B, Ho, Wo, Cout;
  int taps, kw, kchunks, stride;   // taps = kh * kw (tap = ky * kw + kx)
  int kelems, layout;       // K elements per unit (16 / 32 / 64) and the matching UMMA swizzle code
  int ups;                  // K units (taps) per ring stage
  int acc_stages, acc_cols; // TMEM accumulator ring (acc_stages * acc_cols = 512 columns)
  int halo;                 // 3x3 s1 'row-reuse' mode: a stage = one filter column kx; the three ky taps are
                            // 8-row-group offsets into one (TH+2) x TW pixel box (TW = 8)
  int a_slot, b_slot;       // ring slot sizes in bytes
  int b_res_bytes;          // exact bytes of the resident weights (b_res is that, rounded up to 1 KiB)
  int b_res;                // row-reuse mode with the WHOLE weight matrix resident in smem (loaded once per CTA;
                            // the ring then streams activations only): b_res = its size in bytes, 0 = off
  int teams;                // epilogue teams: 2 = two groups of 8 warps drain alternate tiles (steady state of long tile
                            // sequences), 1 = all 16 warps share every tile (launches with <= 1 tile per CTA: halves the tail)
  int stage_c;              // bytes per epilogue staging buffer (8 KiB: one bf16 32-column chunk, 16 KiB: two / one f32)
  unsigned long long* span;    // debug (cft_debug_conv_spans): {min CTA start, max CTA end} of this launch in %globaltimer ns
  unsigned long long* trace;   // debug timeline (cft_debug_conv_trace): kTraceSlots clock samples per CTA, else null
  // chain mode (back-to-back GEMM): y2 = act2(W2 . y + bias2) per pixel, computed from the finished bf16 output tile while
  // it sits in the TMA-store staging buffer (= a K-major SWIZZLE_128B UMMA operand) -- a Bottleneck's cv1 fused into the conv
  // that produces its input (models/common.py:99-109).  Cout in {64, 128}, one n-block, W2 = [Cout, Cout] resident in smem.
  int chain, k2chunks, act2, store_main, w2_bytes;
  const float* bias2;
  int TW, TH, tiles_x, tiles_y;
  int TB, tile_px;         // images per tile (3-D tiles: TW x TH pixels of TB consecutive images); TW * TH * TB <= 128
  int n_blocks, block_n, num_tiles, stages;
  uint32_t mg_nb, mg_tx, mg_ty;   // ceil(2^32 / d) for n_blocks, tiles_x, tiles_y (0 = divide)
  int m_tiles;              // spatial tiles = B * tiles_y * tiles_x; num_tiles counts (pairs of) m-tiles x n-blocks
  int act, out_f32;
  int ldy, y_coff, ldr, r_coff;
  const float* bias;
  void* y;
  const void* res;
};

struct TileCoord {
  int b, y0, x0, n0;
};
// work item -> tile of this CTA.  With CTA pairs a work item is two consecutive spatial tiles (rank 0 / 1) of
// one n-block; a pair's missing second tile (odd count) gets b = B: all-OOB loads (zero fill), clipped stores.
// n / d for the tile decode: multiply-high by ceil(2^32 / d) (exact while n * d < 2^32, checked on the host, which
// otherwise passes magic = 0 -> true division).  Four hardware divisions per tile per warp were ~100 of the
// epilogue's ~490 instructions per warp-tile.
__device__ __forceinline__ int fast_div(int n, int d, uint32_t magic) {
  if (d == 1) return n;
  return magic ? static_cast<int>(__umulhi(static_cast<uint32_t>(n), magic)) : n / d;
}
template <int kCtas>
__device__ __forceinline__ TileCoord decode_tile(const ConvParams& p, int work, int rank) {
  TileCoord t;
  const int wq = fast_div(work, p.n_blocks, p.mg_nb);
  const int nb = work - wq * p.n_blocks;
  int m = wq * kCtas + rank;
  t.n0 = nb * p.block_n;
  if (m >= p.m_tiles) {
    t.b = p.B;
    t.y0 = 0;
    t.x0 = 0;
    return t;
  }
  const int mq = fast_div(m, p.tiles_x, p.mg_tx);
  const int tx = m - mq * p.tiles_x;
  const int bq = fast_div(mq, p.tiles_y, p.mg_ty);
  const int ty = mq - bq * p.tiles_y;
  t.b = bq * p.TB;
  t.y0 = ty * p.TH;
  t.x0 = tx * p.TW;
  return t;
}

constexpr int kTraceSlots = 64;
// slot map: 0 globaltimer at entry | 1 clock at entry | 2 setup done | 3 predecessors done (PDL) | 4 first operand
// stage landed | 5 last MMA committed | 6 epilogue drained | 7 exit | 8+2j / 9+2j accumulator j ready / released
__device__ __forceinline__ void trace_mark(const ConvParams& p, int slot) {
  if (p.trace != nullptr && slot < kTraceSlots) p.trace[blockIdx.x * kTraceSlots + slot] = static_cast<unsigned long long>(clock64());
}

// 32 accumulator columns -> act(acc + bias); bias staged in smem (pre-halved for the tanh-SiLU code 3)
__device__ __forceinline__ void bias_act32(const uint32_t (&v)[32], const float* bias, int act, float (&f)[32]) {
  const float4* bs = reinterpret_cast<const float4*>(bias);
  if (act == 3) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 b4 = bs[i];
      f[4 * i + 0] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 0]), 0.5f, b4.x));
      f[4 * i + 1] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 1]), 0.5f, b4.y));
      f[4 * i + 2] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 2]), 0.5f, b4.z));
      f[4 * i + 3] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 3]), 0.5f, b4.w));
    }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 b4 = bs[i];
      f[4 * i + 0] = __uint_as_float(v[4 * i + 0]) + b4.x;
      f[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
      f[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
      f[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
    }
    if (act == CFT_ACT_SILU) {
#pragma unroll
      for (int i = 0; i < 32; ++i) f[i] = silu_fast(f[i]);
    }
  }
}

// ------------------------------------------------------------------ the kernel
template <int kCtas>
__global__ void __launch_bounds__(kThreads, 1)
cft_conv_tcgen05_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ ConvParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1 KiB alignment by offsetting the __shared__ array (a uintptr_t round trip would make the compiler lose the
  // shared address space and emit generic LD/ST for the epilogue's staging and bias accesses)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int stages = p.stages;
  const int rank = kCtas == 2 ? static_cast<int>(cluster_ctarank()) : 0;    // CTA within the pair
  const int work0 = kCtas == 2 ? (blockIdx.x >> 1) : blockIdx.x;
  const int work_stride = kCtas == 2 ? (gridDim.x >> 1) : gridDim.x;
  const int b_rows = p.block_n / kCtas;                                     // weight rows this CTA stages
  const uint32_t a_stage_bytes = static_cast<uint32_t>(p.a_slot);           // ring slot sizes (>= bytes loaded)
  const uint32_t b_stage_bytes = static_cast<uint32_t>(p.b_slot);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + stages * a_stage_bytes;
  uint8_t* smem_w2 = smem_b + (p.b_res ? p.b_res : stages * b_stage_bytes);  // both multiples of 1024
  uint8_t* smem_c = smem_w2 + p.w2_bytes;                                    // chain mode: W2 resident in front of the staging
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_c + kEpiGroups * p.stage_c);
  uint64_t* full_bar = bars;                          // [kMaxStages]  TMA -> MMA
  uint64_t* empty_bar = bars + kMaxStages;            // [kMaxStages]  MMA -> TMA
  uint64_t* tfull_bar = bars + 2 * kMaxStages;                        // [kMaxAccStages] MMA -> epilogue
  uint64_t* tempty_bar = bars + 2 * kMaxStages + kMaxAccStages;       // [kMaxAccStages] epilogue -> MMA
  uint64_t* res_bar = bars + 2 * kMaxStages + 2 * kMaxAccStages;      // [kEpiGroups] residual TMA -> epilogue group
  uint64_t* bres_bar = bars + 2 * kMaxStages + 2 * kMaxAccStages + kEpiGroups;   // resident weights landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 2 * kMaxAccStages + kEpiGroups + 1);
  float* bias_s = reinterpret_cast<float*>(bars + 2 * kMaxStages + 2 * kMaxAccStages + kEpiGroups + 4);   // [2][256] bias, 16 B aligned
  uint64_t* a2_ready = reinterpret_cast<uint64_t*>(bias_s + 512);   // [2] chain: team's output tile is an operand now
  uint64_t* acc2_full = a2_ready + 2;                               // [2] chain: second accumulator of the team ready
  uint64_t* acc2_empty = a2_ready + 4;                              // [2] chain: ... drained
  uint64_t* w2_bar = a2_ready + 6;                                  // chain: W2 landed
  float* bias2_s = reinterpret_cast<float*>(a2_ready + 8);          // [2][128]

  if (threadIdx.x == 0) {
    if (p.span != nullptr) {
      unsigned long long gt;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
      atomicMin(p.span, gt);
    }
    if (p.trace != nullptr) {
      unsigned long long gt;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
      p.trace[blockIdx.x * kTraceSlots] = gt;
      trace_mark(p, 1);
    }
    prefetch_tmap(&maps.a[0]);
    prefetch_tmap(&maps.b);
    prefetch_tmap(&maps.c);
    if (p.res) prefetch_tmap(&maps.r);
    for (int i = 0; i < stages; ++i) {
      mbar_init(&full_bar[i], kCtas);      // pair: both producers arrive on CTA 0's barrier
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < kMaxAccStages; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], (kEpilogueWarps / p.teams) * kCtas);   // one arrive per warp of the consuming team
    }
    for (int i = 0; i < kEpiGroups; ++i) mbar_init(&res_bar[i], 1);
    mbar_init(bres_bar, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a2_ready[i], kCtas);                               // the team leader of each CTA of the pair
      mbar_init(&acc2_full[i], 1);
      mbar_init(&acc2_empty[i], (kEpilogueWarps / 2) * kCtas);
    }
    mbar_init(w2_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (kCtas == 2) tmem_alloc_2sm(tmem_slot, kTmemCols);
    else tmem_alloc(tmem_slot, kTmemCols);
  }
  tc_fence_before();
  if constexpr (kCtas == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Everything above (barrier init, TMEM allocation, descriptor prefetch) may overlap the tail of the previous kernel
  // in the stream; from here on this kernel reads / overwrites activations, so wait for its predecessors to finish.
  if (threadIdx.x == 0) trace_mark(p, 2);
  pdl_launch_dependents();
  if (p.b_res && warp == 0 && elect_one_sync()) {
    // weights are parameters, never written by a predecessor kernel: fetch them before the dependency wait
    const uint32_t b_unit = static_cast<uint32_t>(p.block_n) * static_cast<uint32_t>(p.kelems) * 2u;
    mbar_arrive_expect_tx(bres_bar, static_cast<uint32_t>(p.b_res_bytes));
    for (int u = 0; u < p.kw * p.kchunks; ++u) {
      const int kx = u / p.kchunks, kc = u - kx * p.kchunks;
      for (int ky = 0; ky < 3; ++ky)
        tma_load_3d(smem_b + (u * 3 + ky) * b_unit, &maps.b, bres_bar, kc * p.kelems, ky * p.kw + kx, 0);
    }
  }
  if (p.chain && warp == 0 && elect_one_sync()) {
    // weights of the chained 1x1: [Cout, Cout], K chunk kc of this CTA's rows at smem_w2 + kc * unit.  A pair splits the rows;
    // both CTAs credit CTA 0's barrier (the MMA issuer lives there), CTA 0 alone arms it with the pair's byte count.
    const int w2rows = p.Cout / kCtas;
    const uint32_t unit = static_cast<uint32_t>(w2rows) * 128u;
    if (rank == 0) mbar_arrive_expect_tx(w2_bar, unit * static_cast<uint32_t>(p.k2chunks) * kCtas);
    for (int kc = 0; kc < p.k2chunks; ++kc) {
      if constexpr (kCtas == 2) tma_load_3d_2sm(smem_w2 + kc * unit, &maps.b2, w2_bar, kc * 64, 0, rank * w2rows);
      else tma_load_3d(smem_w2 + kc * unit, &maps.b2, w2_bar, kc * 64, 0, 0);
    }
  }
  pdl_wait();
  if (threadIdx.x == 0) trace_mark(p, 3);

  // K is walked in units of (tap, kelems-wide channel chunk); a ring stage holds p.ups consecutive units
  // (several taps per stage when the channel count is small, so that per-stage barrier traffic is amortised).
  const int k_units = p.taps * p.kchunks;
  const int k_iters = p.halo ? (p.kw * p.kchunks + p.ups - 1) / p.ups : (k_units + p.ups - 1) / p.ups;
  const uint32_t row_bytes = static_cast<uint32_t>(p.kelems) * 2u;   // operand tile row: 32 / 64 / 128 B
  const uint32_t a_unit_bytes = 128u * row_bytes;                     // one unit's A tile (128 pixel rows)
  const uint32_t b_unit_bytes = static_cast<uint32_t>(b_rows) * row_bytes;

  if (warp == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    long long p_wait = 0, pc0 = 0;      // debug trace: cycles the producer waited for free ring slots (row-reuse path)
    const uint32_t tx_unit = static_cast<uint32_t>(p.tile_px + b_rows) * row_bytes;   // per CTA, per unit
    for (int tile = work0; tile < p.num_tiles; tile += work_stride) {
      const TileCoord t = decode_tile<kCtas>(p, tile, rank);
      auto tap_offsets = [&](int tap, int& mi, int& dy, int& dx) {
        mi = 0; dy = 0; dx = 0;
        if (p.taps > 1) {
          const int ky = tap / p.kw, kx = tap - p.kw * ky;
          if (p.stride == 1) {
            dy = ky - 1;
            dx = kx - (p.kw >> 1);
          } else {  // input row 2*oy + ky - 1 = 2*(oy + dy) + py
            const int py = (ky != 1), px = (kx != 1);
            dy = (ky == 0) ? -1 : 0;
            dx = (kx == 0) ? -1 : 0;
            mi = py * 2 + px;
          }
        }
      };
      if (p.halo) {
        // a unit = (filter column kx, channel chunk): ONE (TH+2) x TW pixel box serves the three taps ky = 0..2;
        // small-Cin layers (kchunks == 1) put up to p.ups filter columns into one ring stage
        const uint32_t a_box = static_cast<uint32_t>((p.TH + 2) * p.TW) * row_bytes;
        const uint32_t tx_halo = a_box + (p.b_res ? 0u : 3u * b_unit_bytes);      // per CTA, per unit
        const int n_hunits = p.kw * p.kchunks;
        for (int u0 = 0; u0 < n_hunits; u0 += p.ups) {
          const int n_units = (n_hunits - u0) < p.ups ? (n_hunits - u0) : p.ups;
          if (p.trace) pc0 = clock64();
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          if (p.trace) p_wait += clock64() - pc0;
          if (elect_one_sync()) {
            if constexpr (kCtas == 2) {
              if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2u * tx_halo * n_units);
              else mbar_arrive_cluster(&full_bar[stage], 0);
            } else {
              mbar_arrive_expect_tx(&full_bar[stage], tx_halo * n_units);
            }
            for (int j = 0; j < n_units; ++j) {
              const int u = u0 + j;
              const int kx = u / p.kchunks, kc = u - kx * p.kchunks;
              const int dxh = kx - (p.kw >> 1);
              uint8_t* sa = smem_a + stage * a_stage_bytes + j * a_box;
              uint8_t* sb = smem_b + stage * b_stage_bytes + j * 3 * b_unit_bytes;
              if constexpr (kCtas == 2) {
                tma_load_4d_2sm(sa, &maps.a[1], &full_bar[stage], kc * p.kelems, t.x0 + dxh, t.y0 - 1, t.b);
                for (int ky = 0; ky < 3; ++ky)
                  tma_load_3d_2sm(sb + ky * b_unit_bytes, &maps.b, &full_bar[stage], kc * p.kelems, ky * p.kw + kx,
                                  t.n0 + rank * b_rows);
              } else {
                tma_load_4d(sa, &maps.a[1], &full_bar[stage], kc * p.kelems, t.x0 + dxh, t.y0 - 1, t.b);
                if (!p.b_res)
                  for (int ky = 0; ky < 3; ++ky)
                    tma_load_3d(sb + ky * b_unit_bytes, &maps.b, &full_bar[stage], kc * p.kelems, ky * p.kw + kx, t.n0);
              }
            }
          }
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      } else if (p.ups == 1) {
        for (int tap = 0; tap < p.taps; ++tap) {
          int mi, dy, dx;
          tap_offsets(tap, mi, dy, dx);
          for (int kc = 0; kc < p.kchunks; ++kc) {
            mbar_wait(&empty_bar[stage], phase ^ 1u);
            if (elect_one_sync()) {
              uint8_t* sa = smem_a + stage * a_stage_bytes;
              uint8_t* sb = smem_b + stage * b_stage_bytes;
              if constexpr (kCtas == 2) {
                tma_load_4d_2sm(sa, &maps.a[mi], &full_bar[stage], kc * p.kelems, t.x0 + dx, t.y0 + dy, t.b);
                tma_load_3d_2sm(sb, &maps.b, &full_bar[stage], kc * p.kelems, tap, t.n0 + rank * b_rows);
                if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2u * tx_unit);
                else mbar_arrive_cluster(&full_bar[stage], 0);
              } else {
                mbar_arrive_expect_tx(&full_bar[stage], tx_unit);
                tma_load_4d(sa, &maps.a[mi], &full_bar[stage], kc * p.kelems, t.x0 + dx, t.y0 + dy, t.b);
                tma_load_3d(sb, &maps.b, &full_bar[stage], kc * p.kelems, tap, t.n0);
              }
            }
            __syncwarp();
            if (++stage == stages) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      } else {
        for (int it = 0; it < k_iters; ++it) {            // kchunks == 1 here: a unit is a tap
          const int u0 = it * p.ups;
          const int n_units = (k_units - u0) < p.ups ? (k_units - u0) : p.ups;
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          if (elect_one_sync()) {
            if constexpr (kCtas == 2) {
              if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2u * tx_unit * n_units);
              else mbar_arrive_cluster(&full_bar[stage], 0);
            } else {
              mbar_arrive_expect_tx(&full_bar[stage], tx_unit * n_units);
            }
            for (int j = 0; j < n_units; ++j) {
              const int tap = u0 + j;
              int mi, dy, dx;
              tap_offsets(tap, mi, dy, dx);
              uint8_t* sa = smem_a + stage * a_stage_bytes + j * a_unit_bytes;
              uint8_t* sb = smem_b + stage * b_stage_bytes + j * b_unit_bytes;
              if constexpr (kCtas == 2) {
                tma_load_4d_2sm(sa, &maps.a[mi], &full_bar[stage], 0, t.x0 + dx, t.y0 + dy, t.b);
                tma_load_3d_2sm(sb, &maps.b, &full_bar[stage], 0, tap, t.n0 + rank * b_rows);
              } else {
                tma_load_4d(sa, &maps.a[mi], &full_bar[stage], 0, t.x0 + dx, t.y0 + dy, t.b);
                tma_load_3d(sb, &maps.b, &full_bar[stage], 0, tap, t.n0);
              }
            }
          }
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
    if (p.trace && lane == 0) p.trace[blockIdx.x * kTraceSlots + kTraceSlots - 4] = static_cast<unsigned long long>(p_wait);
  } else if (warp == 1 && rank == 0) {
    // ===================== MMA issuer (CTA 0 of a pair issues for both) =====================
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t idesc = umma_idesc_ex(128u * kCtas, static_cast<uint32_t>(p.block_n), 0, 0);
    // smem operand descriptor: [0,14) start >> 4 | [32,46) SBO >> 4 | bit 46 version | [61,64) swizzle code
    const uint32_t desc_hi = ((8u * row_bytes) >> 4) | (1u << 14) | (static_cast<uint32_t>(p.layout) << 29);
    const uint32_t a_lo0 = smem_u32(smem_a) >> 4, b_lo0 = smem_u32(smem_b) >> 4;
    const uint32_t a_lo_stride = a_stage_bytes >> 4, b_lo_stride = b_stage_bytes >> 4;
    const int ksteps = p.kelems / 16;
    if (p.b_res) {
      mbar_wait(bres_bar, 0);
      tc_fence_after();
    }
    long long w_full = 0, w_empty = 0, c0 = 0;     // debug trace: cycles this warp waited for operands / accumulators
    // chain mode: the second GEMM of tile jj (the team's finished bf16 output tile x W2) is issued behind the main MMAs of
    // tile jj + 1, by which time the team's first epilogue has normally turned the tile into an operand
    int jt = 0;
    bool w2_seen = false;
    auto issue_gemm2 = [&](int jj) {
      const int tm = jj & 1;
      const uint32_t par = static_cast<uint32_t>(jj >> 1) & 1u;
      if (!w2_seen) {
        mbar_wait(w2_bar, 0);
        w2_seen = true;
      }
      mbar_wait(&a2_ready[tm], par);
      mbar_wait(&acc2_empty[tm], par ^ 1u);
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t idesc2 = umma_idesc_ex(128u * kCtas, static_cast<uint32_t>(p.Cout), 0, 0);
        constexpr uint32_t hi128 = (1024u >> 4) | (1u << 14) | (2u << 29);           // SBO 1024 B, SWIZZLE_128B
        const uint32_t a2_lo = smem_u32(smem_c + tm * (p.k2chunks * 16384)) >> 4;
        const uint32_t w2_lo = smem_u32(smem_w2) >> 4;
        const uint32_t w2_unit16 = (static_cast<uint32_t>(p.Cout / kCtas) * 128u) >> 4;
        const uint32_t d2 = tmem_base + 256u + 128u * tm;
        for (int kc = 0; kc < p.k2chunks; ++kc) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t da = (static_cast<uint64_t>(hi128) << 32) | (a2_lo + kc * 1024 + 2 * k);
            const uint64_t db = (static_cast<uint64_t>(hi128) << 32) | (w2_lo + kc * w2_unit16 + 2 * k);
            if constexpr (kCtas == 2) umma_bf16_2sm(d2, da, db, idesc2, (kc | k) != 0 ? 1u : 0u);
            else umma_bf16(d2, da, db, idesc2, (kc | k) != 0 ? 1u : 0u);
          }
        }
        if constexpr (kCtas == 2) umma_commit_2sm(&acc2_full[tm]);
        else umma_commit(&acc2_full[tm]);
      }
      __syncwarp();
    };
    for (int tile = work0; tile < p.num_tiles; tile += work_stride) {
      if (p.trace) c0 = clock64();
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
      if (p.trace) w_empty += clock64() - c0;
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * p.acc_cols);
      for (int it = 0; it < k_iters; ++it) {
        if (p.trace) c0 = clock64();
        mbar_wait(&full_bar[stage], phase);
        if (p.trace) w_full += clock64() - c0;
        tc_fence_after();
        if (elect_one_sync()) {
          if (tile == work0 && it == 0) trace_mark(p, 4);
          if (p.halo && p.kelems == 64) {   // one (kx, 64-channel) unit per stage: 12 back-to-back MMAs, no inner loops
            // (3 taps ky out of one pixel box: tap ky starts one 8-row swizzle group = 1 KiB further into it)
            const uint32_t b_tap16 = b_unit_bytes >> 4;
            const uint32_t a_lo = a_lo0 + stage * a_lo_stride;
            const uint32_t b_lo = p.b_res ? b_lo0 + it * 3 * b_tap16 : b_lo0 + stage * b_lo_stride;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint64_t da = (static_cast<uint64_t>(desc_hi) << 32) | (a_lo + ky * 64 + 2 * k);
                const uint64_t db = (static_cast<uint64_t>(desc_hi) << 32) | (b_lo + ky * b_tap16 + 2 * k);
                if constexpr (kCtas == 2) umma_bf16_2sm(d_tmem, da, db, idesc, (it | ky | k) != 0 ? 1u : 0u);
                else umma_bf16(d_tmem, da, db, idesc, (it | ky | k) != 0 ? 1u : 0u);
              }
            }
          } else if (p.halo) {      // per unit: 3 taps (ky) out of one pixel box; tap ky starts TW(=8) rows further
            const int n_hunits = p.kw * p.kchunks;
            const int u0 = it * p.ups;
            const int n_units = (n_hunits - u0) < p.ups ? (n_hunits - u0) : p.ups;
            const uint32_t a_box16 = (static_cast<uint32_t>((p.TH + 2) * p.TW) * row_bytes) >> 4;
            const uint32_t b_tap16 = b_unit_bytes >> 4;
            const uint32_t ky_step16 = (8u * row_bytes) >> 4;     // one 8-row swizzle group per tile row
            for (int j = 0; j < n_units; ++j) {
              const uint32_t a_lo = a_lo0 + stage * a_lo_stride + j * a_box16;
              const uint32_t b_lo = p.b_res ? b_lo0 + (u0 + j) * 3 * b_tap16 : b_lo0 + stage * b_lo_stride + j * 3 * b_tap16;
#pragma unroll
              for (int ky = 0; ky < 3; ++ky) {
                for (int k = 0; k < ksteps; ++k) {
                  const uint64_t da = (static_cast<uint64_t>(desc_hi) << 32) | (a_lo + ky * ky_step16 + 2 * k);
                  const uint64_t db = (static_cast<uint64_t>(desc_hi) << 32) | (b_lo + ky * b_tap16 + 2 * k);
                  if constexpr (kCtas == 2) umma_bf16_2sm(d_tmem, da, db, idesc, (it | j | ky | k) != 0 ? 1u : 0u);
                  else umma_bf16(d_tmem, da, db, idesc, (it | j | ky | k) != 0 ? 1u : 0u);
                }
              }
            }
          } else if (p.kelems == 64) {     // one (tap, 64-channel) unit per stage: 4 back-to-back MMAs, no inner loops
            const uint32_t a_lo = a_lo0 + stage * a_lo_stride, b_lo = b_lo0 + stage * b_lo_stride;
#pragma unroll
            for (int k = 0; k < 4; ++k) {             // +32 B along K inside the swizzle atom = +2 in the address field
              const uint64_t da = (static_cast<uint64_t>(desc_hi) << 32) | (a_lo + 2 * k);
              const uint64_t db = (static_cast<uint64_t>(desc_hi) << 32) | (b_lo + 2 * k);
              if constexpr (kCtas == 2) umma_bf16_2sm(d_tmem, da, db, idesc, (it | k) != 0 ? 1u : 0u);
              else umma_bf16(d_tmem, da, db, idesc, (it | k) != 0 ? 1u : 0u);
            }
          } else {                  // small-Cin convs: several 16/32-element units (taps) per stage
            const int u0 = it * p.ups;
            const int n_units = (k_units - u0) < p.ups ? (k_units - u0) : p.ups;
            for (int j = 0; j < n_units; ++j) {
              const uint32_t a_lo = a_lo0 + stage * a_lo_stride + j * (a_unit_bytes >> 4);
              const uint32_t b_lo = b_lo0 + stage * b_lo_stride + j * (b_unit_bytes >> 4);
              for (int k = 0; k < ksteps; ++k) {
                const uint64_t da = (static_cast<uint64_t>(desc_hi) << 32) | (a_lo + 2 * k);
                const uint64_t db = (static_cast<uint64_t>(desc_hi) << 32) | (b_lo + 2 * k);
                if constexpr (kCtas == 2) umma_bf16_2sm(d_tmem, da, db, idesc, (it | j | k) != 0 ? 1u : 0u);
                else umma_bf16(d_tmem, da, db, idesc, (it | j | k) != 0 ? 1u : 0u);
              }
            }
          }
          if constexpr (kCtas == 2) {
            umma_commit_2sm(&empty_bar[stage]);                       // frees the slot in both CTAs
            if (it == k_iters - 1) umma_commit_2sm(&tfull_bar[acc]);  // both CTAs' epilogues
          } else {
            umma_commit(&empty_bar[stage]);                       // smem slot free once these MMAs retire
            if (it == k_iters - 1) umma_commit(&tfull_bar[acc]);  // accumulator complete
          }
          if (it == k_iters - 1) trace_mark(p, 5);
        }
        __syncwarp();
        if (++stage == stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      if (++acc == p.acc_stages) {
        acc = 0;
        acc_phase ^= 1u;
      }
      if (p.chain && jt >= 1) issue_gemm2(jt - 1);
      ++jt;
    }
    if (p.chain && jt >= 1) issue_gemm2(jt - 1);
    if (p.trace && lane == 0) {
      p.trace[blockIdx.x * kTraceSlots + kTraceSlots - 2] = static_cast<unsigned long long>(w_full);
      p.trace[blockIdx.x * kTraceSlots + kTraceSlots - 3] = static_cast<unsigned long long>(w_empty);
    }
  } else if (warp >= 4) {
    // ===================== epilogue: kEpiGroups column groups x 4 warps =====================
    const int ew = warp - 4;
    const int grp = ew >> 2;               // epilogue group 0..3
    const int teams = p.teams, col_groups = kEpiGroups / teams;
    const int team = teams == 2 ? (grp & 1) : 0;      // team t drains the accumulators of this CTA's tiles t, t + teams, ...
    const int cg = teams == 2 ? (grp >> 1) : grp;     // column group inside the team: 32-column chunks cg, cg + col_groups, ...
    const int q = warp & 3;                // TMEM lane quarter this warp may read
    const int row = q * 32 + lane;         // accumulator row = pixel within the tile
    const int gtid = (ew & 3) * 32 + lane; // thread index within the group
    uint8_t* stage_c = smem_c + grp * p.stage_c;      // this group's staging buffer
    uint64_t* rbar = &res_bar[grp];
    float* bias_t = bias_s + team * 256;   // the team's bias copy (teams may be on different n-blocks)
    uint32_t res_phase = 0;
    const int chunks_total = (p.block_n + 31) >> 5;                  // 32-column chunks
    const int my_chunks = chunks_total > cg ? (chunks_total - cg + col_groups - 1) / col_groups : 0;
    const int cps = p.out_f32 ? 1 : (p.stage_c >> 13);               // chunks per staging buffer (8 / 16 KiB)
    const uint32_t c_row_bytes = p.out_f32 ? 128u : 64u;             // one 32-channel row in the staging box
    const uint32_t c_chunk_stride = 128u * c_row_bytes;
    const uint32_t c_box_bytes = static_cast<uint32_t>(p.tile_px) * c_row_bytes;
    const bool use_res = p.res != nullptr;
    int bias_n0 = -1;
    const int bar_id = 1 + grp;
    const int acc_mask = p.acc_stages - 1, acc_shift = p.acc_stages == 4 ? 2 : 1;
    if (p.chain) {
      // ===================== chain mode: y -> staging tile (a UMMA operand) -> second GEMM -> y2 =====================
      // 2 teams x (2 column groups x 4 warps); team t drains tiles t, t + 2, ... of this CTA: main accumulator `t`
      // (2 x 128 columns), second accumulator 256 + 128 t.  The team's staging buffer A2 holds the finished bf16 tile as
      // Cout / 64 boxes of (64 channels x TW x TH) in SWIZZLE_128B = K-major UMMA chunks of 128 rows x 128 B: it is the
      // source of the TMA store of y AND the A operand of the second GEMM; its result (y2) reuses the buffer.
      const int ttid = cg * 128 + gtid;                  // thread within the team
      const bool leader = ttid == 0;
      const int n64 = p.k2chunks;                        // 64-channel boxes per tile
      uint8_t* A2 = smem_c + team * (n64 * 16384);
      float* bias2_t = bias2_s + team * 128;
      uint64_t* rb = &res_bar[team];
      const uint32_t box_bytes = static_cast<uint32_t>(p.tile_px) * 128u;
      const int nch = p.Cout >> 5;                       // 32-column chunks; this column group: cg, cg + 2
      const int tbar = 8 + team;
      const uint32_t lane_q = static_cast<uint32_t>(q * 32) << 16;
      for (int i = ttid; i < p.Cout; i += 256) {         // both bias vectors, once (one n-block)
        const float b1 = p.bias != nullptr ? __ldg(p.bias + i) : 0.f;
        const float b2 = p.bias2 != nullptr ? __ldg(p.bias2 + i) : 0.f;
        bias_t[i] = p.act == 3 ? 0.5f * b1 : b1;
        bias2_t[i] = p.act2 == 3 ? 0.5f * b2 : b2;
      }
      for (int j = team;; j += 2) {
        const int tile = work0 + j * work_stride;
        if (tile >= p.num_tiles) break;
        const uint32_t par = static_cast<uint32_t>(j >> 1) & 1u;          // this team's (j / 2)-th tile
        const TileCoord t = decode_tile<kCtas>(p, tile, rank);
        if (leader) {
          bulk_wait_read<0>();                                           // the previous y2 store has read A2
          if (use_res) {
            mbar_arrive_expect_tx(rb, static_cast<uint32_t>(n64) * box_bytes);
            for (int c = 0; c < n64; ++c) tma_load_4d(A2 + c * 16384, &maps.r, rb, c * 64, t.x0, t.y0, t.b);
          }
        }
        named_bar_sync(tbar, 256);
        mbar_wait(&tfull_bar[team], par);
        tc_fence_after();
        if (use_res) {
          mbar_wait(rb, res_phase);
          res_phase ^= 1u;
        }
        for (int ci = cg; ci < nch; ci += 2) {
          const int c0 = ci * 32;
          uint32_t v[32];
          tmem_ld32(tmem_base + lane_q + static_cast<uint32_t>(team * 128 + c0), v);
          float f[32];
          bias_act32(v, bias_t + c0, p.act, f);
          uint8_t* rowp = A2 + (c0 >> 6) * 16384 + row * 128;
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            bf16x8* s0 = reinterpret_cast<bf16x8*>(rowp + (((((c0 & 63) >> 3) + ch) ^ (row & 7)) << 4));
            if (use_res) {
              float r[8];
              unpack8(*s0, r);
#pragma unroll
              for (int i = 0; i < 8; ++i) f[8 * ch + i] += r[i];
            }
            *s0 = pack8(f + 8 * ch);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCtas == 2 && rank != 0) mbar_arrive_cluster(&tempty_bar[team], 0);
          else mbar_arrive(&tempty_bar[team]);
        }
        fence_proxy_async();
        named_bar_sync(tbar, 256);
        if (leader) {
          if (p.store_main) {
            for (int c = 0; c < n64; ++c) tma_store_4d(&maps.c, A2 + c * 16384, c * 64, t.x0, t.y0, t.b);
            bulk_commit();
          }
          if (kCtas == 2 && rank != 0) mbar_arrive_cluster(&a2_ready[team], 0);      // the tile is an operand now
          else mbar_arrive(&a2_ready[team]);
        }
        // ---- the chained 1x1: second accumulator -> act2(acc + bias2) -> y2
        mbar_wait(&acc2_full[team], par);
        tc_fence_after();
        if (leader) bulk_wait_read<0>();                                 // the store of y has read A2 (GEMM 2 has, too)
        named_bar_sync(tbar, 256);
        for (int ci = cg; ci < nch; ci += 2) {
          const int c0 = ci * 32;
          uint32_t v[32];
          tmem_ld32(tmem_base + lane_q + static_cast<uint32_t>(256 + team * 128 + c0), v);
          float f[32];
          bias_act32(v, bias2_t + c0, p.act2, f);
          uint8_t* rowp = A2 + (c0 >> 6) * 16384 + row * 128;
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)
            *reinterpret_cast<bf16x8*>(rowp + (((((c0 & 63) >> 3) + ch) ^ (row & 7)) << 4)) = pack8(f + 8 * ch);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCtas == 2 && rank != 0) mbar_arrive_cluster(&acc2_empty[team], 0);
          else mbar_arrive(&acc2_empty[team]);
        }
        fence_proxy_async();
        named_bar_sync(tbar, 256);
        if (leader) {
          for (int c = 0; c < n64; ++c) tma_store_4d(&maps.c2, A2 + c * 16384, c * 64, t.x0, t.y0, t.b);
          bulk_commit();
        }
      }
      if (leader) bulk_wait_all();
    } else
    for (int j = team;; j += teams) {          // j = index in this CTA's tile sequence (the MMA warp walks all j)
      const int tile = work0 + j * work_stride;
      if (tile >= p.num_tiles) break;
      const int acc = j & acc_mask;
      const uint32_t acc_phase = static_cast<uint32_t>(j >> acc_shift) & 1u;
      const TileCoord t = decode_tile<kCtas>(p, tile, rank);
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * p.acc_cols);
      bool waited_full = false;
      for (int sg = 0; sg < my_chunks; sg += cps) {        // this group's chunks: cg + kEpiColGroups * (sg + i)
        const int nch = (my_chunks - sg) < cps ? (my_chunks - sg) : cps;
        // acquire the group's staging buffer (its previous store has been read out); prefetch the residual tile
        if (gtid == 0) {
          bulk_wait_read<0>();
          if (use_res) {
            mbar_arrive_expect_tx(rbar, static_cast<uint32_t>(nch) * c_box_bytes);
            for (int i = 0; i < nch; ++i)
              tma_load_4d(stage_c + i * c_chunk_stride, &maps.r, rbar, t.n0 + (cg + col_groups * (sg + i)) * 32, t.x0,
                          t.y0, t.b);
          }
        }
        if (t.n0 != bias_n0) {          // (re)stage this n-block's bias; published by the barrier below
          for (int i = gtid; i < my_chunks * 32; i += 128) {
            const int col = (cg + col_groups * (i >> 5)) * 32 + (i & 31);
            const int n = t.n0 + col;
            const float bv = (p.bias != nullptr && n < p.Cout) ? __ldg(p.bias + n) : 0.f;
            bias_t[col] = p.act == 3 ? 0.5f * bv : bv;     // tanh-SiLU consumes h = (acc + bias) / 2 = fma(acc, .5, bias / 2)
          }
          bias_n0 = t.n0;
        }
        named_bar_sync(bar_id, 128);
        if (!waited_full) {
          mbar_wait(&tfull_bar[acc], acc_phase);
          tc_fence_after();
          waited_full = true;
          if (gtid == 0 && cg == 0) trace_mark(p, 8 + 2 * j);
        }
        if (use_res) {
          mbar_wait(rbar, res_phase);
          res_phase ^= 1u;
        }
        for (int ci = 0; ci < nch; ++ci) {
          const int c0 = (cg + col_groups * (sg + ci)) * 32;
          uint8_t* stage = stage_c + ci * c_chunk_stride;
          uint32_t v[32];
          tmem_ld32(t_row + static_cast<uint32_t>(c0), v);
          // bias (staged in smem once per n-block; zero beyond Cout) + activation on all 32 columns: straight-line,
          // 32 independent dependency chains (columns past Cout/block_n hold garbage that the TMA store clips).
          float f[32];
          const float4* bs = reinterpret_cast<const float4*>(bias_t + c0);
          if (p.act == 3) {     // SiLU as h + h*tanh(h), h = (acc + bias) / 2: FFMA, MUFU.TANH, FFMA per element
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 b4 = bs[i];
              f[4 * i + 0] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 0]), 0.5f, b4.x));
              f[4 * i + 1] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 1]), 0.5f, b4.y));
              f[4 * i + 2] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 2]), 0.5f, b4.z));
              f[4 * i + 3] = silu_tanh_h(fmaf(__uint_as_float(v[4 * i + 3]), 0.5f, b4.w));
            }
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 b4 = bs[i];
              f[4 * i + 0] = __uint_as_float(v[4 * i + 0]) + b4.x;
              f[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
              f[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
              f[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
            }
            if (p.act == CFT_ACT_SILU) {
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = silu_fast(f[i]);
            } else if (p.act == 4) {          // erf-GELU, A&S erf (default; CFT_GELU_ERFF=1 selects erff)
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = gelu_fast(f[i]);
            } else if (p.act == CFT_ACT_GELU) {
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = gelu_f(f[i]);
            }
          }
          // staging tile = TMA box (32 channels x TW x TH), hardware-swizzled rows:
          //   bf16: 64 B rows, SWIZZLE_64B  (16 B chunk ^= (row >> 1) & 3)
          //   f32 : 128 B rows, SWIZZLE_128B (16 B chunk ^= row & 7)
          // The residual tile (if any) was TMA-loaded into the same positions: add in place.
          if (p.out_f32) {
#pragma unroll
            for (int ch = 0; ch < 8; ++ch) {
              float4* s0 = reinterpret_cast<float4*>(stage + row * 128 + ((ch ^ (row & 7)) << 4));
              float4 o = make_float4(f[4 * ch], f[4 * ch + 1], f[4 * ch + 2], f[4 * ch + 3]);
              if (use_res) {
                const float4 r0 = *s0;
                o.x += r0.x; o.y += r0.y; o.z += r0.z; o.w += r0.w;
              }
              *s0 = o;
            }
          } else {
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
              bf16x8* s0 = reinterpret_cast<bf16x8*>(stage + row * 64 + ((ch ^ ((row >> 1) & 3)) << 4));
              if (use_res) {
                float r[8];
                unpack8(*s0, r);
#pragma unroll
                for (int i = 0; i < 8; ++i) f[8 * ch + i] += r[i];
              }
              *s0 = pack8(f + 8 * ch);
            }
          }
        }
        fence_proxy_async();          // generic-proxy smem writes -> visible to the TMA (async proxy)
        named_bar_sync(bar_id, 128);
        if (gtid == 0) {
          for (int i = 0; i < nch; ++i)   // OOB pixels / channels are clipped by the tensor map
            tma_store_4d(&maps.c, stage_c + i * c_chunk_stride, t.n0 + (cg + col_groups * (sg + i)) * 32, t.x0, t.y0, t.b);
          bulk_commit();
        }
      }
      if (!waited_full) {               // a group with no columns still keeps the accumulator handshake in step
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kCtas == 2 && rank != 0) mbar_arrive_cluster(&tempty_bar[acc], 0);   // the MMA issuer lives in CTA 0
        else mbar_arrive(&tempty_bar[acc]);
      }
      if (gtid == 0 && cg == 0) trace_mark(p, 9 + 2 * j);
    }
    if (gtid == 0) bulk_wait_all();   // all bulk stores complete before the CTA exits
    if (gtid == 0 && grp == 0) trace_mark(p, 6);
  }

  tc_fence_before();
  if constexpr (kCtas == 2) {
    cluster_sync_all();     // the peer may still be reading operands / arriving on this CTA's barriers
    if (warp == 2) tmem_dealloc_2sm(tmem_base, kTmemCols);
  } else {
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
  }
  if (threadIdx.x == 0 && p.span != nullptr) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    atomicMax(p.span + 1, gt);
  }
  if (threadIdx.x == 0 && p.trace != nullptr) {
    trace_mark(p, 7);
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    p.trace[blockIdx.x * kTraceSlots + kTraceSlots - 1] = gt;     // calibrates clock64 against wall time
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int encode_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_b,
               const cuuint32_t* box, CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
               CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return CFT_E_CUDA;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, dt, rank, const_cast<void*>(base), dims, strides_b, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d): rank %d dims %llu,%llu,%llu,%llu box %u,%u,%u,%u", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2],
              (unsigned long long)(rank > 3 ? dims[3] : 0), box[0], box[1], box[2], rank > 3 ? box[3] : 0);
    return CFT_E_CUDA;
  }
  return CFT_OK;
}

int round_up(int a, int b) { return (a + b - 1) / b * b; }

// Largest multiple of 16 (<= 256) that divides Cout with the fewest blocks; falls back to 256 + tail.
int pick_block_n(int cout) {
  if (cout <= 256) return round_up(cout, 16);
  int nb = (cout + 255) / 256;
  for (;; ++nb) {
    if (nb > cout / 16) break;
    if (cout % nb == 0 && (cout / nb) % 32 == 0 && cout / nb <= 256) return cout / nb;
    if (nb > 64) break;
  }
  return 256;
}

const bool g_no_tile3d = getenv("CFT_NO_BATCH_TILES") != nullptr;     // tiles never span images (A/B of the 3-D tiles)
// The output-pixel tile of one CTA: TW x TH pixels of TB consecutive images, TW * TH * TB <= 128 (one UMMA M tile; the TMA
// boxes are (channels, TW, TH, TB) of the (C, W, H, B) tensors, so image borders zero-fill per image).  40 x 40 and 20 x 20
// maps have no 2-D tile of 128 pixels without waste (best: 40 x 3 = 120 of 128 rows, 14 tiles per image instead of 12.5);
// 8 x 8 x 2 images / 4 x 4 x 8 images are exact -- 11 % / 22 % fewer tiles and, at batch 32, 3 instead of 4 waves of the
// N = 256 pair tiles of the P4 Bottlenecks.
void pick_spatial_tile(int Ho, int Wo, int B, int* TW, int* TH, int* TB) {
  long best = -1;
  int bw = 1, bh = 1, bb = 1;
  for (int tw = 1; tw <= 128 && tw <= Wo; ++tw) {
    for (int th = 1; th * tw <= 128 && th <= Ho; ++th) {
      int tb = 128 / (tw * th);
      if (tb > B) tb = B;
      if (g_no_tile3d) tb = 1;
      const long tiles = static_cast<long>((Wo + tw - 1) / tw) * ((Ho + th - 1) / th) * ((B + tb - 1) / tb);
      // fewest tiles first, then the fewest images per tile, then the widest rows (longer contiguous runs per TMA box row)
      const long score = (tiles * 256 + tb) * 256 - tw;
      if (best < 0 || score < best) {
        best = score;
        bw = tw;
        bh = th;
        bb = tb;
      }
    }
  }
  *TW = bw;
  *TH = bh;
  *TB = bb;
}

bool g_attr_set = false;
// CFT_CONV_CTAS=1 forces single-CTA tiles, =2 forces CTA pairs wherever legal (tests); unset = heuristic.
const bool g_silu_tanh = getenv("CFT_SILU_EXP2") == nullptr;   // default: one-SFU-op SiLU; CFT_SILU_EXP2=1 -> ex2+rcp form
const bool g_gelu_fast = getenv("CFT_GELU_ERFF") == nullptr;   // default: 2-SFU-op erf-GELU; CFT_GELU_ERFF=1 -> erff
unsigned long long* g_trace_buf = nullptr;   // cft_debug_conv_trace
unsigned long long* g_span_buf = nullptr;    // cft_debug_conv_spans
int g_span_next = 0, g_span_max = 0;
thread_local cft_conv_plan* g_plan_out = nullptr;   // cft_debug_conv_plan: report the plan instead of launching
const bool g_no_bres = getenv("CFT_NO_BRES") != nullptr;     // debug: never keep the weights resident
const bool g_no_pdl = getenv("CFT_NO_PDL") != nullptr;
const bool g_no_halo = getenv("CFT_NO_ROW_REUSE") != nullptr;
const int g_force_ctas = getenv("CFT_CONV_CTAS") ? atoi(getenv("CFT_CONV_CTAS")) : 0;

}  // namespace

extern "C" int cft_conv2d(const cft_conv_args* a, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CFT_REQUIRE(a && a->x && a->w && a->y, "cft_conv2d: null pointer");
  CFT_REQUIRE(a->k == 1 || a->k == 3, "cft_conv2d: k must be 1 or 3 (got %d)", a->k);
  const int kw = a->kw > 0 ? a->kw : a->k;
  CFT_REQUIRE(kw == a->k || (a->k == 3 && kw == 1), "cft_conv2d: kernel %dx%d unsupported", a->k, kw);
  CFT_REQUIRE(a->stride == 1 || (a->stride == 2 && a->k == 3 && kw == 3), "cft_conv2d: stride %d with k %dx%d unsupported",
              a->stride, a->k, kw);
  CFT_REQUIRE(a->B > 0 && a->H > 0 && a->W > 0 && a->Cin > 0 && a->Cout > 0, "cft_conv2d: empty shape");
  CFT_REQUIRE(a->Cin % 8 == 0 && a->ldx % 8 == 0 && a->x_coff % 8 == 0,
              "cft_conv2d: Cin/ldx/x_coff must be multiples of 8 (got %d/%d/%d)", a->Cin, a->ldx, a->x_coff);
  CFT_REQUIRE(a->Cout % 8 == 0 && a->ldy % 8 == 0 && a->y_coff % 8 == 0,
              "cft_conv2d: Cout/ldy/y_coff must be multiples of 8 (got %d/%d/%d)", a->Cout, a->ldy, a->y_coff);
  CFT_REQUIRE(!a->res || (a->ldr % 8 == 0 && a->r_coff % 8 == 0 && reinterpret_cast<uintptr_t>(a->res) % 16 == 0),
              "cft_conv2d: residual ld/coff must be multiples of 8 and the pointer 16-byte aligned");
  CFT_REQUIRE(a->x_coff + a->Cin <= a->ldx && a->y_coff + a->Cout <= a->ldy, "cft_conv2d: channel slice out of range");
  CFT_REQUIRE(reinterpret_cast<uintptr_t>(a->x) % 16 == 0 && reinterpret_cast<uintptr_t>(a->w) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(a->y) % 16 == 0,
              "cft_conv2d: pointers must be 16-byte aligned");
  CFT_REQUIRE(a->stride == 1 || (a->H % 2 == 0 && a->W % 2 == 0), "cft_conv2d: stride 2 needs even H, W");
  CFT_REQUIRE(a->out_dtype == CFT_DT_BF16 || a->out_dtype == CFT_DT_F32, "cft_conv2d: bad out_dtype");
  const bool chain = a->w2 != nullptr;
  if (chain) {
    CFT_REQUIRE(a->y2 != nullptr && a->ldy2 % 8 == 0 && a->y2_coff % 8 == 0 && a->y2_coff + a->Cout <= a->ldy2 &&
                    reinterpret_cast<uintptr_t>(a->y2) % 16 == 0 && reinterpret_cast<uintptr_t>(a->w2) % 16 == 0,
                "cft_conv2d: chained 1x1: bad y2 / w2 (null, misaligned or channel slice out of range)");
    if (a->out_dtype != CFT_DT_BF16 || (a->Cout != 64 && a->Cout != 128)) {
      set_error("cft_conv2d: chained 1x1 needs a bf16 output with 64 or 128 channels (got %d)", a->Cout);
      return CFT_E_UNSUPPORTED;
    }
  }

  // A 1x1 stride-1 conv has no halo: walk its pixels as one flat [B*H*W, C] matrix, so that tiles are 128
  // consecutive pixels (40x40 and 20x20 maps otherwise leave 11 % / 22 % of every 128-row MMA tile empty).
  cft_conv_args flat;
  if (a->k == 1 && kw == 1 && a->stride == 1 && (a->B > 1 || a->H > 1) &&
      static_cast<long long>(a->B) * a->H * a->W < (1LL << 31)) {
    flat = *a;
    flat.W = a->B * a->H * a->W;
    flat.H = 1;
    flat.B = 1;
    a = &flat;
  }
  const int s = a->stride;
  ConvParams p;
  p.B = a->B;
  p.Ho = (a->H + s - 1) / s;
  p.Wo = (a->W + s - 1) / s;
  p.Cout = a->Cout;
  p.taps = a->k * kw;
  p.kw = kw;
  p.kelems = a->Cin <= 16 ? 16 : (a->Cin <= 32 ? 32 : 64);
  p.layout = p.kelems == 64 ? 2 : (p.kelems == 32 ? 4 : 6);   // UMMA LayoutType: SW128 / SW64 / SW32
  p.kchunks = (a->Cin + p.kelems - 1) / p.kelems;
  p.ups = (p.kchunks == 1 && p.taps > 1) ? 64 / p.kelems : 1;   // small-Cin convs: several taps per stage
  p.stride = s;
  // row-reuse mode for L2-bound 3x3 stride-1 layers (measured L2->SM ceiling ~60 B/cycle/SM): 8 x 16 pixel tiles,
  // the 3 vertical taps share one (16+2) x 8 pixel box -> 2.7x less activation traffic than 9 separate boxes
  p.halo = (!g_no_halo && a->k == 3 && s == 1 && p.Wo % 8 == 0 && p.Ho % 16 == 0) ? 1 : 0;
  if (p.halo) {
    // a row-reuse stage = (TH + 2) x TW pixels + three weight taps of the n-block: wide layers (e.g. 256 -> 256 at 64 x 80,
    // BASELINE config 3) would get a ring of fewer than 3 stages -- they take the plain path (one tap per stage, >= 4 stages)
    const int kel = a->Cin <= 16 ? 16 : (a->Cin <= 32 ? 32 : 64);
    const int kch = (a->Cin + kel - 1) / kel;
    const int ups_h = (kch == 1) ? 64 / kel : 1;
    const int bn = pick_block_n(a->Cout);
    const int a_sl = ((ups_h * 18 * 8 * kel * 2 + 1023) / 1024) * 1024;
    const int b_sl = ((ups_h * 3 * (bn / 2) * kel * 2 + 1023) / 1024) * 1024;      // optimistic: a CTA pair halves it
    const int resident = kw * kch * 3 * bn * kel * 2 <= 96 * 1024 && (a->Cout + bn - 1) / bn == 1;
    if (!resident && (kSmemTotal - 1024 - kTailBytes - 4 * kStageCBytes) / (a_sl + b_sl) < 3) p.halo = 0;
  }
  p.TB = 1;
  if (p.halo) {
    p.TW = 8;
    p.TH = 16;
  } else {
    pick_spatial_tile(p.Ho, p.Wo, p.B, &p.TW, &p.TH, &p.TB);
  }
  p.tile_px = p.TW * p.TH * p.TB;
  p.tiles_x = (p.Wo + p.TW - 1) / p.TW;
  p.tiles_y = (p.Ho + p.TH - 1) / p.TH;
  p.block_n = pick_block_n(a->Cout);
  const long long m_tiles = static_cast<long long>((p.B + p.TB - 1) / p.TB) * p.tiles_x * p.tiles_y;
  // too few tiles to fill the GPU (the M = 4096 GEMMs of the CFT blocks): trade tile width for parallelism.  Not with a
  // chained 1x1: its second GEMM needs all Cout channels of y in one tile (n_blocks = 1)
  while (!chain && a->Cin * p.taps <= 1024 && 2 * m_tiles * ((a->Cout + p.block_n - 1) / p.block_n) <= sm_count() &&
         p.block_n >= 128 && (p.block_n / 2) % 32 == 0 && a->Cout % (p.block_n / 2) == 0)
    p.block_n /= 2;
  p.n_blocks = (a->Cout + p.block_n - 1) / p.block_n;
  p.acc_stages = (p.block_n <= 128 && !chain) ? 4 : 2;
  p.acc_cols = chain ? 128 : 512 / p.acc_stages;      // chain mode: main 2 x 128 columns, second accumulators at 256 + 128 t
  CFT_REQUIRE(m_tiles * p.n_blocks < (1LL << 31), "cft_conv2d: too many tiles");
  p.m_tiles = static_cast<int>(m_tiles);
  // CTA pairs (cta_group::2, UMMA M = 256): each CTA stages only half of the weight tile, halving the smem
  // traffic per MMA -- worth it once the layer is tensor-bound (enough K work per tile) and has >= 2 tiles.
  const int k_iters = p.halo ? (kw * p.kchunks + p.ups - 1) / p.ups : (p.taps * p.kchunks + p.ups - 1) / p.ups;
  int ctas = (g_force_ctas == 1) ? 1 : 2;
  if (p.kelems != 64 || p.block_n % 32 != 0 || m_tiles < 2) ctas = 1;
  if (g_force_ctas == 0 && k_iters < 4) ctas = 1;
  p.num_tiles = static_cast<int>(((m_tiles + ctas - 1) / ctas) * p.n_blocks);
  {
    const unsigned long long n_max = static_cast<unsigned long long>(m_tiles + 1) * p.n_blocks + 2;
    auto magic = [&](int d) -> uint32_t {
      if (d <= 1 || n_max * static_cast<unsigned long long>(d) >= (1ULL << 32)) return 0u;
      return static_cast<uint32_t>(((1ULL << 32) + d - 1) / d);
    };
    p.mg_nb = magic(p.n_blocks);
    p.mg_tx = magic(p.tiles_x);
    p.mg_ty = magic(p.tiles_y);
  }
  p.trace = g_trace_buf;
  p.span = nullptr;
  if (g_span_buf != nullptr && g_span_next < g_span_max) p.span = g_span_buf + 2 * (g_span_next++);
  p.out_f32 = a->out_dtype == CFT_DT_F32;
  // epilogue staging: a 32-column chunk is 128 rows x 64 B (bf16) or x 128 B (f32); column groups that own a single
  // bf16 chunk per tile get 8 KiB buffers, which leaves 32 KiB more for the operand ring
  p.teams = kEpiTeams;
  p.chain = chain ? 1 : 0;
  p.k2chunks = chain ? a->Cout / 64 : 0;
  p.act2 = (a->act2 == CFT_ACT_SILU && g_silu_tanh) ? 3 : a->act2;
  p.store_main = a->skip_y ? 0 : 1;
  p.bias2 = a->bias2;
  p.w2_bytes = chain ? (a->Cout / ctas) * a->Cout * 2 : 0;         // [Cout / ctas rows][Cout] bf16, a multiple of 1 KiB
  const int col_groups_h = kEpiGroups / p.teams;
  const int chunks_per_group = ((p.block_n + 31) / 32 + col_groups_h - 1) / col_groups_h;
  p.stage_c = (!p.out_f32 && chunks_per_group <= 1) ? 8 * 1024 : kStageCBytes;
  if (chain) p.stage_c = a->Cout * 128;           // 4 x stage_c = the two teams' [128 px x Cout] bf16 tiles (2 x 16 / 32 KiB)
  const int ring_budget = kSmemTotal - 1024 - kTailBytes - kEpiGroups * p.stage_c - p.w2_bytes;
  p.a_slot = p.halo ? ((p.ups * (p.TH + 2) * p.TW * p.kelems * 2 + 1023) / 1024) * 1024 : kATileBytes;
  p.b_slot = p.halo ? ((p.ups * 3 * (p.block_n / ctas) * p.kelems * 2 + 1023) / 1024) * 1024 : (p.block_n / ctas) * 128;
  // small weight matrices (3x3 convs up to 64 -> 64) stay resident in smem for the whole kernel: they were half of the
  // L2 -> SM traffic of those layers, and TMA-latency x bytes-in-flight is what bounds them
  p.b_res = 0;
  p.b_res_bytes = 0;
  if (p.halo && ctas == 1 && p.n_blocks == 1 && !g_no_bres) {
    const int bytes = kw * p.kchunks * 3 * p.block_n * p.kelems * 2;
    const int rounded = (bytes + 1023) / 1024 * 1024;
    if (rounded <= 96 * 1024 && (ring_budget - rounded) / p.a_slot >= 3) {
      p.b_res = rounded;
      p.b_res_bytes = bytes;
      p.b_slot = 0;
    }
  }
  const int stage_bytes = p.a_slot + p.b_slot;
  p.stages = (ring_budget - p.b_res) / stage_bytes;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  p.act = (a->act == CFT_ACT_SILU && g_silu_tanh) ? 3 : ((a->act == CFT_ACT_GELU && g_gelu_fast) ? 4 : a->act);
  p.ldy = a->ldy;
  p.y_coff = a->y_coff;
  p.ldr = a->ldr;
  p.r_coff = a->r_coff;
  p.bias = a->bias;
  p.y = a->y;
  p.res = a->res;

  if (g_plan_out != nullptr) {      // planning only (host tests): everything below needs the driver / a device
    cft_conv_plan* o = g_plan_out;
    o->ctas = ctas; o->TW = p.TW; o->TH = p.TH; o->TB = p.TB; o->Ho = p.Ho; o->Wo = p.Wo;
    o->tiles_x = p.tiles_x; o->tiles_y = p.tiles_y; o->m_tiles = p.m_tiles;
    o->block_n = p.block_n; o->n_blocks = p.n_blocks; o->num_tiles = p.num_tiles;
    o->kelems = p.kelems; o->kchunks = p.kchunks; o->ups = p.ups; o->halo = p.halo;
    o->stages = p.stages; o->a_slot = p.a_slot; o->b_slot = p.b_slot; o->b_res = p.b_res;
    o->acc_stages = p.acc_stages; o->acc_cols = p.acc_cols; o->teams = p.teams; o->stage_c = p.stage_c;
    o->smem_bytes = 1024 + p.stages * stage_bytes + p.b_res + p.w2_bytes + kEpiGroups * p.stage_c + kTailBytes;
    int units_p = sm_count() / ctas;
    if (units_p > p.num_tiles) units_p = p.num_tiles;
    o->grid = units_p * ctas;
    return CFT_OK;
  }
  TensorMaps maps;
  memset(&maps, 0, sizeof(maps));
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(a->x) + a->x_coff;
  const cuuint64_t eb = 2;
  int rc;
  const CUtensorMapSwizzle op_swz = p.kelems == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                                   : (p.kelems == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  if (s == 1) {
    cuuint64_t dims[4] = {(cuuint64_t)a->Cin, (cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->B};
    cuuint64_t str[3] = {(cuuint64_t)a->ldx * eb, (cuuint64_t)a->W * a->ldx * eb,
                         (cuuint64_t)a->H * a->W * a->ldx * eb};
    cuuint32_t box[4] = {(cuuint32_t)p.kelems, (cuuint32_t)p.TW, (cuuint32_t)p.TH, (cuuint32_t)p.TB};
    rc = encode_map(&maps.a[0], xb, 4, dims, str, box, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, op_swz);
    if (rc) return rc;
    maps.a[1] = maps.a[2] = maps.a[3] = maps.a[0];
    if (p.halo) {
      cuuint32_t hbox[4] = {(cuuint32_t)p.kelems, (cuuint32_t)p.TW, (cuuint32_t)(p.TH + 2), 1};
      rc = encode_map(&maps.a[1], xb, 4, dims, str, hbox, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, op_swz);
      if (rc) return rc;
    }
  } else {
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        cuuint64_t dims[4] = {(cuuint64_t)a->Cin, (cuuint64_t)(a->W / 2), (cuuint64_t)(a->H / 2), (cuuint64_t)a->B};
        cuuint64_t str[3] = {(cuuint64_t)2 * a->ldx * eb, (cuuint64_t)2 * a->W * a->ldx * eb,
                             (cuuint64_t)a->H * a->W * a->ldx * eb};
        cuuint32_t box[4] = {(cuuint32_t)p.kelems, (cuuint32_t)p.TW, (cuuint32_t)p.TH, (cuuint32_t)p.TB};
        const __nv_bfloat16* base = xb + (static_cast<size_t>(py) * a->W + px) * a->ldx;
        rc = encode_map(&maps.a[py * 2 + px], base, 4, dims, str, box, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, op_swz);
        if (rc) return rc;
      }
  }
  {
    const int cin_p = round_up(a->Cin, 8);
    cuuint64_t dims[3] = {(cuuint64_t)a->Cin, (cuuint64_t)p.taps, (cuuint64_t)a->Cout};
    cuuint64_t str[2] = {(cuuint64_t)cin_p * eb, (cuuint64_t)p.taps * cin_p * eb};
    cuuint32_t box[3] = {(cuuint32_t)p.kelems, 1, (cuuint32_t)(p.block_n / ctas)};
    rc = encode_map(&maps.b, a->w, 3, dims, str, box, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, op_swz);
    if (rc) return rc;
  }

  {
    const cuuint64_t es = p.out_f32 ? 4 : 2;
    const uint8_t* yb = reinterpret_cast<const uint8_t*>(a->y) + static_cast<size_t>(a->y_coff) * es;
    cuuint64_t dims[4] = {(cuuint64_t)a->Cout, (cuuint64_t)p.Wo, (cuuint64_t)p.Ho, (cuuint64_t)a->B};
    cuuint64_t str[3] = {(cuuint64_t)a->ldy * es, (cuuint64_t)p.Wo * a->ldy * es, (cuuint64_t)p.Ho * p.Wo * a->ldy * es};
    cuuint32_t box[4] = {chain ? 64u : 32u, (cuuint32_t)p.TW, (cuuint32_t)p.TH, (cuuint32_t)p.TB};
    const CUtensorMapSwizzle c_swz = (p.out_f32 || chain) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    rc = encode_map(&maps.c, yb, 4, dims, str, box,
                    p.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, c_swz);
    if (rc) return rc;
    if (chain) {
      const uint8_t* y2b = reinterpret_cast<const uint8_t*>(a->y2) + static_cast<size_t>(a->y2_coff) * es;
      cuuint64_t str2[3] = {(cuuint64_t)a->ldy2 * es, (cuuint64_t)p.Wo * a->ldy2 * es, (cuuint64_t)p.Ho * p.Wo * a->ldy2 * es};
      rc = encode_map(&maps.c2, y2b, 4, dims, str2, box, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, c_swz);
      if (rc) return rc;
      cuuint64_t wd[3] = {(cuuint64_t)a->Cout, 1, (cuuint64_t)a->Cout};
      cuuint64_t ws[2] = {(cuuint64_t)a->Cout * 2, (cuuint64_t)a->Cout * 2};
      cuuint32_t wb[3] = {64, 1, (cuuint32_t)(a->Cout / ctas)};
      rc = encode_map(&maps.b2, a->w2, 3, wd, ws, wb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
    }
    if (a->res) {
      const uint8_t* rb = reinterpret_cast<const uint8_t*>(a->res) + static_cast<size_t>(a->r_coff) * es;
      cuuint64_t rstr[3] = {(cuuint64_t)a->ldr * es, (cuuint64_t)p.Wo * a->ldr * es, (cuuint64_t)p.Ho * p.Wo * a->ldr * es};
      rc = encode_map(&maps.r, rb, 4, dims, rstr, box,
                      p.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, c_swz);
      if (rc) return rc;
    }
  }

  const int smem_bytes = 1024 + p.stages * stage_bytes + p.b_res + p.w2_bytes + kEpiGroups * p.stage_c + kTailBytes;
  if (!g_attr_set) {
    const int max_smem = kSmemTotal;
    rc = check_cuda(cudaFuncSetAttribute(cft_conv_tcgen05_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem),
                    "cudaFuncSetAttribute(conv_tcgen05<1>)");
    if (rc) return rc;
    rc = check_cuda(cudaFuncSetAttribute(cft_conv_tcgen05_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem),
                    "cudaFuncSetAttribute(conv_tcgen05<2>)");
    if (rc) return rc;
    g_attr_set = true;
  }
  int units = sm_count() / ctas;           // persistent: one CTA (or CTA pair) per SM (pair)
  if (units > p.num_tiles) units = p.num_tiles;
  LaunchScope ls(CFT_K_CONV_TCGEN05, stream);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(units * ctas);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int nattr = 0;
  if (ctas == 2) {
    attr[nattr].id = cudaLaunchAttributeClusterDimension;
    attr[nattr].val.clusterDim.x = 2;
    attr[nattr].val.clusterDim.y = 1;
    attr[nattr].val.clusterDim.z = 1;
    ++nattr;
  }
  if (!g_no_pdl) {   // programmatic dependent launch: this kernel's prologue overlaps the previous kernel's tail
    attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[nattr].val.programmaticStreamSerializationAllowed = 1;
    ++nattr;
  }
  cfg.attrs = attr;
  cfg.numAttrs = nattr;
  cudaError_t e = (ctas == 2) ? cudaLaunchKernelEx(&cfg, cft_conv_tcgen05_kernel<2>, maps, p)
                              : cudaLaunchKernelEx(&cfg, cft_conv_tcgen05_kernel<1>, maps, p);
  if (e != cudaSuccess) {
    ls.finish("cft_conv2d launch");
    return check_cuda(e, "cudaLaunchKernelEx(conv_tcgen05)");
  }
  return ls.finish("cft_conv2d launch");
}

// Debug timeline: `buf` (device, >= grid * 64 u64, zeroed by the caller) receives per-CTA clock samples of every
// cft_conv2d launch that follows (see trace_mark for the slot map); nullptr turns it off.  Not for production use.
extern "C" int cft_debug_conv_trace(void* buf) {
  g_trace_buf = static_cast<unsigned long long*>(buf);
  return CFT_OK;
}

// Debug: the next `max_launches` cft_conv2d launches (in issue order, also when captured into a CUDA graph) write
// {first CTA start, last CTA end} (%globaltimer ns) into buf[2 * i], buf[2 * i + 1]; the caller presets {~0, 0}.
extern "C" int cft_debug_conv_spans(void* buf, int max_launches) {
  g_span_buf = static_cast<unsigned long long*>(buf);
  g_span_next = 0;
  g_span_max = buf ? max_launches : 0;
  return CFT_OK;
}

extern "C" int cft_debug_conv_plan(const cft_conv_args* a, cft_conv_plan* plan) {
  CFT_REQUIRE(plan != nullptr, "cft_debug_conv_plan: null plan");
  memset(plan, 0, sizeof(*plan));
  g_plan_out = plan;
  const int rc = cft_conv2d(a, nullptr);
  g_plan_out = nullptr;
  return rc;
}
