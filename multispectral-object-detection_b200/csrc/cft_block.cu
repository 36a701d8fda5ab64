// The whole transformer stack of one CFT / GPT block (models/common.py:593-639, the n_layer x myTransformerBlock loop
// at :622 plus ln_f at :625; block = :516-546, attention = :475-513) as ONE kernel launch (sm_100a):
//
//   for every layer:  x += out_proj(MHSA(LN1(x)));   x += W2 GELU(W1 LN2(x) + b1) + b2;     finally  y = ln_f(x)
//
// One thread-block CLUSTER of C CTAs owns one image (its 128 x d token tile) for all layers; images are independent,
// so there is no grid-wide synchronisation, only cluster barriers.  CTA `c` of a cluster owns the DC = d / C columns
// [c*DC, (c+1)*DC) of the residual stream (fp32, in REGISTERS for the whole kernel), the heads that live in those
// columns, and the matching N-slices of all four Linear layers:
//
//   LN    row statistics: per-CTA (mean, M2) exchanged through distributed shared memory (one cluster barrier); every
//         CTA normalises its own column slice, writes it (bf16, UMMA K-major SWIZZLE_128B layout) into chunk c of its
//         resident A operand and pushes that 16 KiB chunk into the same place of every peer with a DSMEM bulk copy that
//         signals the peer's chunk mbarrier -- the all-gather never touches L2 and needs no second barrier
//   QKV   A = LN1(x) [128, d] resident; B = this CTA's q|k|v weight rows streamed by TMA; the accumulator is drained
//         (+bias, bf16) straight into UMMA-layout Q / K / V smem tiles -> attention never leaves the SM
//   attn  two local heads at a time (8 compute warps each): S = Q K^T (tcgen05), softmax out of TMEM, P -> smem,
//         O = P V (tcgen05), O / rowsum -> registers -> chunk c of the A operand, all-gathered like the LN output
//   out   A = O resident; N = DC; epilogue: x += acc + bias, then LN2
//   up    A = LN2(x) resident; N = 4 DC in passes; epilogue: +bias, erf-GELU, bf16 hidden slice -> L2
//   down  A = hidden [128, 4d] streamed by TMA through the operand slots; N = DC; epilogue: x += acc + bias, next LN1 / ln_f
//
// Warp roles (640 threads): warp 0 weight (B) producer | warp 1 MMA issuer | warp 2 streamed-A producer + TMEM
// allocator | warp 3 idle (keeps the cluster-barrier count) | warps 4-19 compute: thread (t, qd) owns token row
// t = TMEM lane t and quarter qd of every column range.
// Four cluster barriers per layer: LN1 statistics, attention finished (operand slots free), LN2 statistics, hidden
// published.  The weight producer and the MMA issuer use the split arrive / wait form, so weights of the next GEMM are
// prefetched across a barrier.
//
// Replaces 56 dependent launches per block (7 per layer: LN, QKV GEMM, attention, out-proj, LN, MLP up, MLP down).
#include <stdlib.h>

#include "cft_common.cuh"
#include "tcgen05_ptx.cuh"

namespace {
using namespace cft;
using namespace cft::ptx;

constexpr int kT = 128;                    // tokens per image (2 * 8 * 8)
constexpr int kComputeWarps = 16;
constexpr int kCompute = 32 * kComputeWarps;
constexpr int kThreads = 128 + kCompute;   // 640
constexpr int kAChunk = 16384;             // activation chunk: 128 rows x 64 k (128 B rows, SWIZZLE_128B)
constexpr int kMaxStages = 8;
constexpr int kMaxASlots = 10;
constexpr int kMaxPasses = 12;
constexpr int kTmemCols = 512;
constexpr int kSmemMax = 227 * 1024;
constexpr int kMiscFixed = 512 + 2048 + 2048;   // barriers | softmax max | softmax sum (= LN quarter partials: never live together)

struct __align__(64) BlockMaps {
  CUtensorMap w[4];               // wqkv, wo, w1, w2: box {64 k, rows}
  CUtensorMap hbuf;               // hidden, box {64 k, 128 rows}
};

// one GEMM pass = one accumulator: N weight rows (1-3 row segments) x all of K
struct Pass {
  int map, nseg, seg_rows;
  int row[3];                     // first weight row of each segment (layer 0, cluster rank 0)
  int cta_stride, layer_stride;   // row offset per cluster rank / per layer
  int n, kchunks, kpack;          // MMA N; K / 64; 64-wide K sub-tiles per ring stage
  int tcol;                       // accumulator TMEM column
  int a_mode;                     // 0: resident A, wait for its chunks | 1: resident, already waited | 2: streamed
};

struct BlockParams {
  int B, d, heads, dk, layers, C, hpc;
  int stages, stage_bytes, a_slots, ra_bytes;
  int npass_qkv, npass_up, npass_max;   // passes[0..nq) QKV, [nq] out, [nq+1 .. nq+1+nu) up, [nq+1+nu] down
  Pass passes[kMaxPasses];
  int cw, nch, layout, rowB;      // attention tiles: chunk width (elements), chunks per head, UMMA layout code, row bytes
  int p_off;                      // byte offset of the P tiles inside the operand region (dk < 64), -1: P aliases Q|K
  float scale_log2e, eps1, eps2, epsf;
  const float *bqkv, *bo, *b1, *b2, *ln1g, *ln1b, *ln2g, *ln2b, *lnfg, *lnfb;
  const float* x_in;
  float* x_out;
  const __nv_bfloat16 *wqkv, *wo, *w1, *w2;   // raw weight pointers (L2 prefetch of the next layer)
  __nv_bfloat16* hbuf;            // [B*128][4d]
  float* dbg;                     // optional [layers][B][128][d] dump of x after every layer
  unsigned long long* trace;      // debug (cft_debug_block_trace): [grid][layers][48] clock64 samples: 0-15 compute warp 0, 16+3i.. MMA issuer pass i {start, first operands landed, last MMA issued}
};

// one 16-byte store of 8 bf16 (a plain struct copy is split into four 4-byte stores by the compiler)
__device__ __forceinline__ void st16(void* dst, const float* f) {
  const bf16x8 pk = pack8(f);
  *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(&pk);
}

struct Ring {
  int stage;
  uint32_t phase;
};
__device__ __forceinline__ void ring_advance(Ring& r, int stages) {
  if (++r.stage == stages) {
    r.stage = 0;
    r.phase ^= 1u;
  }
}

// ------------------------------------------------------------------ the kernel
template <int DC, int HP>      // columns per CTA; head PAIRS per CTA
__global__ void __launch_bounds__(kThreads, 1)
cft_gpt_block_kernel(const __grid_constant__ BlockMaps maps, const __grid_constant__ BlockParams p) {
  constexpr int NC = DC / 4;                       // residual-stream columns per compute thread
  constexpr int TB = kT * DC * 2;                  // bytes of this CTA's Q (or K, or V) tiles, all local heads
  constexpr int OWN = DC / 64;                     // A-operand chunks this CTA produces

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* RA = smem;                                          // resident A operand | Q,K,V,P tiles | streamed A slots
  uint8_t* ring = RA + p.ra_bytes;                             // weight stages
  uint8_t* misc = ring + p.stages * p.stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc);
  uint64_t* bfull = bars;                                      // [8]
  uint64_t* bempty = bfull + kMaxStages;                       // [8]
  uint64_t* afull = bempty + kMaxStages;                       // [10]
  uint64_t* aempty = afull + kMaxASlots;                       // [10]
  uint64_t* acc_bar = aempty + kMaxASlots;                     // [4]  GEMM accumulators (round robin: <= 4 passes in flight)
  uint64_t* tiles_bar = acc_bar + 4;                           // [1]  Q, K, V tiles written
  uint64_t* p_bar = tiles_bar + 1;                             // [2]  P of group g written (S consumed)
  uint64_t* s_bar = p_bar + 2;                                 // [2]  S of group g ready
  uint64_t* o_bar = s_bar + 2;                                 // [2]  O of group g ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_bar + 2);
  float* smax = reinterpret_cast<float*>(misc + 512);          // [4][128]  (group * 2 + half)
  float* ssum = smax + 4 * kT;                                 // [4][128]
  float2* part = reinterpret_cast<float2*>(misc + 512);            // [4][128] LayerNorm partials of the column quarters (aliases smax | ssum)
  float2* stats = part + 4 * kT;                               // [2][C][128] per-CTA partial (mean, M2) of its DC columns
  float* lpar = reinterpret_cast<float*>(stats + 2 * p.C * kT);  // [13 DC] this layer's biases / LN parameters of the CTA's columns

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = p.C, d = p.d;
  const int rank = static_cast<int>(cluster_ctarank());
  const int cluster_id = blockIdx.x / C, n_clusters = gridDim.x / C;
  const int kch_d = d / 64;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) prefetch_tmap(&maps.w[i]);
    prefetch_tmap(&maps.hbuf);
    for (int i = 0; i < kMaxStages; ++i) {
      mbar_init(&bfull[i], 1);
      mbar_init(&bempty[i], 1);
    }
    for (int i = 0; i < kMaxASlots; ++i) {
      mbar_init(&afull[i], 1);
      mbar_init(&aempty[i], p.C);      // streamed chunks are multicast: every CTA of the cluster frees the slot
    }
    for (int i = 0; i < 4; ++i) mbar_init(&acc_bar[i], 1);
    mbar_init(tiles_bar, kComputeWarps);
    for (int g = 0; g < 2; ++g) {
      mbar_init(&p_bar[g], kComputeWarps / 2);
      mbar_init(&s_bar[g], 1);
      mbar_init(&o_bar[g], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  // peers write into this CTA's shared memory (LN partials, operand chunks): nobody may run ahead of a CTA that has
  // not initialised its barriers yet
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();      // (no early launch_dependents: a dependent kernel must not take SMs from clusters still to be scheduled)

  const int cpi = 1 + 4 * p.layers;               // cluster barriers per image
  const int n_passes = p.npass_qkv + p.npass_up + 2;

  if (warp == 0) {
    // ===================================================== weight (B) producer
    Ring r{0, 0u};
    bool pend = false;
    auto sp = [&]() {
      if (pend) cluster_wait_acquire();
      cluster_arrive_release();
      pend = true;
    };
    for (int b = cluster_id; b < p.B; b += n_clusters) {
      sp();
      for (int l = 0; l < p.layers; ++l) {
        for (int pi = 0; pi < n_passes; ++pi) {
          const Pass& ps = p.passes[pi];
          const CUtensorMap* map = &maps.w[ps.map];
          const int row_off = rank * ps.cta_stride + l * ps.layer_stride;
          const uint32_t sub_bytes = static_cast<uint32_t>(ps.n) * 128u;
          const uint32_t tx = sub_bytes * static_cast<uint32_t>(ps.kpack);
          for (int s = 0; s < ps.kchunks / ps.kpack; ++s) {
            mbar_wait(&bempty[r.stage], r.phase ^ 1u);
            if (elect_one_sync()) {
              uint8_t* dst = ring + r.stage * p.stage_bytes;
              mbar_arrive_expect_tx(&bfull[r.stage], tx);
              for (int j = 0; j < ps.kpack; ++j)
                for (int sg = 0; sg < ps.nseg; ++sg)
                  tma_load_2d(dst + j * sub_bytes + sg * ps.seg_rows * 128, map, &bfull[r.stage], (s * ps.kpack + j) * 64,
                              ps.row[sg] + row_off);
            }
            __syncwarp();
            ring_advance(r, p.stages);
          }
          // barriers that follow this pass in program order: after QKV (#A), out (#B), the last up pass (#D), down (#E)
          if (pi == p.npass_qkv - 1 || pi == p.npass_qkv || pi == p.npass_qkv + p.npass_up || pi == n_passes - 1) sp();
        }
      }
    }
    if (pend) cluster_wait_acquire();
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    Ring r{0, 0u};
    uint32_t a_par = 0u, ev = 0u;
    uint32_t tiles_n = 0u, pair_n = 0u;
    bool pend = false;
    auto sp = [&]() {
      if (pend) cluster_wait_acquire();
      cluster_arrive_release();
      pend = true;
    };
    const uint32_t ra_addr = smem_u32(RA), ring_addr = smem_u32(ring);
    const uint32_t tile_b = static_cast<uint32_t>(kT * p.dk * 2);           // one head's Q (or K, V) tile
    const uint32_t rowB = static_cast<uint32_t>(p.rowB);
    const uint32_t chunk_b = static_cast<uint32_t>(kT) * rowB;
    const uint32_t idesc_s = umma_idesc_ex(128, 128, 0, 0);
    const uint32_t idesc_o = umma_idesc_ex(128, static_cast<uint32_t>(p.dk), 0, 1);
    constexpr uint32_t op_hi = (1024u >> 4) | (1u << 14) | (2u << 29);      // SBO 1024 B, SWIZZLE_128B
    auto issue_s = [&](int h, int g) {        // S(h) -> TMEM columns [384 - 128 g, +128)
      if (elect_one_sync()) {
        const uint32_t q0 = ra_addr + static_cast<uint32_t>(h) * 2u * tile_b, k0 = q0 + tile_b;
        int kk = 0;
        for (int ci = 0; ci < p.nch; ++ci)
          for (int k = 0; k < p.cw / 16; ++k, ++kk) {
            const uint64_t da = umma_desc(q0 + ci * chunk_b + k * 32, 0, 8u * rowB, p.layout);
            const uint64_t db = umma_desc(k0 + ci * chunk_b + k * 32, 0, 8u * rowB, p.layout);
            umma_bf16(tmem_base + 384u - 128u * g, da, db, idesc_s, kk > 0 ? 1u : 0u);
          }
        umma_commit(&s_bar[g]);
      }
      __syncwarp();
    };
    auto issue_pv = [&](int h, int g) {       // O(h) -> TMEM columns [128 g, +dk)
      if (elect_one_sync()) {
        const uint32_t v0 = ra_addr + 2u * TB + static_cast<uint32_t>(h) * tile_b;
        const uint32_t p0 = p.p_off >= 0 ? ra_addr + static_cast<uint32_t>(p.p_off) + static_cast<uint32_t>(g) * (kT * 256)
                                         : ra_addr + static_cast<uint32_t>(h) * 2u * tile_b;
        for (int k = 0; k < kT / 16; ++k) {
          const uint64_t da = umma_desc(p0 + (k >> 2) * (kT * 128) + (k & 3) * 32, 0, 1024, 2);
          const uint64_t db = umma_desc(v0 + k * 16 * rowB, chunk_b, 8u * rowB, p.layout);
          umma_bf16(tmem_base + 128u * g, da, db, idesc_o, k > 0 ? 1u : 0u);
        }
        umma_commit(&o_bar[g]);
      }
      __syncwarp();
    };
    int tr_l = 0, tr_pass = 0;
    auto mmark = [&](int which) {
      if (p.trace != nullptr && lane == 0 && tr_pass < 10)
        p.trace[(static_cast<size_t>(blockIdx.x) * p.layers + tr_l) * 48 + 16 + 3 * tr_pass + which] = static_cast<unsigned long long>(clock64());
    };
    auto gemm = [&](const Pass& ps) {
      uint64_t* ab = &acc_bar[ev & 3u];
      ++ev;
      mmark(0);
      const uint32_t idesc = umma_idesc_ex(128u, static_cast<uint32_t>(ps.n), 0, 0);
      const uint32_t sub16 = (static_cast<uint32_t>(ps.n) * 128u) >> 4;
      const int n_stage = ps.kchunks / ps.kpack;
      for (int s = 0; s < n_stage; ++s) {
        mbar_wait(&bfull[r.stage], r.phase);
        const uint32_t b_lo0 = (ring_addr + static_cast<uint32_t>(r.stage) * p.stage_bytes) >> 4;
        for (int j = 0; j < ps.kpack; ++j) {
          const int chunk = s * ps.kpack + j;
          const int slot = ps.a_mode == 2 ? chunk % p.a_slots : chunk;
          if (ps.a_mode != 1) {
            mbar_wait(&afull[slot], (a_par >> slot) & 1u);
            a_par ^= 1u << slot;
          }
          tc_fence_after();
          if (s == 0 && j == 0) mmark(1);
          if (elect_one_sync()) {
            const uint32_t a_lo = (ra_addr + static_cast<uint32_t>(slot) * kAChunk) >> 4;
            const uint32_t b_lo = b_lo0 + static_cast<uint32_t>(j) * sub16;
#pragma unroll
            for (int k = 0; k < 4; ++k) {          // four K = 16 steps per 64-wide chunk (+32 B inside the swizzle atom)
              const uint64_t da = (static_cast<uint64_t>(op_hi) << 32) | ((a_lo + 2u * k) & 0x3FFFu);
              const uint64_t db = (static_cast<uint64_t>(op_hi) << 32) | ((b_lo + 2u * k) & 0x3FFFu);
              umma_bf16(tmem_base + static_cast<uint32_t>(ps.tcol), da, db, idesc, (chunk | k) != 0 ? 1u : 0u);
            }
            if (ps.a_mode == 2) umma_commit_mc(&aempty[slot], static_cast<uint16_t>((1u << p.C) - 1u));
            if (j == ps.kpack - 1) {
              umma_commit(&bempty[r.stage]);
              if (s == n_stage - 1) umma_commit(ab);
            }
          }
          __syncwarp();
        }
        ring_advance(r, p.stages);
      }
      mmark(2);
      ++tr_pass;
    };
    for (int b = cluster_id; b < p.B; b += n_clusters) {
      sp();
      for (int l = 0; l < p.layers; ++l) {
        tr_l = l;
        tr_pass = 0;
        int pi = 0;
        for (; pi < p.npass_qkv; ++pi) gemm(p.passes[pi]);
        // attention, two heads at a time (group g = the compute warps that own the head)
        mbar_wait(tiles_bar, (tiles_n++) & 1u);          // Q, K, V tiles written
        tc_fence_after();
        for (int pr = 0; pr < HP; ++pr) {
          issue_s(2 * pr, 0);
          issue_s(2 * pr + 1, 1);
          for (int g = 0; g < 2; ++g) {
            mbar_wait(&p_bar[g], pair_n & 1u);           // P written, S consumed, O of the previous pair read out
            tc_fence_after();
            issue_pv(2 * pr + g, g);
          }
          ++pair_n;
        }
        sp();                                            // #A
        gemm(p.passes[pi++]);                            // out-proj
        sp();                                            // #B
        for (int u = 0; u < p.npass_up; ++u) gemm(p.passes[pi++]);
        sp();                                            // #D
        gemm(p.passes[pi++]);                            // down-proj, A streamed
        sp();                                            // #E
      }
    }
    if (pend) cluster_wait_acquire();
  } else if (warp == 2) {
    // ===================================================== streamed-A producer (hidden -> operand slots)
    uint32_t e_par = 0u;
    auto cb = [&]() {
      cluster_arrive_release();
      cluster_wait_acquire();
    };
    for (int b = cluster_id; b < p.B; b += n_clusters) {
      cb();
      for (int l = 0; l < p.layers; ++l) {
        cb();                                 // #A
        cb();                                 // #B
        cb();                                 // #D: hidden published
        for (int ch = 0; ch < 4 * kch_d; ++ch) {
          const int slot = ch % p.a_slots;
          mbar_wait(&aempty[slot], ((e_par >> slot) & 1u) ^ 1u);
          e_par ^= 1u << slot;
          if (elect_one_sync()) {
            // all C CTAs stream the same image's hidden: chunk ch is fetched once, by CTA ch % C, and multicast
            if (ch == 0) fence_proxy_async_all();
            mbar_arrive_expect_tx(&afull[slot], kAChunk);
            if (ch % C == rank)
              tma_load_2d_mc(RA + slot * kAChunk, &maps.hbuf, &afull[slot], ch * 64, b * kT, static_cast<uint16_t>((1u << C) - 1u));
          }
          __syncwarp();
        }
        cb();                                 // #E
      }
    }
  } else if (warp == 3) {
    // ===================================================== L2 prefetcher: the weight slices this CTA streams in layer l + 1
    // are requested while layer l computes (the forward touches GBs between two uses of a block's weights: L2 is cold)
    auto cb = [&]() {
      cluster_arrive_release();
      cluster_wait_acquire();
    };
    auto prefetch_layer = [&](int l) {
      if (elect_one_sync()) {
        const size_t dd = static_cast<size_t>(d);
        for (int part = 0; part < 3; ++part)
          prefetch_l2_bulk(p.wqkv + (static_cast<size_t>(l) * 3 * d + part * d + rank * DC) * dd, static_cast<uint32_t>(DC * d * 2));
        prefetch_l2_bulk(p.wo + (static_cast<size_t>(l) * d + rank * DC) * dd, static_cast<uint32_t>(DC * d * 2));
        prefetch_l2_bulk(p.w1 + (static_cast<size_t>(l) * 4 * d + rank * 4 * DC) * dd, static_cast<uint32_t>(4 * DC * d * 2));
        prefetch_l2_bulk(p.w2 + (static_cast<size_t>(l) * d + rank * DC) * 4 * dd, static_cast<uint32_t>(DC * 4 * d * 2));
      }
      __syncwarp();
    };
    bool first = true;
    for (int b = cluster_id; b < p.B; b += n_clusters) {
      if (first) prefetch_layer(0);
      cb();
      for (int l = 0; l < p.layers; ++l) {
        if (first && l + 1 < p.layers) prefetch_layer(l + 1);     // later images of this cluster find the block's weights in L2
        cb();
        cb();
        cb();
        cb();
      }
      first = false;
    }
  } else {
    // ===================================================== compute warps: thread (t, qd)
    const int q = warp & 3;                 // TMEM lane quarter
    const int qd = (warp - 4) >> 2;         // column quarter
    const int grp = qd >> 1, hh = qd & 1;   // attention: head group, half of the head's columns / keys
    const int t = q * 32 + lane;            // token row
    const int ctid = threadIdx.x - 128;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const int col0 = rank * DC + qd * NC;   // first residual-stream column of this thread
    const int dk = p.dk, rowB = p.rowB, cw = p.cw;
    const int swz = p.layout == 2 ? (t & 7) : (p.layout == 4 ? ((t >> 1) & 3) : ((t >> 2) & 1));
    const int tile_b = kT * dk * 2;
    uint32_t ev = 0u, pair_n = 0u, sbuf = 0u;
    float xv[NC];
    int cur_l = 0;
    auto mark = [&](int slot) {
      if (p.trace != nullptr && warp == 4 && lane == 0)
        p.trace[(static_cast<size_t>(blockIdx.x) * p.layers + cur_l) * 48 + slot] = static_cast<unsigned long long>(clock64());
    };
    auto acc_wait = [&]() {
      mbar_wait(&acc_bar[ev & 3u], (ev >> 2) & 1u);
      ++ev;
      tc_fence_after();
    };
    auto cb = [&]() {
      cluster_arrive_release();
      cluster_wait_acquire();
    };
    // own-chunk address of (row t, column c of this CTA's slice): K-major SWIZZLE_128B chunk layout
    auto own_chunk_ptr = [&](int c) -> uint8_t* {
      return RA + (rank * OWN + (c >> 6)) * kAChunk + t * 128 + ((((c & 63) >> 3) ^ (t & 7)) << 4);
    };
    // Called by all compute threads right after a cluster barrier that guarantees every CTA's operand slots are free.
    auto arm_chunks = [&]() {
      if (ctid == 0)
        for (int j = 0; j < kch_d; ++j)
          if (j / OWN != rank) mbar_arrive_expect_tx(&afull[j], kAChunk);
    };
    // This CTA's chunk(s) are written: hand them to the local MMA issuer and push them into every peer.
    auto publish_chunks = [&]() {
      fence_proxy_async();
      named_bar_sync(3, kCompute);
      if (ctid == 0) {
        for (int o = 0; o < OWN; ++o) {
          const int j = rank * OWN + o;
          mbar_arrive(&afull[j]);
          const uint32_t src = smem_u32(RA + j * kAChunk), bar = smem_u32(&afull[j]);
          for (int r = 0; r < C; ++r)
            if (r != rank) bulk_copy_s2c(mapa_u32(src, static_cast<uint32_t>(r)), src, kAChunk, mapa_u32(bar, static_cast<uint32_t>(r)));
        }
      }
    };
    // LayerNorm of the cluster-distributed rows.  dst_f32 == null: the normalised slice becomes the next A operand.
    // Row statistics are (mean, M2 = sum of squared deviations) at every level -- two passes over the thread's registers,
    // then Chan's merge of equal counts, M2 = sum M2_i + n * sum (mean_i - mean)^2.  The one-pass Q / d - mean^2 cancels
    // catastrophically in fp32 once |mean| / std passes ~10 (rstd off by 1e-3 at 100, by 10 % at 1000).
    auto ln_step = [&](const float* gamma, const float* beta, float eps, float* dst_f32, int mk) {
      float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;      // two independent chains per pass
#pragma unroll
      for (int i = 0; i < NC; i += 2) {
        s0 += xv[i];
        s1 += xv[i + 1];
      }
      const float m = (s0 + s1) * (1.0f / NC);
#pragma unroll
      for (int i = 0; i < NC; i += 2) {
        const float e0 = xv[i] - m, e1 = xv[i + 1] - m;
        q0 = fmaf(e0, e0, q0);
        q1 = fmaf(e1, e1, q1);
      }
      part[qd * kT + t] = make_float2(m, q0 + q1);
      // gamma / beta of this thread's columns: issue the loads before the barriers
      float4 gg[NC / 4], bb[NC / 4];
#pragma unroll
      for (int i = 0; i < NC / 4; ++i) {
        gg[i] = reinterpret_cast<const float4*>(gamma)[i];      // global (first LN of an image) or staged in smem
        bb[i] = reinterpret_cast<const float4*>(beta)[i];
      }
      named_bar_sync(3, kCompute);
      if (qd == 0) {
        const float2 a0 = part[t], a1 = part[kT + t], a2 = part[2 * kT + t], a3 = part[3 * kT + t];
        const float cm = ((a0.x + a1.x) + (a2.x + a3.x)) * 0.25f;
        const float e0 = a0.x - cm, e1 = a1.x - cm, e2 = a2.x - cm, e3 = a3.x - cm;
        const float cq = ((a0.y + a1.y) + (a2.y + a3.y)) + static_cast<float>(NC) * ((e0 * e0 + e1 * e1) + (e2 * e2 + e3 * e3));
        const uint32_t laddr = smem_u32(&stats[(sbuf * C + rank) * kT + t]);
        for (int r = 0; r < C; ++r) st_cluster_v2f32(mapa_u32(laddr, static_cast<uint32_t>(r)), cm, cq);
      }
      cb();
      mark(mk);
      if (dst_f32 == nullptr) arm_chunks();
      const float2* st = stats + sbuf * C * kT + t;
      float S = 0.f;
      for (int j = 0; j < C; ++j) S += st[j * kT].x;
      const float inv_d = 1.0f / static_cast<float>(d);
      const float mean = S * (static_cast<float>(DC) * inv_d);      // the mean of C equal-count means
      float Q = 0.f, D = 0.f;
      for (int j = 0; j < C; ++j) {
        const float2 v = st[j * kT];
        const float e = v.x - mean;
        Q += v.y;
        D = fmaf(e, e, D);
      }
      sbuf ^= 1u;
      const float var = fmaf(static_cast<float>(DC), D, Q) * inv_d;
      const float rstd = rsqrtf(var + eps);
#pragma unroll
      for (int i = 0; i < NC; i += 8) {
        float f[8];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const float4 g4 = gg[(i >> 2) + j], b4 = bb[(i >> 2) + j];
          f[4 * j + 0] = (xv[i + 4 * j + 0] - mean) * rstd * g4.x + b4.x;
          f[4 * j + 1] = (xv[i + 4 * j + 1] - mean) * rstd * g4.y + b4.y;
          f[4 * j + 2] = (xv[i + 4 * j + 2] - mean) * rstd * g4.z + b4.z;
          f[4 * j + 3] = (xv[i + 4 * j + 3] - mean) * rstd * g4.w + b4.w;
        }
        if (dst_f32 == nullptr) {
          st16(own_chunk_ptr(qd * NC + i), f);
        } else {
          *reinterpret_cast<float4*>(dst_f32 + i) = make_float4(f[0], f[1], f[2], f[3]);
          *reinterpret_cast<float4*>(dst_f32 + i + 4) = make_float4(f[4], f[5], f[6], f[7]);
        }
      }
      if (dst_f32 == nullptr) publish_chunks();
      mark(mk + 1);
    };
    // x += accumulator + bias  (out-proj / down-proj epilogue; accumulator columns [0, DC))
    auto residual_epilogue = [&](const float* bias, int mk) {
      float4 bv[NC / 4];
#pragma unroll
      for (int i = 0; i < NC / 4; ++i) bv[i] = reinterpret_cast<const float4*>(bias)[i];
      acc_wait();
      mark(mk);
#pragma unroll
      for (int c0 = 0; c0 < NC; c0 += 16) {
        uint32_t v[16];
        tmem_ld16_nowait(tmem_base + lane_addr + static_cast<uint32_t>(qd * NC + c0), v);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 b4 = bv[(c0 >> 2) + i];
          xv[c0 + 4 * i + 0] += __uint_as_float(v[4 * i + 0]) + b4.x;
          xv[c0 + 4 * i + 1] += __uint_as_float(v[4 * i + 1]) + b4.y;
          xv[c0 + 4 * i + 2] += __uint_as_float(v[4 * i + 2]) + b4.z;
          xv[c0 + 4 * i + 3] += __uint_as_float(v[4 * i + 3]) + b4.w;
        }
      }
      tc_fence_before();
      mark(mk + 1);
    };

    for (int b = cluster_id; b < p.B; b += n_clusters) {
      const size_t row = static_cast<size_t>(b) * kT + t;
      {
        const float4* xin = reinterpret_cast<const float4*>(p.x_in + row * d + col0);
#pragma unroll
        for (int i = 0; i < NC / 4; ++i) {
          const float4 v = xin[i];
          xv[4 * i + 0] = v.x;
          xv[4 * i + 1] = v.y;
          xv[4 * i + 2] = v.z;
          xv[4 * i + 3] = v.w;
        }
      }
      ln_step(p.ln1g + col0, p.ln1b + col0, p.eps1, nullptr, 14);

      for (int l = 0; l < p.layers; ++l) {
        cur_l = l;
        mark(0);
        // this layer's biases and LayerNorm parameters (this CTA's columns) -> smem, while the QKV MMAs run:
        // [0,3DC) bqkv | [3DC,4DC) bo | [4DC,8DC) b1 | [8DC,9DC) b2 | [9DC,11DC) LN2 gamma, beta | [11DC,13DC) next LN gamma, beta
        for (int i = ctid; i < 13 * DC; i += kCompute) {
          const int seg = i / DC, m = i - seg * DC;
          const bool last = l + 1 == p.layers;
          const float* src;
          if (seg < 3) src = p.bqkv + l * 3 * d + seg * d + rank * DC + m;
          else if (seg == 3) src = p.bo + l * d + rank * DC + m;
          else if (seg < 8) src = p.b1 + l * 4 * d + rank * 4 * DC + (seg - 4) * DC + m;
          else if (seg == 8) src = p.b2 + l * d + rank * DC + m;
          else if (seg == 9) src = p.ln2g + l * d + rank * DC + m;
          else if (seg == 10) src = p.ln2b + l * d + rank * DC + m;
          else if (seg == 11) src = (last ? p.lnfg : p.ln1g + (l + 1) * d) + rank * DC + m;
          else src = (last ? p.lnfb : p.ln1b + (l + 1) * d) + rank * DC + m;
          lpar[i] = __ldg(src);
        }
        named_bar_sync(3, kCompute);
        // ---------------- QKV accumulator -> Q / K / V operand tiles (they overwrite the dead LN1(x) operand)
        for (int z = 0; z < p.npass_qkv; ++z) acc_wait();
        mark(1);
        {
#pragma unroll 1
          for (int z = 0; z < p.npass_qkv; ++z) {
            const int n = p.passes[z].n, g0 = p.passes[z].tcol;    // first q|k|v column of the pass = its TMEM column
#pragma unroll 1
            for (int c0 = qd * (n >> 2); c0 < (qd + 1) * (n >> 2); c0 += 16) {
              const int g = g0 + c0;                               // column within this CTA's [q | k | v], multiple of 16
              uint32_t v[16];
              tmem_ld16_nowait(tmem_base + lane_addr + static_cast<uint32_t>(g), v);
              const int pt = g / DC, m0 = g - pt * DC;
              const float4* b4 = reinterpret_cast<const float4*>(lpar + g);
              const float4 bA = b4[0], bB = b4[1], bC = b4[2], bD = b4[3];
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const float4 b0 = j == 0 ? bA : bC, b1 = j == 0 ? bB : bD;
                float f[8];
                f[0] = __uint_as_float(v[8 * j + 0]) + b0.x;
                f[1] = __uint_as_float(v[8 * j + 1]) + b0.y;
                f[2] = __uint_as_float(v[8 * j + 2]) + b0.z;
                f[3] = __uint_as_float(v[8 * j + 3]) + b0.w;
                f[4] = __uint_as_float(v[8 * j + 4]) + b1.x;
                f[5] = __uint_as_float(v[8 * j + 5]) + b1.y;
                f[6] = __uint_as_float(v[8 * j + 6]) + b1.z;
                f[7] = __uint_as_float(v[8 * j + 7]) + b1.w;
                const int m = m0 + 8 * j;
                const int head = m / dk, e = m - head * dk;
                const int ci = e / cw, ec = e - ci * cw;
                // Q(h) | K(h) interleaved per head, then the V tiles
                uint8_t* tile = pt == 2 ? RA + 2 * TB + head * tile_b : RA + head * 2 * tile_b + pt * tile_b;
                st16(tile + ci * (kT * rowB) + t * rowB + (((ec >> 3) ^ swz) << 4), f);
              }
            }
          }
        }
        fence_proxy_async();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tiles_bar);
        mark(2);

        // ---------------- attention: this thread's group handles head 2 pr + grp of every pair
        uint4 opk[HP][4];                                   // O / rowsum of this thread, bf16 packed (<= 32 values a pair)
#pragma unroll
        for (int pr = 0; pr < HP; ++pr) {
          const int h = 2 * pr + grp;
          const uint32_t par = pair_n & 1u;
          ++pair_n;
          mbar_wait(&s_bar[grp], par);                 // S(h)
          tc_fence_after();
          float sum = 0.f;
          {
            uint32_t v0[16], v1[16], v2[16], v3[16];
            const uint32_t s_addr = tmem_base + lane_addr + 384u - 128u * grp + static_cast<uint32_t>(hh * 64);
            tmem_ld16_nowait(s_addr, v0);
            tmem_ld16_nowait(s_addr + 16, v1);
            tmem_ld16_nowait(s_addr + 32, v2);
            tmem_ld16_nowait(s_addr + 48, v3);
            tmem_wait_ld();
            float mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < 16; ++i)
              mx = fmaxf(fmaxf(mx, fmaxf(__uint_as_float(v0[i]), __uint_as_float(v1[i]))),
                         fmaxf(__uint_as_float(v2[i]), __uint_as_float(v3[i])));
            smax[(grp * 2 + hh) * kT + t] = mx;
            named_bar_sync(1 + grp, kCompute / 2);
            mx = fmaxf(mx, smax[(grp * 2 + (hh ^ 1)) * kT + t]);
            const float mxs = mx * p.scale_log2e;
            uint8_t* ptile = p.p_off >= 0 ? RA + p.p_off + grp * (kT * 256) : RA + h * 2 * tile_b;
            uint8_t* prow = ptile + hh * (kT * 128) + t * 128;           // P chunk hh (64 keys), row = query
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float f[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const uint32_t raw = j < 2 ? v0[8 * j + i] : (j < 4 ? v1[8 * (j - 2) + i] : (j < 6 ? v2[8 * (j - 4) + i] : v3[8 * (j - 6) + i]));
                const float e = exp2f(fmaf(__uint_as_float(raw), p.scale_log2e, -mxs));
                f[i] = __bfloat162float(__float2bfloat16_rn(e));
                sum += f[i];                               // normalise by what the MMA will see
              }
              st16(prow + ((j ^ (t & 7)) << 4), f);
            }
            ssum[(grp * 2 + hh) * kT + t] = sum;
          }
          fence_proxy_async();
          tc_fence_before();
          named_bar_sync(1 + grp, kCompute / 2);          // partner's row sum visible; all S reads of the group retired
          if (lane == 0) mbar_arrive(&p_bar[grp]);
          mbar_wait(&o_bar[grp], par);                 // O(h)
          tc_fence_after();
          const float inv = 1.0f / (ssum[(grp * 2) * kT + t] + ssum[(grp * 2 + 1) * kT + t]);
          const uint32_t o_addr = tmem_base + lane_addr + 128u * grp;
          if (dk >= 64) {                              // this thread: columns [hh dk/2, +dk/2) of O: 32 of them (dk = 64)
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 16) {
              uint32_t v[16];
              tmem_ld16_nowait(o_addr + static_cast<uint32_t>(hh * (dk / 2) + c0), v);
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                float f[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[8 * j + i]) * inv;
                const bf16x8 pk = pack8(f);
                opk[pr][(c0 >> 3) + j] = *reinterpret_cast<const uint4*>(&pk);
              }
            }
          } else {                                     // dk = 16 / 32: pieces of 8 columns out of one 16-column load
            uint32_t v[16];
            tmem_ld16_nowait(o_addr + static_cast<uint32_t>((hh * (dk / 2)) & ~15), v);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              float f[8];
              const int src = dk == 16 ? hh : j;       // dk 16: piece hh of the load; dk 32: both pieces
#pragma unroll
              for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(src == 0 ? v[i] : v[8 + i]) * inv;
              const bf16x8 pk = pack8(f);
              opk[pr][j] = *reinterpret_cast<const uint4*>(&pk);
            }
          }
          tc_fence_before();
        }
        mark(3);
        cb();                                          // #A: every CTA has finished attention -> operand slots free
        arm_chunks();
#pragma unroll
        for (int pr = 0; pr < HP; ++pr) {
          const int cbase = (2 * pr + grp) * dk + hh * (dk / 2);       // column of this CTA's slice
          const int npiece = dk >= 64 ? 4 : (dk / 16);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < npiece) *reinterpret_cast<uint4*>(own_chunk_ptr(cbase + 8 * j)) = opk[pr][j];
        }
        publish_chunks();
        mark(4);

        // ---------------- out-proj epilogue + LN2
        residual_epilogue(lpar + 3 * DC + qd * NC, 5);
        ln_step(lpar + 9 * DC + qd * NC, lpar + 10 * DC + qd * NC, p.eps2, nullptr, 7);       // #B

        // ---------------- MLP up: +bias, erf-GELU -> hidden slice
        {
          const int np = p.npass_max;                           // columns per pass
          __nv_bfloat16* hrow = p.hbuf + row * (4 * d) + rank * 4 * DC + qd * (np >> 2);
          const float* b1 = lpar + 4 * DC + qd * (np >> 2);
#pragma unroll 1
          for (int u = 0; u < p.npass_up; ++u) {
            acc_wait();
            if (u == 0) mark(9);
#pragma unroll 1
            for (int c0 = 0; c0 < (np >> 2); c0 += 16) {
              uint32_t v[16];
              tmem_ld16_nowait(tmem_base + lane_addr + static_cast<uint32_t>(u * np + qd * (np >> 2) + c0), v);
              const float4* b4 = reinterpret_cast<const float4*>(b1 + u * np + c0);
              const float4 bA = b4[0], bB = b4[1], bC = b4[2], bD = b4[3];
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const float4 b0 = j == 0 ? bA : bC, bb1 = j == 0 ? bB : bD;
                float f[8];
                f[0] = gelu_fast(__uint_as_float(v[8 * j + 0]) + b0.x);
                f[1] = gelu_fast(__uint_as_float(v[8 * j + 1]) + b0.y);
                f[2] = gelu_fast(__uint_as_float(v[8 * j + 2]) + b0.z);
                f[3] = gelu_fast(__uint_as_float(v[8 * j + 3]) + b0.w);
                f[4] = gelu_fast(__uint_as_float(v[8 * j + 4]) + bb1.x);
                f[5] = gelu_fast(__uint_as_float(v[8 * j + 5]) + bb1.y);
                f[6] = gelu_fast(__uint_as_float(v[8 * j + 6]) + bb1.z);
                f[7] = gelu_fast(__uint_as_float(v[8 * j + 7]) + bb1.w);
                st16(hrow + u * np + c0 + 8 * j, f);
              }
            }
          }
          tc_fence_before();
        }
        mark(10);
        fence_proxy_async_all();
        cb();                                                    // #D: hidden published
        mark(11);

        // ---------------- down-proj epilogue + next LN1 / ln_f
        residual_epilogue(lpar + 8 * DC + qd * NC, 12);
        if (p.dbg != nullptr) {
          float* dp = p.dbg + ((static_cast<size_t>(l) * p.B * kT) + row) * d + col0;
#pragma unroll
          for (int i = 0; i < NC; ++i) dp[i] = xv[i];
        }
        if (l + 1 < p.layers)
          ln_step(lpar + 11 * DC + qd * NC, lpar + 12 * DC + qd * NC, p.eps1, nullptr, 14);    // #E
        else
          ln_step(lpar + 11 * DC + qd * NC, lpar + 12 * DC + qd * NC, p.epsf, p.x_out + row * d + col0, 14);   // #E
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();          // no CTA leaves while a peer may still address its shared memory
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
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

int encode2d(CUtensorMap* m, const void* base, long long cols, long long rows, int box_cols, int box_rows,
             const char* what) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return CFT_E_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t str[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, str, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(%s: %lld x %lld, box %d x %d) failed (CUresult %d)", what, rows, cols, box_rows,
              box_cols, (int)r);
    return CFT_E_CUDA;
  }
  return CFT_OK;
}

struct Plan {
  int C, DC, hpc, ra_bytes, a_slots, stages, stage_bytes, npass_max, p_off, smem;
};

// Cluster size for (B, d): DC = d / C must be 64 or 128, every CTA gets 2 or 4 heads (they are processed in pairs).
// Prefer the widest split whose B clusters fit on the GPU at once (more SMs per image), else the narrowest.
bool plan_for(int d, int heads, int C, Plan* pl) {
  const int dk = d / heads;
  const int DC = d / C, hpc = heads / C;
  const int TB = kT * DC * 2;
  int ra = kT * d * 2;
  const int tiles = 3 * TB + (dk >= 64 ? 0 : 2 * kT * 256);
  if (tiles > ra) ra = tiles;
  ra = (ra + kAChunk - 1) / kAChunk * kAChunk;
  const int misc = kMiscFixed + 2 * C * kT * 8 + 13 * DC * 4;
  const int ring = kSmemMax - 1024 - ra - misc;
  if (ra / kAChunk > kMaxASlots || ring < 3 * 16384) return false;
  pl->C = C;
  pl->DC = DC;
  pl->hpc = hpc;
  pl->ra_bytes = ra;
  pl->a_slots = ra / kAChunk;
  pl->stage_bytes = ring >= 3 * 32768 ? 32768 : 16384;
  pl->npass_max = pl->stage_bytes / 128;
  pl->stages = ring / pl->stage_bytes;
  if (pl->stages > kMaxStages) pl->stages = kMaxStages;
  pl->p_off = dk >= 64 ? -1 : 3 * TB;
  pl->smem = 1024 + ra + pl->stages * pl->stage_bytes + misc;
  return true;
}
bool make_plan(int B, int d, int heads, int forced_c, Plan* pl) {
  if (heads <= 0 || d % heads) return false;
  const int dk = d / heads;
  if (dk != 16 && dk != 32 && dk != 64) return false;
  if (d % 64 || d > 512) return false;
  int cand[4], n = 0;
  for (int c = 8; c >= 1; c >>= 1) {          // legal splits, widest first
    if (heads % c || d % c) continue;
    const int dc = d / c, hpc = heads / c;
    if ((dc != 64 && dc != 128) || (hpc != 2 && hpc != 4)) continue;
    if (forced_c && c != forced_c) continue;
    cand[n++] = c;
  }
  // first choice: the widest split whose B clusters are resident at once; then whatever fits, widest first
  for (int pass = 0; pass < 2; ++pass)
    for (int i = 0; i < n; ++i) {
      if (pass == 0 && static_cast<long long>(B) * cand[i] > sm_count() - 16) continue;
      if (plan_for(d, heads, cand[i], pl)) return true;
    }
  return false;
}

bool g_attr_set = false;
unsigned long long* g_trace = nullptr;   // cft_debug_block_trace

template <int DC, int HP>
cudaError_t launch_block(const cudaLaunchConfig_t& cfg, const BlockMaps& maps, const BlockParams& p) {
  return cudaLaunchKernelEx(&cfg, cft_gpt_block_kernel<DC, HP>, maps, p);
}

}  // namespace

using namespace cft;

// Debug timeline: `buf` (device, >= grid * layers * 48 u64) receives clock64 samples of the first compute warp of every CTA
// for the cft_gpt_block launches that follow; NULL turns it off.  scripts/trace_block.py only.
extern "C" int cft_debug_block_trace(void* buf) {
  g_trace = static_cast<unsigned long long*>(buf);
  return CFT_OK;
}

extern "C" long long cft_gpt_block_workspace_bytes(int B, int d) {
  if (B <= 0 || d <= 0) return 0;
  return static_cast<long long>(B) * kT * d * 2 * 4;
}

extern "C" int cft_gpt_block_supported(int B, int d, int heads, int tokens) {
  Plan pl;
  return (tokens == kT && B > 0 && make_plan(B, d, heads, 0, &pl)) ? 1 : 0;
}

extern "C" int cft_gpt_block(const cft_gpt_block_args* a, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CFT_REQUIRE(a != nullptr, "cft_gpt_block: null args");
  CFT_REQUIRE(a->wqkv && a->bqkv && a->wo && a->bo && a->w1 && a->b1 && a->w2 && a->b2 && a->ln1_g && a->ln1_b &&
                  a->ln2_g && a->ln2_b && a->lnf_g && a->lnf_b && a->x_in && a->x_out && a->workspace,
              "cft_gpt_block: null pointer");
  CFT_REQUIRE(a->B > 0 && a->layers > 0 && a->tokens == kT, "cft_gpt_block: need B > 0, layers > 0, 128 tokens per image");
  Plan pl;
  if (!make_plan(a->B, a->d, a->heads, a->cluster > 0 ? a->cluster : 0, &pl)) {
    set_error("cft_gpt_block: shape outside the fused kernel (d %d heads %d cluster %d): use the per-op path", a->d,
              a->heads, a->cluster);
    return CFT_E_UNSUPPORTED;
  }
  CFT_REQUIRE(a->workspace_bytes >= cft_gpt_block_workspace_bytes(a->B, a->d), "cft_gpt_block: workspace too small");
  CFT_REQUIRE(reinterpret_cast<uintptr_t>(a->workspace) % 128 == 0 && reinterpret_cast<uintptr_t>(a->wqkv) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(a->wo) % 16 == 0 && reinterpret_cast<uintptr_t>(a->w1) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(a->w2) % 16 == 0 && reinterpret_cast<uintptr_t>(a->x_in) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(a->x_out) % 16 == 0,
              "cft_gpt_block: misaligned pointer");
  const int d = a->d, L = a->layers, B = a->B, DC = pl.DC;
  BlockParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.d = d; p.heads = a->heads; p.dk = d / a->heads; p.layers = L; p.C = pl.C; p.hpc = pl.hpc;
  p.stages = pl.stages; p.stage_bytes = pl.stage_bytes; p.a_slots = pl.a_slots; p.ra_bytes = pl.ra_bytes;
  p.npass_max = pl.npass_max;
  p.p_off = pl.p_off;
  p.cw = p.dk < 64 ? p.dk : 64;
  p.nch = p.dk / p.cw;
  p.rowB = p.cw * 2;
  p.layout = p.cw == 64 ? 2 : (p.cw == 32 ? 4 : 6);
  p.scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(p.dk));
  p.eps1 = a->eps1; p.eps2 = a->eps2; p.epsf = a->epsf;
  p.bqkv = a->bqkv; p.bo = a->bo; p.b1 = a->b1; p.b2 = a->b2;
  p.ln1g = a->ln1_g; p.ln1b = a->ln1_b; p.ln2g = a->ln2_g; p.ln2b = a->ln2_b; p.lnfg = a->lnf_g; p.lnfb = a->lnf_b;
  p.x_in = a->x_in; p.x_out = a->x_out;
  p.hbuf = reinterpret_cast<__nv_bfloat16*>(a->workspace);
  p.wqkv = reinterpret_cast<const __nv_bfloat16*>(a->wqkv);
  p.wo = reinterpret_cast<const __nv_bfloat16*>(a->wo);
  p.w1 = reinterpret_cast<const __nv_bfloat16*>(a->w1);
  p.w2 = reinterpret_cast<const __nv_bfloat16*>(a->w2);
  p.dbg = a->debug_x;
  p.trace = g_trace;

  // ---- the GEMM passes of one layer
  auto kpack_of = [&](int n, int kchunks) {
    int kp = pl.stage_bytes / (n * 128);
    if (kp < 1) kp = 1;
    while (kp > 1 && kchunks % kp) --kp;
    return kp;
  };
  int np = 0;
  {   // QKV: whole parts (q, k, v: DC rows each) packed greedily into passes of <= npass_max rows
    int part = 0;
    while (part < 3) {
      int cnt = pl.npass_max / DC;
      if (cnt < 1) cnt = 1;
      if (cnt > 3 - part) cnt = 3 - part;
      Pass& ps = p.passes[np++];
      ps.map = 0; ps.nseg = cnt; ps.seg_rows = DC;
      for (int s = 0; s < cnt; ++s) ps.row[s] = (part + s) * d;
      ps.cta_stride = DC; ps.layer_stride = 3 * d;
      ps.n = cnt * DC; ps.kchunks = d / 64; ps.kpack = kpack_of(ps.n, ps.kchunks);
      ps.tcol = part * DC; ps.a_mode = part == 0 ? 0 : 1;
      part += cnt;
    }
    p.npass_qkv = np;
  }
  {   // out-proj
    Pass& ps = p.passes[np++];
    ps.map = 1; ps.nseg = 1; ps.seg_rows = DC; ps.row[0] = 0; ps.cta_stride = DC; ps.layer_stride = d;
    ps.n = DC; ps.kchunks = d / 64; ps.kpack = kpack_of(DC, ps.kchunks); ps.tcol = 0; ps.a_mode = 0;
  }
  p.npass_up = 4 * DC / pl.npass_max;
  CFT_REQUIRE(p.npass_up >= 1 && (4 * DC) % pl.npass_max == 0 && np + p.npass_up + 1 <= kMaxPasses,
              "cft_gpt_block: pass table overflow");
  for (int u = 0; u < p.npass_up; ++u) {
    Pass& ps = p.passes[np++];
    ps.map = 2; ps.nseg = 1; ps.seg_rows = pl.npass_max; ps.row[0] = u * pl.npass_max; ps.cta_stride = 4 * DC;
    ps.layer_stride = 4 * d;
    ps.n = pl.npass_max; ps.kchunks = d / 64; ps.kpack = kpack_of(ps.n, ps.kchunks); ps.tcol = u * pl.npass_max;
    ps.a_mode = u == 0 ? 0 : 1;
  }
  {   // down-proj, A streamed
    Pass& ps = p.passes[np++];
    ps.map = 3; ps.nseg = 1; ps.seg_rows = DC; ps.row[0] = 0; ps.cta_stride = DC; ps.layer_stride = d;
    ps.n = DC; ps.kchunks = 4 * d / 64; ps.kpack = kpack_of(DC, ps.kchunks); ps.tcol = 0; ps.a_mode = 2;
  }

  BlockMaps maps;
  memset(&maps, 0, sizeof(maps));
  int rc;
  if ((rc = encode2d(&maps.w[0], a->wqkv, d, static_cast<long long>(L) * 3 * d, 64, DC, "wqkv"))) return rc;
  if ((rc = encode2d(&maps.w[1], a->wo, d, static_cast<long long>(L) * d, 64, DC, "wo"))) return rc;
  if ((rc = encode2d(&maps.w[2], a->w1, d, static_cast<long long>(L) * 4 * d, 64, pl.npass_max, "w1"))) return rc;
  if ((rc = encode2d(&maps.w[3], a->w2, 4 * d, static_cast<long long>(L) * d, 64, DC, "w2"))) return rc;
  if ((rc = encode2d(&maps.hbuf, p.hbuf, 4 * d, static_cast<long long>(B) * kT, 64, kT, "hbuf"))) return rc;

  if (!g_attr_set) {
    cudaError_t e = cudaFuncSetAttribute(cft_gpt_block_kernel<64, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(cft_gpt_block_kernel<64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(cft_gpt_block_kernel<128, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(cft_gpt_block_kernel<128, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
    if ((rc = check_cuda(e, "cudaFuncSetAttribute(gpt_block)"))) return rc;
    g_attr_set = true;
  }
  int clusters = B;
  const int max_clusters = sm_count() / pl.C;
  if (clusters > max_clusters) clusters = max_clusters;
  LaunchScope ls(CFT_K_GPT_BLOCK, stream);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(clusters * pl.C);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = pl.C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e;
  if (DC == 64) e = pl.hpc == 2 ? launch_block<64, 1>(cfg, maps, p) : launch_block<64, 2>(cfg, maps, p);
  else e = pl.hpc == 2 ? launch_block<128, 1>(cfg, maps, p) : launch_block<128, 2>(cfg, maps, p);
  if (e != cudaSuccess) {
    ls.finish("cft_gpt_block launch");
    return check_cuda(e, "cudaLaunchKernelEx(gpt_block)");
  }
  return ls.finish("cft_gpt_block launch");
}
