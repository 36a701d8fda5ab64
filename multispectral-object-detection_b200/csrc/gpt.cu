// CFT / GPT block glue kernels and the Detect tail:
//   adaptive-avg-pool tokeniser, LayerNorm, 128-token multi-head attention core,
//   bilinear un-pool fused with Add2/Add, Detect permute + sigmoid/grid/anchor decode.
// The six Linear layers per transformer block run on the tcgen05 GEMM (conv_tcgen05.cu).
#include <stdlib.h>

#include "cft_common.cuh"

namespace {
using namespace cft;

// ------------------------------------------------------------------ tokeniser
// grid = (2*va*ha, B); block = 128 threads over 8-channel vectors.
// Bin i covers rows [floor(i*H/va), ceil((i+1)*H/va)) -- torch AdaptiveAvgPool2d (models/common.py:578,608-609).
__global__ void __launch_bounds__(256)
pool_tokens_kernel(const __nv_bfloat16* __restrict__ rgb, int ld_rgb, const __nv_bfloat16* __restrict__ ir, int ld_ir,
                   int H, int W, int C, int va, int ha, const float* __restrict__ pos, float* __restrict__ tok) {
  pdl_prologue();
  // 256 threads = (C/8 channel vectors) x (pixel slices): every thread accumulates its slice of the bin, slices are
  // combined through smem.  All 256 threads stay busy for any C (the per-token kernel used C/8 of 128 threads).
  __shared__ float red[256 * 8];
  const int t = blockIdx.x, b = blockIdx.y;
  const int cells = va * ha, T = 2 * cells;
  const int mod = t / cells, cell = t - mod * cells;
  const int bi = cell / ha, bj = cell - bi * ha;
  const int y0 = (bi * H) / va, y1 = ((bi + 1) * H + va - 1) / va;
  const int x0 = (bj * W) / ha, x1 = ((bj + 1) * W + ha - 1) / ha;
  const __nv_bfloat16* src = mod == 0 ? rgb : ir;
  const int ld = mod == 0 ? ld_rgb : ld_ir;
  const int bw = x1 - x0, npix = (y1 - y0) * bw;
  const float inv = 1.0f / static_cast<float>(npix);
  const int nvec = C / 8;
  for (int v0 = 0; v0 < nvec; v0 += 256) {              // C <= 2048: one pass
    const int nv = min(nvec - v0, 256);
    const int slices = 256 / nv > 0 ? 256 / nv : 1;
    const int cv = threadIdx.x % nv, sl = threadIdx.x / nv;
    float s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (sl < slices) {
#pragma unroll 4
      for (int p = sl; p < npix; p += slices) {       // independent 16-byte loads: keep several in flight
        const int y = y0 + p / bw, x = x0 + p % bw;
        float f[8];
        unpack8(*reinterpret_cast<const bf16x8*>(src + ((static_cast<long long>(b) * H + y) * W + x) * ld + (v0 + cv) * 8), f);
#pragma unroll
        for (int i = 0; i < 8; ++i) s[i] += f[i];
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x * 8 + i] = s[i];
    __syncthreads();
    if (sl == 0 && threadIdx.x < nv) {
      for (int q = 1; q < slices; ++q)
#pragma unroll
        for (int i = 0; i < 8; ++i) s[i] += red[(q * nv + cv) * 8 + i];
      float4* o = reinterpret_cast<float4*>(tok + (static_cast<long long>(b) * T + t) * C + (v0 + cv) * 8);
      const float4* pe = reinterpret_cast<const float4*>(pos + static_cast<long long>(t) * C + (v0 + cv) * 8);
      const float4 p0 = __ldg(pe), p1 = __ldg(pe + 1);
      o[0] = make_float4(s[0] * inv + p0.x, s[1] * inv + p0.y, s[2] * inv + p0.z, s[3] * inv + p0.w);
      o[1] = make_float4(s[4] * inv + p1.x, s[5] * inv + p1.y, s[6] * inv + p1.z, s[7] * inv + p1.w);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ LayerNorm (one warp per row)
template <bool kOutF32, int kMaxV>
__global__ void layernorm_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                 const float* __restrict__ be, float eps, long long rows, int C, void* __restrict__ y) {
  pdl_prologue();
  // one warp per row; the row is read from global memory once and kept in registers: kMaxV float4 per lane
  // (C <= 128 kMaxV; 4 / 8 / 16 for C <= 512 / 1024 / 2048 -- 16 costs 98 registers = 16 resident warps per SM)
  const int lane = threadIdx.x & 31;
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + row * C);
  const int n4 = C / 4;
  float4 v[kMaxV];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int i = lane + 32 * j;
    if (i < n4) {
      v[j] = xr[i];
      s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / static_cast<float>(C);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int i = lane + 32 * j;
    if (i < n4) {
      const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q / static_cast<float>(C) + eps);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  const float4* b4 = reinterpret_cast<const float4*>(be);
#pragma unroll
  for (int j = 0; j < kMaxV; ++j) {
    const int i = lane + 32 * j;
    if (i < n4) {
      const float4 gg = g4[i], bb = b4[i];
      const float o0 = (v[j].x - mean) * rstd * gg.x + bb.x, o1 = (v[j].y - mean) * rstd * gg.y + bb.y;
      const float o2 = (v[j].z - mean) * rstd * gg.z + bb.z, o3 = (v[j].w - mean) * rstd * gg.w + bb.w;
      if constexpr (kOutF32) {
        reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + row * C)[i] = make_float4(o0, o1, o2, o3);
      } else {
        const __nv_bfloat162 h0 = __floats2bfloat162_rn(o0, o1), h1 = __floats2bfloat162_rn(o2, o3);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t*>(&h0);
        pk.y = *reinterpret_cast<const uint32_t*>(&h1);
        reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + row * C)[i] = pk;
      }
    }
  }
}

// ------------------------------------------------------------------ attention core, T <= 128 tokens
// One CTA per (image, head); thread t owns query row t.  Q/K/V staged in smem as bf16 with a
// 2-element row pad (conflict-free per-thread row reads; K/V reads are warp broadcasts); scores in
// smem fp32.  softmax in fp32 with the 1/sqrt(dk) scale folded into the exponent.
__global__ void __launch_bounds__(128)
attention_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int T, int C, int heads) {
  pdl_prologue();
  extern __shared__ uint8_t sm[];
  const int dk = C / heads;
  const int ldp = dk + 2;
  __nv_bfloat16* sq = reinterpret_cast<__nv_bfloat16*>(sm);
  __nv_bfloat16* sk = sq + 128 * ldp;
  __nv_bfloat16* sv = sk + 128 * ldp;
  float* ss = reinterpret_cast<float*>(sv + 128 * ldp);  // [128][129]
  const int h = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x;
  const __nv_bfloat16* base = qkv + static_cast<long long>(b) * T * 3 * C + h * dk;
  // cooperative load: 8-element (16 B) global reads, 4-byte smem writes (row pad keeps 4B alignment)
  const int vec_per_row = dk / 8;
  for (int i = tid; i < T * vec_per_row; i += blockDim.x) {
    const int r = i / vec_per_row, cv = i - r * vec_per_row;
    const __nv_bfloat16* g = base + static_cast<long long>(r) * 3 * C + cv * 8;
    const bf16x8 q = *reinterpret_cast<const bf16x8*>(g);
    const bf16x8 k = *reinterpret_cast<const bf16x8*>(g + C);
    const bf16x8 v = *reinterpret_cast<const bf16x8*>(g + 2 * C);
    __nv_bfloat162* dq = reinterpret_cast<__nv_bfloat162*>(sq + r * ldp + cv * 8);
    __nv_bfloat162* dkk = reinterpret_cast<__nv_bfloat162*>(sk + r * ldp + cv * 8);
    __nv_bfloat162* dv = reinterpret_cast<__nv_bfloat162*>(sv + r * ldp + cv * 8);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      dq[j] = q.get(j);
      dkk[j] = k.get(j);
      dv[j] = v.get(j);
    }
  }
  __syncthreads();
  const int t = tid;
  if (t < T) {
    const float scale = rsqrtf(static_cast<float>(dk));
    const __nv_bfloat162* qr = reinterpret_cast<const __nv_bfloat162*>(sq + t * ldp);
    float* srow = ss + t * 129;
    float mx = -INFINITY;
    for (int j = 0; j < T; ++j) {
      const __nv_bfloat162* kr = reinterpret_cast<const __nv_bfloat162*>(sk + j * ldp);
      float a0 = 0.f, a1 = 0.f;
      for (int c = 0; c < dk / 2; ++c) {
        const float2 qa = __bfloat1622float2(qr[c]);
        const float2 ka = __bfloat1622float2(kr[c]);
        a0 = fmaf(qa.x, ka.x, a0);
        a1 = fmaf(qa.y, ka.y, a1);
      }
      const float sc = (a0 + a1) * scale;
      srow[j] = sc;
      mx = fmaxf(mx, sc);
    }
    float sum = 0.f;
    for (int j = 0; j < T; ++j) {
      const float e = __expf(srow[j] - mx);
      srow[j] = e;
      sum += e;
    }
    const float inv = 1.0f / sum;
    __nv_bfloat16* orow = out + (static_cast<long long>(b) * T + t) * C + h * dk;
    for (int c0 = 0; c0 < dk; c0 += 8) {
      float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      for (int j = 0; j < T; ++j) {
        const float pj = srow[j];
        const __nv_bfloat162* vr = reinterpret_cast<const __nv_bfloat162*>(sv + j * ldp + c0);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 va = __bfloat1622float2(vr[i]);
          acc[2 * i] = fmaf(pj, va.x, acc[2 * i]);
          acc[2 * i + 1] = fmaf(pj, va.y, acc[2 * i + 1]);
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] *= inv;
      *reinterpret_cast<bf16x8*>(orow + c0) = pack8(acc);
    }
  }
}

// ------------------------------------------------------------------ bilinear un-pool + Add2 + Add
struct UnpoolArgs {
  const float* tok;
  int B, H, W, C, va, ha;
  const __nv_bfloat16 *x_rgb, *x_ir;
  int ld_xr, ld_xi;
  __nv_bfloat16 *o_rgb, *o_ir, *o_sum;
  int ld_or, ld_oi, ld_os;
};

// torch upsample_bilinear2d, align_corners=False: src = scale*(dst+0.5)-0.5 clamped at 0.
__device__ __forceinline__ void bilin(int dst, int in, int out, int* i0, int* i1, float* l1) {
  const float scale = static_cast<float>(in) / static_cast<float>(out);
  float src = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  if (src < 0.f) src = 0.f;
  const int a = static_cast<int>(src);
  *i0 = a;
  *i1 = a + (a < in - 1 ? 1 : 0);
  *l1 = src - static_cast<float>(a);
}

__global__ void unpool_kernel(UnpoolArgs a) {
  pdl_prologue();
  const int C8 = a.C / 8;
  const int cells = a.va * a.ha;
  const long long total = static_cast<long long>(a.B) * a.H * a.W * C8;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int cv = static_cast<int>(idx % C8);
    long long pix = idx / C8;
    const int x = static_cast<int>(pix % a.W);
    long long t = pix / a.W;
    const int y = static_cast<int>(t % a.H);
    const int b = static_cast<int>(t / a.H);
    int y0, y1, x0, x1;
    float ly, lx;
    bilin(y, a.va, a.H, &y0, &y1, &ly);
    bilin(x, a.ha, a.W, &x0, &x1, &lx);
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    float r[2][8];
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const float* tb = a.tok + (static_cast<long long>(b) * 2 * cells + m * cells) * a.C + cv * 8;
      const float* p00 = tb + static_cast<long long>(y0 * a.ha + x0) * a.C;
      const float* p01 = tb + static_cast<long long>(y0 * a.ha + x1) * a.C;
      const float* p10 = tb + static_cast<long long>(y1 * a.ha + x0) * a.C;
      const float* p11 = tb + static_cast<long long>(y1 * a.ha + x1) * a.C;
#pragma unroll
      for (int i = 0; i < 8; ++i) r[m][i] = w00 * p00[i] + w01 * p01[i] + w10 * p10[i] + w11 * p11[i];
    }
    if (a.x_rgb) {
      float f[8];
      unpack8(*reinterpret_cast<const bf16x8*>(a.x_rgb + pix * a.ld_xr + cv * 8), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) r[0][i] += f[i];
    }
    if (a.x_ir) {
      float f[8];
      unpack8(*reinterpret_cast<const bf16x8*>(a.x_ir + pix * a.ld_xi + cv * 8), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) r[1][i] += f[i];
    }
    *reinterpret_cast<bf16x8*>(a.o_rgb + pix * a.ld_or + cv * 8) = pack8(r[0]);
    *reinterpret_cast<bf16x8*>(a.o_ir + pix * a.ld_oi + cv * 8) = pack8(r[1]);
    if (a.o_sum) {
#pragma unroll
      for (int i = 0; i < 8; ++i) r[0][i] += r[1][i];
      *reinterpret_cast<bf16x8*>(a.o_sum + pix * a.ld_os + cv * 8) = pack8(r[0]);
    }
  }
}


// Row-blocked variant: one CTA per (image, output row, 64-channel chunk).  The two token rows that bracket the
// output row are blended vertically once into smem (2 modalities x ha tokens x 64 channels, fp32); each thread
// then does only the horizontal lerp for its (pixel, 8-channel vector) -- the feature maps are streamed once,
// coalesced, and the token tensor is read ~H/va times less often than by the per-pixel kernel.
constexpr int kUnpoolCC = 64;
constexpr int kUnpoolMaxThreads = 640;   // x 2 CTAs per SM: <= 48 registers per thread (56 unbounded = ONE 640-thread CTA per SM)
__global__ void __launch_bounds__(kUnpoolMaxThreads, 2) unpool_rows_kernel(UnpoolArgs a) {
  pdl_prologue();
  extern __shared__ float srow[];                 // [2][ha][kUnpoolCC]
  const int y = blockIdx.x, cc = blockIdx.y, b = blockIdx.z;
  const int cells = a.va * a.ha;
  int y0, y1;
  float ly;
  bilin(y, a.va, a.H, &y0, &y1, &ly);
  const int c_base = cc * kUnpoolCC;
  const int cw = min(kUnpoolCC, a.C - c_base);    // channels in this chunk (multiple of 8)
  for (int i = threadIdx.x; i < 2 * a.ha * (cw / 4); i += blockDim.x) {
    const int c4 = i % (cw / 4);
    const int t = i / (cw / 4);                   // m * ha + tx
    const int m = t / a.ha, tx = t - m * a.ha;
    const float* tb = a.tok + (static_cast<long long>(b) * 2 * cells + m * cells) * a.C + c_base + c4 * 4;
    const float4 p0 = *reinterpret_cast<const float4*>(tb + static_cast<long long>(y0 * a.ha + tx) * a.C);
    const float4 p1 = *reinterpret_cast<const float4*>(tb + static_cast<long long>(y1 * a.ha + tx) * a.C);
    float4 r;
    r.x = (1.f - ly) * p0.x + ly * p1.x;
    r.y = (1.f - ly) * p0.y + ly * p1.y;
    r.z = (1.f - ly) * p0.z + ly * p1.z;
    r.w = (1.f - ly) * p0.w + ly * p1.w;
    *reinterpret_cast<float4*>(srow + t * kUnpoolCC + c4 * 4) = r;
  }
  __syncthreads();
  const int cv8 = cw / 8;
  const long long row_pix = (static_cast<long long>(b) * a.H + y) * a.W;
  for (int i = threadIdx.x; i < a.W * cv8; i += blockDim.x) {
    const int cv = i % cv8, x = i / cv8;
    int x0, x1;
    float lx;
    bilin(x, a.ha, a.W, &x0, &x1, &lx);
    const long long pix = row_pix + x;
    const int c = c_base + cv * 8;
    float r[2][8];
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const float* s0 = srow + (m * a.ha + x0) * kUnpoolCC + cv * 8;
      const float* s1 = srow + (m * a.ha + x1) * kUnpoolCC + cv * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j) r[m][j] = (1.f - lx) * s0[j] + lx * s1[j];
    }
    if (a.x_rgb) {
      float f[8];
      unpack8(*reinterpret_cast<const bf16x8*>(a.x_rgb + pix * a.ld_xr + c), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) r[0][j] += f[j];
    }
    if (a.x_ir) {
      float f[8];
      unpack8(*reinterpret_cast<const bf16x8*>(a.x_ir + pix * a.ld_xi + c), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) r[1][j] += f[j];
    }
    *reinterpret_cast<bf16x8*>(a.o_rgb + pix * a.ld_or + c) = pack8(r[0]);
    *reinterpret_cast<bf16x8*>(a.o_ir + pix * a.ld_oi + c) = pack8(r[1]);
    if (a.o_sum) {
#pragma unroll
      for (int j = 0; j < 8; ++j) r[0][j] += r[1][j];
      *reinterpret_cast<bf16x8*>(a.o_sum + pix * a.ld_os + c) = pack8(r[0]);
    }
  }
}

// ------------------------------------------------------------------ Detect tail
// One thread per (b, anchor, j, i).  Index math is integer-exact:
//   raw[b][a][j][i][o], z row = z_row0 + a*ny*nx + j*nx + i, grid = (i, j)  (models/yolo_test.py:48-64)
__global__ void detect_decode_kernel(const float* __restrict__ head, int ldh, int B, int ny, int nx, int na, int no,
                                     float stride, const float* __restrict__ anchors, float* __restrict__ raw,
                                     float* __restrict__ z, long long z_rows, long long z_row0) {
  pdl_prologue();
  const long long total = static_cast<long long>(B) * na * ny * nx;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(idx % nx);
    long long t = idx / nx;
    const int j = static_cast<int>(t % ny);
    t /= ny;
    const int a = static_cast<int>(t % na);
    const int b = static_cast<int>(t / na);
    const float* hp = head + ((static_cast<long long>(b) * ny + j) * nx + i) * ldh + a * no;
    float* rp = raw + idx * no;
    float* zp = z + (static_cast<long long>(b) * z_rows + z_row0 + (static_cast<long long>(a) * ny + j) * nx + i) * no;
    const float aw = anchors[2 * a], ah = anchors[2 * a + 1];
    for (int o = 0; o < no; ++o) {
      const float v = hp[o];
      rp[o] = v;
      const float s = 1.0f / (1.0f + expf(-v));
      float d;
      if (o == 0)
        d = __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(s, 2.0f), -0.5f), static_cast<float>(i)), stride);
      else if (o == 1)
        d = __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(s, 2.0f), -0.5f), static_cast<float>(j)), stride);
      else if (o == 2) {
        const float u = __fmul_rn(s, 2.0f);
        d = __fmul_rn(__fmul_rn(u, u), aw);
      } else if (o == 3) {
        const float u = __fmul_rn(s, 2.0f);
        d = __fmul_rn(__fmul_rn(u, u), ah);
      } else
        d = s;
      zp[o] = d;
    }
  }
}

inline int grid_for(long long work, int threads) {
  long long blocks = (work + threads - 1) / threads;
  const long long cap = static_cast<long long>(sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

bool g_attn_attr = false;

}  // namespace

using namespace cft;

extern "C" int cft_gpt_pool_tokens(const void* rgb, int ld_rgb, int coff_rgb, const void* ir, int ld_ir, int coff_ir,
                                   int B, int H, int W, int C, int va, int ha, const float* pos_emb, float* tokens,
                                   void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CFT_REQUIRE(rgb && ir && pos_emb && tokens, "cft_gpt_pool_tokens: null pointer");
  CFT_REQUIRE(C > 0 && C % 8 == 0 && ld_rgb % 8 == 0 && ld_ir % 8 == 0 && coff_rgb % 8 == 0 && coff_ir % 8 == 0,
              "cft_gpt_pool_tokens: channels/ld/coff must be multiples of 8");
  CFT_REQUIRE(B > 0 && H >= 1 && W >= 1 && va >= 1 && ha >= 1 && B <= 65535, "cft_gpt_pool_tokens: bad shape");
  dim3 grid(2 * va * ha, B);
  LaunchScope ls(CFT_K_POOL_TOKENS, stream);
  cft::launch(pool_tokens_kernel, dim3(grid), dim3(256), 0, stream, reinterpret_cast<const __nv_bfloat16*>(rgb) + coff_rgb, ld_rgb,
                                               reinterpret_cast<const __nv_bfloat16*>(ir) + coff_ir, ld_ir, H, W, C, va,
                                               ha, pos_emb, tokens);
  return ls.finish("cft_gpt_pool_tokens launch");
}

extern "C" int cft_layernorm(const float* x, const float* gamma, const float* beta, float eps, long long rows, int C,
                             void* y, int out_dtype, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CFT_REQUIRE(x && gamma && beta && y, "cft_layernorm: null pointer");
  CFT_REQUIRE(rows > 0 && C > 0 && C % 4 == 0 && C <= 2048, "cft_layernorm: C must be a multiple of 4, <= 2048");
  const int warps = 4;
  const long long blocks = (rows + warps - 1) / warps;
  LaunchScope ls(CFT_K_LAYERNORM, stream);
  if (out_dtype != CFT_DT_F32 && out_dtype != CFT_DT_BF16) return fail_arg("cft_layernorm: bad out_dtype");
  const bool f32 = out_dtype == CFT_DT_F32;
  const dim3 grid(static_cast<unsigned>(blocks)), block(warps * 32);
#define CFT_LN_LAUNCH(V)                                                                                          \
  do {                                                                                                            \
    if (f32) cft::launch(layernorm_kernel<true, V>, grid, block, 0, stream, x, gamma, beta, eps, rows, C, y);     \
    else cft::launch(layernorm_kernel<false, V>, grid, block, 0, stream, x, gamma, beta, eps, rows, C, y);        \
  } while (0)
  if (C <= 512) CFT_LN_LAUNCH(4);
  else if (C <= 1024) CFT_LN_LAUNCH(8);
  else CFT_LN_LAUNCH(16);
#undef CFT_LN_LAUNCH
  return ls.finish("cft_layernorm launch");
}

extern "C" int cft_attention(const void* qkv, void* out, int B, int T, int C, int heads, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CFT_REQUIRE(qkv && out, "cft_attention: null pointer");
  CFT_REQUIRE(B > 0 && B <= 65535 && T > 0 && T <= 128 && heads > 0 && C % heads == 0 && (C / heads) % 8 == 0,
              "cft_attention: need T<=128 and head dim multiple of 8 (T %d C %d heads %d)", T, C, heads);
  // both kernels move q / k / v and the output in 16-byte vectors (TMA boxes, bf16x8 loads and stores)
  CFT_REQUIRE(reinterpret_cast<uintptr_t>(qkv) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0,
              "cft_attention: qkv and out must be 16-byte aligned");
  static const bool force_simt = getenv("CFT_ATTENTION_SIMT") != nullptr;   // debug / cross-check
  if (!force_simt) {
    const int rc = attention_tcgen05(qkv, out, B, T, C, heads, stream);
    if (rc != CFT_E_UNSUPPORTED) return rc;
  }
  const int dk = C / heads;
  const int smem = 3 * 128 * (dk + 2) * 2 + 128 * 129 * 4;
  CFT_REQUIRE(smem <= 220 * 1024, "cft_attention: head dim %d too large", dk);
  if (!g_attn_attr) {
    int rc = check_cuda(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024),
                        "cudaFuncSetAttribute(attention)");
    if (rc) return rc;
    g_attn_attr = true;
  }
  dim3 grid(heads, B);
  LaunchScope ls(CFT_K_ATTENTION, stream);
  cft::launch(attention_kernel, dim3(grid), dim3(128), smem, stream, reinterpret_cast<const __nv_bfloat16*>(qkv),
                                                reinterpret_cast<__nv_bfloat16*>(out), T, C, heads);
  return ls.finish("cft_attention launch");
}

extern "C" int cft_gpt_unpool(const float* tok, int B, int H, int W, int C, int va, int ha, const void* x_rgb,
                              int ld_xr, int coff_xr, const void* x_ir, int ld_xi, int coff_xi, void* out_rgb,
                              int ld_or, int coff_or, void* out_ir, int ld_oi, int coff_oi, void* out_sum, int ld_os,
                              int coff_os, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CFT_REQUIRE(tok && out_rgb && out_ir, "cft_gpt_unpool: null pointer");
  CFT_REQUIRE(C > 0 && C % 8 == 0 && B > 0 && H > 0 && W > 0 && va > 0 && ha > 0, "cft_gpt_unpool: bad shape");
  CFT_REQUIRE((ld_or | coff_or | ld_oi | coff_oi) % 8 == 0 && (!x_rgb || (ld_xr | coff_xr) % 8 == 0) &&
                  (!x_ir || (ld_xi | coff_xi) % 8 == 0) && (!out_sum || (ld_os | coff_os) % 8 == 0),
              "cft_gpt_unpool: ld/coff must be multiples of 8");
  UnpoolArgs a;
  a.tok = tok;
  a.B = B; a.H = H; a.W = W; a.C = C; a.va = va; a.ha = ha;
  a.x_rgb = x_rgb ? reinterpret_cast<const __nv_bfloat16*>(x_rgb) + coff_xr : nullptr;
  a.x_ir = x_ir ? reinterpret_cast<const __nv_bfloat16*>(x_ir) + coff_xi : nullptr;
  a.ld_xr = ld_xr; a.ld_xi = ld_xi;
  a.o_rgb = reinterpret_cast<__nv_bfloat16*>(out_rgb) + coff_or;
  a.o_ir = reinterpret_cast<__nv_bfloat16*>(out_ir) + coff_oi;
  a.o_sum = out_sum ? reinterpret_cast<__nv_bfloat16*>(out_sum) + coff_os : nullptr;
  a.ld_or = ld_or; a.ld_oi = ld_oi; a.ld_os = ld_os;
  LaunchScope ls(CFT_K_UNPOOL, stream);
  const int chunks = (C + kUnpoolCC - 1) / kUnpoolCC;
  if (H <= 65535 && chunks <= 65535 && B <= 65535 && ha <= 64) {
    // one (pixel, 8-channel vector) item per thread and pass: balance the passes (640 items = 1 pass of 640 threads, not
    // 512 + 128) so that no pass runs mostly empty
    const int items = W * (kUnpoolCC / 8);
    const int passes = (items + kUnpoolMaxThreads - 1) / kUnpoolMaxThreads;
    int threads = ((items + passes - 1) / passes + 31) / 32 * 32;
    if (threads < 64) threads = 64;
    dim3 grid(H, chunks, B);
    cft::launch(unpool_rows_kernel, dim3(grid), dim3(threads), 2 * ha * kUnpoolCC * sizeof(float), stream, a);
  } else {
    const long long total = static_cast<long long>(B) * H * W * (C / 8);
    cft::launch(unpool_kernel, dim3(grid_for(total, 256)), dim3(256), 0, stream, a);
  }
  return ls.finish("cft_gpt_unpool launch");
}

extern "C" int cft_detect_decode(const float* head, int ldh, int B, int ny, int nx, int na, int no, float stride,
                                 const float* anchors_px, float* raw, float* z, long long z_rows, long long z_row0,
                                 void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CFT_REQUIRE(head && anchors_px && raw && z, "cft_detect_decode: null pointer");
  CFT_REQUIRE(B > 0 && ny > 0 && nx > 0 && na > 0 && no >= 5 && ldh >= na * no, "cft_detect_decode: bad shape");
  CFT_REQUIRE(z_row0 >= 0 && z_row0 + static_cast<long long>(na) * ny * nx <= z_rows, "cft_detect_decode: z rows out of range");
  const long long total = static_cast<long long>(B) * na * ny * nx;
  LaunchScope ls(CFT_K_DETECT, stream);
  cft::launch(detect_decode_kernel, dim3(grid_for(total, 128)), dim3(128), 0, stream, head, ldh, B, ny, nx, na, no, stride, anchors_px, raw,
                                                                 z, z_rows, z_row0);
  return ls.finish("cft_detect_decode launch");
}
