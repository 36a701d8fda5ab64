/*
 * cft_b200.h -- C ABI of the B200-native two-stream CFT (yolov5-CFTx3) forward path.
 *
 * Every entry point takes raw DEVICE pointers, explicit shapes/strides and a CUDA stream
 * (passed as void*, i.e. a cudaStream_t / CUstream handle; NULL = legacy default stream).
 * No torch types, no C++ exceptions, no allocation inside: the caller owns every buffer.
 * Return value: 0 = ok, otherwise a CFT_E_* code; cft_last_error() gives the text.
 *
 * Activations are NHWC ("channels last") bf16.  A tensor argument is described by
 *   (ptr, ld, coff): element (b,y,x,c) lives at ptr[((b*H + y)*W + x)*ld + coff + c]
 * so a producer can write straight into a channel slice of its consumer's buffer
 * (that is how Concat is fused away).
 *
 * The reference has no native code (SURVEY.md section 2.2); each function below names the
 * reference Python it replaces (paths relative to the reference root).
 */
#ifndef CFT_B200_H
#define CFT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CFT_ABI_VERSION 7

enum {
  CFT_OK = 0,
  CFT_E_ARG = 1,        /* bad argument (shape, alignment, null pointer)            */
  CFT_E_CUDA = 2,       /* CUDA runtime / driver error (text in cft_last_error())   */
  CFT_E_UNSUPPORTED = 3 /* valid request this build does not implement              */
};

enum { CFT_ACT_NONE = 0, CFT_ACT_SILU = 1, CFT_ACT_GELU = 2 };
enum { CFT_DT_BF16 = 0, CFT_DT_F32 = 1, CFT_DT_U8 = 2 };

/* kernel ids for the profiling counters */
enum {
  CFT_K_CONV_TCGEN05 = 0, CFT_K_CONV_REF = 1, CFT_K_FOCUS = 2, CFT_K_MAXPOOL = 3,
  CFT_K_UPSAMPLE = 4, CFT_K_ADD = 5, CFT_K_COPY = 6, CFT_K_POOL_TOKENS = 7,
  CFT_K_LAYERNORM = 8, CFT_K_ATTENTION = 9, CFT_K_UNPOOL = 10, CFT_K_DETECT = 11,
  CFT_K_NMS = 12, CFT_K_GPT_BLOCK = 13, CFT_K_COUNT = 14
};

int cft_abi_version(void);
const char* cft_last_error(void);
/* Fails (CFT_E_UNSUPPORTED) unless the current device is compute capability 10.x. */
int cft_check_device(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------------------------------
 * Fused convolution / GEMM:  y = act(conv(x, w) + bias) [+ res]
 *   Replaces Conv.forward / Conv.fuseforward (models/common.py:36-50) with BN folded
 *   (utils/torch_utils.py:181-201), the 1x1/3x3 convs inside Bottleneck (:99-109),
 *   C3 (:131-143), SPP (:154-165), Focus (:168-180), the Detect 1x1 convs
 *   (models/yolo_test.py:46) and, with k=1,B=1,H=1,W=M, every nn.Linear of
 *   SelfAttention / myTransformerBlock (models/common.py:450-453,533-536).
 *
 *   x   : bf16 NHWC [B,H,W,ldx], channels [x_coff, x_coff+Cin)
 *   w   : bf16 packed [Cout][k*k][Cin_p] (Cin_p = Cin rounded up to 8; tap = ky*k+kx)
 *   bias: f32 [Cout] or NULL
 *   k in {1,3} = kernel height; kw = kernel width (0 -> square, kw = k; 1 with k = 3 -> a 3x1 filter, used by Focus);
 *   stride in {1,2} (square 3x3 only); pad = (k/2, kw/2); Ho = ceil(H/stride), Wo = ceil(W/stride)
 *   w   : tap = ky*kw + kx
 *   res : optional residual, added AFTER the activation; dtype = out_dtype
 *   y   : [B,Ho,Wo,ldy] channels [y_coff, y_coff+Cout), bf16 or f32
 * ------------------------------------------------------------------------------------- */
typedef struct cft_conv_args {
  const void* x; int B, H, W, Cin, ldx, x_coff;
  const void* w; const float* bias; int Cout, k, stride, act;
  const void* res; int ldr, r_coff;
  void* y; int ldy, y_coff, out_dtype;
  int kw;
  /* Optional chained 1x1 (back-to-back GEMM in the epilogue): y2 = act2(w2 . y + bias2) per output pixel, computed from the
   * finished bf16 tile of y while it is still on chip -- a Bottleneck's cv1 (models/common.py:104-106) fused into the conv that
   * produces its input.  w2: bf16 packed [Cout][1][Cout] (NULL = no chain); y2: bf16 NHWC channel slice [y2_coff, y2_coff+Cout)
   * of a tensor with the geometry of y; skip_y != 0: y itself is not written (only y2 is wanted).  Needs out_dtype bf16 and
   * Cout in {64, 128}; otherwise CFT_E_UNSUPPORTED and the caller launches the 1x1 separately. */
  const void* w2; const float* bias2; void* y2; int ldy2, y2_coff, act2, skip_y;
} cft_conv_args;

/* tcgen05 / TMA / TMEM implicit-GEMM kernel (the product path). */
int cft_conv2d(const cft_conv_args* a, void* stream);
/* Plain CUDA-core restatement of the same contract; slow; used by the GPU tests to
 * cross-check the tcgen05 kernel.  Never called by the forward path. */
int cft_conv2d_ref(const cft_conv_args* a, void* stream);

/* Focus space-to-depth gather (models/common.py:179): NCHW image [B,3,H,W] -> NHWC bf16 at half resolution.
 * Space-to-depth channel s(dy,dx,c) = (dy + 2*dx)*3 + c (12 channels, padded to 16 with zeros).
 *   layout 0: [B,H/2,W/2,16]  = s(.) of the pixel itself
 *   layout 1: [B,H/2,W/2,64]  = x-direction im2col: channel kx*16 + s holds s(.) of pixel x+kx-1 (kx = 0..2, zero
 *             outside the image), 48..63 = 0.  The Focus 3x3 conv then becomes a 3x1 conv with K = 64 whose
 *             three vertical taps share one TMA box (128-byte TMA rows instead of 32-byte ones).
 * in_dtype: CFT_DT_F32 / CFT_DT_BF16 (values already in [0,1]) or CFT_DT_U8 -- the data loader's wire format
 * (utils/datasets.py:1272-1281), scaled by 1/255 here as train.py:715 / test.py:107-108 do on the device.
 * batch_stride = elements between consecutive images (3*H*W for a dense tensor; 6*H*W when RGB / IR are the two
 * halves of the loader's [B,6,H,W] tensor, train.py:716-717). */
int cft_focus_gather(const void* img, int in_dtype, int B, int H, int W, long long batch_stride,
                     int layout, void* y, void* stream);

/* Fused Focus layer (models/common.py:168-180 = space-to-depth + concat + Conv 3x3 + BN + SiLU) straight from the
 * loader's uint8 image (utils/datasets.py:1272-1281; the 1/255 of train.py:715 / test.py:107-108 is applied to the
 * fp32 accumulator).  img: uint8 [B,3,H,W] (H, W even, W % 16 == 0, batch_stride bytes between images: 6*H*W for the
 * halves of the [B,6,H,W] loader tensor).  w: fp16 [Cout][192], the 3x3x12 filter re-indexed as a 6x6 stride-2 filter
 * on the image: w[o][(c*6 + r)*8 + q] = W[o][(gy + 2*gx)*3 + c][ky][kx] with r = 2*ky + gy, q = 2*kx + gx (q = 6, 7 and
 * columns >= 144 are zero); BN is folded in before the fp16 rounding.  y: NHWC bf16 [B,H/2,W/2,ldy] channel slice.
 * Cout: multiple of 16, <= 128.  act: CFT_ACT_NONE or CFT_ACT_SILU. */
int cft_focus_conv(const void* img, int B, int H, int W, long long batch_stride, const void* w, const float* bias,
                   int Cout, int act, void* y, int ldy, int y_coff, void* stream);

/* MaxPool k x k, stride 1, pad k/2 (-inf padding) on an NHWC bf16 channel slice
 * (SPP, models/common.py:160-165).  src/dst may be slices of the same buffer. */
int cft_maxpool_s1(const void* x, int ldx, int x_coff, void* y, int ldy, int y_coff,
                   int B, int H, int W, int C, int k, void* stream);

/* SPP in one pass (models/common.py:160-165): three stride-1 max pools applied in cascade (windows k0, k1, k2;
 * pool_9 = pool_5 o pool_5 and pool_13 = pool_5 o pool_9, so SPP's (5,9,13) is the cascade (5,5,5)); the result of
 * stage i goes to channel slice y_coff_i of y.  C must be a multiple of 16; H*W*64 bytes of smem per CTA. */
int cft_maxpool_cascade3(const void* x, int ldx, int x_coff, void* y, int ldy, int y_coff0, int y_coff1,
                         int y_coff2, int B, int H, int W, int C, int k0, int k1, int k2, void* stream);

/* nn.Upsample(None, 2, 'nearest') (yaml rows 33/37): [B,H,W,C] -> [B,2H,2W,C]. */
int cft_upsample2x(const void* x, int ldx, int x_coff, void* y, int ldy, int y_coff,
                   int B, int H, int W, int C, void* stream);

/* Add / Add2 (models/common.py:222-243): y = a + b on bf16 channel slices, npix = B*H*W. */
int cft_add(const void* a, int lda, int a_coff, const void* b, int ldb, int b_coff,
            void* y, int ldy, int y_coff, long long npix, int C, void* stream);

/* Concat fallback (models/common.py:219): copy a channel slice. */
int cft_copy(const void* x, int ldx, int x_coff, void* y, int ldy, int y_coff,
             long long npix, int C, void* stream);

/* GPT front end (models/common.py:608-621): AdaptiveAvgPool2d((va,ha)) of both modalities,
 * tokenise (RGB tokens first, token = row*ha+col), + pos_emb.  Output f32 [B, 2*va*ha, C]. */
int cft_gpt_pool_tokens(const void* rgb, int ld_rgb, int coff_rgb,
                        const void* ir, int ld_ir, int coff_ir,
                        int B, int H, int W, int C, int va, int ha,
                        const float* pos_emb, float* tokens, void* stream);

/* LayerNorm over the last dim (models/common.py:529-530,572), f32 in, eps explicit.
 * out_dtype selects bf16 (GEMM operand) or f32 output. */
int cft_layernorm(const float* x, const float* gamma, const float* beta, float eps,
                  long long rows, int C, void* y, int out_dtype, void* stream);

/* Multi-head self-attention core (models/common.py:497-510): qkv bf16 [B*T, 3*C] holding
 * q|k|v (head h at columns h*dk of each third), T tokens per image (T <= 128),
 * out bf16 [B*T, C] = softmax(q k^T / sqrt(dk)) v with heads merged.
 * dk = C / heads must be a multiple of 8; qkv and out must be 16-byte aligned (CFT_E_ARG otherwise).
 * T = 128 with 16 <= dk <= 256 runs on the tensor cores when the head dim splits into at most 4 chunks of 64 / 32 / 16
 * (a last chunk of 16 may cover the final 8 columns); every other shape runs on a CUDA-core kernel whose shared memory
 * (3 * 128 * (dk + 2) * 2 + 128 * 129 * 4 bytes) must stay within 220 KiB, i.e. dk <= 200 -- beyond that CFT_E_ARG. */
int cft_attention(const void* qkv, void* out, int B, int T, int C, int heads, void* stream);

/* ---------------------------------------------------------------------------------------
 * The transformer stack of one CFT / GPT block in ONE launch (models/common.py:622 `self.trans_blocks(x)` + :625
 * `self.ln_f(x)`; per layer myTransformerBlock.forward :540-546 with SelfAttention.forward :475-513):
 *     x += out_proj(softmax(q k^T / sqrt(dk)) v),  q|k|v = Linear(LN1(x));    x += W2 GELU(W1 LN2(x) + b1) + b2
 * One thread-block cluster per image keeps the 128 x d token tile on chip / in L2 for all layers (csrc/cft_block.cu).
 *   x_in   f32 [B, 128, d]   tokens (output of cft_gpt_pool_tokens)         x_out  f32 [B, 128, d] = ln_f(x)
 *   wqkv   bf16 [layers*3d, d]  rows of layer l: que_proj | key_proj | val_proj weights (nn.Linear [out, in])
 *   wo     bf16 [layers*d, d]   w1 bf16 [layers*4d, d]   w2 bf16 [layers*d, 4d];  biases f32, same row order
 *   ln1_*, ln2_*  f32 [layers*d] (ln_input / ln_output of every layer),  lnf_*  f32 [d]
 *   workspace: cft_gpt_block_workspace_bytes(B, d) bytes, 128-byte aligned (all-gathered bf16 operands)
 *   cluster: CTAs per image (0 = automatic);  debug_x: optional f32 [layers, B, 128, d] dump of x after each layer
 * Supported: 128 tokens, head dim 16/32/64, d <= 512 with d / cluster in {64, 128}
 * (cft_gpt_block_supported() tells); anything else returns CFT_E_UNSUPPORTED and the caller runs the per-op path
 * (cft_layernorm / cft_conv2d / cft_attention).
 * ------------------------------------------------------------------------------------- */
typedef struct cft_gpt_block_args {
  int B, tokens, d, heads, layers, cluster;
  const void* wqkv; const float* bqkv;
  const void* wo;   const float* bo;
  const void* w1;   const float* b1;
  const void* w2;   const float* b2;
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *lnf_g, *lnf_b;
  float eps1, eps2, epsf;
  const float* x_in; float* x_out;
  void* workspace; long long workspace_bytes;
  float* debug_x;
} cft_gpt_block_args;
long long cft_gpt_block_workspace_bytes(int B, int d);
int cft_gpt_block_supported(int B, int d, int heads, int tokens);
int cft_gpt_block(const cft_gpt_block_args* a, void* stream);
/* debug: per-CTA, per-layer clock samples of the compute warps (16 u64 slots each); NULL = off */
int cft_debug_block_trace(void* buf);

/* GPT back end (models/common.py:626-637) fused with Add2 (:239-242) and Add (:229):
 * tok f32 [B, 2*va*ha, C] (after ln_f) is bilinearly upsampled (align_corners=False) to HxW
 * per modality; out_rgb = x_rgb + up_rgb, out_ir = x_ir + up_ir, out_sum = out_rgb + out_ir.
 * x_rgb/x_ir NULL -> the upsampled map alone is written (plain GPT.forward output).
 * out_sum may be NULL.  All maps NHWC bf16 with (ld, coff). */
int cft_gpt_unpool(const float* tok, int B, int H, int W, int C, int va, int ha,
                   const void* x_rgb, int ld_xr, int coff_xr,
                   const void* x_ir, int ld_xi, int coff_xi,
                   void* out_rgb, int ld_or, int coff_or,
                   void* out_ir, int ld_oi, int coff_oi,
                   void* out_sum, int ld_os, int coff_os, void* stream);

/* Detect tail (models/yolo_test.py:48-59) for one level: head f32 [B*ny*nx, ldh] holding
 * na*no conv outputs per pixel (channel = a*no + o) ->
 *   raw f32 [B,na,ny,nx,no]   (the permuted head, :48)
 *   z   f32 [B, z_rows, no] rows [z_row0 + a*ny*nx + j*nx + i]  (sigmoid + grid/anchor decode)
 * anchors_px: na*2 floats (anchor_grid of this level, pixels). */
int cft_detect_decode(const float* head, int ldh, int B, int ny, int nx, int na, int no,
                      float stride, const float* anchors_px,
                      float* raw, float* z, long long z_rows, long long z_row0, void* stream);

/* Batched non-maximum suppression of Detect's z (the step after the forward: detect_twostream.py:86, test.py:129).
 * Replaces utils/general.py:455-544 (non_max_suppression), :299-306 (xywh2xyxy) and the torchvision.ops.nms call at
 * :527 -- results are bit-identical to them (fp32, same operation order, stable descending sort).
 *   pred   f32 [B, rows, no]: cx, cy, w, h, obj, cls[no-5]   (z of cft_detect_decode)
 *   keeps obj > conf_thres and conf = cls*obj > conf_thres (best class; every class when multi_label && nc > 1),
 *   classes/n_classes: optional HOST array of allowed class ids (n_classes = 0: all),
 *   boxes of different classes never suppress each other unless agnostic (class offset 4096 px, :525),
 *   at most 30000 candidates per image enter the suppression (:466, :521-522), at most max_det (<= 1024) leave it.
 *   out    f32 [B, max_det, 6]: x1, y1, x2, y2, conf, cls -- rows [0, counts[b]) valid, descending conf
 *   counts i32 [B]
 *   workspace: device scratch of cft_nms_workspace_bytes(B, rows, no - 5, multi_label) bytes, 8-byte aligned.
 * Not covered: the `labels` (autolabelling) branch (:482-489) and merge-NMS (hard-wired off at :470). */
long long cft_nms_workspace_bytes(int B, int rows, int nc, int multi_label);
int cft_nms(const float* pred, int B, int rows, int no, float conf_thres, float iou_thres, int max_det,
            int multi_label, int agnostic, const int* classes, int n_classes,
            void* workspace, long long workspace_bytes, float* out, int* counts, void* stream);

/* ---- profiling counters (CUDA events around every launch while enabled) ---- */
int cft_prof_enable(int on);            /* resets counters when turned on           */
int cft_prof_get(int kernel_id, double* total_ms, long long* launches);
long long cft_launch_count(void);       /* kernels launched by this library so far  */
/* debug: per-CTA clock samples (64 u64 slots per CTA, device buffer zeroed by the caller) written by the following
 * cft_conv2d launches; NULL turns the trace off.  Used by scripts/trace_conv.py only.                            */
int cft_debug_conv_trace(void* buf);
/* debug: {first CTA start, last CTA end} in %globaltimer ns of each of the next max_launches conv launches */
int cft_debug_conv_spans(void* buf, int max_launches);

/* The launch plan cft_conv2d would use for `a` (tiling, pipeline depth, shared memory) WITHOUT touching the device:
 * pointers in `a` are only checked for null / alignment.  Host-side tests walk every conv / linear shape of the
 * yolov5{s,l,x}-x3 graphs through it (tests/test_conv_plan_cpu.py). */
typedef struct cft_conv_plan {
  int ctas;                 /* 1, or 2 = CTA pairs (cta_group::2, UMMA M = 256)                         */
  int TW, TH;               /* output-pixel tile of one CTA (TW * TH * TB <= 128)                         */
  int Ho, Wo, tiles_x, tiles_y, m_tiles;
  int block_n, n_blocks;    /* N tile and their number (n_blocks * block_n >= Cout)                        */
  int num_tiles;            /* work items (pairs of m-tiles with ctas == 2) x n-blocks                     */
  int kelems, kchunks, ups; /* K unit (16 / 32 / 64 elements), units per tap, units per ring stage         */
  int halo;                 /* 3x3 row-reuse mode                                                          */
  int stages, a_slot, b_slot, b_res;   /* operand ring depth, slot bytes, resident-weight bytes           */
  int acc_stages, acc_cols; /* TMEM accumulator ring (acc_stages * acc_cols == 512)                        */
  int teams, stage_c;       /* epilogue teams, bytes per epilogue staging buffer                           */
  int smem_bytes;           /* dynamic shared memory of the launch                                          */
  int grid;                 /* CTAs launched                                                               */
  int TB;                   /* images per tile: the tile is TW x TH pixels of TB consecutive images, <= 128 px */
} cft_conv_plan;
int cft_debug_conv_plan(const cft_conv_args* a, cft_conv_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* CFT_B200_H */
