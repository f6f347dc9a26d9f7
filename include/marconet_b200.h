/*
 * marconet_b200.h -- C ABI of libmarconet_b200.so (sm_100a).
 *
 * The reference (csxmli2016/MARCONet) has no FFI/plugin boundary of its own: its hot
 * path is Python modules in models/networks.py that call torch.nn.functional ops
 * (cuDNN / cuBLAS / ATen kernels) plus one third-party CUDA extension
 * (basicsr.ops.fused_act, models/networks.py:10).  This header is the boundary a
 * maintainer would bind instead of those calls: every entry point names the
 * reference call site(s) it replaces.  All functions
 *   - take raw DEVICE pointers and sizes (no torch types),
 *   - are asynchronous on the given stream (a cudaStream_t passed as void*),
 *   - never allocate persistent device memory (the caller owns every buffer,
 *     including workspaces),
 *   - return 0 on success or a negative mn_status; mn_last_error() returns a
 *     message for the calling thread.
 *
 * Activation layout everywhere: NHWC, fp32, channel stride given explicitly as
 * `*_cs` (floats per pixel in the underlying buffer) so that operators can read
 * from / write into channel slices of concatenated buffers without copies.
 */
#ifndef MARCONET_B200_H
#define MARCONET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    MN_OK = 0,
    MN_ERR_INVALID = -1,   /* bad argument (shape, alignment, null pointer)      */
    MN_ERR_CUDA = -2,      /* a CUDA runtime/driver call failed (see last error) */
    MN_ERR_UNSUPPORTED = -3,
    MN_ERR_WORKSPACE = -4  /* workspace too small                                 */
} mn_status;

typedef enum {
    MN_ACT_NONE = 0,
    MN_ACT_RELU = 1,       /* models/resnet.py:24,29                              */
    MN_ACT_LRELU02 = 2,    /* nn.LeakyReLU(0.2) / fused_leaky_relu slope          */
    MN_ACT_TANH = 3,       /* models/networks.py:321,375                          */
    MN_ACT_GELU = 4,       /* exact erf GELU, models/textvit_arch.py:47,87        */
    MN_ACT_SIGMOID = 5,    /* models/textvit_arch.py:50                           */
    MN_ACT_RSQRT_EPS = 6   /* rsqrt(v + 1e-8): demodulation, networks.py:286      */
} mn_act;

typedef enum {
    MN_PREC_FP32_SIMT = 0,   /* CUDA-core fp32 FMA implicit GEMM                       */
    MN_PREC_F16X3_TC = 1,    /* tcgen05 kind::f16, fp16 hi/lo split, 3 MMAs (~fp32)    */
    MN_PREC_BF16X3_TC = 2,   /* tcgen05 kind::f16, bf16 hi/lo split, 3 MMAs            */
    MN_PREC_F16X1_TC = 3     /* tcgen05 single pass fp16 (NOT parity grade)            */
} mn_precision;

const char* mn_last_error(void);
int mn_version(void);
/* Cap the number of CTAs the persistent tensor-core kernels launch (0 = one per SM).  Leaving a few SMs free lets NCCL's
 * copy kernels run beside them, so an asynchronous all-gather overlaps the next chunk of compute.  Returns the old value. */
int mn_set_max_ctas(int n);

/* Programmatic dependent launch (every kernel is launched with the programmatic-stream-serialization attribute so that its
 * launch overlaps the previous kernel's tail).  mn_set_pdl(0) turns the attribute off process-wide (returns the old
 * setting); the environment variable MN_PDL=0 does the same at load time. */
int mn_set_pdl(int on);
/* 1 when the current device is compute capability 10.x (tcgen05/TMA paths usable). */
int mn_device_is_sm100(void);

/* ------------------------------------------------------------------------------------
 * Implicit-GEMM convolution / linear layer.
 *
 * Replaces: every F.conv2d / nn.Conv2d / nn.Linear / F.linear on the path
 *   models/resnet.py:5-8,36,21-30 ; models/networks.py:294,299 (ModulatedConv2d, via the
 *   shared-weight reformulation y = demod[n,o] * sum_k W[o,k] * (s[n,c(k)] * x[n,k]) ),
 *   :336-408,501-505 (TSPSRNet convs, spectral norm folded at pack time),
 *   models/textvit_arch.py:34,42,46-51,57,61,86-88,101-102 (Linear = 1x1 conv on [M,1,1,K]),
 *   and the fused bias+leaky-relu of basicsr fused_act (networks.py:195,244-245).
 *
 *   y[n,oy,ox,o] = act( out_scale[n,o] * sum_{ky,kx,c} x[n,oy*sh+ky-ph,ox*sw+kx-pw,c] * w[(ky*KW+kx)*Cin+c][o]
 *                       + bias[o] + residual[n,oy,ox,o] ) * act_gain
 *   y2[n,oy,ox,o] = y[n,oy,ox,o] * y2_scale[n,o]      (optional second output: the
 *                   pre-modulated operand of the next modulated conv)
 *   Columns ox >= valid_w[n] are written as 0 when valid_w != NULL (ragged per-character
 *   windows keep their zero padding, models/networks.py:442-447).
 * ------------------------------------------------------------------------------------ */
typedef struct {
    const float* x;  int N, H, W, Cin, x_cs;
    const float* w;  int KH, KW, stride_h, stride_w, pad_h, pad_w, Cout;   /* w: [KH*KW*Cin][Cout] */
    float* y;        int y_cs;                 /* may be NULL when only y2 is wanted           */
    const float* bias;                         /* [Cout] or NULL                               */
    const float* out_scale; int out_scale_stride; /* [N][stride] (stride 0 -> Cout) or NULL      */
    const float* residual; int res_cs;         /* NHWC [N,OH,OW,res_cs] or NULL                */
    int res_broadcast_n;                       /* 1: residual has no batch dim (positional emb) */
    int act;  float act_gain;
    float* y2;       int y2_cs;  const float* y2_scale; int y2_scale_stride;   /* optional      */
    const int32_t* valid_w;                    /* [N] or NULL                                   */
    float* workspace; int64_t workspace_bytes; /* split-K partial sums; may be NULL (no split)  */
    int split_k;                               /* 0 = choose automatically, 1 = never split     */
    int precision;                             /* mn_precision                                  */
    /* tensor-core precisions only: weights pre-split by mn_conv_pack_weights_tc()                */
    const void* w_tc_hi; const void* w_tc_lo;  /* 16-bit [KH*KW][Cout][Cin] (K-major)            */
    const float* w_tc_scale;                   /* the 2-float scale record written by the packer */
    /* optional input transform fused into the tcgen05 kernel's operand-split stage (tensor-core path only):
     *   x' = swish( (x - mean[n,g]) * rstd[n,g] * gamma[c] + beta[c] ),  zero outside the image / beyond valid_w[n]
     * i.e. GroupNorm(32 channels per group) + swish of models/networks.py:508-512 applied while the A operand is built (its own
     * kernel instantiation: four lanes per halo row, constants in registers).  Needs OH*OW >= 128 (one sample per 128-pixel tile);
     * the sigmoid uses ex2.approx / rcp.approx (~2e-7 relative).  */
    const float* gn_mean_rstd;                 /* [N][Cin/32][2] from mn_groupnorm_stats, or NULL                          */
    const float* gn_gamma; const float* gn_beta;   /* [Cin]                                                                */
    int gn_swish;
    /* fp16-range management of the tensor-core precisions (the fp16 hi/lo split needs |x * x_scale| < 65504; the reference
     * computes in fp32, models/networks.py:294,299 / F.conv2d everywhere, and has no such limit):
     *   x_scale   power of two applied to the A operand before it is split and undone exactly in the epilogue (0 -> 1);
     *   x_absmax  optional DEVICE float: atomic max of |x * x_scale| over every element the kernel consumed (calibration);
     *   range_flag optional int32 the kernel STORES range_tag into when an operand element left the representable range
     *             (fp16 modes: |x * x_scale| >= 65504; every mode: Inf).  May point to pinned host memory (plain store). */
    float x_scale;
    float* x_absmax;
    int32_t* range_flag;
    int32_t range_tag;
    /* Per-sample base pointers of the SECOND output: sample n's [OH][OW][y2_cs] block is written at y2_ptrs[n] instead of
     * y2 + n*OH*OW*y2_cs (y2 must still be non-NULL to enable the output; it is not dereferenced).  The pointers may address the
     * memory of PEER GPUs (NVLink-mapped symmetric memory): the epilogue's stores then deliver every character's prior features
     * straight into the buffer of the rank that runs that character's SR decoder, tile by tile, while the MMAs of the next tile run
     * -- the exchange of the character-sharded path (reference consumer: models/networks.py:442-445, 475-478) without a separate
     * collective.  Tensor-core path only, layers whose samples are whole pixel tiles (OH*OW >= 128), no split-K. */
    float* const* y2_ptrs;
    /* GroupNorm statistics of the OUTPUT accumulated by the epilogue (models/networks.py:508-512: the tensor this convolution writes
     * is normalised next): per (sample, group of 32 output channels) sum and sum of squares of y, fp32 partials per warp and tile
     * added into [N][Cout/32][2] doubles with atomics (the caller zeroes the buffer; columns beyond valid_w contribute 0).
     * Tensor-core path only, whole-tile samples (OH*OW >= 128), no split-K; finish with mn_groupnorm_finalize. */
    double* gn_stats_out;
} mn_conv_params;

int mn_conv2d_nhwc(const mn_conv_params* p, void* stream);
/* Bytes of workspace mn_conv2d_nhwc wants for this problem (0 if it will not split). */
int64_t mn_conv2d_workspace_bytes(const mn_conv_params* p);
/* 1 if the tcgen05 path can run this geometry (stride 1, 3x3/pad1 or 1x1, Cin%64==0, Cout%64==0, H a multiple of 8 or a
 * power of two below 8, W a multiple of 128/min(H,8) or a power of two below that, a halo tile of at most 208 rows, 16-byte
 * aligned operands); 0 otherwise (mn_last_error() says why). */
int mn_conv2d_tc_supported(const mn_conv_params* p);
/* Split fp32 weights w:[taps*Cin][Cout] (the layout mn_conv2d_nhwc takes) into hi/lo 16-bit planes
 * [taps][Cout][Cin], pre-scaled by a power of two so the lo plane stays in the fp16 normal range.
 * hi, lo: taps*Cin*Cout 16-bit elements each; scale2: 2 floats {abs-max, 2^-S}. */
int mn_conv_pack_weights_tc(const float* w, int taps, int Cin, int Cout, int precision, void* hi, void* lo,
                            float* scale2, void* stream);

/* ------------------------------------------------------------------------------------
 * Generator (TSPGAN) operators
 * ------------------------------------------------------------------------------------ */
/* PixelNorm, models/networks.py:170-171:  y = x * rsqrt(mean(x^2, dim=1) + 1e-8), x:[N][C]. */
int mn_pixelnorm(const float* x, float* y, int N, int C, void* stream);

/* SelectText (models/networks.py:205-215) fused with the first conv's input modulation:
 *   out[n, yy, l*4+xx, c] = emb[labels[n*L+l]][c] * s[n*s_stride + c],   yy,xx in [0,4)
 * labels are int64 on the DEVICE and must already be range-checked by the host. */
int mn_select_text(const float* emb, const int64_t* labels, const float* s, int s_stride,
                   float* out, int N, int L, int C, void* stream);

/* Device-side range check of the character labels (the reference fails on the empty embedding slice at
 * models/networks.py:211): clamped[i] = clamp(labels[i], 0, classes-1); bit 0 of *err is raised when any label was out
 * of range.  For callers that must not touch the host between launches (CUDA-graph capture, SURVEY 8f n1). */
int mn_check_labels(const int64_t* labels, int64_t* clamped, int n, int classes, int32_t* err, void* stream);

/* Demodulation factors, models/networks.py:284-287 restated on the shared weight:
 *   demod[n][o] = rsqrt( sum_c s[n][c]^2 * wsq[c][o] + 1e-8 ),
 *   wsq[c][o] = scale^2 * sum_{ky,kx} W[o][c][ky][kx]^2 (packed once at load time). */
int mn_demod(const float* s, int s_stride, const float* wsq, float* demod, int N, int Cin, int Cout, void* stream);

/* All demodulation tables of one generator pass in a single launch.  descs: DEVICE array of n_layers records;
 * demod of layer l lands in out_all[n*out_stride + out_off .. + cout). */
typedef struct {
    const float* wsq;   /* [cin][cout] */
    int32_t s_off;      /* column offset of this layer's style inside s_all rows */
    int32_t cin, cout;
    int32_t out_off;
} mn_demod_desc;
int mn_demod_batched(const float* s_all, int s_stride, const mn_demod_desc* descs, int n_layers, int max_cout,
                     float* out_all, int out_stride, int N, void* stream);

/* y = (bilinear x2 upsample, align_corners=False, of x) * s[n][c]   (up=1)
 * y = x * s[n][c]                                                   (up=0);  s may be NULL.
 * Replaces nn.Upsample / F.interpolate(scale_factor=2, mode='bilinear') at
 * models/networks.py:268,293,318,360,370,415-416 (and the per-sample style multiply of :284). */
int mn_resample_modulate(const float* x, int x_cs, float* y, int y_cs, const float* s, int s_stride,
                         int N, int H, int W, int C, int up, void* stream);

/* ToRGB, models/networks.py:313-321: 1x1 modulated conv to 3 channels WITHOUT demodulation
 * + bias + bilinear-x2(skip) + tanh.
 *   out[n,p,o] = tanh( sum_c x[n,p,c]*s[n][c]*w[o][c] + bias[o] + up2(skip)[n,p,o] )
 * w:[3][C] already multiplied by 1/sqrt(C); skip:[N,H/2,W/2,3] or NULL; out:[N,H,W,3]. */
int mn_torgb(const float* x, int x_cs, const float* s, int s_stride, const float* w, const float* bias,
             const float* skip, float* out, int N, int H, int W, int C, void* stream);

/* ------------------------------------------------------------------------------------
 * SR decoder (TSPSRNet) operators
 * ------------------------------------------------------------------------------------ */
/* GroupNorm(32 channels/group, eps) + optional swish, models/networks.py:487-493,508-512.
 * Statistics run over H x valid_w[n] pixels per sample (valid_w NULL -> W); columns beyond
 * valid_w[n] are written as 0.  stats_ws: >= N*(C/cpg)*3 doubles of scratch. */
int mn_groupnorm_swish(const float* x, int x_cs, float* y, int y_cs, const float* gamma, const float* beta,
                       int N, int H, int W, int C, int cpg, float eps, int swish,
                       const int32_t* valid_w, double* stats_ws, void* stream);
/* The two halves of mn_groupnorm_swish, for fusing the normalisation into the consuming convolution:
 * statistics -> mean_rstd [N][C/cpg][2] fp32 (stats_ws: >= 2*N*(C/cpg) doubles), and the elementwise apply. */
int mn_groupnorm_stats(const float* x, int x_cs, int N, int H, int W, int C, int cpg, float eps,
                       const int32_t* valid_w, double* stats_ws, float* mean_rstd, void* stream);
/* Second half of mn_groupnorm_stats alone: sums [N][C/cpg][2] (sum, sum of squares; fp64) -> mean_rstd.  Used when the PRODUCING
 * convolution accumulated the sums in its epilogue (mn_conv_params.gn_stats_out): no separate read pass over the tensor. */
int mn_groupnorm_finalize(const double* stats_ws, int N, int H, int W, int C, int cpg, float eps, const int32_t* valid_w,
                          float* mean_rstd, void* stream);
int mn_groupnorm_apply(const float* x, int x_cs, float* y, int y_cs, const float* gamma, const float* beta,
                       const float* mean_rstd, int N, int H, int W, int C, int cpg, int swish,
                       const int32_t* valid_w, void* stream);

/* Per-character window table entry (host computes the integers bit-exactly like
 * models/networks.py:426-441 / :460-474). */
typedef struct {
    int32_t line;     /* b: which LR line the character belongs to                          */
    int32_t x1, x2;   /* window [x1,x2) in the line feature map                              */
    int32_t y1;       /* first column of the centred crop of the character prior            */
} mn_window;

/* AdaIN + concat, models/networks.py:442-445,518-533:
 *   out[i,:,:wv,0:C]  = (prior[i,:,y1:y1+wv,:] - mean_p)/std_p * std_l + mean_l
 *   out[i,:,:wv,C:2C] = feat[line,:,x1:x2,:]
 *   out[i,:,wv:,:]    = 0                        (wv = x2-x1, slot width = Wp)
 * std uses the unbiased variance + 1e-5.  prior:[Nc,H,Wp,C], feat:[B,H,W,C], out:[Nc,H,Wp,2C].
 * stats_ws: >= 6*Nc*C doubles of scratch. */
int mn_adain_concat(const float* prior, int prior_cs, const float* feat, int feat_cs, const mn_window* win,
                    float* out, int Nc, int H, int Wp, int W, int C, double* stats_ws, void* stream);

/* Write-back of the per-character modulation, models/networks.py:448-449 / :481-482:
 *   out[b,:,x,:] = feat + (feat*scale[i,:,x-x1,:] + shift[i,:,x-x1,:])  if column x of line b is
 *   owned by character i = owner[b*W + x] (the LAST character in program order whose window
 *   covers x; -1: none -> out = feat).  scale/shift:[Nc,H,Wp,C]. */
int mn_window_scatter(const float* feat, int feat_cs, const float* scale, const float* shift,
                      const int32_t* owner, const mn_window* win, float* out, int out_cs,
                      int B, int H, int W, int Wp, int C, void* stream);

/* The window integers of models/networks.py:426-441 / :460-474 computed on the device (no host round trip):
 *   center = (int)(locs[b*locs_stride + 2c] * W)   (fp32 multiply, truncation), x1 = max(center-half,0) as coded,
 *   x2 = min(center+half, W), y1 = half - (x2-x1)/2; valid[i] = x2-x1; owner[b*W+x] = last character whose window
 *   covers column x, else -1.  Characters of line b are win[line_first[b] .. line_first[b+1]) (device int32[B+1]);
 *   max_chars >= the longest line.  An empty window (reference: error at networks.py:443) raises bit 1 of *err and
 *   becomes a zero-width window. */
int mn_char_windows(const float* locs, int locs_stride, const int32_t* line_first, int B, int max_chars, int W, int half,
                    mn_window* win, int32_t* valid, int32_t* owner, int32_t* err, void* stream);

/* Style per character of a line wider than the encoder's input (pipeline.restore_wide_image, DESIGN "Wide lines").  The
 * encoder (TextViT: 64 tokens, LayerNorm(64) + Linear(64->16) over the token axis, models/textvit_arch.py) only takes 512
 * columns, so line b of a W-wide canvas is encoded as `segs` segments of seg_w columns, w[b*segs + s][0..dim) (row stride
 * w_stride).  Character c of line b (characters line_first[b] .. line_first[b+1], device int32[B+1]) gets
 *   center = (int)(locs[b*locs_stride + 2c] * W)     (fp32 multiply, truncation: the 32-level window centre,
 *                                                      models/networks.py:426, same arithmetic as mn_char_windows)
 *   seg    = clamp(floor(center / seg_w), 0, segs-1)
 *   styles[i*styles_stride + k] = w[(b*segs + seg)*w_stride + k],  seg_out[i] = seg  (seg_out may be NULL),  i = line_first[b]+c.
 * With segs == 1 every character gets its line's w, which is what test_sr.py:147-181 feeds TSPGAN (w0.repeat(n, 1)).
 * max_chars >= the longest line. */
int mn_char_segment_styles(const float* w, int w_stride, const float* locs, int locs_stride, const int32_t* line_first,
                           int B, int max_chars, int W, int seg_w, int segs, int dim, float* styles, int styles_stride,
                           int32_t* seg_out, void* stream);

/* The reference module's standalone helper functions on NCHW-contiguous tensors (rows = B*C, len = H*W); the hot path uses
 * the fused NHWC kernels above.
 *   mn_swish         x * sigmoid(x)                                                models/networks.py:492-493
 *   mn_row_mean_std  mean, sqrt(unbiased var + eps) of every row                   calc_mean_std_4D, :518-525
 *   mn_adain_rows    (prior - prior_mean)/prior_std * lq_std + lq_mean per row     adaptive_instance_normalization, :528-533 */
int mn_swish(const float* x, float* y, long long n, void* stream);
int mn_row_mean_std(const float* x, float* mean, float* stdv, int rows, int len, float eps, void* stream);
int mn_adain_rows(const float* prior, const float* prior_mean, const float* prior_std, const float* lq_mean,
                  const float* lq_std, float* out, int rows, int len, void* stream);

/* ------------------------------------------------------------------------------------
 * TextViT operators
 * ------------------------------------------------------------------------------------ */
/* nn.LayerNorm over the last dim (eps 1e-5), models/textvit_arch.py:41,46,53,58,85,99. */
int mn_layernorm(const float* x, float* y, const float* gamma, const float* beta, int rows, int dim,
                 float eps, void* stream);

/* nn.Linear for M <= 64 rows (the tokens of one text line), models/textvit_arch.py:42,46-51,57,61,86-88,101-102:
 *   y[M][N] = act(x[M][K] w[K][N] + bias[N] + residual[M][N]) * gain, K % 32 == 0, N % 16 == 0.  (Note: residual is added
 *   BEFORE the activation, like mn_conv2d_nhwc.) */
int mn_linear_small_m(const float* x, const float* w, const float* bias, const float* residual, float* y,
                      int M, int K, int N, int act, float gain, void* stream);

/* The same layer over a GATHERED x and `batches` independent row blocks (text lines): element (r, k) of batch z is
 *   x[z*x_batch_stride + r*x_row_stride + (k / x_seg_len)*x_seg_stride + k % x_seg_len]      (x_seg_len % 32 == 0),
 * y is dense [batches][M][N]; residual (optional) is [M][N] per batch at residual + z*res_batch_stride (0 = shared).
 * This is the TextViT patch embedding (models/textvit_arch.py:33-36: Rearrange 'b c (h p1) (w p2) -> b h w (p1 p2 c)' +
 * Linear(32768, 512) + positional embedding) reading the NHWC ResNet feature map [B,8,512,512] in place:
 *   M = 64 tokens, K = 8*8*512, x_row_stride = 8*512, x_seg_len = 8*512, x_seg_stride = 512*512, x_batch_stride = 8*512*512. */
int mn_linear_small_m_ex(const float* x, long long x_row_stride, long long x_batch_stride, int x_seg_len, long long x_seg_stride,
                         const float* w, const float* bias, const float* residual, long long res_batch_stride, float* y,
                         int batches, int M, int K, int N, int act, float gain, void* stream);

/* mn_linear_small_m_ex with a caller-owned scratch: deep-K layers (the patch embedding, K = 32768) are additionally split into
 * outer K slices whose raw partial tiles go to `workspace` (>= slices*batches*M*N floats are used when available) and are added
 * in slice order by a second kernel that runs the bias / residual / activation epilogue -- deterministic, no atomics.
 * workspace may be NULL (then identical to mn_linear_small_m_ex). */
int mn_linear_small_m_ws(const float* x, long long x_row_stride, long long x_batch_stride, int x_seg_len, long long x_seg_stride,
                         const float* w, const float* bias, const float* residual, long long res_batch_stride, float* y,
                         int batches, int M, int K, int N, int act, float gain, float* workspace, long long workspace_bytes,
                         void* stream);

/* LayerNorm over the TOKEN axis followed by Linear(T -> To) over the token axis, i.e. the
 * `x.permute(0,2,1)` -> LayerNorm(T) -> Linear -> permute(0,2,1) idiom at
 * models/textvit_arch.py:154 (T=64 -> 16) and :72 (64 -> 1).  x:[B,T,D] -> out:[B,To,D]. */
int mn_token_mix(const float* x, const float* gamma, const float* beta, const float* w, const float* bias,
                 float* out, int B, int T, int To, int D, float eps, void* stream);

/* Fused multi-head attention, models/textvit_arch.py:104-111: softmax(q k^T * scale) v for every
 * (batch, head) in one CTA.  qkv:[B,S,3*heads*dh] (q|k|v thirds, head-major inside), out:[B,S,heads*dh].
 * S <= 64, dh == 64. */
int mn_attention(const float* qkv, float* out, int B, int S, int heads, int dh, float scale, void* stream);

/* ------------------------------------------------------------------------------------
 * Layout conversion at the module boundary (the reference API is NCHW, models/networks.py:42,61,411)
 * ------------------------------------------------------------------------------------ */
int mn_nchw_to_nhwc(const float* x, float* y, int N, int C, int H, int W, int y_cs, void* stream);
int mn_nhwc_to_nchw(const float* x, int x_cs, float* y, int N, int C, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------
 * Script pre/post-processing on the device (SURVEY 8f n2; the reference does this on the host with cv2 / torchvision)
 * ------------------------------------------------------------------------------------ */
/* test_sr.py:98-111:  LQ = cv2.resize(img, (0,0), fx, fy, INTER_CUBIC)  (8-bit HWC image, OpenCV's own algorithm, bit-exact:
 * see csrc/image_ops.cu), pasted into a zero out_h x out_w canvas, ToTensor, Normalize((.5,.5,.5),(.5,.5,.5)).
 *   img:[h][w][cn] uint8 (device), dh = round_half_even(h*fy), dw = round_half_even(w*fx) (computed by the caller, as cv::resize
 *   does), lq:[cn][out_h][out_w] fp32, lq_u8 (optional): the resized bytes [dh][dw][cn].  Fails when dw > out_w (the script skips
 *   such images, test_sr.py:107-109). */
int mn_preprocess_lq_u8(const uint8_t* img, int h, int w, int cn, double fx, double fy, int dh, int dw,
                        float* lq, uint8_t* lq_u8, int out_h, int out_w, void* stream);

/* test_sr.py:198-201 (+ the uint8 rounding of cv2.imwrite, :231):
 *   out[b][y][x][C-1-c] = saturate_u8(round_half_even(clip(sr[b,c,y,x]*0.5 + 0.5, 0, 1) * 255)).
 * sr is addressed through element strides so that the channels_last view the SR module returns is read in place. */
int mn_postprocess_sr_u8(const float* sr, long long stride_n, long long stride_c, long long stride_h, long long stride_w,
                         uint8_t* out, int B, int C, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MARCONET_B200_H */
