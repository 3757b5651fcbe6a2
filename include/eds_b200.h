/*
 * eds_b200.h -- C ABI of libeds_b200.so, the B200 (sm_100a) hot path of
 * duylebkHCM/EyeDiseaseSegmentation's inference-and-scoring pipeline.
 *
 * The reference is 100 % Python and has no FFI of its own; every entry point below
 * replaces a span of reference Python (cited as file:line relative to the reference
 * root) that the Python shim in eyediseasesegmentation_b200/ calls through ctypes.
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 (EDS_OK) or a negative error code; the message of the
 *     last failure on the calling thread is eds_last_error();
 *   - all tensor pointers are caller-owned DEVICE pointers unless the parameter
 *     name ends in _host; nothing is allocated, freed or synchronised inside;
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued on it and the
 *     call returns immediately;
 *   - activations are NHWC (channels innermost) with storage type `dtype`
 *     (EDS_BF16 or EDS_F32); arithmetic is fp32 (tensor-core convs: bf16 inputs,
 *     fp32 accumulate);
 *   - there is no CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef EDS_B200_H
#define EDS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define EDS_API __attribute__((visibility("default")))
#else
#define EDS_API
#endif

#define EDS_OK 0
#define EDS_ERR_INVALID (-1)
#define EDS_ERR_CUDA (-2)
#define EDS_ERR_UNSUPPORTED (-3)

#define EDS_BF16 0
#define EDS_F32 1

/* PR/ROC histogram geometry (see DESIGN.md "score key").  The key of a probability p (fp32) is monotone in p
 * and SYMMETRIC about 1/2, so a confident positive (p -> 1) is resolved as finely as a confident negative
 * (p -> 0) -- fp32 itself has 2^-24 steps just below 1, and a segmentation net's sigmoid lives there:
 *     q    = p >= 0.5 ? 1 - p : p                     (exact in fp32 for p in [0.5, 1])
 *     k    = clamp((int)(bits(q) >> EDS_PR_KEY_SHIFT) - EDS_PR_KEY_BIAS, 0, EDS_PR_HALF - 1)
 *     key  = p >= 0.5 ? EDS_PR_BINS - 1 - k : k
 * k = 0 is q < 2^-24, then 9 mantissa bits per binade for 2^-24 <= q < 1/2 (23 * 512 bins), and k =
 * EDS_PR_HALF - 1 is q = 1/2 exactly.  Scores that share a key are treated as tied. */
#define EDS_PR_KEY_SHIFT 14
#define EDS_PR_KEY_BIAS ((103 << 9) - 1)
#define EDS_PR_HALF (23 * 512 + 2)
#define EDS_PR_BINS (2 * EDS_PR_HALF)
/* thresholds of aucpr.py:53,128: 0,1e-5,1e-4,1e-3,1e-2,.1,...,.9,.99,.999,.9999,.99999,1 */
#define EDS_PR_NTHRESH 19

/* interpolation of the x2 decoder upsample */
#define EDS_UP_NEAREST 0   /* deep_supunetplusplus.py:49, smp Unet decoder */
#define EDS_UP_BILINEAR 1  /* unetplusplusstar.py:128 (align_corners=False) */
#define EDS_UP_NONE 2      /* plain torch.cat: x0 already has the output resolution */

EDS_API int eds_version(void);
EDS_API const char* eds_last_error(void);
/* 1 if a CUDA device with compute capability 10.x is present, else 0. */
EDS_API int eds_device_ok(void);
/* One-time per-process setup on the current device (constant tables, shared-memory
 * opt-ins, driver entry points).  Must be called once before any entry point is
 * used under CUDA-graph capture; otherwise the first call of each entry does it. */
EDS_API int eds_init(void);

/* ------------------------------------------------------------------ scoring
 * Replaces sklearn average_precision_score / roc_auc_score as called from
 * src/main/aucpr.py:24,38 and the 19-threshold loops of aucpr.py:60-81,136-170. */

/* Per-image score histograms.  prob: [n_images][n_pixels] fp32, gt: same shape u8
 * (non-zero = positive).  hist: [n_images][2][EDS_PR_BINS] u32 (class 0 = negatives),
 * straddle: [n_images][EDS_PR_NTHRESH][2] u32 = pixels that share the key of
 * threshold k and are strictly above it.  Both are ACCUMULATED into (caller zeroes).
 * splits = 0: one persistent wave of CTAs shares the linear range of all images' pixels (a CTA flushes
 * where its share crosses an image boundary); splits > 0: exactly that many CTAs per image. */
EDS_API int eds_pr_hist_f32(const float* prob, const uint8_t* gt, int64_t n_pixels, int n_images,
                    uint32_t* hist, uint32_t* straddle, int splits, void* stream);

/* The same histogram over a list of rectangles of ONE image (prob / gt: [img_h][img_w]); rects_host:
 * n_rects x (y, x, h, w), n_rects <= 32.  Used by the (image, tile) partition: every rank bins only the
 * pixels its tiles own, the per-image integer histograms of all ranks are summed by one all-reduce and
 * equal the single-process histogram bin for bin.  Accumulates into hist [2][EDS_PR_BINS] and
 * straddle [EDS_PR_NTHRESH][2] of that image. */
EDS_API int eds_pr_hist_rects_f32(const float* prob, const uint8_t* gt, int img_h, int img_w, int n_rects,
                          const int* rects_host, uint32_t* hist, uint32_t* straddle, void* stream);

/* Scan of the histograms.  Per image: ap[i] (sklearn AP on key-quantised scores),
 * roc[i] (trapezoid ROC-AUC), counts[i][k] = {tp, pp} at threshold k (strict >,
 * aucpr.py:63-66), totals[i] = {n_pos, n_neg}.  NaN when a class is empty. */
EDS_API int eds_pr_scan(const uint32_t* hist, const uint32_t* straddle, int n_images, double* ap,
                double* roc, uint64_t* counts, uint64_t* totals, void* stream);

/* --------------------------------------------------------------- TTA + paste
 * Replaces ttach.SegmentationTTAWrapper's de-augment + Merger('mean') (tta.py:92-99,
 * 173-180), the sigmoid (tta.py:114,210), the cv2.resize of the tile and the
 * overwrite paste (tta.py:211-213) / center-crop + resize (tta.py:117-119). */

/* logits: [V][B][S][S] fp32 (view-major).  view_maps_host: V*6 ints, de-augment map
 * of view v: out[i][j] += logits_v[a*i+b*j+c][d*i+e*j+f].  prob: [B][S][S] fp32 =
 * sigmoid((((l0+l1)+l2)+...)/V) in view order, or the raw mean when apply_sigmoid=0. */
EDS_API int eds_tta_merge(const float* logits, int V, int B, int S, const int* view_maps_host,
                  int apply_sigmoid, float* prob, void* stream);

/* Bilinear (half-pixel centres, edge clamp == cv2.INTER_LINEAR on fp32 ==
 * F.interpolate(align_corners=False)) resize of the crop
 * src[crop_y:crop_y+crop_h, crop_x:crop_x+crop_w] to out_h x out_w, written over
 * dst[dst_y:dst_y+out_h, dst_x:dst_x+out_w] (clipped to the dst extent). */
EDS_API int eds_resize_paste_f32(const float* src, int src_h, int src_w, int crop_y, int crop_x,
                         int crop_h, int crop_w, float* dst, int dst_h, int dst_w, int dst_y,
                         int dst_x, int out_h, int out_w, void* stream);

/* The sliding-window case of the above for a whole batch of tiles in one launch: dst[ys[b]+oy][xs[b]+ox] =
 * bilinear x2 of src[b] ([n_tiles][S][S] -> 2S x 2S each), pasted in index order with last-writer-wins
 * (tta.py:211-213); bit-identical to n_tiles calls of eds_resize_paste_f32.  n_tiles <= 32. */
EDS_API int eds_paste_tiles_x2_f32(const float* src, int n_tiles, int S, const int* ys_host, const int* xs_host,
                                   float* dst, int dst_h, int dst_w, void* stream);

/* One rank's share of the same paste under the (image, tile) partition (SURVEY.md 8e; replaces the
 * single-GPU tile loop of tta.py:170,207): src holds the n_src tiles first_tile .. first_tile+n_src-1 of the
 * image's tile list (ys/xs list ALL n_tiles tiles of the image, in make_grid order).  A pixel is written only
 * if no LATER tile of the list covers it, whether that tile is in src or on another rank -- every rank writes
 * exactly the pixels its tiles own, and the ranks' canvases sum to the single-process image.  dst_w % 4 == 0. */
EDS_API int eds_paste_tiles_owned_x2_f32(const float* src, int n_src, int first_tile, int n_tiles, int S,
                                 const int* ys_host, const int* xs_host, float* dst, int dst_h, int dst_w,
                                 void* stream);

/* The blend of one batch of tiles in ONE kernel (SURVEY.md 8d): eds_tta_merge (with sigmoid) followed by
 * eds_paste_tiles_owned_x2_f32, bit-identical to that pair, without the [B][S][S] intermediate; blocks that a later
 * tile covers completely are never read.  logits: [V][Bt][S][S]; the n_src tiles b0 .. b0+n_src-1 of that batch are
 * the tiles first_tile .. first_tile+n_src-1 of the image's list (ys/xs: all n_tiles origins, make_grid order).
 * Needs S % 64 == 0, dst_w % 4 == 0 and view offsets that keep 16-byte loads aligned (every flip / rot90 of a
 * square tile does): eds_tta_blend_supported() returns 1 when the arguments qualify. */
EDS_API int eds_tta_blend_supported(int V, int S, const int* view_maps_host, int dst_w);
EDS_API int eds_tta_blend_x2_f32(const float* logits, int V, int Bt, int b0, int n_src, int S,
                         const int* view_maps_host, int first_tile, int n_tiles, const int* ys_host,
                         const int* xs_host, float* dst, int dst_h, int dst_w, void* stream);

/* OPT-IN blend mode, not the reference's behaviour (the reference overwrites, tta.py:213; overwrite stays the
 * default and the parity mode): Gaussian-weighted accumulation of overlapping tiles.  For ONE tile src [S][S]:
 * acc[y][x] += w * v and wsum[y][x] += w over its 2S x 2S window at (dst_y, dst_x), v = the bilinear x2 value
 * the paste kernels write, w = window[oy] * window[ox] (device table of 2S floats).  Call once per tile in tile
 * order (deterministic fp32 sums), then eds_blend_finalize_f32: out = acc / wsum (0 where no tile wrote). */
EDS_API int eds_blend_tile_gaussian_x2_f32(const float* src, int S, int dst_y, int dst_x, const float* window,
                                   float* acc, float* wsum, int dst_h, int dst_w, void* stream);
EDS_API int eds_blend_finalize_f32(const float* acc, const float* wsum, int64_t n, float* out, void* stream);

/* Sliding-window tile fetch (tta.py:201-204): window [y0,y0+2S) x [x0,x0+2S) of an
 * HWC u8 RGB image -> 2x2 box mean with round-half-up (== cv2.resize of uint8 by
 * exactly 1/2) -> x/255, -mean, /std (archs/__init__.py:88-97) -> out [3][S][S] fp32. */
EDS_API int eds_preprocess_tile_u8(const uint8_t* img, int img_h, int img_w, int y0, int x0, int S,
                           const double* mean3_host, const double* std3_host, float* out,
                           void* stream);

/* ------------------------------------------------------------- network ops */

/* Encoder stem: 7x7 stride-2 pad-3 conv 3->64 + folded BN + ReLU (SENet layer0 /
 * ResNet conv1,bn1,relu).  x: [B][3][H][W] fp32 NCHW as the reference feeds it.
 * The V TTA views are folded into the loader: view v reads x through
 * aug_maps_host (V*6 ints, aug_v(x)[i][j] = x[a*i+b*j+c][d*i+e*j+f]); output image
 * index is v*B+b.  w: [7][7][3][64] fp32 (cout innermost, BN folded), bias: [64] fp32.
 * y: [V*B][H/2][W/2][64]. */
EDS_API int eds_stem_conv7x7s2(const float* x, int B, int H, int W, int V, const int* aug_maps_host,
                       const float* w, const float* bias, void* y, int dtype, void* stream);

/* The same stem on the tensor cores for bf16 outputs (stem_mma.cu): weights are packed once with
 * eds_stem_pack_weights (w [7][7][3][64] fp32 -> EDS_STEM_PACKED_ELEMS bf16: [64 couts][184], K ordered
 * (c, r, s') with the 7 horizontal taps padded to 8), then every call is
 * im2col-in-shared-memory + mma.sync.m16n8k16.  y: [V*B][H/2][W/2][64] bf16. */
#define EDS_STEM_PACKED_ELEMS (64 * 184)
EDS_API int eds_stem_pack_weights(const float* w, void* w_packed, void* stream);
EDS_API int eds_stem_conv7x7s2_mma(const float* x, int B, int H, int W, int V, const int* aug_maps_host,
                                   const void* w_packed, const float* bias, void* y, void* stream);

/* Implicit-GEMM convolution on the tcgen05 tensor cores (bf16 in, fp32 accumulate in
 * TMEM, TMA-staged NHWC tiles).  x: [N][H][W][C] bf16, w: [Cout][R][S][C] bf16 (BN
 * folded), bias: [Cout] fp32 or NULL, residual: [N][Ho][Wo][Cout] bf16 or NULL (added
 * before the ReLU), y: [N][Ho][Wo][Cout] bf16.  R=S in {1,3}, stride in {1,2},
 * C % 16 == 0, Cout % 16 == 0.  Replaces cuDNN for unetplusplusstar.py:40-63 and the
 * SENet / ResNet / axial-block convolutions. */
EDS_API int eds_conv2d_igemm_bf16(const void* x, int N, int H, int W, int C, const void* w,
                          const float* bias, int Cout, int R, int S, int stride, int pad,
                          int relu, const void* residual, void* y, void* stream);

/* The same with a squeeze-excitation scale in the epilogue: y = relu((conv + bias) * gate[n][co] + residual),
 * gate [N][Cout] fp32.  The SE bottleneck's conv3 has no activation, so the channel means its SE module squeezes
 * are an affine function of the channel means of conv3's INPUT (eds_affine_rows): the gate is known before conv3
 * runs, and `x * se(x) + residual -> ReLU` (Cadene SENet bottleneck, SURVEY A.1) happens on the accumulators
 * instead of in three more passes over the 4x wider map. */
EDS_API int eds_conv2d_igemm_bf16_gated(const void* x, int N, int H, int W, int C, const void* w,
                                const float* bias, const float* gate, int Cout, int R, int S, int stride,
                                int pad, int relu, const void* residual, void* y, void* stream);

/* Grouped convolution on the same tcgen05 pipeline (ResNeXt 3x3 conv2 with 32 groups: the torchvision Bottleneck
 * of resnext50_32x4d and the Cadene SEResNeXtBottleneck of se_resnext50_32x4d, both reached through smp 0.1.3's
 * get_encoder; replaces their cuDNN nn.Conv2d(groups=32)).  C == Cout, C % 64 == 0 and the channels per group
 * (C / groups) divide 64, so every 64-channel cout tile reads one 64-channel input chunk.  w_packed is the
 * block-diagonal [Cout][R][S][64] bf16 matrix: row co holds the 64 input channels of co's chunk, zero outside
 * co's group (BN folded in fp32 before the cast).  Other arguments as eds_conv2d_igemm_bf16.
 * eds_conv2d_igemm_grouped_supported returns 1 for the shapes the kernel takes; the others are rejected with
 * an eds_last_error() message. */
EDS_API int eds_conv2d_igemm_grouped_supported(int C, int Cout, int groups, int R, int S, int stride);
EDS_API int eds_conv2d_igemm_bf16_grouped(const void* x, int N, int H, int W, int C, const void* w_packed,
                                          const float* bias, int groups, int Cout, int R, int S, int stride, int pad,
                                          int relu, const void* residual, void* y, void* stream);

/* out[n][co] = sum_ci w[co][ci] * m[n][ci] + b[co]   (fp32; w [Cout][Cin] row-major, b may be NULL). */
EDS_API int eds_affine_rows(const float* m, int N, int Cin, const float* w, const float* b, int Cout, float* out,
                    void* stream);

/* Same contract on CUDA cores with fp32 accumulate for either storage type; used for
 * the fp32 parity mode and as the cross-check of the tensor-core kernel.  w has the
 * activation dtype. */
EDS_API int eds_conv2d_simt(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                    int Cout, int R, int S, int stride, int pad, int relu, const void* residual,
                    void* y, int dtype, void* stream);

/* Grouped form of eds_conv2d_simt (fp32 parity mode of the ResNeXt conv2, nn.Conv2d(groups=...)):
 * w [Cout][R][S][C / groups] in the activation dtype, output channel co reads the input channels of group
 * co / (Cout / groups).  Any group size. */
EDS_API int eds_conv2d_simt_grouped(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                    int groups, int Cout, int R, int S, int stride, int pad, int relu,
                                    const void* residual, void* y, int dtype, void* stream);

/* Segmentation head: 3x3 pad-1 conv C->classes with bias, fp32 logits out
 * ([N][classes][H][W], NCHW like the reference output).  w: [classes][3][3][C] fp32. */
EDS_API int eds_head_conv3x3(const void* x, int N, int H, int W, int C, const float* w, const float* bias,
                     int classes, float* logits, int dtype, void* stream);

/* MaxPool2d(k, stride, pad, ceil_mode): SENet layer0.pool (3,2,0,ceil), ResNet
 * maxpool (3,2,1), MHCA init_conv pool (2,2,0). */
EDS_API int eds_maxpool2d(const void* x, int N, int H, int W, int C, int k, int stride, int pad,
                  int ceil_mode, void* y, int dtype, void* stream);

/* AvgPool2d(2) followed by a per-channel affine (folded BN) and optional ReLU
 * (axial_attention_v2.py:256-259,277-279). */
EDS_API int eds_avgpool2_affine(const void* x, int N, int H, int W, int C, const float* scale,
                        const float* shift, int relu, void* y, int dtype, void* stream);

/* Global average pool: x [N][HW][C] -> mean [N][C] fp32. */
EDS_API int eds_channel_mean(const void* x, int N, int HW, int C, float* mean, int dtype, void* stream);

/* Squeeze-excite MLP on pooled features: gate = sigmoid(w2 * relu(w1 * mean + b1) + b2).
 * mean/gate: [N][C] fp32, w1: [Cr][C], w2: [C][Cr] fp32. */
EDS_API int eds_se_gate(const float* mean, int N, int C, int Cr, const float* w1, const float* b1,
                const float* w2, const float* b2, float* gate, void* stream);

/* y = relu(x * gate[n][c] + residual): tail of a SENet bottleneck. */
EDS_API int eds_se_scale_add_relu(const void* x, const float* gate, const void* residual, int N, int HW,
                          int C, void* y, int dtype, void* stream);

/* Decoder concat: y[N][2h][2w][C0 + sum Ci] = cat(up2x(x0), skip_1 .. skip_n) with
 * nearest or bilinear(align_corners=False) upsampling of x0 [N][h][w][C0]; with
 * EDS_UP_NONE the output is [N][h][w][...] (torch.cat of same-size maps,
 * unetplusplusstar.py:253-254).
 * skips_host / skip_channels_host: n_skips (<= 5) device pointers / channel counts. */
EDS_API int eds_upsample2x_concat(const void* x0, int N, int h, int w, int C0, int mode,
                          const void* const* skips_host, const int* skip_channels_host,
                          int n_skips, void* y, int dtype, void* stream);

/* 3x3 / stride 1 / pad 1 convolution for narrow outputs (Cout <= 128), same contract as
 * eds_conv2d_igemm_bf16 (bf16 NHWC in/out, w [Cout][3][3][C] with BN folded, fp32 bias, optional
 * residual and ReLU): persistent CTAs, halo-slab reuse of the input tile across the nine taps,
 * double-buffered TMEM accumulators (conv3x3_halo_sm100.cu).  eds_conv3x3_halo_supported returns 1
 * when a layer shape is eligible. */
EDS_API int eds_conv3x3_halo_supported(int C, int Cout, int R, int S, int stride, int pad);
EDS_API int eds_conv3x3_halo_bf16(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                  int Cout, int relu, const void* residual, void* y, void* stream);

/* 3x3 / stride 1 / pad 1 convolution for very narrow outputs (Cout <= 64), same contract as
 * eds_conv3x3_halo_bf16: the three horizontal taps of a kernel row run as ONE tcgen05.mma of N = 3 * Cout on a
 * shared A operand and the epilogue combines the three accumulators with a one-lane warp shuffle
 * (conv3x3_wide_sm100.cu) -- at N = Cout <= 64 a per-tap MMA is bound by shared-memory operand reads. */
EDS_API int eds_conv3x3_wide_supported(int C, int Cout, int R, int S, int stride, int pad);
EDS_API int eds_conv3x3_wide_bf16(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                  int Cout, int relu, const void* residual, void* y, void* stream);
EDS_API int eds_conv3x3_wide_bf16_2src(const void* x0, int C0, const void* x1, int C1, int N, int H, int W,
                                       const void* w, const float* bias, int Cout, int relu, const void* residual,
                                       void* y, void* stream);

/* 3x3 / stride 1 / pad 1 convolution for the full-resolution decoder tail on mma.sync (conv3x3_small.cu):
 * x [N][H][W][C], w [Cout][3][3][C] bf16, fp32 bias (may be NULL), optional ReLU -> y [N][H][W][Cout] bf16.
 * eds_conv3x3_small_supported returns 1 for C = 16 and Cout in {16, 32}, the only shapes it takes. */
EDS_API int eds_conv3x3_small_supported(int C, int Cout);
EDS_API int eds_conv3x3_small_bf16(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                   int Cout, int relu, void* y, void* stream);

/* Convolution of the channel concatenation cat(x0 [N][H][W][C0], x1 [N][H][W][C1]) without building it:
 * the K loop walks the channel chunks of x0, then of x1, through two tensor maps (stride 1; w is
 * [Cout][R][S][C0+C1]).  Same contract otherwise as the single-input forms above. */
EDS_API int eds_conv2d_igemm_bf16_2src(const void* x0, int C0, const void* x1, int C1, int N, int H, int W,
                                       const void* w, const float* bias, int Cout, int R, int S, int pad, int relu,
                                       const void* residual, void* y, void* stream);
EDS_API int eds_conv3x3_halo_bf16_2src(const void* x0, int C0, const void* x1, int C1, int N, int H, int W,
                                       const void* w, const float* bias, int Cout, int relu, const void* residual,
                                       void* y, void* stream);

/* ---- SCSE with deferred gates (the product path of the decoders; scse_gated.cu) ----------------
 * A "gated source" is a map whose SCSE gate has not been applied yet:
 *     value[n][p][c] = x[n][p][c] * (cgate[n][c] + sgate[n][p])     (cgate == sgate == NULL: plain map)
 * with cgate [N][C] fp32 (cSE, smp SCSEModule) and sgate [N][P] fp32 (sSE, already a probability).
 * Replaces attention1 / attention2 of DecoderBlock.forward (unetplusplusstar.py:151-161). */
typedef struct {
    const void* x;        /* [N][P][C] activations */
    const float* cgate;   /* [N][C] or NULL */
    const float* sgate;   /* [N][P] or NULL */
    int C;
} eds_gated_src;

/* Pass A over ONE source at its own resolution (P pixels):
 *   chan_mean[n][c_off + c] += mean_p value[n][p][c]      (row stride mean_stride; zero_mean clears
 *                                                           the whole [N][mean_stride] block first)
 *   dot[n][p] (+)= sum_c w_sse[c] * value[n][p][c]         (w_sse: this source's C-slice; dot may be
 *                                                           NULL; accumulate=0 starts a new map) */
EDS_API int eds_gated_stats(const void* x, const float* cgate, const float* sgate, int N, int P, int C,
                            const float* w_sse, float* chan_mean, int mean_stride, int c_off, int zero_mean,
                            float* dot, int accumulate, int dtype, void* stream);

/* The same pass for ALL consumers of a same-resolution skip source at once (dense decoder: a block output is
 * the skip of up to 4 later blocks; unetplusplusstar.py:239-263).  One read of the source; for consumer k:
 *   chan_mean[k][n][c_off[k] + c] += mean_p value[n][p][c]      (row stride mean_stride[k]; caller zeroes)
 *   dot[k][n][p]                  += sum_c w_sse[k][c] * value[n][p][c]              (caller zeroes)
 * n_consumers <= 4; the pointer arrays are host arrays of device pointers. */
EDS_API int eds_gated_stats_multi(const void* x, const float* cgate, const float* sgate, int N, int P, int C,
                                  int n_consumers, const float* const* w_sse, float* const* chan_mean,
                                  const int* mean_stride, const int* c_off, float* const* dot, int dtype,
                                  void* stream);

/* sgate[n][p] = sigmoid(up(dot0)[p] + dot1[p] + b_sse) on the output grid (up*h x up*w; mode as in
 * eds_upsample2x_concat; dot0 [N][h][w] or NULL, dot1 [N][up*h][up*w] or NULL; sgate may alias dot1). */
EDS_API int eds_sse_finalize(const float* dot0, const float* dot1, int N, int h, int w, int mode, float b_sse,
                             float* sgate, void* stream);

/* Pass B: y [N][2h][2w][sum C] = cat(up2x(value(src 0)), value(src 1..)) * (cgate[n][c] + sgate[n][p]);
 * source 0 is [N][h][w][C0] (nearest or bilinear x2), the others [N][2h][2w][Ck]; cgate/sgate NULL =
 * plain concat of the (gated) sources. */
EDS_API int eds_concat_gated(const eds_gated_src* srcs, int n_srcs, int N, int h, int w, int mode,
                             const float* cgate, const float* sgate, void* y, int dtype, void* stream);

/* The same with TWO dense destinations: y_up [N][2h][2w][C0] holds the upsampled source 0, y_skip
 * [N][2h][2w][sum C1..] the other sources, so every pixel row of either map is written whole (a single
 * Ctot-wide map is written in two interleaved passes, which costs DRAM write efficiency).  The pair is
 * consumed by eds_conv2d_igemm_bf16_2src / eds_conv3x3_halo_bf16_2src. */
EDS_API int eds_concat_gated_split(const eds_gated_src* srcs, int n_srcs, int N, int h, int w, int mode,
                                   const float* cgate, const float* sgate, void* y_up, void* y_skip, int dtype,
                                   void* stream);

/* y = x * (cgate[n][c] + sgate[n][p]) (materialise a gated map; y may alias x). */
EDS_API int eds_apply_gate(const void* x, const float* cgate, const float* sgate, int N, int HW, int C, void* y,
                           int dtype, void* stream);

/* Axial attention core (axial_attention_v2.py:100-135,178-213) for one axis.
 * qk: per pixel `heads` groups of [q(dqk) | k(dqk) | (v(dv) if v == NULL)] channels,
 * pixel stride qk_cstride elements; v: optional separate tensor with `heads` groups
 * of dv channels (MHCA), pixel stride v_cstride.  Tensors are [N][H][W][*]; axis 0
 * attends along H (one sequence per (n,w)), axis 1 along W.  L = length of that axis.
 * rel: [2*dqk+dv][2L-1] fp32 relative table; sim_scale: [heads][3] (qr, kr, dots BN
 * scales); out_scale/out_shift: [2][heads*dv] (kv part, out part) folded out_norm.
 * relu: apply the block's trailing ReLU (axial_attention_v2.py:279) to the output.
 * y: [N][H][W][heads*dv]. */
EDS_API int eds_axial_attention(const void* qk, int qk_cstride, const void* v, int v_cstride, int N, int H,
                        int W, int axis, int heads, int dqk, int dv, const float* rel,
                        const float* sim_scale, const float* out_scale, const float* out_shift,
                        int relu, void* y, int dtype, void* stream);

/* MHCA gate (unetplusplusstar.py:146-147): y = ori * up2x_bilinear(sigmoid(att)),
 * ori/y: [N][2h][2w][C], att: [N][h][w][C]. */
EDS_API int eds_mhca_gate(const void* ori, const void* att, int N, int h, int w, int C, void* y, int dtype,
                  void* stream);

/* Confusion counts of two uint8 masks binarised with `x > thr` (stat_result.py:30-57,
 * stat_result_vessel.py): counts[img][3] += { sum(gt & pred), sum(gt), sum(pred) } over n_pixels
 * bytes per image (the caller zeroes counts). */
EDS_API int eds_confusion_u8(const uint8_t* pred, const uint8_t* gt, int64_t n_pixels, int n_images, int thr_pred,
                             int thr_gt, uint64_t* counts, void* stream);

/* dtype conversion helpers for weights / debugging (n elements). */
EDS_API int eds_cast_f32_to_bf16(const float* x, void* y, int64_t n, void* stream);
EDS_API int eds_cast_bf16_to_f32(const void* x, float* y, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EDS_B200_H */
