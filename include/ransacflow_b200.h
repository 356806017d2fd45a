/*
 * ransacflow_b200 - C ABI of the B200 (sm_100a) implementation of RANSAC-Flow's
 * per-pair inference hot path.
 *
 * The reference (XiSHEN0220/RANSAC-Flow) is pure Python on PyTorch: it has no
 * FFI.  Its drop-in boundary is a set of Python modules (`outil`, `model`,
 * `coarseAlignFeatMatch`, `kornia.geometry`; SURVEY.md section 8b).  The Python
 * mirror of those modules (package `ransac-flow_b200/`) is a thin layer over
 * THIS library; every entry point below names the reference code it replaces
 * (paths relative to the reference checkout).
 *
 * Conventions
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers
 *     unless the parameter name ends in `_host`;
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = default stream);
 *     every call is asynchronous on that stream unless stated otherwise;
 *   - return value 0 = OK, non-zero = error (message: rf_last_error_string());
 *   - no allocation inside: scratch memory comes from the caller (`ws`), sized
 *     by the matching `*_workspace()` query;
 *   - activations are NHWC fp32, "ragged batch": `nimg` images of different
 *     (H, W) packed back to back in one buffer (`hw_host[2*i] = H_i`,
 *     `hw_host[2*i+1] = W_i`); outputs are packed the same way;
 *   - there is NO CPU fallback anywhere in this library.
 */
#ifndef RANSACFLOW_B200_H
#define RANSACFLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RF_MAX_IMGS 16

/* status written by rf_ransac_homography to *status_out (device int) */
#define RF_RANSAC_OK 0          /* H_out / nbInlier_out / mask_out valid                          */
#define RF_RANSAC_NONE 1        /* reference returns (None, 0, [], []): utils/outil.py:145-146      */
#define RF_RANSAC_NO_MODEL 2    /* reference raises TypeError at utils/outil.py:162 (bestParams None) */
#define RF_RANSAC_TOO_FEW 3     /* fewer than 4 matches (callers return None before calling)      */

int rf_version(void);
/* sha256 of the sources (csrc/, this header, compiler flags) the library was built from; the Python binding refuses a library
 * whose digest differs from the sources next to it */
const char* rf_source_digest(void);
const char* rf_last_error_string(void);
/* number of kernel launches issued through this library since load (bench.py's gpu_launches) */
uint64_t rf_launch_count(void);

/* ---------------------------------------------------------------- matching --
 * utils/outil.py:32-45 mutualMatching, fused: the NA x NB score matrix is never
 * written.  featA [NA][C], featB [NB][C] (K-major rows = one feature vector).
 * Outputs: idx1/idx2 (int64, capacity >= min(NA,NB)) sorted by idx1, *count.
 * precision: 0 = exact fp32 FMA (SIMT); 1 = 3xTF32 on tcgen05 tensor cores (hi*hi + lo*hi + hi*lo, C % 32 == 0);
 * 2 = fp16 split on tcgen05 (x = hi + lo * 2^-11 in fp16, cross terms in a second TMEM accumulator, C % 64 == 0): the
 * same 22 significand bits with half the MMAs per channel.
 * Precision 2 runs the persistent correlation kernel (one CTA per SM, two TMEM accumulator pairs, arg-max epilogue
 * overlapped with the next tile's MMAs) between a fused split / key-zeroing launch and a fused mutual-test + compaction
 * launch.  rf_corr_mutual_nn_launches() (host only) returns the number of launches a call with this precision makes
 * (NA, NB > 0): 4 / 6 / 3 for precision 0 / 1 / 2. */
size_t rf_corr_mutual_nn_workspace(int NA, int NB, int C, int precision);
int rf_corr_mutual_nn_launches(int precision);
int rf_corr_mutual_nn(const float* featA, int NA, const float* featB, int NB, int C,
                      int64_t* idx1_out, int64_t* idx2_out, int* count_out,
                      void* ws, size_t ws_bytes, int precision, void* stream);

/* The same with operands their producer already split (rf_l2norm_split_nhwc writes the normalised rows as fp16 hi / lo * 2^11
 * planes): no split pass.  A_hi / A_lo [NA][C], B_hi / B_lo [NB][C] fp16, C % 64 == 0.  Three graph nodes: memset of the
 * arg-max keys, the persistent fp16-split tcgen05 kernel (precision 2 of rf_corr_mutual_nn, identical arithmetic), the
 * column-driven mutual test + compaction. */
size_t rf_corr_mutual_nn_presplit_workspace(int NA, int NB);
int rf_corr_mutual_nn_presplit(const void* A_hi, const void* A_lo, int NA, const void* B_hi, const void* B_lo, int NB, int C,
                               int64_t* idx1_out, int64_t* idx2_out, int* count_out, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ RANSAC --
 * utils/outil.py:117-164 RANSAC + :102-113 ScoreRANSAC + :68-87 Homography +
 * :97-100 Prediction as ONE persistent kernel.  `samples` is the (nbIter,4)
 * int64 tensor `torch.randint` returned at utils/outil.py:120 (the draw stays
 * on the host side so the generator stream is the reference's).
 * match1/match2 [M][3] fp32 (x, y, 1).  `M_dev` (nullable) overrides M with a
 * device-side count (<= M) so no host sync is needed after matching.
 * Outputs: H_out[9] fp32, nbInlier_out int64, mask_out[M] u8, status_out int. */
/* `sample_mode`: how `samples` (nbIter x 4 int64) becomes match indices.
 *   RF_SAMPLES_INDEX    the tensor torch.randint(M, (nbIter, 4)) returned (utils/outil.py:120), used as is;
 *   RF_SAMPLES_MOD      arbitrary non-negative integers, reduced `% M` on the device (M = *M_dev);
 *   RF_SAMPLES_PHILOX64 full-range 64-bit generator words (`Tensor.random_(-2**63, None)` on CUDA = (x << 32) | y of one
 *                       curand4 call per element): index = x % M, which IS what torch.randint(M, (nbIter, 4), device='cuda')
 *                       returns from the same generator state (ATen random_from_to_kernel, range < 2^28, nbIter * 4 <=
 *                       256 * SMs * blocks-per-SM so that every element has its own Philox subsequence) - the reference's
 *                       seeded sample stream without knowing M on the host, usable inside a CUDA graph. */
#define RF_SAMPLES_INDEX 0
#define RF_SAMPLES_MOD 1
#define RF_SAMPLES_PHILOX64 2
size_t rf_ransac_workspace(int nbIter);
int rf_ransac_homography(const float* match1, const float* match2, int M, const int* M_dev,
                         const int64_t* samples, int sample_mode, int nbIter, float tolerance, int chunk,
                         float* H_out, int64_t* nbInlier_out, uint8_t* mask_out, int* status_out,
                         void* ws, size_t ws_bytes, void* stream);
/* utils/outil.py:68-87 Homography alone: X,Y [N][4][3] -> H [N][9] (for tests). */
int rf_homography_dlt(const float* X, const float* Y, int N, float* H_out, void* stream);
/* utils/outil.py:97-100 Prediction: err [N][M]. */
int rf_prediction(const float* match1, const float* match2, int M, const float* H, int N, float* err_out, void* stream);
/* coarseAlignFeatMatch.py (variant A :158-168, variant C :146-155): gather the
 * matched cell-centre coordinates into match1/match2 [M][3] = (x=H, y=W, 1).
 * valid16 (nullable, u8 [NB]) drops matches whose target cell is masked; the
 * surviving count goes to *count_out, order preserved. */
int rf_build_matches(const int64_t* idx1, const int64_t* idx2, const int* count_in,
                     const float* W1, const float* H1, const float* W2, const float* H2,
                     const uint8_t* valid16, float* match1_out, float* match2_out,
                     int64_t* idx2_kept_out, int* count_out, int capacity, void* stream);

/* ---------------------------------------------------------------- networks --
 * conv + folded BatchNorm (eval) + optional residual add + optional ReLU:
 * model/model.py:27-56,59-125,167-322; torchvision ResNet-50 bottlenecks.
 * x: ragged NHWC [sum HW][Cin]; w: [R*S*Cin][Cout] (tap-major, Cout contiguous);
 * bias [Cout] (nullable); residual: packed like y (nullable).
 * engine: 0 = fp32 SIMT implicit GEMM everywhere; 1 = TF32 tcgen05 implicit GEMM for the layers it
 * supports (stride 1, Cin % 32 == 0, 1x1 / 3x3; w_tc = same weights as [Cout][R*S*Cin]), the exact-fp32
 * SIMT kernel for the rest (3-channel stems, stride-2 convs);
 * 2 = fp16 tcgen05 implicit GEMM: x, residual, y and w_tc ([Cout][R*S*Cin]) hold IEEE fp16 elements behind the
 * same pointers (10-bit mantissa like TF32, half the HBM bytes, twice the tensor rate), fp32 accumulation and fp32
 * bias, outputs saturated to +-65504; needs Cin % 64 == 0, Cout % 8 == 0, 1x1 / 3x3, stride 1 / 2 and fails otherwise
 * (no fallback).  Used for the ResNet-50 conv4 trunk. */
#define RF_ENGINE_FP32 0
#define RF_ENGINE_TF32 1
#define RF_ENGINE_F16 2
#define RF_ENGINE_F16_OUT32 3   /* engine 2 operands, fp32 output rounded to TF32 after ReLU (3x3 / stride 1 / no residual):
                                   the layer that hands over from fp16 activations to a TF32 layer */
/* 4 = fp32-GRADE tcgen05 implicit GEMM ("f16x3"): every activation / weight element is carried as two fp16 values,
 * v = hi + lo * 2^-11 (hi = fp16(v), lo = fp16((v - hi) * 2^11): 22 significand bits), and every MAC is three kind::f16 MMAs
 * (hi*hi | hi*lo + lo*hi in a second TMEM accumulator).  x, residual and y are SPLIT tensors behind the same pointers:
 * [2][sum HW][C] fp16, plane 0 = hi, plane 1 = lo * 2^11 (4 bytes per element like fp32); w_tc = [2][Cout][R*S*Cin] fp16,
 * split the same way.  fp32 accumulation, bias, residual add and ReLU; needs Cin % 64 == 0, Cout % 8 == 0, 1x1 / 3x3,
 * stride 1 / 2 (no fallback).  This is the engine whose features reproduce the reference's fp32 arg-max (match set).
 * 5 = engine 4 operands with a plain fp32 [sum HoWo][Cout] output (any Cout, no residual): the heads' 49- / 1-channel layers. */
#define RF_ENGINE_SPLIT 4
#define RF_ENGINE_SPLIT_OUT32 5
int rf_conv2d_nhwc(const float* x, int nimg, const int* hw_host, int Cin,
                   const float* w, const float* w_tc, const float* bias, const float* residual,
                   int Cout, int R, int S, int stride, int pad, int relu, int engine,
                   float* y, void* stream);
/* Engine 4 only: a 1x1 convolution over TWO inputs whose channels are concatenated along K,
 *   y = act(W[:, :Cin1] x1 + W[:, Cin1:] x2[::stride2, ::stride2] + bias),
 * i.e. a ResNet bottleneck's conv3 + bn3 and its down-sampling branch (downsample.0 + downsample.1 of torchvision's Bottleneck,
 * which quick_start/coarseAlignFeatMatch.py:31-38 runs up to layer3) + the residual add + ReLU as ONE GEMM: the branch's output
 * never goes to HBM.  x1 / x2 / y split tensors; hw1 = sizes of x1 and y, hw2 = sizes of x2 ((h2 - 1) / stride2 + 1 == h1);
 * w_split = [2][Cout][Cin1 + Cin2] fp16; Cin1 % 64 == Cin2 % 64 == 0, Cout % 8 == 0, stride2 1 or 2. */
int rf_conv1x1_dual_split(const void* x1, const void* x2, int nimg, const int* hw1_host, const int* hw2_host, int Cin1, int Cin2,
                          int stride2, const void* w_split, const float* bias, int Cout, int relu, void* y, void* stream);
/* A whole network in one call: `layers_host[n]` executed in order over a ragged batch.  Buffers are numbered
 * "slots" (`slots_host[i]` = device pointer, caller-allocated); slot `layers[0].src` holds the input images
 * (`hw_host` = their sizes) and every layer's output sizes follow from its input's.  This is what the Python
 * mirrors of FeatureExtractor / NetFlowCoarse / NetMatchability / ResNet-50 conv4 call (one host call per
 * network instead of one per layer). */
#define RF_OP_CONV 0      /* conv + bias (+ residual slot) (+ ReLU) */
#define RF_OP_MAXPOOL 1   /* k, stride, pad */
#define RF_OP_BLUR 2      /* model/downsample.py: reflect-pad 1 + [1 2 1]^2/16, stride */
#define RF_OP_IM2COL 3    /* k x k x Cin patches (r, s, c order) zero-padded to Cout floats per output pixel: few-channel stems */
#define RF_OP_POOLBLUR 4  /* MaxPool2d(2, stride 1) + blur stride 2 fused (model/model.py:71-72) */
#define RF_OP_STEM7 5     /* engines 2 / 4 only: ResNet-50 stem fused (7x7 / stride 2 / pad 3 on the 3-channel fp32 image + bias + ReLU ->
                             fp16 / split, 64 channels) without the im2col matrix; w_f16 = [64][192] ([2][64][192] for engine 4) in
                             (r, s, c) order, zero padded */
#define RF_OP_CONV_DUAL 6  /* engine 4 only: rf_conv1x1_dual_split; src = x1 (Cin channels), src2 = x2 (Cin2 channels, stride2), w_f16 = [2][Cout][Cin + Cin2] */
#define RF_MAX_SLOTS 32
typedef struct rf_layer {
    int op;
    int src, dst, res;              /* slot indices; res < 0 = none */
    int Cin, Cout, k, stride, pad, relu;
    const float* w;                 /* [k*k*Cin][Cout] */
    const float* w_tc;              /* [Cout][k*k*Cin] */
    const float* bias;              /* [Cout] or NULL */
    const void* w_f16;              /* engine 2: [Cout][k*k*Cin] fp16; engine 4: [2][Cout][k*k*Cin] fp16 hi / lo planes (NULL otherwise) */
    int flags;                      /* engines 2 / 4: RF_LAYER_* */
    int src2, Cin2, stride2;        /* RF_OP_CONV_DUAL: second input slot, its channels and sampling stride (ignored otherwise) */
} rf_layer_t;
#define RF_LAYER_OUT_F32 1          /* conv: fp16 operands, fp32 output (RF_ENGINE_F16_OUT32; engine 4: RF_ENGINE_SPLIT_OUT32) */
#define RF_LAYER_TF32 2             /* conv: fp32 input and output on the TF32 engine (e.g. a 49-channel head after an OUT_F32 layer) */
/* engine 2: slots hold fp16 except the input of an RF_OP_IM2COL (the fp32 image; row length = Cout % 64 == 0), the
 * output of an RF_LAYER_OUT_F32 conv and the input / output of an RF_LAYER_TF32 conv; pooling and blur run in fp16. */
/* engine 4: slots hold split tensors ([2][P][C] fp16) except the fp32 input image of an RF_OP_IM2COL / RF_OP_STEM7 and the fp32
 * output of an RF_LAYER_OUT_F32 conv; pooling and blur rebuild the fp32 values and split their results again. */
int rf_run_layers(const rf_layer_t* layers_host, int n, void* const* slots_host, int nimg, const int* hw_host,
                  int engine, void* stream);
/* max pooling k x k / stride / zero-free padding: nn.MaxPool2d (model/model.py:71; torchvision resnet maxpool) */
int rf_maxpool2d_nhwc(const float* x, int nimg, const int* hw_host, int C, int k, int stride, int pad,
                      float* y, void* stream);
/* model/downsample.py:12-46: reflect-pad 1 + depthwise [1 2 1]x[1 2 1]/16, stride */
int rf_blur_downsample_nhwc(const float* x, int nimg, const int* hw_host, int C, int stride, float* y, void* stream);
/* F.normalize(x, dim=1): y = x / max(||x||_2, 1e-12) per pixel over C (P = total pixels).
 * mask (nullable, u8 [P]): masked pixels are written as zeros (quick_start/coarseAlignFeatMatch.py:143). */
int rf_l2norm_nhwc(const float* x, long long P, int C, const uint8_t* mask, float* y, void* stream);
/* same with a split input (engine 4: [2][P][C] fp16), fp32 output y (nullable); y_hi / y_lo (nullable, together): write the
 * normalised rows as fp16 hi / lo * 2^11 planes [P][C] - the operands of rf_corr_mutual_nn_presplit; C % 8 == 0 */
int rf_l2norm_split_nhwc(const void* x_split, long long P, int C, const uint8_t* mask, float* y, void* y_hi, void* y_lo, void* stream);
/* same with fp16 input (the engine-2 trunk's output), fp32 output; C % 8 == 0 */
int rf_l2norm_f16_nhwc(const void* x_f16, long long P, int C, const uint8_t* mask, float* y, void* stream);
/* model/model.py:129-160 CorrNeigh: x,y NHWC [N][h][w][C] -> out NHWC [N][h][w][ldo], channels >= k*k are
 * written as zeros (ldo = 64 makes the 49-channel volume a 128-byte-aligned operand for the conv engines);
 * round_tf32_out = 1 stores the values rounded to nearest TF32 (operand of the tensor-core heads);
 * round_tf32_out = 2 stores fp16 (out then holds N*h*w*ldo halves: the operand of the engine-2 heads) */
int rf_corr_neigh_nhwc(const float* x, const float* y, int N, int h, int w, int C, int k, int ldo, int round_tf32_out,
                       float* out, void* stream);
/* CorrNeigh(x, y) -> out_xy AND CorrNeigh(y, x) -> out_yx in one launch: the two volumes every PredFlowMask computes
 * (evaluation/evalHpatch/evaluation.py:29-30; evalCorr/evaluation.py:36-37) hold the same dot products,
 * out_yx[p][d] = out_xy[p+d][-d], so each product is computed once and stored twice (bit-identical to two
 * rf_corr_neigh_nhwc calls). */
int rf_corr_neigh_pair_nhwc(const float* x, const float* y, int N, int h, int w, int C, int k, int ldo, int round_tf32_out,
                            float* out_xy, float* out_yx, void* stream);
/* engine 4 form of the pair call: split outputs (fp16 hi / lo * 2^11 planes).  out12_split = CorrNeigh(x, y) as [2][P][ldo] (the
 * flow head's input), both_split = the two-image tensor [2][2P][ldo] = [CorrNeigh(x, y) ; CorrNeigh(y, x)] the matchability head
 * runs on (P = N*h*w; also usable with both_split = NULL for a single volume). */
int rf_corr_neigh_pair_split(const float* x, const float* y, int N, int h, int w, int C, int k, int ldo, void* out12_split, void* both_split,
                             void* stream);
/* model/model.py:226-233: softmax over k*k logits + expected offset -> flow NCHW [N][2][h][w] */
int rf_softmax_flow(const float* logits, int N, int h, int w, int k, float* flow_nchw, void* stream);
/* model/model.py:306: sigmoid, NHWC [P][1] -> [P] */
int rf_sigmoid(const float* x, long long n, float* y, void* stream);
/* ToTensor (+ Normalize): u8 HWC -> fp32 NHWC, (v/255 - mean)/std, exact torchvision op order.
 * normalize = 0 gives plain ToTensor.  (coarseAlignFeatMatch.py:63-66,106) */
int rf_preproc_u8(const uint8_t* img, long long npix, int normalize, float* out_nhwc, void* stream);
/* PIL ImagingResample (LANCZOS, 8bpc fixed point) on device: one pass.
 * coefficients come from rf_lanczos_coeffs_host (exact PIL arithmetic). */
int rf_resample_u8(const uint8_t* in, int in_h, int in_w, int channels, int horizontal,
                   const int* bounds, const int* kk, int ksize, int out_size, uint8_t* out, void* stream);
int rf_lanczos_coeffs_host(int in_size, int out_size, int* bounds_host, int* kk_host, int kk_capacity, int* ksize_out);

/* -------------------------------------------------------------------- warp --
 * kornia 0.1.4 HomographyWarper.warp_grid: H [N][9] -> grid [N][h][w][2] */
int rf_warp_grid(const float* H, int N, int h, int w, float* grid_out, void* stream);
/* F.grid_sample(bilinear, zeros).  Generic element strides so NCHW and NHWC both work.
 * in: (N,C,Hin,Win) with strides in_s[4] (N,C,H,W); grid [N][Hout][Wout][2]; out strides out_s[4]. */
int rf_grid_sample(const float* in, int N, int C, int Hin, int Win, const long long* in_s_host,
                   const float* grid, int Hout, int Wout, int align_corners,
                   float* out, const long long* out_s_host, void* stream);
/* F.interpolate(mode='bilinear', align_corners=False): NCHW [NC][h][w] -> [NC][H][W] */
int rf_upsample_bilinear(const float* in, int NC, int h, int w, int H, int W, float* out, void* stream);
/* PredFlowMask tail, evaluation/evalHpatch/evaluation.py:37-51 fused:
 * flowUp = clamp(interp(flowDown8) + grid); flow12 = grid_sample(coarse, flowUp);
 * match = interp(match12) [* grid_sample(interp(match21), flowUp)] * inside(flow12).
 * flowDown8 NCHW [2][h8][w8]; match12/match21 [h8][w8] (match21 nullable);
 * coarse [H][W][2]; outputs flow12 [H][W][2], match [H][W] (nullable), flowUp [H][W][2] (nullable). */
int rf_compose_fine(const float* flowDown8, const float* match12, const float* match21, int h8, int w8,
                    const float* coarse, int H, int W, int clamp, int align_corners,
                    float* flow12_out, float* match_out, float* flowUp_out, void* stream);
/* The same with a coarse grid of its own size, coarse [Hc][Wc][2] sampled at the (H, W) output positions: the second
 * level of the KITTI flow (evaluation/evalKITTI/evaluation.py:296-302: PredFlowMask with the resized image's flow and
 * the original image's grid) and the two-level recomposition of evaluation/evalKITTI/getResults.py:104-113. */
int rf_compose_fine_ex(const float* flowDown8, const float* match12, const float* match21, int h8, int w8,
                       const float* coarse, int Hc, int Wc, int H, int W, int clamp, int align_corners,
                       float* flow12_out, float* match_out, float* flowUp_out, void* stream);
/* remove_small_cc, evaluation/evalKITTI/evaluation.py:85-100 and evalKITTI/getResults.py:66-83, in place on
 * match [N][H][W]: every 8-connected component (skimage.measure.label's default for 2-D) of (match > match_th) whose
 * area fraction count / (H*W) is <= cc_th gets its matchability zeroed; cc_th == 0 leaves the map untouched. */
size_t rf_remove_small_cc_workspace(int H, int W);
int rf_remove_small_cc(float* match, int N, int H, int W, float match_th, double cc_th, void* ws, size_t ws_bytes, void* stream);

/* interpolate_flow_match, evaluation/evalKITTI/getResults.py:87-93: flow_out[p] = flow[nearest matched pixel of p]
 * (exact Euclidean distance; a matched pixel keeps its own flow).  flow / flow_out [H][W][2] (distinct buffers), matched
 * u8 [H][W] (non-zero = matched), index_out (nullable) int32 [H][W][2] = (row, col) of the chosen pixel.  Between
 * equidistant matched pixels the choice is this library's (documented at the kernel), not scipy's. */
size_t rf_fill_nearest_matched_workspace(int H, int W);
int rf_fill_nearest_matched(const float* flow, const uint8_t* matched, int H, int W, float* flow_out, int* index_out,
                            void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif
