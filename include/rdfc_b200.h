/*
 * rdfc_b200.h -- C ABI of librdfc_b200.so, the sm_100a implementation of the RDF-GAN / RDFC-GAN generator hot path.
 *
 * Plain pointers and sizes only (no torch / ATen types).  Every pointer is a DEVICE pointer unless its name ends in
 * `_host`.  Every entry point enqueues work on `stream` (a cudaStream_t passed as void*, NULL = legacy default
 * stream), never synchronises, and returns 0 on success or a negative rdfc_status; rdfc_last_error() then returns a
 * thread-local message.  Nothing here falls back to the CPU: without an sm_100 device the calls fail.
 *
 * Reference interfaces replaced (paths are relative to
 * /root/reference/RDFC-GAN/lib/models/generator/rdf_generator/ ; D = nlspn/deformconv):
 *
 *   rdfc_dcn_forward / rdfc_dcn_backward
 *       D/src/vision.cpp:7-12 -- pybind module `DCN`: deform_conv_forward/backward (mask == NULL) and
 *       modulated_deform_conv_forward/backward; dispatch D/src/modulated_deform_conv.h:10-44,46-86 and
 *       D/src/deform_conv.h; CUDA bodies D/src/cuda/modulated_deform_conv_cuda.cu:19-121,124-280.
 *   rdfc_nlspn_affinity_forward
 *       nlspn/nlspn_model.py:68-138  NLPSN._get_offset_affinity (conv_offset_aff + 8 confidence gathers + normalisation).
 *   rdfc_nlspn_propagate_forward
 *       nlspn/nlspn_model.py:140-144,157-173  the prop_time x ModulatedDeformConvFunction loop (C = 1, ones weight).
 *   rdfc_fuse_depth_forward
 *       rdf_generator.py:401-406  clamp + 2-way confidence softmax + weighted sum.
 *   rdfc_conv_forward
 *       encoder_decoder/common.py:29-61 conv_bn_relu / convt_bn_relu, torchvision BasicBlock convs
 *       (encoder_decoder/encoder_decoder.py:39-59), decode heads (rdf_generator.py:68-102) and the per-pixel
 *       EqualLinear of W-AdaIN (model_utils.py:39-50,72-75): NHWC implicit GEMM with a fused
 *       scale/shift (+residual) + activation epilogue.  `path` selects the tcgen05 bf16 kernel or the fp32 SIMT kernel.
 *   rdfc_heads_forward
 *       rdf_generator.py:374-398  the five Cout<=8 *_dec0 heads (+tanh / sigmoid), fused per branch.
 *   rdfc_instnorm_stats / rdfc_adain_apply
 *       model_utils.py:53-90 (AdaptiveInstanceNorm = W-AdaIN), :92-116 (AdaIN), :119-129 (IN).
 */
#ifndef RDFC_B200_H
#define RDFC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RDFC_ABI_VERSION 2

typedef enum {
    RDFC_OK = 0,
    RDFC_ERR_INVALID = -1,   /* bad argument (shape / divisibility / null pointer): the reference's AT_ASSERTM cases */
    RDFC_ERR_CUDA = -2,      /* CUDA runtime error (message carries cudaGetErrorString) */
    RDFC_ERR_UNSUPPORTED = -3
} rdfc_status;

/* RDFC_F16: the fp16 [hi | lo] split tensors of the fp32_tc training entry points only */
typedef enum { RDFC_F32 = 0, RDFC_F64 = 1, RDFC_BF16 = 2, RDFC_F16 = 3 } rdfc_dtype;

int rdfc_abi_version(void);
const char *rdfc_last_error(void);
/* number of kernels this library has launched in the calling process (for bench.py's gpu_launches) */
uint64_t rdfc_launch_count(void);

/* ------------------------------------------------------------------ DCN boundary ------------------------------ */
/* Shapes follow D/src/cuda/modulated_deform_conv_cuda.cu:47-76.
 *   input (B,Cin,H,W)  weight (Cout,Cin/group,kh,kw)  bias (Cout)  offset (B,dg*2*kh*kw,Ho,Wo)  mask (B,dg*kh*kw,Ho,Wo)
 *   output (B,Cout,Ho,Wo) contiguous NCHW, Ho = (H + 2 ph - (dh (kh-1) + 1)) / sh + 1.
 * `im2col_step` is validated exactly like the reference (B % min(B, im2col_step) == 0) and otherwise ignored. */
typedef struct {
    int B, Cin, H, W, Cout;
    int kh, kw, sh, sw, ph, pw, dh, dw;
    int group, deformable_group, im2col_step;
} rdfc_dcn_shape;

int rdfc_dcn_out_size(const rdfc_dcn_shape *s, int *Ho, int *Wo);

/* mask == NULL => DCN v1 (deform_conv_forward).  dtype: RDFC_F32 or RDFC_F64. */
int rdfc_dcn_forward(const void *input, const void *weight, const void *bias, const void *offset, const void *mask,
                     void *output, const rdfc_dcn_shape *s, int dtype, void *stream);

/* Any grad_* may be NULL (skipped).  grad_input is zero-filled by the callee before the scatter.
 * mask == NULL => DCN v1 (grad_mask must be NULL). */
int rdfc_dcn_backward(const void *input, const void *weight, const void *offset, const void *mask,
                      const void *grad_output, void *grad_input, void *grad_offset, void *grad_mask,
                      void *grad_weight, void *grad_bias, const rdfc_dcn_shape *s, int dtype, void *stream);

/* Flags of the *_ex backward entry points.  RDFC_DETERMINISTIC: the scatters that rdfc_dcn_backward,
 * rdfc_nlspn_affinity_backward and rdfc_nlspn_propagate_backward do with floating-point atomics (so that their last bits depend
 * on the execution order) accumulate instead in 64-bit fixed point, scaled by a power of two taken on the device from a bound on
 * the largest possible sum; the results are then bit-identical from run to run on the same GPU and build.  A NaN or Inf input
 * still gives non-finite results.  flags == 0 calls the entry point without _ex; other bits are refused before any launch.
 * The deterministic paths allocate their workspace stream-ordered (cudaMallocAsync) and free it before returning.  Bindings that
 * follow torch.use_deterministic_algorithms pass RDFC_DETERMINISTIC when torch.are_deterministic_algorithms_enabled(). */
#define RDFC_DETERMINISTIC 1

/* rdfc_dcn_backward's arguments plus flags */
int rdfc_dcn_backward_ex(const void *input, const void *weight, const void *offset, const void *mask,
                         const void *grad_output, void *grad_input, void *grad_offset, void *grad_mask,
                         void *grad_weight, void *grad_bias, const rdfc_dcn_shape *s, int dtype, void *stream, int flags);

/* ------------------------------------------------------------------ NLSPN ------------------------------------- */
typedef enum { RDFC_AFF_AS = 0, RDFC_AFF_ASS = 1, RDFC_AFF_TC = 2, RDFC_AFF_TGASS = 3 } rdfc_affinity;

/* guidance (B,8,H,W) fp32 NCHW; confidence (B,1,H,W) or NULL when conf_prop == 0;
 * conv_w (24,8,3,3), conv_b (24) = conv_offset_aff; aff_scale = aff_scale_const (device pointer to 1 float).
 * Writes offset (B,18,H,W) and aff (B,9,H,W) in the reference layout (centre tap inserted at index 4). k_f = 3 only. */
int rdfc_nlspn_affinity_forward(const float *guidance, const float *confidence, const float *conv_w,
                                const float *conv_b, const float *aff_scale, int affinity, int conf_prop,
                                float *offset, float *aff, int B, int H, int W, void *stream);

/* Optional output fusion applied by the LAST propagation iteration (rdf_generator.py:401-406): the result is clamped to [-1,1]
 * (= depth_map_2, written to `out`) and  pred = softmax([c1, c2]) . [d1, clamp(result)]  is written as well.  All (B,1,H,W) fp32. */
typedef struct {
    const float *d1, *c1, *c2;
    float *pred;
} rdfc_fuse_out;

/* feat_init (B,1,H,W); offset (B,18,H,W); aff (B,9,H,W); feat_fix (B,1,H,W) or NULL; out (B,1,H,W);
 * scratch: B*H*W floats (ping-pong buffer, may not alias anything else);
 * inter: NULL or prop_time*B*H*W floats receiving every iteration's result (the reference's list_feat).
 * preserve_input: every iteration reads feat blended with feat_fix where feat_fix > 0 (nlspn_model.py:159-160,169; folded into the
 * kernel's staging).  clamp_out != 0 additionally clamps the final result to [-1,1] (rdf_generator.py:401); fuse: NULL or the
 * output fusion above (implies the clamp). */
int rdfc_nlspn_propagate_forward(const float *feat_init, const float *offset, const float *aff,
                                 const float *feat_fix, int preserve_input, float *out, float *scratch,
                                 float *inter, int B, int H, int W, int prop_time, int clamp_out,
                                 const rdfc_fuse_out *fuse, void *stream);

/* The same two stages over a PACKED fp16 stream instead of the fp32 offset / aff planes (bf16 inference mode): per pixel 24
 * halves = (dy, dx) of the 8 non-centre taps + their 8 affinities (the centre tap's offset is zero and its affinity is
 * 1 - sum of the rounded others, so every iteration stays an exact affine combination): 48 B instead of 100 B streamed per
 * pixel and iteration.  Pixel g = b*H*W + y*W + x is stored as three 16-byte chunks at byte offset
 * (g/32)*1536 + c*512 + (g%32)*16, c = 0..2.  `packed`: 16-byte aligned, rdfc_nlspn_packed_bytes(B,H,W) bytes. */
size_t rdfc_nlspn_packed_bytes(int B, int H, int W);
int rdfc_nlspn_affinity_forward_packed(const float *guidance, const float *confidence, const float *conv_w,
                                       const float *conv_b, const float *aff_scale, int affinity, int conf_prop,
                                       void *packed, int B, int H, int W, void *stream);
int rdfc_nlspn_propagate_forward_packed(const float *feat_init, const void *packed, const float *feat_fix,
                                        int preserve_input, float *out, float *scratch, int B, int H, int W,
                                        int prop_time, int clamp_out, const rdfc_fuse_out *fuse, void *stream);

/* Backward of rdfc_nlspn_affinity_forward up to the conv output (training): grad_offset (B,18,H,W), grad_aff (B,9,H,W) ->
 * grad_conv (B,24,H,W) = dL/d conv_offset_aff(guidance) (the caller back-propagates the 8 -> 24 channel conv itself),
 * grad_confidence (B,1,H,W, overwritten; required when conf_prop) through the 1x1 DCN gathers of nlspn_model.py:96-119 (their
 * offsets are detached in the reference), grad_aff_scale (1 float, overwritten; NULL to skip) for TGASS's learnable scale
 * (nlspn_model.py:86-87).  offset = the forward's output.  fp32 atomics in the confidence scatter and the scale reduction
 * (rdfc_nlspn_affinity_backward_ex with RDFC_DETERMINISTIC has none). */
int rdfc_nlspn_affinity_backward(const float *guidance, const float *confidence, const float *conv_w, const float *conv_b,
                                 const float *aff_scale, int affinity, int conf_prop, const float *offset,
                                 const float *grad_offset, const float *grad_aff, float *grad_conv, float *grad_confidence,
                                 float *grad_aff_scale, int B, int H, int W, void *stream);

/* Backward of rdfc_nlspn_propagate_forward (training; replaces the reference's 18 ModulatedDeformConvFunction.backward calls,
 * modulated_deform_conv_cuda.cu:124-280 with weight = 1, bias = 0, as nlspn_model.py:140-175 issues them).
 * grad_out (B,1,H,W) = dL/d out; grad_inter NULL or (prop_time,B,1,H,W) = dL/d list_feat[t]; feat_init, offset, aff, feat_fix,
 * preserve_input as in the forward; inter = the forward's `inter` buffer (required when prop_time > 1).
 * Writes grad_feat_init (B,1,H,W), grad_offset (B,18,H,W), grad_aff (B,9,H,W) (overwritten, not accumulated).
 * scratch: (prop_time + 1) * B*H*W floats.  The input-gradient scatter uses fp32 atomics (as the reference's col2im does), so
 * the last bits depend on the execution order (rdfc_nlspn_propagate_backward_ex with RDFC_DETERMINISTIC: they do not). */
int rdfc_nlspn_propagate_backward(const float *grad_out, const float *grad_inter, const float *feat_init,
                                  const float *inter, const float *offset, const float *aff, const float *feat_fix,
                                  int preserve_input, float *grad_feat_init, float *grad_offset, float *grad_aff,
                                  float *scratch, int B, int H, int W, int prop_time, void *stream);

/* The two NLSPN backwards with a trailing flags argument (RDFC_DETERMINISTIC, see rdfc_dcn_backward_ex).  Deterministic, the
 * propagation backward runs two kernels per iteration instead of one (the fixed-point scatter, then its conversion fused with the
 * per-iteration finalisation) and the affinity backward four instead of one. */
int rdfc_nlspn_affinity_backward_ex(const float *guidance, const float *confidence, const float *conv_w, const float *conv_b,
                                    const float *aff_scale, int affinity, int conf_prop, const float *offset,
                                    const float *grad_offset, const float *grad_aff, float *grad_conv, float *grad_confidence,
                                    float *grad_aff_scale, int B, int H, int W, void *stream, int flags);
int rdfc_nlspn_propagate_backward_ex(const float *grad_out, const float *grad_inter, const float *feat_init,
                                     const float *inter, const float *offset, const float *aff, const float *feat_fix,
                                     int preserve_input, float *grad_feat_init, float *grad_offset, float *grad_aff,
                                     float *scratch, int B, int H, int W, int prop_time, void *stream, int flags);

/* pred = softmax([c1,c2]) . [d1, clamp(d2)] ; d2_clamped receives clamp(d2,-1,1) (may alias d2). n = B*H*W. */
int rdfc_fuse_depth_forward(const float *d1, const float *c1, const float *d2, const float *c2, float *d2_clamped,
                            float *pred, size_t n, void *stream);

/* ------------------------------------------------------------------ dense part (NHWC) ------------------------- */
typedef enum { RDFC_ACT_NONE = 0, RDFC_ACT_RELU = 1, RDFC_ACT_LEAKY02 = 2, RDFC_ACT_TANH = 3, RDFC_ACT_SIGMOID = 4 }
    rdfc_act;
/* RDFC_PATH_UMMA_F32X3: fp32 NHWC in / out on the bf16 tensor cores with split operands (x = x_hi + x_lo, W = W_hi + W_lo;
 * x_hi W_hi + x_hi W_lo + x_lo W_hi accumulated in fp32): the <= 1e-4 parity mode at tensor-core speed.  `weight` is the UMMA
 * packing of [W_hi ; W_lo ; W_hi] along Cin (3 * Cin input channels); needs `workspace`. */
typedef enum { RDFC_PATH_SIMT_F32 = 0, RDFC_PATH_UMMA_BF16 = 1, RDFC_PATH_UMMA_F32X3 = 2 } rdfc_conv_path;

/* A view of an NHWC tensor: element (b,y,x,c) lives at ptr[((b*H + y)*W + x)*pix_stride + c].
 * nchw != 0 switches to (B,C,H,W) contiguous addressing (pix_stride ignored) -- SIMT path only. */
typedef struct {
    void *ptr;
    int dtype;       /* RDFC_F32 or RDFC_BF16 */
    int C;           /* channels of the view */
    int pix_stride;  /* elements between consecutive pixels (>= C; lets a view be a channel slice of a concat buffer) */
    int nchw;
} rdfc_view;

typedef struct {
    int B, Hi, Wi;          /* input spatial size */
    int Ho, Wo;             /* output spatial size actually written (ConvTranspose: may be cropped, rdf_generator.py:249-256) */
    int kh, kw, stride, pad;
    int transposed;         /* 1 = ConvTranspose2d(k3,s2,p1,op1) gather form; weights packed accordingly */
    int act;                /* rdfc_act */
    int path;               /* rdfc_conv_path */
    rdfc_view in;           /* Cin = in.C */
    rdfc_view in2;          /* optional second source concatenated after `in` along C (ptr == NULL: unused); SIMT only */
    rdfc_view out;          /* Cout = out.C */
    rdfc_view residual;     /* optional (ptr == NULL: none): added after scale/shift, before the activation */
    const void *weight;     /* packed by rdfc_gan_b200.engine: SIMT: fp32 [kh*kw][Cin][Cout]; UMMA: bf16 [kh*kw][Cin/8][Cout padded to 16][8] */
    const float *scale;     /* per-Cout multiplier (folded BN gamma/sqrt(var+eps)) or NULL (= 1) */
    const float *shift;     /* per-Cout addend (folded BN beta - mean*scale, or the conv bias) or NULL (= 0) */
    void *workspace;        /* RDFC_PATH_UMMA_F32X3 only: B*Hi*Wi*Cin*4 bytes, 128-byte aligned (the split input) */
    size_t workspace_bytes;
} rdfc_conv_desc;

int rdfc_conv_forward(const rdfc_conv_desc *d, void *stream);

/* Fused decode heads (rdf_generator.py:372-398): the <= 16 *_dec0 output columns that read one NHWC bf16 view, each a
 * 3x3 / stride-1 / pad-1 convolution with its own bias and activation, as ONE launch: a tensor-core 1x1 GEMM to
 * 9 * ncols columns  Y[p, t * ncols + q] = W_q[:, tap t] . x[p, :]  followed (same kernel, through shared memory) by
 * out_q[p] = act_q(bias_q + sum_t Y[p + d_t, t * ncols + q]).  Column q is written as an fp32 plane:
 * out[q][b * out_bstride[q] + y * W + x]  -- so depth / confidence maps and the NCHW guidance tensor the NLSPN
 * kernels read come straight out of the epilogue. */
typedef struct {
    int B, H, W;
    rdfc_view in;                /* bf16 (or fp32, see workspace) NHWC, C % 32 == 0 */
    const void *weight;          /* bf16 [1][C/8][NP][8], NP = 9 * ncols padded to 16, row t * ncols + q = tap t (= ky*3+kx) of column q */
    const float *shift;          /* device, NP floats: bias of column q at index q (q < ncols), the rest unused */
    int ncols;                   /* 1..16 */
    int act[16];                 /* rdfc_act per column */
    float *out[16];              /* device plane base pointers */
    long long out_bstride[16];   /* elements between consecutive images of a plane */
    void *workspace;             /* only when `in` is an fp32 view (tensor-core fp32 mode: weight packs [W_hi ; W_lo ; W_hi], fp16): */
    size_t workspace_bytes;      /*   B*H*W*C*4 bytes, 128-byte aligned, receives the split input */
} rdfc_heads_desc;

int rdfc_heads_forward(const rdfc_heads_desc *d, void *stream);

/* Fused input stems (rdf_generator.py:286-292: rgb_branch_en1, depth_branch_en1_rgb, depth_branch_en1_depth; each a
 * conv_bn_relu 3x3 / stride 1 / pad 1 of encoder_decoder/common.py:29-43 over 3 / 3 / 1 input channels): ONE
 * tensor-core launch.  The producer warps build the im2col rows k = ci*9 + ky*3 + kx (in0's channels first, then
 * in1's nine taps, zero-padded to 64) straight from the fp32 NCHW inputs; the filter bank is a 1x1 UMMA weight with
 * Cin = 64 whose columns [0, out.C) are written to `out` and [out.C, out.C + out2.C) to `out2` (bf16 NHWC slices). */
typedef struct {
    int B, H, W;
    const float *in0;            /* fp32 NCHW (B, C0, H, W) */
    int C0;                      /* C0 + (in1 != NULL) <= 4 input planes */
    const float *in1;            /* fp32 NCHW (B, 1, H, W) or NULL */
    rdfc_view out, out2;         /* bf16 NHWC; out2.ptr == NULL: single destination */
    const void *weight;          /* bf16 [1][8][CoutP][8], CoutP = out.C + out2.C padded to 16 */
    const float *scale, *shift;  /* per column (folded BatchNorm / bias) */
    int act;                     /* rdfc_act: none / ReLU / LeakyReLU(0.2) */
} rdfc_stem_desc;

int rdfc_stem_forward(const rdfc_stem_desc *d, void *stream);

/* Stem inputs with many channels (RDF-GAN's 40-channel guidance, rdf_gan_generator.py:235-245): fp32 NCHW in0 (B,C0,H,W)
 * and optional in1 (B,1,H,W) -> one bf16 NHWC tensor (B,H,W,Cpad) = [in0 | in1 | zeros], which rdfc_conv_forward then reads
 * on the tensor cores.  Cpad % 8 == 0, Cpad <= 128. */
int rdfc_pack_stem_input(const float *in0, int C0, const float *in1, void *out_bf16, int Cpad, int B, int H, int W, void *stream);

/* W-AdaIN with the style projection fused (model_utils.py:53-90 without `weighting`): ONE tensor-core launch computes
 * the per-pixel EqualLinear  [gamma | beta] = style[p, :] . W^T + bias  (a 1x1 convolution Cd -> 2C) and applies
 *   out[p, c] = gamma[p, c] * (x[p, c] - mean[b, c]) * rstd[b, c] + beta[p, c]
 * (times the optional per-pixel weights of `weighting=True`) in its epilogue, so the (B,H,W,2C) gamma/beta tensor never exists.  The filter rows are packed in tiles of
 * `rdfc_wadain_tile(C)` columns: tile t = gamma rows of channels [t*h, (t+1)*h) followed by their beta rows, h = tile/2;
 * `bias` is permuted the same way.  mean / rstd: (B, C) fp32 from rdfc_instnorm_stats. */
typedef struct {
    int B, H, W;
    rdfc_view style;             /* bf16 NHWC, Cd % 32 == 0 */
    rdfc_view x;                 /* bf16 NHWC, C channels, C % 64 == 0 */
    rdfc_view out;               /* bf16 NHWC, C channels */
    const void *weight;          /* bf16 [1][Cd/8][2C][8], rows permuted as described */
    const float *bias;           /* 2C floats, permuted */
    const float *mean, *rstd;    /* (B, C) */
    rdfc_view gwbw;              /* optional (ptr NULL: none): bf16 NHWC, 2C channels [gamma weight | beta weight] =
                                  * gamma/beta_weight_layer(x) (model_utils.py:84-88): out = gw*gamma*IN(x) + bw*beta */
} rdfc_wadain_conv_desc;

int rdfc_wadain_tile(int C);
int rdfc_wadain_conv_forward(const rdfc_wadain_conv_desc *d, void *stream);

/* per-(b,c) mean and 1/sqrt(var+eps) over the pixels of an NHWC view.  unbiased != 0 divides by (n-1) (AdaIN,
 * model_utils.py:98) and returns sqrt(var+eps) in `rstd` instead of its reciprocal when want_std != 0.
 * partial: workspace of B*nchunk*C*2 floats with nchunk = rdfc_instnorm_nchunk(H*W). mean/rstd: (B,C) fp32. */
int rdfc_instnorm_nchunk(int npix);
int rdfc_instnorm_stats(const rdfc_view *x, int B, int H, int W, float eps, int unbiased, int want_std,
                        float *partial, float *mean, float *rstd, void *stream);

/* W-AdaIN apply (model_utils.py:76-88): out[p,c] = gw*gamma*(x-mean)*rstd + bw*beta with
 * gamma = gb[p, c], beta = gb[p, C + c]  (gb = EqualLinear output, NHWC view with 2C channels) and optional
 * gw/bw = gamma/beta_weight_layer(x) views (ptr NULL = 1). */
int rdfc_wadain_apply(const rdfc_view *x, const rdfc_view *gb, const rdfc_view *gw, const rdfc_view *bw,
                      const float *mean, const float *rstd, const rdfc_view *out, int B, int H, int W, void *stream);

/* AdaIN apply (model_utils.py:102-116): out = (x - cmean)/cstd * sstd + smean, all (B,C) statistics. */
int rdfc_adain_apply(const rdfc_view *x, const float *cmean, const float *cstd, const float *smean,
                     const float *sstd, const rdfc_view *out, int B, int H, int W, void *stream);

/* plain per-channel affine normalise (IN fuse, model_utils.py:119-129): out = (x - mean) * rstd, written into `out`
 * (a channel slice of the concat buffer that feeds down_channel). */
int rdfc_norm_apply(const rdfc_view *x, const float *mean, const float *rstd, const rdfc_view *out, int B, int H,
                    int W, void *stream);

/* ------------------------------------------------------------------ evaluation glue --------------------------- */
/* The sums behind RDFGANMetric (lib/metrics/rdf_gan_metric.py:59-151: RMSE, MAE, iRMSE, iMAE, REL, D^1..D^3), with the
 * de-normalisation x * std + mean of Eval.inference (lib/evaluator/evaluator.py:27-29) fused in.  pred, gt: B images of n fp32
 * pixels; evaluate_mask: NULL or B*n bytes (non-zero = evaluate).  A pixel counts when gt > t_valid (and its mask byte is set).
 * sums (B,9) doubles: count, sum d^2, sum |d|, sum dinv^2, sum |dinv|, sum |d|/(gt+1e-8), #(ratio < 1.25), #(< 1.25^2),
 * #(< 1.25^3); partial: scratch of B * rdfc_depth_metric_nchunk(n) * 9 doubles.  Deterministic (no atomics). */
int rdfc_depth_metric_nchunk(long long n);
int rdfc_depth_metric_sums(const float *pred, const float *gt, const unsigned char *evaluate_mask, float std, float mean,
                           float t_valid, double *sums, double *partial, int B, long long n, void *stream);

/* ------------------------------------------------------------------ training step ---------------------------- */
/* Batch-statistics BatchNorm fused with the activation and the residual add, and the conv filter gradient: what the
 * reference's train() mode leaves to nn.BatchNorm2d / cuDNN inside conv_bn_relu / convt_bn_relu / BasicBlock
 * (encoder_decoder/common.py:29-61, encoder_decoder/encoder_decoder.py:39-59; training step lib/models/rdf_gan.py:135-207).
 * Activations: NHWC views over npix = B*H*W pixels -- bf16, or fp32 for the BatchNorm entry points (one dtype per call; fp32 pixel
 * strides a multiple of 4); statistics and parameter gradients fp32; deterministic reductions. */

/* floats of workspace for rdfc_bn_stats / rdfc_bn_act_backward */
int rdfc_bn_workspace_floats(long long npix, int C);
/* per-channel mean and BIASED variance of x over npix pixels (Chan-combined partials, fixed order) */
int rdfc_bn_stats(const rdfc_view *x, long long npix, float *workspace, float *mean, float *var, void *stream);
/* out = act(x * scale[c] + shift[c] + residual)   (scale = gamma * rstd, shift = beta - mean * scale; residual may be NULL;
 * act: none / ReLU / LeakyReLU(0.2)) */
int rdfc_affine_act_forward(const rdfc_view *x, const float *scale, const float *shift, const rdfc_view *residual, int act,
                            const rdfc_view *out, long long npix, void *stream);
/* Backward of out = act(gamma * (y - mean) * rstd + beta + residual) with batch statistics (mean, rstd) of y:
 *   dz = dout * act'(out)  (act' from the sign of `out`),   sum_dz[c] = sum dz (= d beta),   sum_dz_xhat[c] = sum dz * xhat (= d gamma),
 *   dy = gamma * rstd * (dz - sum_dz / npix - xhat * sum_dz_xhat / npix),   dres = dz (written when dres is not NULL). */
int rdfc_bn_act_backward(const rdfc_view *dout, const rdfc_view *out, const rdfc_view *y, const float *mean, const float *rstd,
                         const float *gamma, int act, const rdfc_view *dy, const rdfc_view *dres, float *workspace,
                         float *sum_dz, float *sum_dz_xhat, long long npix, void *stream);

/* Filter gradient of y = conv2d(input, W (O, I, k, k), stride, padding (k-1)/2):
 *   grad_weight[o][i][ky][kx] = sum_{b,py,px} grad_out[b,py,px,o] * input[b, stride*py - pad + ky, stride*px - pad + kx, i]
 * (fp32, torch's (O, I, kh, kw) layout, overwritten).  A ConvTranspose2d(k3, s2, p1, op1) layer's filter gradient (Cin, Cout, 3, 3)
 * is the same sum with grad_out := the layer's INPUT and input := the gradient w.r.t. its (uncropped) output.
 * workspace: rdfc_conv_wgrad_workspace_floats(d) floats (split-K partials, reduced in a fixed order). */
typedef struct {
    int B;
    int Hg, Wg;             /* grid of grad_out */
    int Hi, Wi;             /* grid of input */
    int k, stride, pad;     /* k in {1, 3}, stride in {1, 2}, pad = (k - 1) / 2 */
    rdfc_view grad_out;     /* bf16 NHWC, O channels, O % 8 == 0 */
    rdfc_view input;        /* bf16 NHWC, I channels, I % 8 == 0 */
} rdfc_wgrad_desc;
long long rdfc_conv_wgrad_workspace_floats(const rdfc_wgrad_desc *d);
int rdfc_conv_wgrad(const rdfc_wgrad_desc *d, float *grad_weight, float *workspace, void *stream);
/* The training step's fp32_tc mode: fp32 activations and gradients, contractions on the tensor cores with split fp16 operands
 * (x = x_hi + x_lo; x_hi W_hi + x_hi W_lo + x_lo W_hi accumulated in fp32).  Each tensor is first scaled by a power of two taken
 * from its own largest magnitude (fp16's exponent range is narrow: gradients near 1e-5 would lose their low half), and the
 * factors stay on the device.  C % 32 == 0 everywhere; views 16-byte aligned; invalid arguments fail before any launch.
 *
 * rdfc_split_scaled: x = fp32 NHWC view (C channels, pixel stride a multiple of 4) -> out = RDFC_F16 view of 2C channels
 *   [hi | lo] of s * x per pixel (pixel stride a multiple of 8); *factor (device float) = s, the power of two with
 *   max|x| * s in [1024, 2048), 1 for an all-zero tensor. */
int rdfc_split_scaled(const rdfc_view *x, long long npix, const rdfc_view *out, float *factor, void *stream);
/* rdfc_conv_forward on an already split input: d->in = the RDFC_F16 [hi | lo] view (2 Cin channels), d->path =
 * RDFC_PATH_UMMA_F32X3 (weight = that path's [W_hi ; W_lo ; W_hi] packing, of the filter scaled by its own power of two),
 * d->out fp32 NHWC, d->scale REQUIRED: the per-Cout factor 1 / (s_x s_w) that undoes the scaling; no residual, no workspace. */
int rdfc_conv_forward_split(const rdfc_conv_desc *d, void *stream);
/* Filter gradient of split operands: d->grad_out / d->input = RDFC_F16 [hi | lo] views (2 O / 2 I channels) of s_g * grad_out and
 * s_x * input; inv_scale = device float 1 / (s_g s_x).  The three products g_hi x_hi, g_hi x_lo, g_lo x_hi run on the tcgen05
 * filter-gradient kernel into consecutive chunk ranges of the workspace (rdfc_conv_wgrad_split_workspace_floats(d) floats,
 * 16-byte aligned); one reduction in a fixed order writes grad_weight (O, I, k, k) fp32: bit-reproducible. */
long long rdfc_conv_wgrad_split_workspace_floats(const rdfc_wgrad_desc *d);
int rdfc_conv_wgrad_split(const rdfc_wgrad_desc *d, const float *inv_scale, float *grad_weight, float *workspace, void *stream);

/* ------------------------------------------------------------------ ESANet guidance glue ---------------------- */
/* The non-GEMM layers of RDF-GAN's global_guidance_module (F/lib/models/segmentator/esa_net/esa_net_one_modality.py:145-172,
 * decoder.py:137-191, model_utils.py:34-49,99-134; F = /root/reference/RDF-GAN); its GEMM-shaped layers go through
 * rdfc_conv_forward.  Views are NHWC, bf16 or fp32, C % 8 == 0, 16-byte aligned, pixel stride a multiple of 8 (bf16) or 4 (fp32)
 * elements; the views of one call share a dtype (else RDFC_ERR_INVALID).  The up-sampling's fp32 NCHW result takes either input dtype. */

/* encoder.conv1 + folded bn1 + ReLU: k x k (<= 7) conv, any stride, from fp32 NCHW x (B, Cin <= 4, Hi, Wi); weight (Cout, Cin, k, k) fp32 */
int rdfc_first_conv_forward(const float *x_nchw, int B, int Cin, int Hi, int Wi, const float *weight, int k, int stride, int pad,
                            const float *scale, const float *shift, int relu, const rdfc_view *out, void *stream);
/* F.max_pool2d(kernel 3, stride 2, padding 1) */
int rdfc_maxpool3x3s2_forward(const rdfc_view *x, const rdfc_view *out, int B, int Hi, int Wi, void *stream);
/* SqueezeAndExcitation.fc on the per-image channel means (B, C) -> weights (B, C): sigmoid(W2 relu(W1 m + b1) + b2), W1 (R, C), W2 (C, R);
 * the scaling x * w is rdfc_norm_apply with mean = 0, rstd = w */
int rdfc_se_weights(const float *mean, const float *w1, const float *b1, const float *w2, const float *b2, float *out, int B, int C, int R,
                    void *stream);
/* nn.AdaptiveAvgPool2d(bins) -> out (B, bins, bins, C) */
int rdfc_adaptive_avgpool_forward(const rdfc_view *x, const rdfc_view *out, int B, int H, int W, int bins, void *stream);
/* F.interpolate(mode='nearest') of a (hs, ws) map to (H, W), written into `out` (a channel slice of a concat buffer) */
int rdfc_upsample_nearest_forward(const rdfc_view *x, const rdfc_view *out, int B, int hs, int ws, int H, int W, void *stream);
/* Upsample('learned-3x3-zeropad'): nearest resize (Hi, Wi) -> (Ho, Wo), depth-wise 3x3 conv (weight (C, 1, 3, 3), bias (C)) with zero
 * padding, + skip (or NULL); result to `out` (NHWC, x's dtype) or, when out_nchw != NULL, to fp32 NCHW (B, C, Ho, Wo) */
int rdfc_upsample_dw_forward(const rdfc_view *x, const float *weight, const float *bias, const rdfc_view *skip, const rdfc_view *out,
                             float *out_nchw, int B, int Hi, int Wi, int Ho, int Wo, void *stream);

/* ------------------------------------------------------------------ development aids ------------------------- */
/* Not part of the drop-in boundary.  rdfc_dev_set_knob overrides a development knob (the RDFC_* environment variables, which
 * the library reads once per name); value INT64_MIN restores the default.  rdfc_dev_umma_timers copies the per-role cycle
 * counters of the last conv launch made under RDFC_UMMA_DBG=1 (a -DRDFC_UMMA_TIMERS build) to `host`. */
int rdfc_dev_set_knob(const char *name, long long value);
int rdfc_dev_umma_timers(long long *host, int n);

#ifdef __cplusplus
}
#endif
#endif /* RDFC_B200_H */
