// The fp32_tc training mode's pieces (train_ops.py): fp32 activations and gradients contracted on the 16-bit tensor cores with
// split operands, x = x_hi + x_lo (both fp16), at fp32 fidelity.
//
//   rdfc_split_scaled       amax of an fp32 NHWC view -> power-of-two factor s (device) -> fp16 [hi | lo] of s * x
//   rdfc_conv_wgrad_split   the filter gradient of wgrad_umma.cu on fp16 halves, run for the three products g_hi.x_hi, g_hi.x_lo,
//                           g_lo.x_hi into consecutive chunk ranges of one workspace, then ONE reduction in a fixed order that also
//                           applies 1 / (s_g s_x)  (bit-reproducible)
// (the conv forward / data gradient on an already split input is rdfc_conv_forward_split, conv.cu.)  The split kernel also serves,
// unscaled, the fp32 inputs of the inference path's RDFC_PATH_UMMA_F32X3 convs and fp32 heads (split_f32_forward).
//
// Why the scaling: fp16 keeps 11 significant bits down to 6.1e-5 only, and the training step's gradients start near 1e-5 (the
// reference's image_loss_weight = mask / mask.sum()).  Scaled so that the largest magnitude lies in [1024, 2048), the low half keeps
// 11 bits down to ~3e-5 of the largest element -- the scheme of the DCN path (common.cuh, pow2_scale).  The factor never leaves the
// device: no host synchronisation per conv.
#include <cuda_fp16.h>

#include "common.cuh"

namespace rdfc {
long long wgrad_umma_workspace_floats(const rdfc_wgrad_desc *d);
int wgrad_umma_partials(const rdfc_wgrad_desc *d, float *workspace, int fp16, cudaStream_t st, int *nchunk);

namespace {

// max |x| over an NHWC view, as the bit pattern of a non-negative float (which orders like an unsigned integer)
__global__ void __launch_bounds__(256) split_amax_kernel(const float *__restrict__ x, int C, int stride, long long npix, unsigned *__restrict__ am) {
    const int cgs = C >> 2;
    const long long total = npix * cgs;
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i / cgs;
        const float4 v = __ldg(reinterpret_cast<const float4 *>(x + p * stride) + (i - p * cgs));
        m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, sft));
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(am, __float_as_uint(m));
}

// fp32 NHWC view -> fp16 [pixel][hi(C) | lo(C)] of s * x, hi = fp16(s x), lo = fp16(s x - hi).  8 channels per thread.
// kScaled: s = pow2_scale(max |x|), read from `am`; otherwise s = 1 -- no load of `am`, no multiply (the inference path's split).
template <bool kScaled>
__global__ void __launch_bounds__(256) split_kernel(const float *__restrict__ x, int C, int stride, __half *__restrict__ out, int out_stride,
                                                    long long npix, const unsigned *__restrict__ am) {
    float s = 1.f;
    if (kScaled) s = pow2_scale(__uint_as_float(__ldg(am)));
    const int cgs = C >> 3;
    const long long total = npix * cgs;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i / cgs;
        const int c0 = (int)(i - p * cgs) * 8;
        const float4 a = __ldg(reinterpret_cast<const float4 *>(x + p * stride + c0)), b = __ldg(reinterpret_cast<const float4 *>(x + p * stride + c0) + 1);
        float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        if (kScaled)
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] *= s;
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const __half2 h = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
            const float2 hf = __half22float2(h);
            const __half2 l = __floats2half2_rn(v[2 * q] - hf.x, v[2 * q + 1] - hf.y);
            hi[q] = *reinterpret_cast<const uint32_t *>(&h);
            lo[q] = *reinterpret_cast<const uint32_t *>(&l);
        }
        __half *o = out + p * out_stride + c0;
        *reinterpret_cast<uint4 *>(o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4 *>(o + C) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

// the maximum's slot becomes the factor (after every reader of the maximum, stream order)
__global__ void split_factor_kernel(float *f) { *f = pow2_scale(__uint_as_float(*reinterpret_cast<const unsigned *>(f))); }

// dW[o][i][tap] (torch's (O, I, k, k)) = inv * sum over the chunk blocks partial[c][tap][o][i], c = 0 .. nchunk-1 in order
__global__ void __launch_bounds__(256) wgrad_split_reduce_kernel(const float *__restrict__ partial, float *__restrict__ dw, int O, int Ich, int nchunk,
                                                                 int ntap, const float *__restrict__ inv_scale) {
    const long long per = (long long)O * Ich, total = ntap * per;
    const float inv = __ldg(inv_scale);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int tap = (int)(e / per);
        const long long oi = e - (long long)tap * per;
        float s = 0.f;
        for (int c = 0; c < nchunk; ++c) s += __ldg(partial + (long long)c * total + e);
        dw[oi * ntap + tap] = s * inv;
    }
}

}  // namespace
}  // namespace rdfc

using namespace rdfc;

// a split [hi | lo] view: fp16, 2 * C channels, C % 32 == 0, 16-byte aligned, pixel stride a multiple of 8
static int check_split_view(const rdfc_view *v, const char *what) {
    RDFC_REQUIRE(v && v->ptr, "%s: NULL view", what);
    RDFC_REQUIRE(v->dtype == RDFC_F16 && !v->nchw, "%s: an fp16 NHWC [hi | lo] view expected", what);
    RDFC_REQUIRE(v->C > 0 && v->C % 64 == 0 && v->pix_stride >= v->C && v->pix_stride % 8 == 0 && ((uintptr_t)v->ptr % 16) == 0,
                 "%s: 2 x C channels with C %% 32 == 0 (got %d), pixel stride a multiple of 8, 16-byte aligned", what, v->C);
    return 0;
}

template <bool kScaled>
static int split_launch(const rdfc_view *x, __half *out, int out_stride, long long npix, const unsigned *am, cudaStream_t st) {
    const int nblk = (int)min((long long)cdiv(npix * (x->C / 8), 256), (long long)sm_count() * 16);
    split_kernel<kScaled><<<nblk, 256, 0, st>>>((const float *)x->ptr, x->C, x->pix_stride, out, out_stride, npix, am);
    RDFC_CHECK_LAUNCH("split_kernel");
    return 0;
}

namespace rdfc {
// the unscaled split into a dense [hi | lo] workspace: the fp32 input of the RDFC_PATH_UMMA_F32X3 conv and of the fp32 heads (conv.cu)
int split_f32_forward(const rdfc_view *x, void *out, long long npix, cudaStream_t st) {
    RDFC_REQUIRE(x && x->ptr && out && x->dtype == RDFC_F32 && !x->nchw && x->C % 8 == 0 && x->pix_stride % 4 == 0 &&
                     ((uintptr_t)x->ptr % 16) == 0,
                 "split: 16-byte aligned fp32 NHWC view with C % 8 == 0 expected");
    return split_launch<false>(x, (__half *)out, 2 * x->C, npix, nullptr, st);
}
}  // namespace rdfc

extern "C" int rdfc_split_scaled(const rdfc_view *x, long long npix, const rdfc_view *out, float *factor, void *stream) {
    RDFC_REQUIRE(x && out && factor && npix > 0, "split: bad argument");
    RDFC_REQUIRE(x->ptr && x->dtype == RDFC_F32 && !x->nchw, "split: the source must be an fp32 NHWC view");
    RDFC_REQUIRE(x->C > 0 && x->C % 32 == 0 && x->pix_stride >= x->C && x->pix_stride % 4 == 0 && ((uintptr_t)x->ptr % 16) == 0,
                 "split: source channels (%d) must be a multiple of 32, 16-byte aligned with a pixel stride that is a multiple of 4", x->C);
    if (int rc = check_split_view(out, "split destination")) return rc;
    RDFC_REQUIRE(out->C == 2 * x->C, "split: destination has %d channels, 2 x %d expected", out->C, x->C);
    RDFC_REQUIRE(((uintptr_t)factor % 4) == 0, "split: factor must be 4-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    RDFC_CUDA(cudaMemsetAsync(factor, 0, sizeof(float), st));
    const int ablk = (int)min((long long)cdiv(npix * (x->C / 4), 256 * 8), (long long)sm_count() * 4);
    split_amax_kernel<<<ablk, 256, 0, st>>>((const float *)x->ptr, x->C, x->pix_stride, npix, (unsigned *)factor);
    RDFC_CHECK_LAUNCH("split_amax_kernel");
    if (int rc = split_launch<true>(x, (__half *)out->ptr, out->pix_stride, npix, (const unsigned *)factor, st)) return rc;
    split_factor_kernel<<<1, 1, 0, st>>>(factor);
    RDFC_CHECK_LAUNCH("split_factor_kernel");
    return 0;
}

// the per-product descriptor: `part` 0 = (g_hi, x_hi), 1 = (g_hi, x_lo), 2 = (g_lo, x_hi); 16-bit views of C channels
static rdfc_wgrad_desc split_part(const rdfc_wgrad_desc *d, int part) {
    rdfc_wgrad_desc e = *d;
    const int O = d->grad_out.C / 2, I = d->input.C / 2;
    e.grad_out.C = O; e.input.C = I;
    e.grad_out.dtype = e.input.dtype = RDFC_BF16;       // 16-bit operands; wgrad_umma_partials(fp16 = 1) reads them as fp16
    e.grad_out.ptr = (char *)d->grad_out.ptr + (part == 2 ? (size_t)O * 2 : 0);
    e.input.ptr = (char *)d->input.ptr + (part == 1 ? (size_t)I * 2 : 0);
    return e;
}

static int check_wgrad_split(const rdfc_wgrad_desc *d) {
    RDFC_REQUIRE(d, "wgrad (split): descriptor is NULL");
    if (int rc = check_split_view(&d->grad_out, "wgrad (split) grad_out")) return rc;
    if (int rc = check_split_view(&d->input, "wgrad (split) input")) return rc;
    RDFC_REQUIRE((d->k == 1 || d->k == 3) && (d->stride == 1 || d->stride == 2) && d->pad == (d->k - 1) / 2,
                 "wgrad (split): 3x3 / 1x1 kernels, stride 1 / 2, padding (k-1)/2");
    RDFC_REQUIRE(d->B > 0 && d->Hg > 0 && d->Wg > 0 && d->Hi > 0 && d->Wi > 0, "wgrad (split): empty dimension");
    RDFC_REQUIRE(d->Hg == (d->Hi + 2 * d->pad - d->k) / d->stride + 1 && d->Wg == (d->Wi + 2 * d->pad - d->k) / d->stride + 1,
                 "wgrad (split): gradient grid (%d,%d) does not match the input grid (%d,%d)", d->Hg, d->Wg, d->Hi, d->Wi);
    return 0;
}

extern "C" long long rdfc_conv_wgrad_split_workspace_floats(const rdfc_wgrad_desc *d) {
    if (check_wgrad_split(d) != 0) return -1;
    const rdfc_wgrad_desc e = split_part(d, 0);
    const long long per = wgrad_umma_workspace_floats(&e);
    return per < 0 ? -1 : 3 * per;
}

extern "C" int rdfc_conv_wgrad_split(const rdfc_wgrad_desc *d, const float *inv_scale, float *grad_weight, float *workspace, void *stream) {
    if (int rc = check_wgrad_split(d)) return rc;
    RDFC_REQUIRE(inv_scale && grad_weight && workspace, "wgrad (split): NULL inverse scale / output / workspace");
    RDFC_REQUIRE(((uintptr_t)workspace % 16) == 0 && ((uintptr_t)grad_weight % 4) == 0 && ((uintptr_t)inv_scale % 4) == 0,
                 "wgrad (split): the workspace must be 16-byte aligned");
    rdfc_wgrad_desc parts[3];
    for (int t = 0; t < 3; ++t) parts[t] = split_part(d, t);
    cudaStream_t st = (cudaStream_t)stream;
    const int O = parts[0].grad_out.C, I = parts[0].input.C, ntap = d->k * d->k;
    const long long blk = (long long)ntap * O * I;
    int nchunk = 0;
    for (int t = 0; t < 3; ++t) {                                       // hi.hi, hi.lo, lo.hi into consecutive chunk ranges
        int nc = 0;
        if (int rc = wgrad_umma_partials(&parts[t], workspace + (long long)nchunk * blk, 1, st, &nc)) return rc;
        nchunk += nc;
    }
    const int nblk = (int)min((long long)cdiv(blk, 256), (long long)sm_count() * 8);
    wgrad_split_reduce_kernel<<<nblk, 256, 0, st>>>(workspace, grad_weight, O, I, nchunk, ntap, inv_scale);
    RDFC_CHECK_LAUNCH("wgrad_split_reduce_kernel");
    return 0;
}
