// Training-step kernels (SURVEY 8f rank 1): batch-statistics BatchNorm forward / backward fused with the activation and the
// residual add, the backward of a frozen (running-statistics) BatchNorm folded into its conv, and the entry points of the
// convolution filter gradient (its tcgen05 kernel is in wgrad_umma.cu).
//
// Replaces, for conv_bn_relu / convt_bn_relu / torchvision BasicBlock in train() mode (encoder_decoder/common.py:29-61,
// encoder_decoder/encoder_decoder.py:39-59), what the reference leaves to cuDNN / ATen: nn.BatchNorm2d's batch statistics and
// its backward, the (Leaky)ReLU backward, and Conv2d / ConvTranspose2d's weight gradient.  Activations are NHWC views (pointer,
// channels, pixel stride): bf16, or fp32 in the BatchNorm kernels (the fp32_tc training mode); statistics and gradients of parameters fp32, all reductions deterministic (fixed
// combination order, no atomics).
#include "common.cuh"

namespace rdfc {
namespace {

// ---------------------------------------------------------------------------------------------------------------------------
// 8 consecutive channels of one pixel as fp32
__device__ __forceinline__ void ld8(const __nv_bfloat16 *p, float (&v)[8]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p));
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&w[q]));
        v[2 * q] = f.x;
        v[2 * q + 1] = f.y;
    }
}
__device__ __forceinline__ void st8(__nv_bfloat16 *p, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * q], v[2 * q + 1]);
        w[q] = *reinterpret_cast<const uint32_t *>(&h);
    }
    *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

// the same for fp32 activations (the fp32_tc training mode): two 16-byte loads / stores
__device__ __forceinline__ void ld8(const float *p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4 *>(p)), b = __ldg(reinterpret_cast<const float4 *>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void st8(float *p, const float (&v)[8]) {
    reinterpret_cast<float4 *>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4 *>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f(float v) { return v; }

// an NHWC view of bf16 (the default training mode) or fp32 (fp32_tc) activations
template <typename T>
struct View {
    const T *ptr;
    int stride;
};

// ---- per-channel batch statistics ---------------------------------------------------------------------------------------
// Pass 1: grid (nblk, ceil(C/64)), block 256 = 8 channel groups x 32 pixel lanes.  A CTA owns pixels [p0, p1) and emits the
// (mean, M2) of every channel over them (sums shifted by the CTA's first pixel, so nothing cancels).
template <typename T>
__global__ void __launch_bounds__(256) bn_partial_kernel(View<T> x, int C, long long npix, int per_blk, float *__restrict__ partial) {
    __shared__ float red[32][8][17];
    const int cg = threadIdx.x & 7, lane = threadIdx.x >> 3;
    const int c0 = blockIdx.y * 64 + cg * 8;
    const long long p0 = (long long)blockIdx.x * per_blk;
    const long long p1 = p0 + per_blk < npix ? p0 + per_blk : npix;
    const int n = (int)(p1 - p0);
    float s[8], ss[8], pivot[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) s[q] = ss[q] = pivot[q] = 0.f;
    if (c0 < C && n > 0) {
        const T *base = x.ptr + p0 * x.stride + c0;
        ld8(base, pivot);
        for (int p = lane; p < n; p += 32) {
            float v[8];
            ld8(base + (long long)p * x.stride, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float d = v[q] - pivot[q];
                s[q] += d;
                ss[q] = fmaf(d, d, ss[q]);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        red[lane][cg][q] = s[q];
        red[lane][cg][8 + q] = ss[q];
    }
    __syncthreads();
    if (threadIdx.x < 64) {
        const int g2 = threadIdx.x >> 3, q = threadIdx.x & 7, c = blockIdx.y * 64 + g2 * 8 + q;
        if (c < C) {
            float ts = 0.f, tss = 0.f;
            for (int l = 0; l < 32; ++l) {
                ts += red[l][g2][q];
                tss += red[l][g2][8 + q];
            }
            float mean = 0.f, m2 = 0.f;
            if (n > 0) {
                const float pv = to_f(x.ptr[p0 * x.stride + c]);
                mean = pv + ts / n;
                m2 = fmaxf(tss - ts * ts / n, 0.f);
            }
            float *o = partial + ((long long)blockIdx.x * C + c) * 2;
            o[0] = mean;
            o[1] = m2;
        }
    }
}

// Chan's pairwise combination of (n, mean, M2)
__device__ __forceinline__ void chan(float &n, float &mean, float &m2, float nb, float mb, float m2b) {
    if (nb <= 0.f) return;
    const float nn = n + nb, delta = mb - mean;
    mean += delta * nb / nn;
    m2 += m2b + delta * delta * n * nb / nn;
    n = nn;
}

// Pass 2: one warp per channel; lane l folds blocks l, l + 32, ... in order, then the lanes fold in a fixed butterfly order.
__global__ void __launch_bounds__(256) bn_final_kernel(const float *__restrict__ partial, int C, long long npix, int per_blk, int nblk,
                                                       float *__restrict__ mean_o, float *__restrict__ var_o) {
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= C) return;
    float n = 0.f, mean = 0.f, m2 = 0.f;
    for (int k = lane; k < nblk; k += 32) {
        const long long p0 = (long long)k * per_blk;
        const float nb = (float)((p0 + per_blk < npix ? p0 + per_blk : npix) - p0);
        const float2 v = __ldg(reinterpret_cast<const float2 *>(partial + ((long long)k * C + c) * 2));
        chan(n, mean, m2, nb, v.x, v.y);
    }
    for (int o = 1; o < 32; o <<= 1) {
        const float nb = __shfl_xor_sync(0xffffffffu, n, o), mb = __shfl_xor_sync(0xffffffffu, mean, o), m2b = __shfl_xor_sync(0xffffffffu, m2, o);
        // both partners must compute the same value: combine in a canonical order (lower lane first)
        if (lane & o) {
            float n2 = nb, mean2 = mb, m22 = m2b;
            chan(n2, mean2, m22, n, mean, m2);
            n = n2; mean = mean2; m2 = m22;
        } else {
            chan(n, mean, m2, nb, mb, m2b);
        }
    }
    if (lane == 0) {
        mean_o[c] = mean;
        var_o[c] = m2 / n;          // biased variance (what BatchNorm normalises with)
    }
}

// ---- out = act(x * scale[c] + shift[c] + residual) ---------------------------------------------------------------------
// kHoist (C / 8 a power of two <= 256, i.e. a divisor of the 256-thread block): a thread's channel group is the same in every iteration
// of the grid-stride loop, so its eight (scale, shift) pairs are read once and the pixel index advances by an add -- the plain form reads
// 16 per-channel values through the LSU per 2-3 vector loads of data and divides a 64-bit index per iteration.
template <typename T, bool kHoist>
__global__ void __launch_bounds__(256) affine_act_kernel(View<T> x, const float *__restrict__ scale, const float *__restrict__ shift, View<T> res,
                                                         float slope, T *__restrict__ out, int out_stride, int C, long long npix) {
    const int cgs = C >> 3;
    if (kHoist) {
        const long long tid = (long long)blockIdx.x * 256 + threadIdx.x, T = (long long)gridDim.x * 256;
        const int c0 = (int)(tid % cgs) * 8;
        const long long pstep = T / cgs;
        float sc[8], sh[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { sc[q] = __ldg(scale + c0 + q); sh[q] = __ldg(shift + c0 + q); }
        for (long long p = tid / cgs; p < npix; p += pstep) {
            float v[8], r[8];
            ld8(x.ptr + p * x.stride + c0, v);
            if (res.ptr) ld8(res.ptr + p * res.stride + c0, r);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                float y = fmaf(v[q], sc[q], sh[q]);
                if (res.ptr) y += r[q];
                v[q] = fmaxf(y, slope * y);
            }
            st8(out + p * out_stride + c0, v);
        }
        return;
    }
    const long long total = npix * cgs;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i / cgs;
        const int c0 = (int)(i - p * cgs) * 8;
        float v[8], r[8];
        ld8(x.ptr + p * x.stride + c0, v);
        if (res.ptr) ld8(res.ptr + p * res.stride + c0, r);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float y = fmaf(v[q], __ldg(scale + c0 + q), __ldg(shift + c0 + q));
            if (res.ptr) y += r[q];
            v[q] = fmaxf(y, slope * y);           // slope 1: identity, 0: ReLU, 0.2: LeakyReLU
        }
        st8(out + p * out_stride + c0, v);
    }
}

// ---- backward: dz = dout * act'(out);  sums of dz and dz * xhat per channel ----------------------------------------------
// act' from the sign of the activation's OUTPUT (ReLU / LeakyReLU keep the sign; slope 1 = no activation).
__device__ __forceinline__ float dact(float out, float slope) { return out > 0.f ? 1.f : slope; }

template <typename T>
__global__ void __launch_bounds__(256) bn_bwd_partial_kernel(View<T> dout, View<T> out, View<T> y, const float *__restrict__ mean,
                                                             const float *__restrict__ rstd, float slope, int C, long long npix, int per_blk,
                                                             float *__restrict__ partial) {
    __shared__ float red[32][8][17];
    const int cg = threadIdx.x & 7, lane = threadIdx.x >> 3;
    const int c0 = blockIdx.y * 64 + cg * 8;
    const long long p0 = (long long)blockIdx.x * per_blk;
    const long long p1 = p0 + per_blk < npix ? p0 + per_blk : npix;
    const int n = (int)(p1 - p0);
    float s[8], ss[8], mu[8], rs[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) s[q] = ss[q] = mu[q] = rs[q] = 0.f;
    if (c0 < C && n > 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) { mu[q] = __ldg(mean + c0 + q); rs[q] = __ldg(rstd + c0 + q); }
        for (int p = lane; p < n; p += 32) {
            float g[8], o[8], v[8];
            ld8(dout.ptr + (p0 + p) * dout.stride + c0, g);
            ld8(out.ptr + (p0 + p) * out.stride + c0, o);
            ld8(y.ptr + (p0 + p) * y.stride + c0, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float dz = g[q] * dact(o[q], slope);
                s[q] += dz;
                ss[q] = fmaf(dz, (v[q] - mu[q]) * rs[q], ss[q]);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        red[lane][cg][q] = s[q];
        red[lane][cg][8 + q] = ss[q];
    }
    __syncthreads();
    if (threadIdx.x < 64) {
        const int g2 = threadIdx.x >> 3, q = threadIdx.x & 7, c = blockIdx.y * 64 + g2 * 8 + q;
        if (c < C) {
            float ts = 0.f, tss = 0.f;
            for (int l = 0; l < 32; ++l) {
                ts += red[l][g2][q];
                tss += red[l][g2][8 + q];
            }
            float *o = partial + ((long long)blockIdx.x * C + c) * 2;
            o[0] = ts;
            o[1] = tss;
        }
    }
}

__global__ void __launch_bounds__(256) sum_final_kernel(const float *__restrict__ partial, int C, int nblk, float *__restrict__ s0,
                                                        float *__restrict__ s1) {
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= C) return;
    double a = 0.0, b = 0.0;
    for (int k = lane; k < nblk; k += 32) {
        const float2 v = __ldg(reinterpret_cast<const float2 *>(partial + ((long long)k * C + c) * 2));
        a += v.x;
        b += v.y;
    }
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane == 0) {
        s0[c] = (float)a;
        s1[c] = (float)b;
    }
}

// dy = gamma * rstd * (dz - sum_dz / N - xhat * sum_dz_xhat / N);  dres = dz.   kHoist: as in affine_act_kernel (same arithmetic order).
template <typename T, bool kHoist>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(View<T> dout, View<T> out, View<T> y, const float *__restrict__ mean,
                                                           const float *__restrict__ rstd, const float *__restrict__ gamma,
                                                           const float *__restrict__ sum_dz, const float *__restrict__ sum_dzx, float slope,
                                                           T *__restrict__ dy, int dy_stride, T *__restrict__ dres,
                                                           int dres_stride, int C, long long npix) {
    const int cgs = C >> 3;
    const float invn = 1.f / (float)npix;
    if (kHoist) {
        const long long tid = (long long)blockIdx.x * 256 + threadIdx.x, T = (long long)gridDim.x * 256;
        const int c0 = (int)(tid % cgs) * 8;
        const long long pstep = T / cgs;
        float mu[8], rs[8], grs[8], k1[8], sx[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            mu[q] = __ldg(mean + c0 + q); rs[q] = __ldg(rstd + c0 + q); grs[q] = __ldg(gamma + c0 + q) * rs[q];
            k1[q] = __ldg(sum_dz + c0 + q) * invn; sx[q] = __ldg(sum_dzx + c0 + q);
        }
        for (long long p = tid / cgs; p < npix; p += pstep) {
            float g[8], o[8], v[8], dzv[8];
            ld8(dout.ptr + p * dout.stride + c0, g);
            ld8(out.ptr + p * out.stride + c0, o);
            ld8(y.ptr + p * y.stride + c0, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float dz = g[q] * dact(o[q], slope);
                const float xh = (v[q] - mu[q]) * rs[q];
                dzv[q] = dz;
                v[q] = grs[q] * (dz - k1[q] - xh * sx[q] * invn);
            }
            st8(dy + p * dy_stride + c0, v);
            if (dres) st8(dres + p * dres_stride + c0, dzv);
        }
        return;
    }
    const long long total = npix * cgs;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i / cgs;
        const int c0 = (int)(i - p * cgs) * 8;
        float g[8], o[8], v[8];
        ld8(dout.ptr + p * dout.stride + c0, g);
        ld8(out.ptr + p * out.stride + c0, o);
        ld8(y.ptr + p * y.stride + c0, v);
        float dzv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int c = c0 + q;
            const float dz = g[q] * dact(o[q], slope);
            const float rs = __ldg(rstd + c), xh = (v[q] - __ldg(mean + c)) * rs;
            dzv[q] = dz;
            // __fmul_rn: sum_dz / N rounded on its own, as the hoisted form's k1 is -- contracted into dz - sum_dz * invn, one fma
            // would round once and the two forms would differ in the last bit
            v[q] = __ldg(gamma + c) * rs * (dz - __fmul_rn(__ldg(sum_dz + c), invn) - xh * __ldg(sum_dzx + c) * invn);
        }
        st8(dy + p * dy_stride + c0, v);
        if (dres) st8(dres + p * dres_stride + c0, dzv);
    }
}

// ---- frozen BatchNorm backward: dz = dout * act'(out) (written when dz is not NULL), per-CTA partial sums of dz ------------
template <typename T> __device__ __forceinline__ float rnd(float v);
template <> __device__ __forceinline__ float rnd<float>(float v) { return v; }
template <> __device__ __forceinline__ float rnd<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// Same grid and CTA layout as bn_bwd_partial_kernel; partial[blk][C] holds one float per channel, summed by sum1_final_kernel.
template <typename T>
__global__ void __launch_bounds__(256) bn_frozen_partial_kernel(View<T> dout, View<T> out, float slope, T *__restrict__ dz, int dz_stride,
                                                                int C, long long npix, int per_blk, float *__restrict__ partial) {
    __shared__ float red[32][8][9];
    const int cg = threadIdx.x & 7, lane = threadIdx.x >> 3;
    const int c0 = blockIdx.y * 64 + cg * 8;
    const long long p0 = (long long)blockIdx.x * per_blk;
    const long long p1 = p0 + per_blk < npix ? p0 + per_blk : npix;
    const int n = (int)(p1 - p0);
    float s[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) s[q] = 0.f;
    if (c0 < C && n > 0) {
#pragma unroll 1                                    // unrolled, the bf16 instantiation spills
        for (int p = lane; p < n; p += 32) {
            float g[8];
            ld8(dout.ptr + (p0 + p) * dout.stride + c0, g);
            if (out.ptr) {                      // an activation: its derivative from the sign of the output
                float o[8];
                ld8(out.ptr + (p0 + p) * out.stride + c0, o);
#pragma unroll
                for (int q = 0; q < 8; ++q) g[q] = rnd<T>(g[q] * dact(o[q], slope));
            }
            if (dz) st8(dz + (p0 + p) * dz_stride + c0, g);
#pragma unroll
            for (int q = 0; q < 8; ++q) s[q] += g[q];      // the sum of dz as stored: d gamma = rstd (<W, G(dz)> - rm sum dz) cancels exactly
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) red[lane][cg][q] = s[q];
    __syncthreads();
    if (threadIdx.x < 64) {
        const int g2 = threadIdx.x >> 3, q = threadIdx.x & 7, c = blockIdx.y * 64 + g2 * 8 + q;
        if (c < C) {
            float ts = 0.f;
            for (int l = 0; l < 32; ++l) ts += red[l][g2][q];
            partial[(long long)blockIdx.x * C + c] = ts;
        }
    }
}

// one warp per channel: lane l sums blocks l, l + 32, ... in order (fp64), then a fixed butterfly
__global__ void __launch_bounds__(256) sum1_final_kernel(const float *__restrict__ partial, int C, int nblk, float *__restrict__ s0) {
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= C) return;
    double a = 0.0;
    for (int k = lane; k < nblk; k += 32) a += __ldg(partial + (long long)k * C + c);
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) s0[c] = (float)a;
}

}  // namespace
}  // namespace rdfc

using namespace rdfc;

template <typename T>
static inline View<T> mk(const rdfc_view *v) { return View<T>{(const T *)v->ptr, v->pix_stride}; }
// `dtype`: the dtype every view of the call must have -- bf16 (pixel stride a multiple of 8) or fp32 (a multiple of 4); 16-byte aligned
static int check_view(const rdfc_view *v, int C, const char *what, int dtype) {
    RDFC_REQUIRE(v && v->ptr, "%s: NULL view", what);
    RDFC_REQUIRE((dtype == RDFC_BF16 || dtype == RDFC_F32) && v->dtype == dtype && !v->nchw,
                 "%s: NHWC views of one dtype (bf16 or fp32) expected", what);
    RDFC_REQUIRE(v->C == C && C % 8 == 0 && v->pix_stride % (dtype == RDFC_BF16 ? 8 : 4) == 0 && ((uintptr_t)v->ptr % 16) == 0,
                 "%s: %d channels expected, multiples of 8, 16-byte aligned", what, C);
    return 0;
}
static int red_blocks(long long npix, int *per_blk) {
    long long nblk = (long long)sm_count() * 4;
    long long per = (npix + nblk - 1) / nblk;
    if (per < 64) per = 64;
    *per_blk = (int)per;
    return (int)((npix + per - 1) / per);
}

extern "C" int rdfc_bn_workspace_floats(long long npix, int C) {
    int per;
    return red_blocks(npix, &per) * C * 2;
}

template <typename T>
static int bn_stats(const rdfc_view *x, long long npix, float *workspace, float *mean, float *var, cudaStream_t st) {
    int per;
    const int nblk = red_blocks(npix, &per), C = x->C;
    bn_partial_kernel<T><<<dim3(nblk, cdiv(C, 64)), 256, 0, st>>>(mk<T>(x), C, npix, per, workspace);
    RDFC_CHECK_LAUNCH("bn_partial_kernel");
    bn_final_kernel<<<cdiv(C, 8), 256, 0, st>>>(workspace, C, npix, per, nblk, mean, var);
    RDFC_CHECK_LAUNCH("bn_final_kernel");
    return 0;
}

extern "C" int rdfc_bn_stats(const rdfc_view *x, long long npix, float *workspace, float *mean, float *var, void *stream) {
    RDFC_REQUIRE(x && workspace && mean && var && npix > 0, "bn stats: bad argument");
    if (int rc = check_view(x, x->C, "bn stats", x->dtype)) return rc;
    if (x->dtype == RDFC_F32) return bn_stats<float>(x, npix, workspace, mean, var, (cudaStream_t)stream);
    return bn_stats<__nv_bfloat16>(x, npix, workspace, mean, var, (cudaStream_t)stream);
}

static float act_slope(int act) { return act == RDFC_ACT_RELU ? 0.f : (act == RDFC_ACT_LEAKY02 ? 0.2f : 1.f); }

template <typename T>
static int affine_act(const rdfc_view *x, const float *scale, const float *shift, const rdfc_view *residual, int act, const rdfc_view *out,
                      long long npix, cudaStream_t st) {
    const int C = x->C;
    const View<T> r = (residual && residual->ptr) ? mk<T>(residual) : View<T>{nullptr, 0};
    const int nblk = (int)min((long long)cdiv(npix * (C / 8), 256), (long long)sm_count() * 16);
    if (256 % (C >> 3) == 0 && knob("RDFC_BN_HOIST", 1) != 0)
        affine_act_kernel<T, true><<<nblk, 256, 0, st>>>(mk<T>(x), scale, shift, r, act_slope(act), (T *)out->ptr, out->pix_stride, C, npix);
    else
        affine_act_kernel<T, false><<<nblk, 256, 0, st>>>(mk<T>(x), scale, shift, r, act_slope(act), (T *)out->ptr, out->pix_stride, C, npix);
    RDFC_CHECK_LAUNCH("affine_act_kernel");
    return 0;
}

extern "C" int rdfc_affine_act_forward(const rdfc_view *x, const float *scale, const float *shift, const rdfc_view *residual, int act,
                                       const rdfc_view *out, long long npix, void *stream) {
    RDFC_REQUIRE(x && scale && shift && out && npix > 0, "affine act: bad argument");
    RDFC_REQUIRE(act == RDFC_ACT_NONE || act == RDFC_ACT_RELU || act == RDFC_ACT_LEAKY02, "affine act: none / ReLU / LeakyReLU(0.2) only");
    const int C = x->C, dt = x->dtype;
    if (int rc = check_view(x, C, "affine act x", dt)) return rc;
    if (int rc = check_view(out, C, "affine act out", dt)) return rc;
    if (residual && residual->ptr) if (int rc = check_view(residual, C, "affine act residual", dt)) return rc;
    if (dt == RDFC_F32) return affine_act<float>(x, scale, shift, residual, act, out, npix, (cudaStream_t)stream);
    return affine_act<__nv_bfloat16>(x, scale, shift, residual, act, out, npix, (cudaStream_t)stream);
}

template <typename T>
static int bn_act_backward(const rdfc_view *dout, const rdfc_view *out, const rdfc_view *y, const float *mean, const float *rstd, const float *gamma,
                           int act, const rdfc_view *dy, const rdfc_view *dres, float *workspace, float *sum_dz, float *sum_dz_xhat, long long npix,
                           cudaStream_t st) {
    const int C = y->C;
    int per;
    const int nblk = red_blocks(npix, &per);
    const float slope = act_slope(act);
    bn_bwd_partial_kernel<T><<<dim3(nblk, cdiv(C, 64)), 256, 0, st>>>(mk<T>(dout), mk<T>(out), mk<T>(y), mean, rstd, slope, C, npix, per, workspace);
    RDFC_CHECK_LAUNCH("bn_bwd_partial_kernel");
    sum_final_kernel<<<cdiv(C, 8), 256, 0, st>>>(workspace, C, nblk, sum_dz, sum_dz_xhat);
    RDFC_CHECK_LAUNCH("sum_final_kernel");
    const int ablk = (int)min((long long)cdiv(npix * (C / 8), 256), (long long)sm_count() * 16);
    T *dr = (dres && dres->ptr) ? (T *)dres->ptr : nullptr;
    const int dr_stride = dr ? dres->pix_stride : 0;
    if (256 % (C >> 3) == 0 && knob("RDFC_BN_HOIST", 1) != 0)
        bn_bwd_apply_kernel<T, true><<<ablk, 256, 0, st>>>(mk<T>(dout), mk<T>(out), mk<T>(y), mean, rstd, gamma, sum_dz, sum_dz_xhat, slope, (T *)dy->ptr,
                                                           dy->pix_stride, dr, dr_stride, C, npix);
    else
        bn_bwd_apply_kernel<T, false><<<ablk, 256, 0, st>>>(mk<T>(dout), mk<T>(out), mk<T>(y), mean, rstd, gamma, sum_dz, sum_dz_xhat, slope, (T *)dy->ptr,
                                                            dy->pix_stride, dr, dr_stride, C, npix);
    RDFC_CHECK_LAUNCH("bn_bwd_apply_kernel");
    return 0;
}

extern "C" int rdfc_bn_act_backward(const rdfc_view *dout, const rdfc_view *out, const rdfc_view *y, const float *mean, const float *rstd,
                                    const float *gamma, int act, const rdfc_view *dy, const rdfc_view *dres, float *workspace,
                                    float *sum_dz, float *sum_dz_xhat, long long npix, void *stream) {
    RDFC_REQUIRE(dout && out && y && mean && rstd && gamma && dy && workspace && sum_dz && sum_dz_xhat && npix > 0, "bn backward: bad argument");
    RDFC_REQUIRE(act == RDFC_ACT_NONE || act == RDFC_ACT_RELU || act == RDFC_ACT_LEAKY02, "bn backward: none / ReLU / LeakyReLU(0.2) only");
    const int C = y->C, dt = y->dtype;
    if (int rc = check_view(dout, C, "bn backward dout", dt)) return rc;
    if (int rc = check_view(out, C, "bn backward out", dt)) return rc;
    if (int rc = check_view(y, C, "bn backward y", dt)) return rc;
    if (int rc = check_view(dy, C, "bn backward dy", dt)) return rc;
    if (dres && dres->ptr) if (int rc = check_view(dres, C, "bn backward dres", dt)) return rc;
    if (dt == RDFC_F32)
        return bn_act_backward<float>(dout, out, y, mean, rstd, gamma, act, dy, dres, workspace, sum_dz, sum_dz_xhat, npix, (cudaStream_t)stream);
    return bn_act_backward<__nv_bfloat16>(dout, out, y, mean, rstd, gamma, act, dy, dres, workspace, sum_dz, sum_dz_xhat, npix, (cudaStream_t)stream);
}

template <typename T>
static int bn_frozen_backward(const rdfc_view *dout, const rdfc_view *out, int act, const rdfc_view *dz, float *workspace, float *sum_dz,
                              long long npix, cudaStream_t st) {
    const int C = dout->C;
    int per;
    const int nblk = red_blocks(npix, &per);
    const View<T> o = act == RDFC_ACT_NONE ? View<T>{nullptr, 0} : mk<T>(out);
    T *d = (dz && dz->ptr) ? (T *)dz->ptr : nullptr;
    bn_frozen_partial_kernel<T><<<dim3(nblk, cdiv(C, 64)), 256, 0, st>>>(mk<T>(dout), o, act_slope(act), d, d ? dz->pix_stride : 0, C, npix,
                                                                         per, workspace);
    RDFC_CHECK_LAUNCH("bn_frozen_partial_kernel");
    sum1_final_kernel<<<cdiv(C, 8), 256, 0, st>>>(workspace, C, nblk, sum_dz);
    RDFC_CHECK_LAUNCH("sum1_final_kernel");
    return 0;
}

extern "C" int rdfc_bn_frozen_backward(const rdfc_view *dout, const rdfc_view *out, int act, const rdfc_view *dz, float *workspace,
                                       float *sum_dz, long long npix, void *stream) {
    RDFC_REQUIRE(dout && workspace && sum_dz && npix > 0, "bn frozen backward: bad argument");
    RDFC_REQUIRE(act == RDFC_ACT_NONE || act == RDFC_ACT_RELU || act == RDFC_ACT_LEAKY02,
                 "bn frozen backward: none / ReLU / LeakyReLU(0.2) only");
    const bool has_dz = dz && dz->ptr;
    RDFC_REQUIRE(act == RDFC_ACT_NONE || has_dz, "bn frozen backward: an activation needs a dz destination");
    const int C = dout->C, dt = dout->dtype;
    if (int rc = check_view(dout, C, "bn frozen backward dout", dt)) return rc;
    if (act != RDFC_ACT_NONE) if (int rc = check_view(out, C, "bn frozen backward out", dt)) return rc;
    if (has_dz) if (int rc = check_view(dz, C, "bn frozen backward dz", dt)) return rc;
    if (dt == RDFC_F32) return bn_frozen_backward<float>(dout, out, act, dz, workspace, sum_dz, npix, (cudaStream_t)stream);
    return bn_frozen_backward<__nv_bfloat16>(dout, out, act, dz, workspace, sum_dz, npix, (cudaStream_t)stream);
}

// argument checks shared by the workspace query and the launch
static int check_wgrad(const rdfc_wgrad_desc *d) {
    RDFC_REQUIRE(d && (d->k == 1 || d->k == 3) && (d->stride == 1 || d->stride == 2) && d->pad == (d->k - 1) / 2,
                 "wgrad: 3x3 / 1x1 kernels, stride 1 / 2, padding (k-1)/2");
    RDFC_REQUIRE(d->B > 0 && d->Hg > 0 && d->Wg > 0 && d->Hi > 0 && d->Wi > 0, "wgrad: empty dimension");
    RDFC_REQUIRE(d->Hg == (d->Hi + 2 * d->pad - d->k) / d->stride + 1 && d->Wg == (d->Wi + 2 * d->pad - d->k) / d->stride + 1,
                 "wgrad: gradient grid (%d,%d) does not match the input grid (%d,%d)", d->Hg, d->Wg, d->Hi, d->Wi);
    RDFC_REQUIRE(d->grad_out.C % 8 == 0 && d->input.C % 8 == 0, "wgrad: channel counts must be multiples of 8");
    return 0;
}

namespace rdfc {
long long wgrad_umma_workspace_floats(const rdfc_wgrad_desc *d);    // wgrad_umma.cu: the filter gradient on tcgen05
int wgrad_umma(const rdfc_wgrad_desc *d, float *grad_weight, float *workspace, cudaStream_t st);
}  // namespace rdfc

extern "C" long long rdfc_conv_wgrad_workspace_floats(const rdfc_wgrad_desc *d) {
    return check_wgrad(d) == 0 ? wgrad_umma_workspace_floats(d) : -1;
}

extern "C" int rdfc_conv_wgrad(const rdfc_wgrad_desc *d, float *grad_weight, float *workspace, void *stream) {
    if (int rc = check_wgrad(d)) return rc;
    RDFC_REQUIRE(grad_weight && workspace, "wgrad: NULL output / workspace");
    if (int rc = check_view(&d->grad_out, d->grad_out.C, "wgrad grad_out", RDFC_BF16)) return rc;
    if (int rc = check_view(&d->input, d->input.C, "wgrad input", RDFC_BF16)) return rc;
    return wgrad_umma(d, grad_weight, workspace, (cudaStream_t)stream);
}
