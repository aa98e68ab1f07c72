// NHWC reflection / replication padding with one padding p on all four sides: nn.ReflectionPad2d / nn.ReplicationPad2d of
// RDFC-GAN's ResnetGenerator (G_B2A, C/lib/models/generator/resnet_generator.py:6-98) -- the 1-channel input and the 64-channel
// map before the two 7x7 convolutions (p = 3), the residual blocks' 256-channel activations (p = 1).
//
// Forward: a copy, bit for bit F.pad(x, (p,) * 4, mode).  Backward: a GATHER, not PyTorch's atomicAdd scatter -- each input pixel
// sums, rows ascending and columns ascending, every padded position that maps onto it (reflect: up to 3 rows x 3 columns;
// replicate: up to (2p + 1)^2 at a corner), in fp32 with a compensated sum, rounded once to the output dtype.  The order is fixed,
// so the gradient is bit-reproducible by construction.  Views: bf16 or fp32 (pointer, channels, pixel stride), any channel count;
// 16-byte channel chunks when the channel count, the pixel strides and the pointers allow, one element per thread otherwise.
#include "common.cuh"

namespace rdfc {
namespace {

// padded index o in [0, n + 2p) -> the source index in [0, n) it copies (reflect: p < n)
__device__ __forceinline__ int pad_src(int o, int n, int p, int mode) {
    int i = o - p;
    if (mode == RDFC_PAD_REFLECT) {
        i = i < 0 ? -i : i;
        return i >= n ? 2 * (n - 1) - i : i;
    }
    return i < 0 ? 0 : (i >= n ? n - 1 : i);
}

// the padded indices that copy source index i, ascending, as three runs [lo[r], lo[r] + len[r]): before the source range, the
// position itself, after it (reflect: single mirrored positions; replicate: the whole border when i is the first / last index)
__device__ __forceinline__ void pad_runs(int i, int n, int p, int mode, int (&lo)[3], int (&len)[3]) {
    lo[1] = i + p;
    len[1] = 1;
    if (mode == RDFC_PAD_REFLECT) {
        lo[0] = p - i;
        len[0] = (i >= 1 && i <= p) ? 1 : 0;
        lo[2] = 2 * (n - 1) - i + p;
        len[2] = (i <= n - 2 && i >= n - 1 - p) ? 1 : 0;
    } else {
        lo[0] = 0;
        len[0] = i == 0 ? p : 0;
        lo[2] = n + p;
        len[2] = i == n - 1 ? p : 0;
    }
}

// 16 bytes of bf16 / fp32 as fp32 and back
__device__ __forceinline__ void unpack(uint4 a, float (&v)[8]) {
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&w[q]));
        v[2 * q] = f.x;
        v[2 * q + 1] = f.y;
    }
}
__device__ __forceinline__ void unpack(uint4 a, float (&v)[4]) {
    v[0] = __uint_as_float(a.x); v[1] = __uint_as_float(a.y); v[2] = __uint_as_float(a.z); v[3] = __uint_as_float(a.w);
}
__device__ __forceinline__ uint4 pack(const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * q], v[2 * q + 1]);
        w[q] = *reinterpret_cast<const uint32_t *>(&h);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ uint4 pack(const float (&v)[4]) {
    return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
}

// N elements per thread: 16 / sizeof(T) (one 16-byte chunk) or 1 (the scalar path)
template <typename T, int N>
__device__ __forceinline__ void load_f(const T *p, float (&v)[N]) {
    if constexpr (N == 1) v[0] = ldf(p);
    else unpack(__ldg(reinterpret_cast<const uint4 *>(p)), v);
}
template <typename T, int N>
__device__ __forceinline__ void store_f(T *p, const float (&v)[N]) {
    if constexpr (N == 1) stf(p, v[0]);
    else *reinterpret_cast<uint4 *>(p) = pack(v);
}

// one CTA per output row (b, oy); its threads stride over the row's (column, channel chunk) pairs
template <typename T, int N>
__global__ void __launch_bounds__(256) pad_fwd_kernel(const T *__restrict__ x, int xs, T *__restrict__ out, int os, int H, int W, int C,
                                                      int p, int mode) {
    const int Ho = H + 2 * p, Wo = W + 2 * p, nc = C / N;
    const int b = blockIdx.x / Ho, oy = blockIdx.x - b * Ho;
    const T *src = x + ((long long)b * H + pad_src(oy, H, p, mode)) * W * xs;
    T *dst = out + (long long)blockIdx.x * Wo * os;
    for (int j = threadIdx.x; j < Wo * nc; j += blockDim.x) {
        const int ox = j / nc, c = (j - ox * nc) * N;
        const T *s = src + (long long)pad_src(ox, W, p, mode) * xs + c;
        T *d = dst + (long long)ox * os + c;
        if constexpr (N == 1) *d = *s;
        else *reinterpret_cast<uint4 *>(d) = __ldg(reinterpret_cast<const uint4 *>(s));
    }
}

// one CTA per input row (b, iy); each thread gathers one (column, channel chunk) of it
template <typename T, int N>
__global__ void __launch_bounds__(256) pad_bwd_kernel(const T *__restrict__ g, int gs, T *__restrict__ dx, int ds, int H, int W, int C,
                                                      int p, int mode) {
    const int Ho = H + 2 * p, Wo = W + 2 * p, nc = C / N;
    const int b = blockIdx.x / H, iy = blockIdx.x - b * H;
    int ylo[3], ylen[3];
    pad_runs(iy, H, p, mode, ylo, ylen);
    const T *gimg = g + (long long)b * Ho * Wo * gs;
    T *drow = dx + (long long)blockIdx.x * W * ds;
    for (int j = threadIdx.x; j < W * nc; j += blockDim.x) {
        const int ix = j / nc, c = (j - ix * nc) * N;
        int xlo[3], xlen[3];
        pad_runs(ix, W, p, mode, xlo, xlen);
        float s[N], e[N];
#pragma unroll
        for (int k = 0; k < N; ++k) s[k] = e[k] = 0.f;
#pragma unroll
        for (int r = 0; r < 3; ++r)
            for (int oy = ylo[r]; oy < ylo[r] + ylen[r]; ++oy)
#pragma unroll
                for (int q = 0; q < 3; ++q)
                    for (int ox = xlo[q]; ox < xlo[q] + xlen[q]; ++ox) {
                        float v[N];
                        load_f<T, N>(gimg + ((long long)oy * Wo + ox) * gs + c, v);
#pragma unroll
                        for (int k = 0; k < N; ++k) {          // Neumaier: s + e is the sum to ~1 ulp whatever the count
                            const float t = s[k] + v[k];
                            e[k] += fabsf(s[k]) >= fabsf(v[k]) ? (s[k] - t) + v[k] : (v[k] - t) + s[k];
                            s[k] = t;
                        }
                    }
#pragma unroll
        for (int k = 0; k < N; ++k) s[k] += e[k];
        store_f<T, N>(drow + (long long)ix * ds + c, s);
    }
}

}  // namespace
}  // namespace rdfc

using namespace rdfc;

static int elem_bytes(int dtype) { return dtype == RDFC_F32 ? 4 : 2; }

// `small` (B, H, W, C) and `big` (B, H + 2 pad, W + 2 pad, C): one dtype, one channel count; *vec: both allow 16-byte chunks
static int check_pad(const rdfc_view *small, const rdfc_view *big, int B, int H, int W, int pad, int mode, const char *what, bool *vec) {
    RDFC_REQUIRE(small && big && small->ptr && big->ptr, "%s: NULL view", what);
    RDFC_REQUIRE(mode == RDFC_PAD_REFLECT || mode == RDFC_PAD_REPLICATE, "%s: unknown mode %d (0 = reflect, 1 = replicate)", what, mode);
    RDFC_REQUIRE(pad >= 0, "%s: padding %d < 0", what, pad);
    RDFC_REQUIRE(B > 0 && H > 0 && W > 0, "%s: empty dimension (B %d, H %d, W %d)", what, B, H, W);
    RDFC_REQUIRE(mode != RDFC_PAD_REFLECT || (pad < H && pad < W),
                 "%s: reflection padding %d needs padding < H and < W, got H %d, W %d", what, pad, H, W);
    RDFC_REQUIRE((long long)B * (H + 2 * pad) < (1ll << 31) && (long long)(W + 2 * pad) * small->C < (1ll << 31), "%s: tensor too large", what);
    const int dt = small->dtype;
    RDFC_REQUIRE((dt == RDFC_BF16 || dt == RDFC_F32) && big->dtype == dt && !small->nchw && !big->nchw,
                 "%s: NHWC views of one dtype (bf16 or fp32) expected", what);
    RDFC_REQUIRE(small->C > 0 && big->C == small->C && small->pix_stride >= small->C && big->pix_stride >= big->C,
                 "%s: both views need the same channel count (%d vs %d), pixel strides >= it", what, small->C, big->C);
    const int eb = elem_bytes(dt);
    RDFC_REQUIRE((uintptr_t)small->ptr % eb == 0 && (uintptr_t)big->ptr % eb == 0, "%s: views not aligned to their %d-byte elements", what, eb);
    const int n = 16 / eb;
    *vec = small->C % n == 0 && small->pix_stride % n == 0 && big->pix_stride % n == 0 && (uintptr_t)small->ptr % 16 == 0 &&
           (uintptr_t)big->ptr % 16 == 0;
    return 0;
}

template <typename T>
static int pad_forward(const rdfc_view *x, int B, int H, int W, int pad, int mode, const rdfc_view *out, bool vec, cudaStream_t st) {
    const int rows = B * (H + 2 * pad);
    if (vec)
        pad_fwd_kernel<T, 16 / sizeof(T)><<<rows, 256, 0, st>>>((const T *)x->ptr, x->pix_stride, (T *)out->ptr, out->pix_stride, H, W, x->C, pad, mode);
    else
        pad_fwd_kernel<T, 1><<<rows, 256, 0, st>>>((const T *)x->ptr, x->pix_stride, (T *)out->ptr, out->pix_stride, H, W, x->C, pad, mode);
    RDFC_CHECK_LAUNCH("pad_fwd_kernel");
    return 0;
}

template <typename T>
static int pad_backward(const rdfc_view *g, int B, int H, int W, int pad, int mode, const rdfc_view *gi, bool vec, cudaStream_t st) {
    if (vec)
        pad_bwd_kernel<T, 16 / sizeof(T)><<<B * H, 256, 0, st>>>((const T *)g->ptr, g->pix_stride, (T *)gi->ptr, gi->pix_stride, H, W, g->C, pad, mode);
    else
        pad_bwd_kernel<T, 1><<<B * H, 256, 0, st>>>((const T *)g->ptr, g->pix_stride, (T *)gi->ptr, gi->pix_stride, H, W, g->C, pad, mode);
    RDFC_CHECK_LAUNCH("pad_bwd_kernel");
    return 0;
}

extern "C" int rdfc_pad_nhwc_forward(const rdfc_view *x, int B, int H, int W, int pad, int mode, const rdfc_view *out, void *stream) {
    bool vec;
    if (int rc = check_pad(x, out, B, H, W, pad, mode, "pad forward", &vec)) return rc;
    if (x->dtype == RDFC_F32) return pad_forward<float>(x, B, H, W, pad, mode, out, vec, (cudaStream_t)stream);
    return pad_forward<__nv_bfloat16>(x, B, H, W, pad, mode, out, vec, (cudaStream_t)stream);
}

extern "C" int rdfc_pad_nhwc_backward(const rdfc_view *grad_out, int B, int H, int W, int pad, int mode, const rdfc_view *grad_in,
                                      void *stream) {
    bool vec;
    if (int rc = check_pad(grad_in, grad_out, B, H, W, pad, mode, "pad backward", &vec)) return rc;
    if (grad_out->dtype == RDFC_F32) return pad_backward<float>(grad_out, B, H, W, pad, mode, grad_in, vec, (cudaStream_t)stream);
    return pad_backward<__nv_bfloat16>(grad_out, B, H, W, pad, mode, grad_in, vec, (cudaStream_t)stream);
}
