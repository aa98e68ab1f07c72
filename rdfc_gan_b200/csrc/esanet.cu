// Glue kernels of the ESANet guidance network (RDF-GAN's global_guidance_module,
// F/lib/models/segmentator/esa_net/esa_net_one_modality.py:11-194, F = /root/reference/RDF-GAN) over NHWC activations, bf16 (the
// throughput mode) or fp32 (the parity modes).  Every kernel is a template over the activation type T; the bf16 instantiations
// keep the arithmetic and store order they had before fp32 existed, so the bf16 network's outputs are unchanged.
//
// The GEMM-shaped layers of ESANet (ResNet BasicBlocks, 1x1 skip / context convs, decoder 3x3 and factorised 3x1 / 1x3 convs,
// conv_out) run on conv_umma_kernel; what is left are HBM-bound layers with a handful of input channels or no contraction at
// all: the 7x7 stride-2 stem, max pooling, squeeze-and-excitation, the pyramid-pooling module's average pools and nearest
// up-sampling, and the decoder's "learned" x2 up-sampling (nearest + depth-wise 3x3, + skip add).
#include "common.cuh"

namespace rdfc {
namespace {

// eight consecutive channels of an NHWC pixel: one 16-byte access in bf16, two in fp32
template <typename T>
__device__ __forceinline__ void load8(const T *p, float (&v)[8]);
template <>
__device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16 *p, float (&v)[8]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p));
    const __nv_bfloat162 *h = reinterpret_cast<const __nv_bfloat162 *>(&a);
#pragma unroll
    for (int q = 0; q < 4; ++q) { const float2 f = __bfloat1622float2(h[q]); v[2 * q] = f.x; v[2 * q + 1] = f.y; }
}
template <>
__device__ __forceinline__ void load8<float>(const float *p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4 *>(p)), b = __ldg(reinterpret_cast<const float4 *>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void store8(__nv_bfloat16 *p, const float (&v)[8]) {
    uint32_t o[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) { const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * q], v[2 * q + 1]); o[q] = *reinterpret_cast<const uint32_t *>(&h); }
    *reinterpret_cast<uint4 *>(p) = make_uint4(o[0], o[1], o[2], o[3]);
}
__device__ __forceinline__ void store8(float *p, const float (&v)[8]) {
    reinterpret_cast<float4 *>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4 *>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
// copy of eight channels without conversion
__device__ __forceinline__ void copy8(__nv_bfloat16 *d, const __nv_bfloat16 *s) {
    *reinterpret_cast<uint4 *>(d) = __ldg(reinterpret_cast<const uint4 *>(s));
}
__device__ __forceinline__ void copy8(float *d, const float *s) {
    reinterpret_cast<float4 *>(d)[0] = __ldg(reinterpret_cast<const float4 *>(s));
    reinterpret_cast<float4 *>(d)[1] = __ldg(reinterpret_cast<const float4 *>(s) + 1);
}

// ---- encoder.conv1 + bn1 + ReLU: k x k (k <= 7) stride-s conv from fp32 NCHW (Cin <= 4) to T NHWC (Cout = 64) -------------
// block = 64 threads (one per output channel) x 4 pixels; the filter bank sits in shared memory as [tap][ci][cout].
template <typename T>
__global__ void __launch_bounds__(256) first_conv_kernel(const float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ scale,
                                                         const float *__restrict__ shift, T *__restrict__ out, int out_stride, int B,
                                                         int Cin, int Hi, int Wi, int Ho, int Wo, int k, int s, int pad, int Cout, int relu) {
    extern __shared__ float sw[];                       // [k*k*Cin][Cout]
    const int ntaps = k * k * Cin;
    for (int e = threadIdx.x; e < ntaps * Cout; e += blockDim.x) {
        const int co = e % Cout, t = e / Cout;           // t = (ky*k + kx)*Cin + ci ; torch layout w[co][ci][ky][kx]
        const int ci = t % Cin, kk = t / Cin;
        sw[e] = w[((long long)co * Cin + ci) * k * k + kk];
    }
    __syncthreads();
    const int co = threadIdx.x % Cout, sub = threadIdx.x / Cout, npb = blockDim.x / Cout;
    const long long npix = (long long)B * Ho * Wo;
    for (long long p = (long long)blockIdx.x * npb + sub; p < npix; p += (long long)gridDim.x * npb) {
        const int ox = (int)(p % Wo), oy = (int)((p / Wo) % Ho), b = (int)(p / ((long long)Wo * Ho));
        float acc = 0.f;
        for (int ky = 0; ky < k; ++ky) {
            const int iy = oy * s - pad + ky;
            if (iy < 0 || iy >= Hi) continue;
            for (int kx = 0; kx < k; ++kx) {
                const int ix = ox * s - pad + kx;
                if (ix < 0 || ix >= Wi) continue;
#pragma unroll 1                                    // unrolled (Cin <= 4), ptxas spills 16 bytes
                for (int ci = 0; ci < Cin; ++ci)
                    acc = fmaf(__ldg(x + (((long long)b * Cin + ci) * Hi + iy) * Wi + ix), sw[((ky * k + kx) * Cin + ci) * Cout + co], acc);
            }
        }
        float y = fmaf(acc, scale[co], shift[co]);
        if (relu) y = fmaxf(y, 0.f);
        stf(out + p * out_stride + co, y);
    }
}

// ---- the same for the case ESANet runs (7 x 7, stride 2, pad 3, 64 outputs): register-tiled --------------------------------------------
// A CTA computes 8 x 16 output pixels x 64 channels: the input patch (Cin x 21 x 37, zero padded) and the whole filter bank ([tap][ci][cout],
// 37 KB at Cin = 3) sit in shared memory; a warp owns one output row, a lane 4 adjacent pixels x 8 channels (32 accumulators).  Per (ci, ky)
// the lane reads the 13 patch values its four pixels touch once (three 16-byte loads + one) and per kx eight filter values (two 16-byte,
// warp-broadcast loads): 224 FMAs per 18 shared-memory loads instead of 1 per 2 in the kernel above (7.1 ms -> 0.3 ms at B = 32, 228 x 304).
constexpr int FC_TY = 8, FC_TX = 16, FC_PR = 2 * FC_TY + 5, FC_PC = 40;
template <typename T>
__global__ void __launch_bounds__(256) first_conv7s2_kernel(const float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ scale,
                                                            const float *__restrict__ shift, T *__restrict__ out, int out_stride, int B,
                                                            int Cin, int Hi, int Wi, int Ho, int Wo, int relu) {
    extern __shared__ __align__(16) float fsm[];
    float *sw = fsm;                                    // [49 * Cin][64]
    float *patch = fsm + 49 * Cin * 64;                 // [Cin][FC_PR][FC_PC]
    for (int e = threadIdx.x; e < 49 * Cin * 64; e += 256) {
        const int co = e & 63, t = e >> 6, ci = t % Cin, kk = t / Cin;          // torch layout w[co][ci][ky][kx]
        sw[e] = w[((long long)co * Cin + ci) * 49 + kk];
    }
    const int tiles_x = (Wo + FC_TX - 1) / FC_TX, tiles_y = (Ho + FC_TY - 1) / FC_TY;
    const long long ntiles = (long long)B * tiles_y * tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cg = lane & 7, pg = lane >> 3;
    float sc[8], sh[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) { sc[c] = scale[cg * 8 + c]; sh[c] = shift[cg * 8 + c]; }
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int tx = (int)(tile % tiles_x), ty = (int)((tile / tiles_x) % tiles_y), b = (int)(tile / ((long long)tiles_x * tiles_y));
        const int oy0 = ty * FC_TY, ox0 = tx * FC_TX, iy0 = 2 * oy0 - 3, ix0 = 2 * ox0 - 3;
        __syncthreads();                                // the previous tile's patch has been consumed (and the filters are in place)
        for (int e = threadIdx.x; e < Cin * FC_PR * FC_PC; e += 256) {
            const int c = e % FC_PC, r = (e / FC_PC) % FC_PR, ci = e / (FC_PC * FC_PR);
            const int iy = iy0 + r, ix = ix0 + c;
            patch[e] = (iy >= 0 && iy < Hi && ix >= 0 && ix < Wi) ? __ldg(x + (((long long)b * Cin + ci) * Hi + iy) * Wi + ix) : 0.f;
        }
        __syncthreads();
        float acc[4][8];
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[p][c] = 0.f;
        for (int ci = 0; ci < Cin; ++ci)
#pragma unroll 1
            for (int ky = 0; ky < 7; ++ky) {
                const float *prow = patch + (ci * FC_PR + 2 * warp + ky) * FC_PC + 8 * pg;
                float in[13];
                {
                    const float4 a = *reinterpret_cast<const float4 *>(prow), b4 = *reinterpret_cast<const float4 *>(prow + 4),
                                 c4 = *reinterpret_cast<const float4 *>(prow + 8);
                    in[0] = a.x; in[1] = a.y; in[2] = a.z; in[3] = a.w; in[4] = b4.x; in[5] = b4.y; in[6] = b4.z; in[7] = b4.w;
                    in[8] = c4.x; in[9] = c4.y; in[10] = c4.z; in[11] = c4.w; in[12] = prow[12];
                }
#pragma unroll
                for (int kx = 0; kx < 7; ++kx) {
                    const float *wp = sw + ((ky * 7 + kx) * Cin + ci) * 64 + cg * 8;
                    const float4 w0 = *reinterpret_cast<const float4 *>(wp), w1 = *reinterpret_cast<const float4 *>(wp + 4);
                    const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                    for (int p = 0; p < 4; ++p)
#pragma unroll
                        for (int c = 0; c < 8; ++c) acc[p][c] = fmaf(in[2 * p + kx], wv[c], acc[p][c]);
                }
            }
        const int oy = oy0 + warp;
        if (oy < Ho) {
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const int ox = ox0 + 4 * pg + p;
                if (ox >= Wo) continue;
                float y[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    y[c] = fmaf(acc[p][c], sc[c], sh[c]);
                    if (relu) y[c] = fmaxf(y[c], 0.f);
                }
                store8(out + (((long long)b * Ho + oy) * Wo + ox) * out_stride + cg * 8, y);
            }
        }
    }
}

// ---- max pooling 3x3 / stride 2 / pad 1 over NHWC, 8 channels per thread ------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) maxpool_kernel(const T *__restrict__ x, int x_stride, T *__restrict__ out,
                                                      int out_stride, int B, int C, int Hi, int Wi, int Ho, int Wo) {
    const int cgs = C >> 3;
    const long long total = (long long)B * Ho * Wo * cgs;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int cg = (int)(i % cgs);
        const long long p = i / cgs;
        const int ox = (int)(p % Wo), oy = (int)((p / Wo) % Ho), b = (int)(p / ((long long)Wo * Ho));
        float m[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) m[q] = -3.0e38f;
        for (int ky = 0; ky < 3; ++ky) {
            const int iy = 2 * oy - 1 + ky;
            if (iy < 0 || iy >= Hi) continue;
            for (int kx = 0; kx < 3; ++kx) {
                const int ix = 2 * ox - 1 + kx;
                if (ix < 0 || ix >= Wi) continue;
                float v[8];
                load8(x + (((long long)b * Hi + iy) * Wi + ix) * x_stride + cg * 8, v);
#pragma unroll
                for (int q = 0; q < 8; ++q) m[q] = fmaxf(m[q], v[q]);
            }
        }
        store8(out + p * out_stride + cg * 8, m);
    }
}

// ---- squeeze-and-excitation weights: w[b, :] = sigmoid(W2 relu(W1 mean[b, :] + b1) + b2), one CTA per image ----------------
__global__ void __launch_bounds__(256) se_weights_kernel(const float *__restrict__ mean, const float *__restrict__ w1, const float *__restrict__ b1,
                                                         const float *__restrict__ w2, const float *__restrict__ b2, float *__restrict__ out, int C,
                                                         int R) {
    extern __shared__ float sm[];                       // mean[C], hidden[R]
    float *m = sm, *h = sm + C;
    const int b = blockIdx.x;
    for (int c = threadIdx.x; c < C; c += blockDim.x) m[c] = mean[(long long)b * C + c];
    __syncthreads();
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        float a = b1[r];
        for (int c = 0; c < C; ++c) a = fmaf(w1[(long long)r * C + c], m[c], a);
        h[r] = fmaxf(a, 0.f);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float a = b2[c];
        for (int r = 0; r < R; ++r) a = fmaf(w2[(long long)c * R + r], h[r], a);
        out[(long long)b * C + c] = 1.f / (1.f + expf(-a));
    }
}

// ---- adaptive average pooling to bins x bins (torch's window rule: [floor(i*H/n), ceil((i+1)*H/n))) ------------------------
template <typename T>
__global__ void __launch_bounds__(256) adaptive_avgpool_kernel(const T *__restrict__ x, int x_stride, T *__restrict__ out,
                                                               int out_stride, int B, int C, int H, int W, int bins) {
    const long long total = (long long)B * bins * bins * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const long long p = i / C;
        const int bx = (int)(p % bins), by = (int)((p / bins) % bins), b = (int)(p / ((long long)bins * bins));
        const int y0 = (by * H) / bins, y1 = ((by + 1) * H + bins - 1) / bins, x0 = (bx * W) / bins, x1 = ((bx + 1) * W + bins - 1) / bins;
        float s = 0.f;
        for (int y = y0; y < y1; ++y)
            for (int xx = x0; xx < x1; ++xx) s += ldf(x + (((long long)b * H + y) * W + xx) * x_stride + c);
        stf(out + p * out_stride + c, s / (float)((y1 - y0) * (x1 - x0)));
    }
}

// ---- nearest up-sampling of a (hs x ws) map into a channel slice of a (H x W) NHWC buffer (torch 'nearest': floor(dst*in/out)) --
template <typename T>
__global__ void __launch_bounds__(256) upsample_nearest_kernel(const T *__restrict__ x, int x_stride, T *__restrict__ out,
                                                               int out_stride, int B, int C, int hs, int ws, int H, int W) {
    const int cgs = C >> 3;
    const long long total = (long long)B * H * W * cgs;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int cg = (int)(i % cgs);
        const long long p = i / cgs;
        const int ox = (int)(p % W), oy = (int)((p / W) % H), b = (int)(p / ((long long)W * H));
        const int sy = min((int)floorf(oy * ((float)hs / H)), hs - 1), sx = min((int)floorf(ox * ((float)ws / W)), ws - 1);
        copy8(out + p * out_stride + cg * 8, x + (((long long)b * hs + sy) * ws + sx) * x_stride + cg * 8);
    }
}

// ---- the decoder's learned up-sampling (Upsample, decoder.py:137-191, mode 'learned-3x3-zeropad'): nearest resize to (Ho, Wo),
// depth-wise 3x3 conv with zero padding + bias, optional skip add.  Output: T NHWC, or fp32 NCHW planes (the network's result).
template <typename T, bool kNCHW>
__global__ void __launch_bounds__(256) upsample_dw_kernel(const T *__restrict__ x, int x_stride, const float *__restrict__ w,
                                                          const float *__restrict__ bias, const T *__restrict__ skip, int skip_stride,
                                                          void *__restrict__ out, int out_stride, int B, int C, int Hi, int Wi, int Ho, int Wo) {
    const long long total = (long long)B * Ho * Wo * C;
    const float fy = (float)Hi / Ho, fx = (float)Wi / Wo;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        // NHWC output: channel fastest; NCHW output: x fastest (coalesced stores either way)
        int c, ox, oy, b;
        if (kNCHW) {
            ox = (int)(i % Wo); oy = (int)((i / Wo) % Ho); c = (int)((i / ((long long)Wo * Ho)) % C); b = (int)(i / ((long long)Wo * Ho * C));
        } else {
            c = (int)(i % C); ox = (int)((i / C) % Wo); oy = (int)((i / ((long long)C * Wo)) % Ho); b = (int)(i / ((long long)C * Wo * Ho));
        }
        float acc = bias[c];
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const int uy = oy - 1 + ky;                 // position in the up-sampled map
            if (uy < 0 || uy >= Ho) continue;
            const int sy = min((int)floorf(uy * fy), Hi - 1);
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int ux = ox - 1 + kx;
                if (ux < 0 || ux >= Wo) continue;
                const int sx = min((int)floorf(ux * fx), Wi - 1);
                acc = fmaf(w[c * 9 + ky * 3 + kx], ldf(x + (((long long)b * Hi + sy) * Wi + sx) * x_stride + c), acc);
            }
        }
        const long long p = ((long long)b * Ho + oy) * Wo + ox;
        if (skip) acc += ldf(skip + p * skip_stride + c);
        if (kNCHW) reinterpret_cast<float *>(out)[(((long long)b * C + c) * Ho + oy) * Wo + ox] = acc;
        else stf(reinterpret_cast<T *>(out) + p * out_stride + c, acc);
    }
}

// The two shapes ESANet runs, restructured (the kernel above stays as the general fallback; same arithmetic order, identical results):
// (1) fp32 NCHW result (the network's last up-sampling, 40 planes at full resolution): with x fastest across the lanes the plain kernel reads
// 2 bytes out of a different pixel per lane and tap.  Here a CTA owns 64 output pixels of one row x all channels: the (<= 3) source rows are
// staged in shared memory with coalesced channel-fastest reads, the outputs leave as 256-byte runs per plane (1.36 ms -> ~0.1 ms at B = 32).
// The staged rows are fp32 whatever T is, so the tile's shared memory (3 x 70 x (C | 1) floats, 34 KB at C = 40) is the same for a
// bf16 and an fp32 input; an fp32 input takes two 16-byte reads per eight channels instead of one.
constexpr int UP_TX = 64, UP_NCOL = 70;
template <typename T>
__global__ void __launch_bounds__(256) upsample_dw_nchw_kernel(const T *__restrict__ x, int x_stride, const float *__restrict__ w,
                                                               const float *__restrict__ bias, const T *__restrict__ skip, int skip_stride,
                                                               float *__restrict__ out, int C, int Hi, int Wi, int Ho, int Wo) {
    extern __shared__ float usrc[];                     // [3][UP_NCOL][CP]
    const int CP = C | 1;
    const float fy = (float)Hi / Ho, fx = (float)Wi / Wo;
    const int oy = blockIdx.y, ox0 = blockIdx.x * UP_TX, b = blockIdx.z;
    int sy[3];
    bool vy[3];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int uy = oy - 1 + ky;
        vy[ky] = uy >= 0 && uy < Ho;
        sy[ky] = vy[ky] ? min((int)floorf(uy * fy), Hi - 1) : 0;
    }
    const int ux_lo = max(ox0 - 1, 0), ux_hi = min(ox0 + UP_TX, Wo - 1);
    const int sx_lo = min((int)floorf(ux_lo * fx), Wi - 1), ncol = min((int)floorf(ux_hi * fx), Wi - 1) - sx_lo + 1;
    const int cgs = C >> 3;                             // 16-byte loads: eight channels per thread
    for (int e = threadIdx.x; e < 3 * ncol * cgs; e += 256) {
        const int cg = e % cgs, col = (e / cgs) % ncol, ky = e / (cgs * ncol);
        float *dst = usrc + (ky * UP_NCOL + col) * CP + cg * 8;
        if (vy[ky]) {
            float v[8];
            load8(x + (((long long)b * Hi + sy[ky]) * Wi + sx_lo + col) * x_stride + cg * 8, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) dst[q] = v[q];
        } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) dst[q] = 0.f;
        }
    }
    __syncthreads();
    const int ox = ox0 + (threadIdx.x & (UP_TX - 1));
    if (ox >= Wo) return;
    int scol[3];
    bool vx[3];
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
        const int ux = ox - 1 + kx;
        vx[kx] = ux >= 0 && ux < Wo;
        scol[kx] = vx[kx] ? min((int)floorf(ux * fx), Wi - 1) - sx_lo : 0;
    }
    for (int c = threadIdx.x / UP_TX; c < C; c += 256 / UP_TX) {
        float acc = bias[c];
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            if (!vy[ky]) continue;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx)
                if (vx[kx]) acc = fmaf(w[c * 9 + ky * 3 + kx], usrc[(ky * UP_NCOL + scol[kx]) * CP + c], acc);
        }
        if (skip) acc += ldf(skip + (((long long)b * Ho + oy) * Wo + ox) * skip_stride + c);
        out[(((long long)b * C + c) * Ho + oy) * Wo + ox] = acc;
    }
}

// (2) NHWC result: eight channels per thread (16-byte loads / stores), the depth-wise filters in shared memory as [tap][channel]
template <typename T>
__global__ void __launch_bounds__(256) upsample_dw_nhwc8_kernel(const T *__restrict__ x, int x_stride, const float *__restrict__ w,
                                                                const float *__restrict__ bias, const T *__restrict__ skip, int skip_stride,
                                                                T *__restrict__ out, int out_stride, int B, int C, int Hi, int Wi, int Ho,
                                                                int Wo) {
    extern __shared__ float usw[];                      // [9][C] then bias[C]
    for (int e = threadIdx.x; e < 9 * C; e += 256) usw[e] = w[(e % C) * 9 + e / C];
    for (int e = threadIdx.x; e < C; e += 256) usw[9 * C + e] = bias[e];
    __syncthreads();
    const int cgs = C >> 3;
    const long long total = (long long)B * Ho * Wo * cgs;
    const float fy = (float)Hi / Ho, fx = (float)Wi / Wo;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c0 = (int)(i % cgs) * 8;
        const long long p = i / cgs;
        const int ox = (int)(p % Wo), oy = (int)((p / Wo) % Ho), b = (int)(p / ((long long)Wo * Ho));
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] = usw[9 * C + c0 + q];
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const int uy = oy - 1 + ky;
            if (uy < 0 || uy >= Ho) continue;
            const int sy = min((int)floorf(uy * fy), Hi - 1);
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int ux = ox - 1 + kx;
                if (ux < 0 || ux >= Wo) continue;
                const int sx = min((int)floorf(ux * fx), Wi - 1);
                float v[8];
                load8(x + (((long long)b * Hi + sy) * Wi + sx) * x_stride + c0, v);
                const float *wt = usw + (ky * 3 + kx) * C + c0;
#pragma unroll
                for (int q = 0; q < 8; ++q) acc[q] = fmaf(wt[q], v[q], acc[q]);
            }
        }
        if (skip) {
            float v[8];
            load8(skip + p * skip_stride + c0, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[q] += v[q];
        }
        store8(out + p * out_stride + c0, acc);
    }
}

int grid_for(long long total) { return (int)min((long long)cdiv(total, 256), (long long)sm_count() * 16); }

}  // namespace
}  // namespace rdfc

using namespace rdfc;

// NHWC activation view: bf16 or fp32, C % 8 == 0, 16-byte aligned at every pixel (eight channels are one or two 16-byte accesses)
static int act_view_ok(const rdfc_view *v, const char *what) {
    RDFC_REQUIRE(v && v->ptr && (v->dtype == RDFC_BF16 || v->dtype == RDFC_F32) && !v->nchw && v->C % 8 == 0 &&
                     v->pix_stride % (v->dtype == RDFC_BF16 ? 8 : 4) == 0 && ((uintptr_t)v->ptr % 16) == 0,
                 "%s: 16-byte aligned bf16 or fp32 NHWC view with C %% 8 == 0 expected", what);
    return 0;
}

// both views valid and of one dtype
static int act_pair_ok(const rdfc_view *x, const rdfc_view *out, const char *what) {
    if (int rc = act_view_ok(x, what)) return rc;
    if (int rc = act_view_ok(out, what)) return rc;
    RDFC_REQUIRE(x->dtype == out->dtype, "%s: input and output views must share a dtype", what);
    return 0;
}

template <typename T>
static int first_conv_launch(const float *x_nchw, int B, int Cin, int Hi, int Wi, const float *weight, int k, int stride, int pad,
                             const float *scale, const float *shift, int relu, const rdfc_view *out, cudaStream_t st) {
    const int Ho = (Hi + 2 * pad - k) / stride + 1, Wo = (Wi + 2 * pad - k) / stride + 1;
    if (k == 7 && stride == 2 && pad == 3 && out->C == 64 && knob("RDFC_FIRSTCONV_FAST", 1) != 0) {     // ESANet's stem: the register-tiled kernel
        const size_t fsmem = (size_t)(49 * Cin * 64 + Cin * FC_PR * FC_PC) * sizeof(float);
        static bool attr[64] = {};
        int dev = 0;
        RDFC_CUDA(cudaGetDevice(&dev));
        if (!attr[dev & 63]) {
            RDFC_CUDA(cudaFuncSetAttribute(first_conv7s2_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024));
            attr[dev & 63] = true;
        }
        const long long ntiles = (long long)B * cdiv(Ho, FC_TY) * cdiv(Wo, FC_TX);
        const int grid = (int)min(ntiles, (long long)sm_count() * 3);
        first_conv7s2_kernel<T><<<grid, 256, fsmem, st>>>(x_nchw, weight, scale, shift, (T *)out->ptr, out->pix_stride, B, Cin, Hi, Wi, Ho, Wo, relu);
        RDFC_CHECK_LAUNCH("first_conv7s2_kernel");
        return 0;
    }
    const size_t smem = (size_t)k * k * Cin * out->C * sizeof(float);
    RDFC_REQUIRE(smem <= 48 * 1024, "first conv: filter bank exceeds 48 KB of shared memory");
    const long long npix = (long long)B * Ho * Wo;
    const int npb = 256 / out->C;
    const int grid = (int)min((long long)cdiv(npix, npb), (long long)sm_count() * 8);
    first_conv_kernel<T><<<grid, 256, smem, st>>>(x_nchw, weight, scale, shift, (T *)out->ptr, out->pix_stride, B, Cin, Hi, Wi, Ho, Wo, k, stride, pad,
                                                  out->C, relu);
    RDFC_CHECK_LAUNCH("first_conv_kernel");
    return 0;
}

extern "C" int rdfc_first_conv_forward(const float *x_nchw, int B, int Cin, int Hi, int Wi, const float *weight, int k, int stride, int pad,
                                       const float *scale, const float *shift, int relu, const rdfc_view *out, void *stream) {
    RDFC_REQUIRE(x_nchw && weight && scale && shift && out, "first conv: NULL argument");
    if (int rc = act_view_ok(out, "first conv out")) return rc;
    RDFC_REQUIRE(B > 0 && Cin >= 1 && Cin <= 4 && k >= 1 && k <= 7 && stride >= 1 && out->C <= 256 && 256 % out->C == 0,
                 "first conv: Cin <= 4, k <= 7, Cout a divisor of 256");
    return out->dtype == RDFC_F32
               ? first_conv_launch<float>(x_nchw, B, Cin, Hi, Wi, weight, k, stride, pad, scale, shift, relu, out, (cudaStream_t)stream)
               : first_conv_launch<__nv_bfloat16>(x_nchw, B, Cin, Hi, Wi, weight, k, stride, pad, scale, shift, relu, out, (cudaStream_t)stream);
}

extern "C" int rdfc_maxpool3x3s2_forward(const rdfc_view *x, const rdfc_view *out, int B, int Hi, int Wi, void *stream) {
    if (int rc = act_pair_ok(x, out, "maxpool")) return rc;
    RDFC_REQUIRE(x->C == out->C && B > 0 && Hi > 0 && Wi > 0, "maxpool: channel mismatch / empty");
    const int Ho = (Hi - 1) / 2 + 1, Wo = (Wi - 1) / 2 + 1;
    const int grid = grid_for((long long)B * Ho * Wo * (x->C / 8));
    if (x->dtype == RDFC_F32)
        maxpool_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float *)x->ptr, x->pix_stride, (float *)out->ptr, out->pix_stride, B, x->C,
                                                                      Hi, Wi, Ho, Wo);
    else
        maxpool_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16 *)x->ptr, x->pix_stride, (__nv_bfloat16 *)out->ptr,
                                                                              out->pix_stride, B, x->C, Hi, Wi, Ho, Wo);
    RDFC_CHECK_LAUNCH("maxpool_kernel");
    return 0;
}

extern "C" int rdfc_se_weights(const float *mean, const float *w1, const float *b1, const float *w2, const float *b2, float *out, int B, int C,
                               int R, void *stream) {
    RDFC_REQUIRE(mean && w1 && b1 && w2 && b2 && out && B > 0 && C > 0 && R > 0 && (size_t)(C + R) * 4 <= 48 * 1024, "SE weights: bad argument");
    se_weights_kernel<<<B, 256, (size_t)(C + R) * sizeof(float), (cudaStream_t)stream>>>(mean, w1, b1, w2, b2, out, C, R);
    RDFC_CHECK_LAUNCH("se_weights_kernel");
    return 0;
}

extern "C" int rdfc_adaptive_avgpool_forward(const rdfc_view *x, const rdfc_view *out, int B, int H, int W, int bins, void *stream) {
    if (int rc = act_pair_ok(x, out, "adaptive avgpool")) return rc;
    RDFC_REQUIRE(x->C == out->C && B > 0 && bins > 0 && H > 0 && W > 0, "adaptive avgpool: bad shape");
    const int grid = grid_for((long long)B * bins * bins * x->C);
    if (x->dtype == RDFC_F32)
        adaptive_avgpool_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float *)x->ptr, x->pix_stride, (float *)out->ptr, out->pix_stride,
                                                                               B, x->C, H, W, bins);
    else
        adaptive_avgpool_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(
            (const __nv_bfloat16 *)x->ptr, x->pix_stride, (__nv_bfloat16 *)out->ptr, out->pix_stride, B, x->C, H, W, bins);
    RDFC_CHECK_LAUNCH("adaptive_avgpool_kernel");
    return 0;
}

extern "C" int rdfc_upsample_nearest_forward(const rdfc_view *x, const rdfc_view *out, int B, int hs, int ws, int H, int W, void *stream) {
    if (int rc = act_pair_ok(x, out, "upsample nearest")) return rc;
    RDFC_REQUIRE(x->C == out->C && B > 0 && hs > 0 && ws > 0 && H > 0 && W > 0, "upsample nearest: bad shape");
    const int grid = grid_for((long long)B * H * W * (x->C / 8));
    if (x->dtype == RDFC_F32)
        upsample_nearest_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float *)x->ptr, x->pix_stride, (float *)out->ptr, out->pix_stride,
                                                                               B, x->C, hs, ws, H, W);
    else
        upsample_nearest_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(
            (const __nv_bfloat16 *)x->ptr, x->pix_stride, (__nv_bfloat16 *)out->ptr, out->pix_stride, B, x->C, hs, ws, H, W);
    RDFC_CHECK_LAUNCH("upsample_nearest_kernel");
    return 0;
}

template <typename T>
static int upsample_dw_launch(const rdfc_view *x, const float *weight, const float *bias, const T *sk, int sk_stride, const rdfc_view *out,
                              float *out_nchw, int B, int Hi, int Wi, int Ho, int Wo, cudaStream_t st) {
    const T *xp = (const T *)x->ptr;
    const long long total = (long long)B * Ho * Wo * x->C;
    const bool fast = knob("RDFC_UPSAMPLE_FAST", 1) != 0;
    if (out_nchw && fast && Hi <= Ho && Wi <= Wo && (size_t)3 * UP_NCOL * (x->C | 1) * 4 <= 48 * 1024 && B <= 65535 && Ho <= 65535) {
        upsample_dw_nchw_kernel<T><<<dim3(cdiv(Wo, UP_TX), Ho, B), 256, (size_t)3 * UP_NCOL * (x->C | 1) * 4, st>>>(
            xp, x->pix_stride, weight, bias, sk, sk_stride, out_nchw, x->C, Hi, Wi, Ho, Wo);
    } else if (out_nchw) {
        upsample_dw_kernel<T, true><<<grid_for(total), 256, 0, st>>>(xp, x->pix_stride, weight, bias, sk, sk_stride, out_nchw, 0, B, x->C, Hi, Wi, Ho, Wo);
    } else if (fast && (size_t)10 * x->C * 4 <= 48 * 1024) {
        upsample_dw_nhwc8_kernel<T><<<grid_for(total / 8), 256, (size_t)10 * x->C * 4, st>>>(xp, x->pix_stride, weight, bias, sk, sk_stride,
                                                                                             (T *)out->ptr, out->pix_stride, B, x->C, Hi, Wi, Ho, Wo);
    } else {
        upsample_dw_kernel<T, false><<<grid_for(total), 256, 0, st>>>(xp, x->pix_stride, weight, bias, sk, sk_stride, out->ptr, out->pix_stride, B, x->C,
                                                                      Hi, Wi, Ho, Wo);
    }
    RDFC_CHECK_LAUNCH("upsample_dw_kernel");
    return 0;
}

extern "C" int rdfc_upsample_dw_forward(const rdfc_view *x, const float *weight, const float *bias, const rdfc_view *skip, const rdfc_view *out,
                                        float *out_nchw, int B, int Hi, int Wi, int Ho, int Wo, void *stream) {
    if (int rc = act_view_ok(x, "upsample dw x")) return rc;
    RDFC_REQUIRE(weight && bias && B > 0 && Hi > 0 && Wi > 0 && Ho > 0 && Wo > 0, "upsample dw: bad argument");
    RDFC_REQUIRE((out && out->ptr) != (out_nchw != nullptr), "upsample dw: exactly one of out (NHWC) / out_nchw (fp32 NCHW)");
    if (!out_nchw) {
        if (int rc = act_pair_ok(x, out, "upsample dw")) return rc;
        RDFC_REQUIRE(out->C == x->C, "upsample dw: output channel mismatch");
    }
    const void *sk = nullptr;
    int sk_stride = 0;
    if (skip && skip->ptr) {
        if (int rc = act_pair_ok(x, skip, "upsample dw skip")) return rc;
        RDFC_REQUIRE(skip->C == x->C, "upsample dw: skip channel mismatch");
        sk = skip->ptr; sk_stride = skip->pix_stride;
    }
    if (x->dtype == RDFC_F32)
        return upsample_dw_launch<float>(x, weight, bias, (const float *)sk, sk_stride, out, out_nchw, B, Hi, Wi, Ho, Wo, (cudaStream_t)stream);
    return upsample_dw_launch<__nv_bfloat16>(x, weight, bias, (const __nv_bfloat16 *)sk, sk_stride, out, out_nchw, B, Hi, Wi, Ho, Wo,
                                             (cudaStream_t)stream);
}
