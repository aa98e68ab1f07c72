// Training-step kernels (SURVEY 8f rank 1): batch-statistics BatchNorm forward / backward fused with the activation and the
// residual add, and the convolution filter gradient.
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
            v[q] = __ldg(gamma + c) * rs * (dz - __ldg(sum_dz + c) * invn - xh * __ldg(sum_dzx + c) * invn);
        }
        st8(dy + p * dy_stride + c0, v);
        if (dres) st8(dres + p * dres_stride + c0, dzv);
    }
}

// ---------------------------------------------------------------------------------------------------------------------------
// Filter gradient.   dW[o][i][ky][kx] = sum over (b, py, px) of  G[b, py, px, o] * I[b, s*py - pad + ky, s*px - pad + kx, i]
// G = gradient w.r.t. the conv output (grid Hg x Wg, O channels), I = the conv input (grid Hi x Wi, I channels); the transposed
// convolution's filter gradient is the same sum with the roles of its input and its output gradient exchanged (host side).
// A GEMM with K = pixels: per CTA a 64 (o) x 64 (i) block of every tap over a chunk of G rows ("split K"), partial results to a
// workspace, reduced in chunk order by wgrad_reduce_kernel.  Both operands sit pixel-major in shared memory ([pixel][channel],
// rows padded to 144 bytes against bank conflicts), i.e. "transposed" for the tensor-core fragments: ldmatrix.trans delivers
// them.  Warp-level mma.sync (m16n8k16, bf16 -> fp32): this first version does not use tcgen05 (DESIGN.md, open items).
constexpr int WG_OB = 64, WG_IB = 64, WG_ROWP = 72;      // block sizes; smem row pitch in elements (64 channels + 8 pad)
constexpr int WG_TW = 32;                                  // G pixels per tile row (two K = 16 steps)

__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp16(uint32_t dst, const void *src, bool ok) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(ok ? 16u : 0u) : "memory");
}

struct WgradParams {
    const __nv_bfloat16 *G, *I;
    int g_stride, i_stride, O, Ich;
    int B, Hg, Wg, Hi, Wi, k, s, pad;
    int rows_per_cta;            // G rows (over all images) per CTA
    int TR;                      // G rows per tile
    int ksplit;                  // warps that share one (tap, half) by taking K steps round-robin (k = 1 layers)
    float *partial;              // [chunk][tap][64][64]
    int nchunk_cta;              // CTAs along the pixel dimension
};

// warp w: tap = w / (2 * ksplit), half = (w / ksplit) & 1, ks = w % ksplit.  Accumulators: 64 (o) x 32 (i) = 4 x 4 mma tiles.
__global__ void __launch_bounds__(576) wgrad_kernel(WgradParams P) {
    extern __shared__ __align__(16) unsigned char wsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntap = P.k * P.k, nwarps = blockDim.x >> 5;
    const int tap = warp / (2 * P.ksplit), half = (warp / P.ksplit) & 1, ks = warp % P.ksplit;
    const int ky = tap / P.k, kx = tap - ky * P.k;
    const int o0 = blockIdx.y * WG_OB, i0 = blockIdx.z * WG_IB;
    // tile geometry: TR rows x WG_TW columns of G; the I patch that its taps touch
    const int TR = P.TR, IR = P.s * (TR - 1) + P.k, IC = P.s * (WG_TW - 1) + P.k;
    const int g_tile = TR * WG_TW * WG_ROWP * 2, i_tile = IR * IC * WG_ROWP * 2;       // bytes per buffer
    const uint32_t sG = (uint32_t)__cvta_generic_to_shared(wsm), sI = sG + 2u * (uint32_t)g_tile;
    const long long total_rows = (long long)P.B * P.Hg;
    const long long row0 = (long long)blockIdx.x * P.rows_per_cta;
    const long long row1 = row0 + P.rows_per_cta < total_rows ? row0 + P.rows_per_cta : total_rows;
    const int xtiles = (P.Wg + WG_TW - 1) / WG_TW;

    float acc[4][4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;

    // tiles of this CTA: (row group, x tile); a row group never crosses an image
    // enumerate lazily: state (row, xt)
    auto issue_tile = [&](long long row, int xt, int buf) {
        const int b = (int)(row / P.Hg), gy0 = (int)(row - (long long)b * P.Hg), gx0 = xt * WG_TW;
        long long nr = row1 - row;
        if (nr > P.Hg - gy0) nr = P.Hg - gy0;
        if (nr > TR) nr = TR;
        // G tile: TR x WG_TW pixels x 64 channels (8 chunks of 16 bytes per pixel)
        for (int e = threadIdx.x; e < TR * WG_TW * 8; e += blockDim.x) {
            const int ch = e & 7, px = (e >> 3) % WG_TW, r = (e >> 3) / WG_TW;
            const int gy = gy0 + r, gx = gx0 + px, c = o0 + ch * 8;
            const bool ok = r < nr && gx < P.Wg && c < P.O;
            const __nv_bfloat16 *src = ok ? P.G + (((long long)b * P.Hg + gy) * P.Wg + gx) * P.g_stride + c : P.G;
            cp16(sG + (uint32_t)buf * g_tile + (uint32_t)((r * WG_TW + px) * WG_ROWP + ch * 8) * 2u, src, ok);
        }
        const int iy0 = P.s * gy0 - P.pad, ix0 = P.s * gx0 - P.pad;
        for (int e = threadIdx.x; e < IR * IC * 8; e += blockDim.x) {
            const int ch = e & 7, px = (e >> 3) % IC, r = (e >> 3) / IC;
            const int iy = iy0 + r, ix = ix0 + px, c = i0 + ch * 8;
            const bool ok = iy >= 0 && iy < P.Hi && ix >= 0 && ix < P.Wi && c < P.Ich && r < P.s * ((int)nr - 1) + P.k;
            const __nv_bfloat16 *src = ok ? P.I + (((long long)b * P.Hi + iy) * P.Wi + ix) * P.i_stride + c : P.I;
            cp16(sI + (uint32_t)buf * i_tile + (uint32_t)((r * IC + px) * WG_ROWP + ch * 8) * 2u, src, ok);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        return (int)nr;
    };

    long long row = row0;
    int xt = 0, buf = 0;
    int nr_cur = 0;
    if (row < row1) nr_cur = issue_tile(row, 0, 0);
    // lane-constant parts of the ldmatrix row addresses
    const int lrow = lane & 7, lmat = lane >> 3;
    while (row < row1) {
        // next tile
        long long nrow = row;
        int nxt = xt + 1;
        if (nxt == xtiles) { nxt = 0; nrow = row + nr_cur; }
        int nr_next = 0;
        if (nrow < row1) nr_next = issue_tile(nrow, nxt, buf ^ 1);
        else asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        if (tap < ntap) {
            const uint32_t gb = sG + (uint32_t)buf * g_tile, ib = sI + (uint32_t)buf * i_tile;
            const int nsteps = TR * (WG_TW / 16);
            for (int st = ks; st < nsteps; st += P.ksplit) {
                const int r = st / (WG_TW / 16), x16 = (st - r * (WG_TW / 16)) * 16;
                // A fragments (o x pixels): matrices (k0, m0), (k0, m0 + 8), (k0 + 8, m0), (k0 + 8, m0 + 8) of S[k = pixel][m = o]
                uint32_t afr[4][4];
#pragma unroll
                for (int mb = 0; mb < 4; ++mb) {
                    const int kk = x16 + lrow + 8 * (lmat >> 1), mm = mb * 16 + 8 * (lmat & 1);
                    ldsm_x4_t(gb + (uint32_t)((r * WG_TW + kk) * WG_ROWP + mm) * 2u, afr[mb]);
                }
                // B fragments (pixels x i): matrices (k0, n0), (k0 + 8, n0), (k0, n0 + 8), (k0 + 8, n0 + 8) of S'[k = pixel][n = i];
                // the pixel of K index kk under this tap is (s * r + ky, s * (x16 + kk) + kx) of the I patch
                uint32_t bfr[2][4];
#pragma unroll
                for (int nb = 0; nb < 2; ++nb) {
                    const int kk = lrow + 8 * (lmat & 1), nn = half * 32 + nb * 16 + 8 * (lmat >> 1);
                    const int pr = P.s * r + ky, pc = P.s * (x16 + kk) + kx;
                    ldsm_x4_t(ib + (uint32_t)((pr * IC + pc) * WG_ROWP + nn) * 2u, bfr[nb]);
                }
#pragma unroll
                for (int mb = 0; mb < 4; ++mb)
#pragma unroll
                    for (int nb = 0; nb < 2; ++nb) {
                        mma16816(acc[mb][2 * nb], afr[mb], bfr[nb][0], bfr[nb][1]);
                        mma16816(acc[mb][2 * nb + 1], afr[mb], bfr[nb][2], bfr[nb][3]);
                    }
            }
        }
        __syncthreads();
        row = nrow; xt = nxt; buf ^= 1; nr_cur = nr_next;
    }
    // partial results: chunk id = (CTA along pixels) * ksplit + ks
    if (tap < ntap) {
        const int g = lane >> 2, t = lane & 3;
        const long long chunk = (long long)blockIdx.x * P.ksplit + ks;
        const long long nchunks = (long long)P.nchunk_cta * P.ksplit;
        const int nob = gridDim.y, nib = gridDim.z;
        float *base = P.partial + ((((long long)(blockIdx.y * nib + blockIdx.z) * nchunks + chunk) * ntap + tap) * WG_OB) * WG_IB;
        (void)nob;
#pragma unroll
        for (int mb = 0; mb < 4; ++mb)
#pragma unroll
            for (int nb = 0; nb < 4; ++nb) {
                const int m = mb * 16 + g, n = half * 32 + nb * 8 + 2 * t;
                *reinterpret_cast<float2 *>(base + m * WG_IB + n) = make_float2(acc[mb][nb][0], acc[mb][nb][1]);
                *reinterpret_cast<float2 *>(base + (m + 8) * WG_IB + n) = make_float2(acc[mb][nb][2], acc[mb][nb][3]);
            }
    }
    (void)nwarps;
}

// dW[o][i][tap] (torch layout (O, I, kh, kw)) = sum over chunks, in chunk order
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float *__restrict__ partial, float *__restrict__ dw, int O, int Ich, int ntap,
                                                           int nchunks, int nib) {
    const long long total = (long long)O * Ich * ntap;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        // consecutive threads walk i fastest inside a 64 x 64 block for coalesced partial reads
        const int i = (int)(e % Ich);
        const int tap = (int)((e / Ich) % ntap);
        const int o = (int)(e / ((long long)Ich * ntap));
        const int ob = o / WG_OB, ib = i / WG_IB;
        const float *src = partial + (((long long)(ob * nib + ib) * nchunks * ntap + tap) * WG_OB + (o % WG_OB)) * WG_IB + (i % WG_IB);
        const long long cstride = (long long)ntap * WG_OB * WG_IB;
        float s = 0.f;
        for (int c = 0; c < nchunks; ++c) s += __ldg(src + (long long)c * cstride);
        dw[((long long)o * Ich + i) * ntap + tap] = s;
    }
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

// geometry shared by the workspace query and the launch
struct WgGeom { int nob, nib, nchunk_cta, rows_per_cta, TR, ksplit, nwarps; size_t smem; long long ws_floats; };
static int wgrad_geom(const rdfc_wgrad_desc *d, WgGeom *g) {
    RDFC_REQUIRE(d && (d->k == 1 || d->k == 3) && (d->stride == 1 || d->stride == 2) && d->pad == (d->k - 1) / 2,
                 "wgrad: 3x3 / 1x1 kernels, stride 1 / 2, padding (k-1)/2");
    RDFC_REQUIRE(d->B > 0 && d->Hg > 0 && d->Wg > 0 && d->Hi > 0 && d->Wi > 0, "wgrad: empty dimension");
    RDFC_REQUIRE(d->Hg == (d->Hi + 2 * d->pad - d->k) / d->stride + 1 && d->Wg == (d->Wi + 2 * d->pad - d->k) / d->stride + 1,
                 "wgrad: gradient grid (%d,%d) does not match the input grid (%d,%d)", d->Hg, d->Wg, d->Hi, d->Wi);
    const int O = d->grad_out.C, I = d->input.C;
    RDFC_REQUIRE(O % 8 == 0 && I % 8 == 0, "wgrad: channel counts must be multiples of 8");
    g->nob = cdiv(O, WG_OB); g->nib = cdiv(I, WG_IB);
    g->ksplit = d->k == 1 ? 8 : 1;
    g->nwarps = d->k * d->k * 2 * g->ksplit;             // 18 (3x3) or 16 (1x1)
    g->TR = d->stride == 1 ? 4 : 2;
    const int IR = d->stride * (g->TR - 1) + d->k, IC = d->stride * (WG_TW - 1) + d->k;
    g->smem = 2 * ((size_t)g->TR * WG_TW + (size_t)IR * IC) * WG_ROWP * 2;
    RDFC_REQUIRE(g->smem <= 220 * 1024, "wgrad: tile does not fit shared memory");
    const long long rows = (long long)d->B * d->Hg;
    long long want = (long long)sm_count() * 2 / ((long long)g->nob * g->nib);     // ~2 CTAs' worth of work per SM in total
    if (want < 1) want = 1;
    long long rpc = (rows + want - 1) / want;
    if (rpc < g->TR) rpc = g->TR;
    g->rows_per_cta = (int)rpc;
    g->nchunk_cta = (int)((rows + rpc - 1) / rpc);
    g->ws_floats = (long long)g->nob * g->nib * g->nchunk_cta * g->ksplit * d->k * d->k * WG_OB * WG_IB;
    return 0;
}

namespace rdfc {
bool wgrad_umma_ok(const rdfc_wgrad_desc *d);                       // wgrad_umma.cu: 3x3 filter gradients on tcgen05
long long wgrad_umma_workspace_floats(const rdfc_wgrad_desc *d);
int wgrad_umma(const rdfc_wgrad_desc *d, float *grad_weight, float *workspace, cudaStream_t st);
}  // namespace rdfc

extern "C" long long rdfc_conv_wgrad_workspace_floats(const rdfc_wgrad_desc *d) {
    WgGeom g;
    if (wgrad_geom(d, &g) != 0) return -1;
    if (wgrad_umma_ok(d)) {                                         // either path may serve the call (knob): size for both
        const long long u = wgrad_umma_workspace_floats(d);
        return u > g.ws_floats ? u : g.ws_floats;
    }
    return wgrad_geom(d, &g) == 0 ? g.ws_floats : -1;
}

extern "C" int rdfc_conv_wgrad(const rdfc_wgrad_desc *d, float *grad_weight, float *workspace, void *stream) {
    WgGeom g;
    if (int rc = wgrad_geom(d, &g)) return rc;
    RDFC_REQUIRE(grad_weight && workspace, "wgrad: NULL output / workspace");
    if (int rc = check_view(&d->grad_out, d->grad_out.C, "wgrad grad_out", RDFC_BF16)) return rc;
    if (int rc = check_view(&d->input, d->input.C, "wgrad input", RDFC_BF16)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (wgrad_umma_ok(d)) return wgrad_umma(d, grad_weight, workspace, st);
    WgradParams P{};
    P.G = (const __nv_bfloat16 *)d->grad_out.ptr; P.I = (const __nv_bfloat16 *)d->input.ptr;
    P.g_stride = d->grad_out.pix_stride; P.i_stride = d->input.pix_stride; P.O = d->grad_out.C; P.Ich = d->input.C;
    P.B = d->B; P.Hg = d->Hg; P.Wg = d->Wg; P.Hi = d->Hi; P.Wi = d->Wi; P.k = d->k; P.s = d->stride; P.pad = d->pad;
    P.rows_per_cta = g.rows_per_cta; P.TR = g.TR; P.ksplit = g.ksplit; P.partial = workspace; P.nchunk_cta = g.nchunk_cta;
    static bool attr[64] = {};
    int dev = 0;
    RDFC_CUDA(cudaGetDevice(&dev));
    if (!attr[dev & 63]) {
        RDFC_CUDA(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        attr[dev & 63] = true;
    }
    wgrad_kernel<<<dim3(g.nchunk_cta, g.nob, g.nib), g.nwarps * 32, g.smem, st>>>(P);
    RDFC_CHECK_LAUNCH("wgrad_kernel");
    const int ntap = d->k * d->k;
    const long long total = (long long)P.O * P.Ich * ntap;
    const int nblk = (int)min((long long)cdiv(total, 256), (long long)sm_count() * 8);
    wgrad_reduce_kernel<<<nblk, 256, 0, st>>>(workspace, grad_weight, P.O, P.Ich, ntap, g.nchunk_cta * g.ksplit, g.nib);
    RDFC_CHECK_LAUNCH("wgrad_reduce_kernel");
    return 0;
}
