// fp32-compute convolution kernels on CUDA cores (NHWC implicit GEMM), used for
//   * the fp32 parity mode of the whole generator (max-abs <= 1e-4 against the reference needs fp32 products), and
//   * in bf16 mode, the layers that are not GEMM shaped: the 3/1-channel stems and the Cout <= 8 decode heads
//     (memory bound; a warp per output pixel).
// Epilogue (both kernels): y = act(acc * scale[co] + shift[co] + residual), written into an NHWC channel slice or an
// NCHW tensor.  Reference layers: encoder_decoder/common.py:29-61, rdf_generator.py:60-102.
#include <type_traits>

#include "common.cuh"

namespace rdfc {
namespace {

struct SrcView {
    const void *ptr;
    int C, stride, nchw;
};

struct ConvGeo {
    int B, Hi, Wi, Ho, Wo, kh, kw, stride, pad, transposed, act;
    SrcView in, in2;
    void *out;
    int Cout, out_stride, out_nchw;
    const void *res;
    int res_stride;
    const float *weight, *scale, *shift;
    int CinT;   // in.C + in2.C
};

// input coordinate of output (oy,ox) for tap (ky,kx); false if the tap does not touch the input
__device__ __forceinline__ bool tap_coord(const ConvGeo &g, int oy, int ox, int ky, int kx, int &iy, int &ix) {
    if (!g.transposed) {
        iy = oy * g.stride - g.pad + ky;
        ix = ox * g.stride - g.pad + kx;
    } else {  // ConvTranspose2d(k, s=2, p): oy = 2*iy - p + ky
        const int ty = oy + g.pad - ky, tx = ox + g.pad - kx;
        if (ty < 0 || tx < 0 || (ty & 1) || (tx & 1)) return false;
        iy = ty >> 1;
        ix = tx >> 1;
    }
    return iy >= 0 && iy < g.Hi && ix >= 0 && ix < g.Wi;
}

template <typename T>
__device__ __forceinline__ float load_elem(const SrcView &v, int Hi, int Wi, int b, int iy, int ix, int c) {
    const T *p = (const T *)v.ptr;
    if (v.nchw) return ldf(p + (((long long)b * v.C + c) * Hi + iy) * Wi + ix);
    return ldf(p + (((long long)b * Hi + iy) * Wi + ix) * v.stride + c);
}

// ------------------------------------------------------------------------------------------------------------------
// Tiled implicit GEMM: CTA = 64 output pixels x 64 output channels, 256 threads, 4x4 register tile, K step 16.
constexpr int BM = 64, BN = 64, BK = 16, NTH = 256;

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(NTH) conv_tile_kernel(ConvGeo g) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const long long M = (long long)g.B * g.Ho * g.Wo;
    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    // A-load mapping: 4 consecutive threads fetch 16 consecutive channels of one pixel
    const int a_pl = tid >> 2, a_k4 = (tid & 3) * 4;
    const long long a_m = m0 + a_pl;
    int a_b = 0, a_oy = 0, a_ox = 0;
    const bool a_ok = a_m < M;
    if (a_ok) {
        a_b = (int)(a_m / (g.Ho * g.Wo));
        const int r = (int)(a_m % (g.Ho * g.Wo));
        a_oy = r / g.Wo;
        a_ox = r % g.Wo;
    }
    // B-load mapping: thread -> (k = tid/16, 4 consecutive couts)
    const int b_k = tid >> 4, b_n4 = (tid & 15) * 4;
    // compute mapping
    const int tx = tid & 15, ty = tid >> 4;   // tx -> couts tx*4.., ty -> pixels ty*4..
    float acc[4][4] = {};

    const int ntaps = g.kh * g.kw;
    for (int t = 0; t < ntaps; ++t) {
        const int ky = t / g.kw, kx = t % g.kw;
        int iy = 0, ix = 0;
        const bool hit = a_ok && tap_coord(g, a_oy, a_ox, ky, kx, iy, ix);
        for (int c0 = 0; c0 < g.CinT; c0 += BK) {
            // ---- stage A
            float av[4] = {0.f, 0.f, 0.f, 0.f};
            if (hit) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int c = c0 + a_k4 + i;
                    if (c < g.in.C) av[i] = load_elem<TIn>(g.in, g.Hi, g.Wi, a_b, iy, ix, c);
                    else if (c < g.CinT) av[i] = load_elem<TIn>(g.in2, g.Hi, g.Wi, a_b, iy, ix, c - g.in.C);
                }
            }
            // ---- stage B: weight[t][c][co]
            float bv[4] = {0.f, 0.f, 0.f, 0.f};
            {
                const int c = c0 + b_k;
                if (c < g.CinT) {
                    const float *wp = g.weight + ((long long)t * g.CinT + c) * g.Cout + n0 + b_n4;
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (n0 + b_n4 + i < g.Cout) bv[i] = __ldg(wp + i);
                }
            }
            __syncthreads();
#pragma unroll
            for (int i = 0; i < 4; ++i) As[a_k4 + i][a_pl] = av[i];
#pragma unroll
            for (int i = 0; i < 4; ++i) Bs[b_k][b_n4 + i] = bv[i];
            __syncthreads();
#pragma unroll
            for (int k = 0; k < BK; ++k) {
                const float4 a4 = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
                const float4 b4 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
                const float a_[4] = {a4.x, a4.y, a4.z, a4.w}, b_[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a_[i], b_[j], acc[i][j]);
            }
        }
    }
    // ---- epilogue
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long long m = m0 + ty * 4 + i;
        if (m >= M) continue;
        const int b = (int)(m / (g.Ho * g.Wo)), r = (int)(m % (g.Ho * g.Wo));
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = n0 + tx * 4 + j;
            if (co >= g.Cout) continue;
            float v = acc[i][j] * (g.scale ? __ldg(g.scale + co) : 1.f) + (g.shift ? __ldg(g.shift + co) : 0.f);
            if (g.res) v += ldf((const TOut *)g.res + m * g.res_stride + co);
            v = apply_act(v, g.act);
            TOut *o = (TOut *)g.out;
            if (g.out_nchw) stf(o + ((long long)b * g.Cout + co) * g.Ho * g.Wo + r, v);
            else stf(o + m * g.out_stride + co, v);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Small-Cout kernel (Cout <= 8): one warp per output pixel, lanes split the input channels, weights in shared
// memory as [tap][cin][cout]; a butterfly reduction finishes each output.  grid-stride over pixels.
constexpr int SC_MAX = 8;

template <typename TIn, typename TOut, int COUT>
__global__ void __launch_bounds__(256) conv_smallc_kernel(ConvGeo g) {
    extern __shared__ float s_w[];   // ntaps * CinT * COUT
    const int ntaps = g.kh * g.kw;
    for (int e = threadIdx.x; e < ntaps * g.CinT * COUT; e += blockDim.x) {
        const int co = e % COUT, rest = e / COUT;
        s_w[e] = co < g.Cout ? __ldg(g.weight + (long long)rest * g.Cout + co) : 0.f;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const long long M = (long long)g.B * g.Ho * g.Wo;
    for (long long m = (long long)blockIdx.x * wpb + (threadIdx.x >> 5); m < M; m += (long long)gridDim.x * wpb) {
        const int b = (int)(m / (g.Ho * g.Wo)), r = (int)(m % (g.Ho * g.Wo));
        const int oy = r / g.Wo, ox = r % g.Wo;
        float acc[COUT];
#pragma unroll
        for (int j = 0; j < COUT; ++j) acc[j] = 0.f;
        for (int t = 0; t < ntaps; ++t) {
            int iy, ix;
            if (!tap_coord(g, oy, ox, t / g.kw, t % g.kw, iy, ix)) continue;   // warp-uniform
            const float *wt = s_w + (long long)t * g.CinT * COUT;
            for (int c = lane; c < g.CinT; c += 32) {
                const float v = c < g.in.C ? load_elem<TIn>(g.in, g.Hi, g.Wi, b, iy, ix, c)
                                           : load_elem<TIn>(g.in2, g.Hi, g.Wi, b, iy, ix, c - g.in.C);
#pragma unroll
                for (int j = 0; j < COUT; ++j) acc[j] = fmaf(v, wt[c * COUT + j], acc[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < COUT; ++j)
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], s);
        if (lane < g.Cout) {
            float v = 0.f;
#pragma unroll
            for (int j = 0; j < COUT; ++j) v = (lane == j) ? acc[j] : v;
            v = v * (g.scale ? __ldg(g.scale + lane) : 1.f) + (g.shift ? __ldg(g.shift + lane) : 0.f);
            if (g.res) v += ldf((const TOut *)g.res + m * g.res_stride + lane);
            v = apply_act(v, g.act);
            TOut *o = (TOut *)g.out;
            if (g.out_nchw) stf(o + ((long long)b * g.Cout + lane) * g.Ho * g.Wo + r, v);
            else stf(o + m * g.out_stride + lane, v);
        }
    }
}


// ------------------------------------------------------------------------------------------------------------------
// Stem kernel: NCHW fp32 input with <= 4 channels (normal map / sparse depth, rdf_generator.py:60-61,77-80), 3x3,
// stride 1, pad 1.  CTA = 32x8 pixels; the input tile + halo and the whole filter bank sit in shared memory; a thread
// produces one pixel x 16 output channels per pass and writes them as one 32/64-byte NHWC vector.
constexpr int ST_TX = 32, ST_TY = 8, ST_MAXC = 4;

// 16 consecutive channels of one pixel: vector stores when the slice is 16-byte aligned, scalar tail otherwise
__device__ __forceinline__ void store16(float *p, const float (&y)[16], int nvalid, bool vec_ok) {
    if (vec_ok && nvalid >= 16) {
        float4 *q = reinterpret_cast<float4 *>(p);
#pragma unroll
        for (int i = 0; i < 4; ++i) q[i] = make_float4(y[4 * i], y[4 * i + 1], y[4 * i + 2], y[4 * i + 3]);
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (j < nvalid) p[j] = y[j];
    }
}
__device__ __forceinline__ void store16(__nv_bfloat16 *p, const float (&y)[16], int nvalid, bool vec_ok) {
    if (vec_ok && nvalid >= 16) {
        uint32_t o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(y[2 * i], y[2 * i + 1]);
            o[i] = *reinterpret_cast<const uint32_t *>(&h2);
        }
        uint4 *q = reinterpret_cast<uint4 *>(p);
        q[0] = make_uint4(o[0], o[1], o[2], o[3]);
        q[1] = make_uint4(o[4], o[5], o[6], o[7]);
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (j < nvalid) p[j] = __float2bfloat16_rn(y[j]);
    }
}

template <typename TOut>
__global__ void __launch_bounds__(ST_TX *ST_TY) conv_stem_kernel(ConvGeo g) {
    extern __shared__ float st_smem[];
    float *s_in = st_smem;                                           // [Cin][ST_TY+2][ST_TX+2]
    float *s_w = s_in + ST_MAXC * (ST_TY + 2) * (ST_TX + 2);        // [Cin*9][CoutP]  (CoutP = Cout rounded up to 16)
    const int Cin = g.in.C, CoutP = (g.Cout + 15) / 16 * 16;
    const int tid = threadIdx.y * ST_TX + threadIdx.x;
    const int b = blockIdx.z, x0 = blockIdx.x * ST_TX, y0 = blockIdx.y * ST_TY;
    const float *in = (const float *)g.in.ptr;
    for (int e = tid; e < Cin * (ST_TY + 2) * (ST_TX + 2); e += ST_TX * ST_TY) {
        const int c = e / ((ST_TY + 2) * (ST_TX + 2)), r = e % ((ST_TY + 2) * (ST_TX + 2));
        const int yy = y0 + r / (ST_TX + 2) - 1, xx = x0 + r % (ST_TX + 2) - 1;
        s_in[e] = (yy >= 0 && yy < g.Hi && xx >= 0 && xx < g.Wi) ? __ldg(in + (((long long)b * Cin + c) * g.Hi + yy) * g.Wi + xx) : 0.f;
    }
    // packed SIMT weights are [tap][cin][cout]; re-index to [(cin*9+tap)][coutP]
    for (int e = tid; e < Cin * 9 * CoutP; e += ST_TX * ST_TY) {
        const int co = e % CoutP, q = e / CoutP, ci = q / 9, t = q % 9;
        s_w[e] = co < g.Cout ? __ldg(g.weight + ((long long)t * Cin + ci) * g.Cout + co) : 0.f;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= g.Wi || y >= g.Hi) return;
    float v[ST_MAXC * 9];
    for (int ci = 0; ci < Cin; ++ci)
#pragma unroll
        for (int t = 0; t < 9; ++t) v[ci * 9 + t] = s_in[(ci * (ST_TY + 2) + threadIdx.y + t / 3) * (ST_TX + 2) + threadIdx.x + t % 3];
    const long long pix = ((long long)b * g.Ho + y) * g.Wo + x;
    TOut *op = (TOut *)g.out + pix * g.out_stride;
    const bool vec_ok = ((uintptr_t)g.out % 16) == 0 && (g.out_stride * sizeof(TOut)) % 16 == 0;
    for (int c0 = 0; c0 < g.Cout; c0 += 16) {
        float acc[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] = 0.f;
        for (int q = 0; q < Cin * 9; ++q) {
            const float4 *w4 = reinterpret_cast<const float4 *>(s_w + q * CoutP + c0);
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
                const float4 w = w4[j4];
                acc[4 * j4 + 0] = fmaf(v[q], w.x, acc[4 * j4 + 0]);
                acc[4 * j4 + 1] = fmaf(v[q], w.y, acc[4 * j4 + 1]);
                acc[4 * j4 + 2] = fmaf(v[q], w.z, acc[4 * j4 + 2]);
                acc[4 * j4 + 3] = fmaf(v[q], w.w, acc[4 * j4 + 3]);
            }
        }
        float y[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int co = c0 + j;
            const float r = co < g.Cout ? acc[j] * (g.scale ? __ldg(g.scale + co) : 1.f) + (g.shift ? __ldg(g.shift + co) : 0.f) : 0.f;
            y[j] = apply_act(r, g.act);
        }
        store16(op + c0, y, g.Cout - c0, vec_ok);
    }
}

template <typename TIn, typename TOut>
int launch(const ConvGeo &g, cudaStream_t st) {
    if constexpr (std::is_same<TIn, float>::value) {
        if (g.in.nchw && !g.in2.ptr && g.in.C <= ST_MAXC && g.kh == 3 && g.kw == 3 && g.stride == 1 && g.pad == 1 &&
            !g.transposed && !g.res && !g.out_nchw && g.Cout <= 256) {
            const int CoutP = (g.Cout + 15) / 16 * 16;
            const size_t smem = sizeof(float) * (ST_MAXC * (ST_TY + 2) * (ST_TX + 2) + g.in.C * 9 * CoutP);
            dim3 grid(cdiv(g.Wi, ST_TX), cdiv(g.Hi, ST_TY), g.B), block(ST_TX, ST_TY);
            RDFC_REQUIRE(g.B <= 65535 && smem <= 48 * 1024, "stem conv: batch / filter bank too large");
            conv_stem_kernel<TOut><<<grid, block, smem, st>>>(g);
            RDFC_CHECK_LAUNCH("conv_stem_kernel");
            return 0;
        }
    }
    const long long M = (long long)g.B * g.Ho * g.Wo;
    if (g.Cout <= SC_MAX && g.CinT >= 32) {
        const size_t smem = sizeof(float) * g.kh * g.kw * g.CinT * (g.Cout <= 1 ? 1 : (g.Cout <= 2 ? 2 : (g.Cout <= 4 ? 4 : 8)));
        RDFC_REQUIRE(smem <= 96 * 1024, "small-Cout conv: filter bank does not fit shared memory");
        const int blocks = (int)min((long long)cdiv(M, 8), (long long)sm_count() * 8);
#define RDFC_SC(N)                                                                                         \
    do {                                                                                                   \
        RDFC_CUDA(cudaFuncSetAttribute(conv_smallc_kernel<TIn, TOut, N>,                                   \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));           \
        conv_smallc_kernel<TIn, TOut, N><<<blocks, 256, smem, st>>>(g);                                    \
    } while (0)
        if (g.Cout <= 1) RDFC_SC(1);
        else if (g.Cout <= 2) RDFC_SC(2);
        else if (g.Cout <= 4) RDFC_SC(4);
        else RDFC_SC(8);
#undef RDFC_SC
        RDFC_CHECK_LAUNCH("conv_smallc_kernel");
        return 0;
    }
    dim3 grid(cdiv(M, BM), cdiv(g.Cout, BN));
    RDFC_REQUIRE(grid.y <= 65535, "Cout too large");
    conv_tile_kernel<TIn, TOut><<<grid, NTH, 0, st>>>(g);
    RDFC_CHECK_LAUNCH("conv_tile_kernel");
    return 0;
}

}  // namespace

int conv_simt_forward(const rdfc_conv_desc *d, cudaStream_t st) {
    ConvGeo g{};
    g.B = d->B; g.Hi = d->Hi; g.Wi = d->Wi; g.Ho = d->Ho; g.Wo = d->Wo;
    g.kh = d->kh; g.kw = d->kw; g.stride = d->stride; g.pad = d->pad; g.transposed = d->transposed; g.act = d->act;
    g.in = SrcView{d->in.ptr, d->in.C, d->in.pix_stride, d->in.nchw};
    g.in2 = SrcView{d->in2.ptr, d->in2.ptr ? d->in2.C : 0, d->in2.pix_stride, d->in2.nchw};
    g.CinT = g.in.C + g.in2.C;
    g.out = d->out.ptr; g.Cout = d->out.C; g.out_stride = d->out.pix_stride; g.out_nchw = d->out.nchw;
    g.res = d->residual.ptr; g.res_stride = d->residual.pix_stride;
    g.weight = (const float *)d->weight; g.scale = d->scale; g.shift = d->shift;
    RDFC_REQUIRE(!d->in2.ptr || d->in2.dtype == d->in.dtype, "both sources must share a dtype");
    RDFC_REQUIRE(!d->residual.ptr || (d->residual.dtype == d->out.dtype && !d->residual.nchw && !d->out.nchw),
                 "residual must be NHWC with the output's dtype");
    RDFC_REQUIRE(!d->transposed || d->stride == 2, "transposed convolution supports stride 2 only");
    const int it = d->in.dtype, ot = d->out.dtype;
    if (it == RDFC_F32 && ot == RDFC_F32) return launch<float, float>(g, st);
    if (it == RDFC_F32 && ot == RDFC_BF16) return launch<float, __nv_bfloat16>(g, st);
    if (it == RDFC_BF16 && ot == RDFC_BF16) return launch<__nv_bfloat16, __nv_bfloat16>(g, st);
    if (it == RDFC_BF16 && ot == RDFC_F32) return launch<__nv_bfloat16, float>(g, st);
    return fail(RDFC_ERR_UNSUPPORTED, "conv (SIMT): unsupported dtype pair (%d,%d)", it, ot);
}

}  // namespace rdfc
