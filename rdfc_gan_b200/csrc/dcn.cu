// General deformable convolution (DCN v1 / modulated v2), forward and backward, fp32 / fp64, NCHW.
//
// This is the drop-in for the reference's pybind module `DCN`
// (nlspn/deformconv/src/vision.cpp:7-12; semantics restated in SURVEY.md Appendix C).  Unlike the reference there is
// no `columns` buffer and no per-im2col_step chunking: a CTA samples a strip of output pixels once into shared
// memory and contracts it against the filter bank in registers.  The NLSPN-shaped calls (Cin = Cout = 1) never come
// here from the generator -- they run in nlspn.cu -- but the Function / Module API does.
#include <cuda_fp16.h>

#include "common.cuh"
#include "fixed_point.cuh"

namespace rdfc {
int conv_umma_forward(const rdfc_conv_desc *d, cudaStream_t st, const rdfc_heads_desc *heads, const rdfc_stem_desc *stem,
                      const rdfc_wadain_conv_desc *wad, int split_c);
long long wgrad_umma_workspace_floats(const rdfc_wgrad_desc *d);
int wgrad_umma_partials(const rdfc_wgrad_desc *d, float *workspace, int fp16, cudaStream_t st, int *nchunk);
namespace {

constexpr int TP = 32;        // output pixels per CTA strip (one warp lane per pixel in the contraction)
constexpr int NT = 256;       // threads per CTA
constexpr int CHUNK = 64;     // (ci,k) rows sampled per pass
constexpr int RMAX = 16;      // output channels per thread per pass (8 warps x 16 = 128 per pass)

struct Geo {
    int B, Cin, H, W, Cout, kh, kw, sh, sw, ph, pw, dh, dw, group, dg, Ho, Wo;
};

template <typename T>
__device__ __forceinline__ T ld(const T *p) { return __ldg(p); }

// value at (y,x) with the reference's validity rule and per-corner zeroing
// (modulated_deform_im2col_cuda.cuh:25-54,180)
template <typename T>
__device__ __forceinline__ T sample(const T *im, int H, int W, T y, T x) {
    if (!(y > (T)-1 && x > (T)-1 && y < (T)H && x < (T)W)) return (T)0;
    const int yl = (int)floor(y), xl = (int)floor(x);
    const int yh = yl + 1, xh = xl + 1;
    const T ly = y - yl, lx = x - xl, hy = (T)1 - ly, hx = (T)1 - lx;
    const T v1 = (yl >= 0 && xl >= 0) ? ld(im + (size_t)yl * W + xl) : (T)0;
    const T v2 = (yl >= 0 && xh <= W - 1) ? ld(im + (size_t)yl * W + xh) : (T)0;
    const T v3 = (yh <= H - 1 && xl >= 0) ? ld(im + (size_t)yh * W + xl) : (T)0;
    const T v4 = (yh <= H - 1 && xh <= W - 1) ? ld(im + (size_t)yh * W + xh) : (T)0;
    return hy * hx * v1 + hy * lx * v2 + ly * hx * v3 + ly * lx * v4;
}

// d val / d y and d val / d x (modulated_deform_im2col_cuda.cuh:84-125)
template <typename T>
__device__ __forceinline__ void sample_grad(const T *im, int H, int W, T y, T x, T &val, T &gy, T &gx) {
    val = gy = gx = (T)0;
    if (y <= (T)-1 || y >= (T)H || x <= (T)-1 || x >= (T)W) return;
    const int yl = (int)floor(y), xl = (int)floor(x);
    const int yh = yl + 1, xh = xl + 1;
    const T ly = y - yl, lx = x - xl, hy = (T)1 - ly, hx = (T)1 - lx;
    const T v1 = (yl >= 0 && xl >= 0) ? ld(im + (size_t)yl * W + xl) : (T)0;
    const T v2 = (yl >= 0 && xh <= W - 1) ? ld(im + (size_t)yl * W + xh) : (T)0;
    const T v3 = (yh <= H - 1 && xl >= 0) ? ld(im + (size_t)yh * W + xl) : (T)0;
    const T v4 = (yh <= H - 1 && xh <= W - 1) ? ld(im + (size_t)yh * W + xh) : (T)0;
    val = hy * hx * v1 + hy * lx * v2 + ly * hx * v3 + ly * lx * v4;
    gy = hx * (v3 - v1) + lx * (v4 - v2);
    gx = hy * (v2 - v1) + ly * (v4 - v3);
}

// ---------------------------------------------------------------- forward -------------------------------------
// grid: (ceil(Ho*Wo / TP), B, group).  Each CTA: TP pixels of image b, all Cout/group outputs of group g.
template <typename T, bool kMask>
__global__ void __launch_bounds__(NT) dcn_fwd_kernel(const T *__restrict__ input, const T *__restrict__ weight,
                                                      const T *__restrict__ bias, const T *__restrict__ offset,
                                                      const T *__restrict__ mask, T *__restrict__ output, Geo g) {
    __shared__ T col[CHUNK][TP + 1];
    const int K = g.kh * g.kw, P = g.Ho * g.Wo;
    const int cpg = g.Cin / g.group, opg = g.Cout / g.group, cpdg = g.Cin / g.dg;
    const int pix0 = blockIdx.x * TP, b = blockIdx.y, grp = blockIdx.z;
    const int lane = threadIdx.x % TP, wrp = threadIdx.x / TP;  // wrp in [0,8)
    const int rows = cpg * K;                                    // contraction length of this group

    for (int co0 = 0; co0 < opg; co0 += (NT / TP) * RMAX) {
        T acc[RMAX];
#pragma unroll
        for (int r = 0; r < RMAX; ++r) acc[r] = (T)0;
        for (int q0 = 0; q0 < rows; q0 += CHUNK) {
            __syncthreads();
            // phase 1: sample CHUNK x TP values
            for (int e = threadIdx.x; e < CHUNK * TP; e += NT) {
                const int qq = e / TP, pl = e % TP, q = q0 + qq, pix = pix0 + pl;
                T v = (T)0;
                if (q < rows && pix < P) {
                    const int ci = grp * cpg + q / K, k = q % K, i = k / g.kw, j = k % g.kw;
                    const int ho = pix / g.Wo, wo = pix % g.Wo, gd = ci / cpdg;
                    const T *off = offset + ((size_t)(b * g.dg + gd) * 2 * K) * P;
                    const T y = (T)(ho * g.sh - g.ph + i * g.dh) + ld(off + (size_t)(2 * k) * P + pix);
                    const T x = (T)(wo * g.sw - g.pw + j * g.dw) + ld(off + (size_t)(2 * k + 1) * P + pix);
                    v = sample(input + ((size_t)b * g.Cin + ci) * g.H * g.W, g.H, g.W, y, x);
                    if (kMask) v *= ld(mask + ((size_t)(b * g.dg + gd) * K + k) * P + pix);
                }
                col[qq][pl] = v;
            }
            __syncthreads();
            // phase 2: contract against the filters; weight address is warp-uniform (broadcast load)
            const int qn = min(CHUNK, rows - q0);
#pragma unroll
            for (int r = 0; r < RMAX; ++r) {
                const int col_o = co0 + wrp + r * (NT / TP);
                if (col_o < opg) {
                    const T *wrow = weight + (size_t)(grp * opg + col_o) * rows + q0;
                    T a = acc[r];
                    for (int qq = 0; qq < qn; ++qq) a += ld(wrow + qq) * col[qq][lane];
                    acc[r] = a;
                }
            }
        }
        const int pix = pix0 + lane;
        if (pix < P) {
#pragma unroll
            for (int r = 0; r < RMAX; ++r) {
                const int col_o = co0 + wrp + r * (NT / TP);
                if (col_o < opg) {
                    const int co = grp * opg + col_o;
                    output[((size_t)b * g.Cout + co) * P + pix] = acc[r] + (bias ? ld(bias + co) : (T)0);
                }
            }
        }
    }
}

// ---------------------------------------------------------------- backward: data ------------------------------
// One thread per (b, gd, k, pixel): loops the channels of the deformable group, forms
// gcol = sum_co W[co,ci,k] * gout[b,co,pix]  (modulated_deform_conv_cuda.cu:217-222), then
// grad_mask / grad_offset (col2im_coord, cuh:257-328) and the grad_input scatter (col2im, cuh:197-254).
// kDet (RDFC_DETERMINISTIC): the scatter goes to gacc in fixed point, bounded per destination by K * P contributions of at most
// am[0] = max |grad_output| x am[1] = max over (ci, tap) of sum_o |W| x am[2] = max |mask|.
template <typename T, bool kMask, bool kDet>
__global__ void __launch_bounds__(NT) dcn_bwd_data_kernel(const T *__restrict__ input, const T *__restrict__ weight,
                                                           const T *__restrict__ offset, const T *__restrict__ mask,
                                                           const T *__restrict__ gout, T *__restrict__ gin,
                                                           T *__restrict__ goff, T *__restrict__ gmask, Geo g,
                                                           long long *__restrict__ gacc, const unsigned long long *__restrict__ am) {
    const int K = g.kh * g.kw, P = g.Ho * g.Wo;
    const Fx<T> fx(kDet ? (double)K * P : 1.0, am, kDet ? (kMask ? 3 : 2) : 0);
    const bool scatter = kDet ? gacc != nullptr : gin != nullptr;
    const int cpg = g.Cin / g.group, opg = g.Cout / g.group, cpdg = g.Cin / g.dg;
    const long long total = (long long)g.B * g.dg * K * P;
    for (long long idx = (long long)blockIdx.x * NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
        const int pix = (int)(idx % P);
        const int k = (int)((idx / P) % K);
        const int gd = (int)((idx / P / K) % g.dg);
        const int b = (int)(idx / P / K / g.dg);
        const int i = k / g.kw, j = k % g.kw, ho = pix / g.Wo, wo = pix % g.Wo;
        const T *off = offset + ((size_t)(b * g.dg + gd) * 2 * K) * P;
        const T y = (T)(ho * g.sh - g.ph + i * g.dh) + ld(off + (size_t)(2 * k) * P + pix);
        const T x = (T)(wo * g.sw - g.pw + j * g.dw) + ld(off + (size_t)(2 * k + 1) * P + pix);
        const T m = kMask ? ld(mask + ((size_t)(b * g.dg + gd) * K + k) * P + pix) : (T)1;
        const bool valid = (y > (T)-1 && x > (T)-1 && y < (T)g.H && x < (T)g.W);
        const int yl = (int)floor(y), xl = (int)floor(x);
        const T ly = y - yl, lx = x - xl;
        T s_mask = (T)0, s_y = (T)0, s_x = (T)0;
        for (int c = 0; c < cpdg; ++c) {
            const int ci = gd * cpdg + c, grp = ci / cpg, cil = ci % cpg;
            T gcol = (T)0;
            for (int o = 0; o < opg; ++o) {
                const int co = grp * opg + o;
                gcol += ld(weight + ((size_t)co * cpg + cil) * K + k) * ld(gout + ((size_t)b * g.Cout + co) * P + pix);
            }
            const T *im = input + ((size_t)b * g.Cin + ci) * g.H * g.W;
            T val, gy, gx;
            sample_grad(im, g.H, g.W, y, x, val, gy, gx);
            s_mask += gcol * val;
            s_y += gcol * m * gy;
            s_x += gcol * m * gx;
            if (scatter && valid) {
                const size_t plane = ((size_t)b * g.Cin + ci) * g.H * g.W;
                const T top = gcol * m;
#pragma unroll
                for (int a = 0; a < 2; ++a)
#pragma unroll
                    for (int c2 = 0; c2 < 2; ++c2) {
                        const int yy = yl + a, xx = xl + c2;
                        if (yy >= 0 && yy <= g.H - 1 && xx >= 0 && xx <= g.W - 1) {
                            const T wgt = (a ? ly : (T)1 - ly) * (c2 ? lx : (T)1 - lx);
                            if (kDet) fx_add(gacc + plane + (size_t)yy * g.W + xx, fx.to_fixed(wgt * top));
                            else atomicAdd(gin + plane + (size_t)yy * g.W + xx, wgt * top);
                        }
                    }
            }
        }
        if (goff) {
            T *go = goff + ((size_t)(b * g.dg + gd) * 2 * K) * P;
            go[(size_t)(2 * k) * P + pix] = s_y;
            go[(size_t)(2 * k + 1) * P + pix] = s_x;
        }
        if (kMask && gmask) gmask[((size_t)(b * g.dg + gd) * K + k) * P + pix] = s_mask;
    }
}

// am[0] = max over (ci, tap) of sum_o |W[o, ci, tap]| (the bound of one column gradient per unit grad_output)
template <typename T>
__global__ void __launch_bounds__(NT) dcn_wsum_max_kernel(const T *__restrict__ weight, Geo g, unsigned long long *__restrict__ am) {
    const int K = g.kh * g.kw, cpg = g.Cin / g.group, opg = g.Cout / g.group;
    unsigned long long m = 0;
    for (int e = blockIdx.x * NT + threadIdx.x; e < g.Cin * K; e += gridDim.x * NT) {
        const int ci = e / K, k = e % K, grp = ci / cpg, cil = ci % cpg;
        T s = (T)0;
        for (int o = 0; o < opg; ++o) s += fabs(ld(weight + ((size_t)(grp * opg + o) * cpg + cil) * K + k));
        const unsigned long long bits = fx_bits((double)s);
        m = bits > m ? bits : m;
    }
    fx_warp_max(m, am);
}

// ---------------------------------------------------------------- backward: filters ---------------------------
// grid: (Cin * K).  grad_weight[co, cil, k] = sum_{b,pix} gout[b,co,pix] * col(ci,k,b,pix)   (cu:248-272).
// Deterministic: fixed tile order, warp-shuffle reduction, one owner per output element.
template <typename T, bool kMask>
__global__ void __launch_bounds__(NT) dcn_bwd_weight_kernel(const T *__restrict__ input,
                                                             const T *__restrict__ offset,
                                                             const T *__restrict__ mask, const T *__restrict__ gout,
                                                             T *__restrict__ gweight, Geo g) {
    extern __shared__ unsigned char smem_raw[];
    T *colv = reinterpret_cast<T *>(smem_raw);          // NT
    T *acc_s = colv + NT;                               // opg
    const int K = g.kh * g.kw, P = g.Ho * g.Wo;
    const int cpg = g.Cin / g.group, opg = g.Cout / g.group, cpdg = g.Cin / g.dg;
    const int ci = blockIdx.x / K, k = blockIdx.x % K;
    const int grp = ci / cpg, cil = ci % cpg, gd = ci / cpdg, i = k / g.kw, j = k % g.kw;
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    for (int o = threadIdx.x; o < opg; o += NT) acc_s[o] = (T)0;
    const long long total = (long long)g.B * P;
    for (long long t0 = 0; t0 < total; t0 += NT) {
        __syncthreads();
        const long long p = t0 + threadIdx.x;
        T v = (T)0;
        if (p < total) {
            const int b = (int)(p / P), pix = (int)(p % P), ho = pix / g.Wo, wo = pix % g.Wo;
            const T *off = offset + ((size_t)(b * g.dg + gd) * 2 * K) * P;
            const T y = (T)(ho * g.sh - g.ph + i * g.dh) + ld(off + (size_t)(2 * k) * P + pix);
            const T x = (T)(wo * g.sw - g.pw + j * g.dw) + ld(off + (size_t)(2 * k + 1) * P + pix);
            v = sample(input + ((size_t)b * g.Cin + ci) * g.H * g.W, g.H, g.W, y, x);
            if (kMask) v *= ld(mask + ((size_t)(b * g.dg + gd) * K + k) * P + pix);
        }
        colv[threadIdx.x] = v;
        __syncthreads();
        for (int o = wrp; o < opg; o += NT / 32) {
            const int co = grp * opg + o;
            T part = (T)0;
#pragma unroll
            for (int jj = 0; jj < NT / 32; ++jj) {
                const long long pp = t0 + lane + 32 * jj;
                if (pp < total) {
                    const int b = (int)(pp / P), pix = (int)(pp % P);
                    part += ld(gout + ((size_t)b * g.Cout + co) * P + pix) * colv[lane + 32 * jj];
                }
            }
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) part += __shfl_xor_sync(0xffffffffu, part, s);
            if (lane == 0) acc_s[o] += part;
        }
    }
    __syncthreads();
    for (int o = threadIdx.x; o < opg; o += NT)
        gweight[((size_t)(grp * opg + o) * cpg + cil) * K + k] = acc_s[o];
}

// grid: (Cout).  grad_bias[co] = sum gout[:,co,:]  (cu:271-273)
template <typename T>
__global__ void __launch_bounds__(NT) dcn_bwd_bias_kernel(const T *__restrict__ gout, T *__restrict__ gbias, int B,
                                                           int Cout, int P) {
    __shared__ T red[NT / 32];
    const int co = blockIdx.x;
    T s = (T)0;
    for (long long p = threadIdx.x; p < (long long)B * P; p += NT)
        s += ld(gout + ((size_t)(p / P) * Cout + co) * P + (p % P));
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) s += __shfl_xor_sync(0xffffffffu, s, sft);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        T t = (T)0;
        for (int w = 0; w < NT / 32; ++w) t += red[w];
        gbias[co] = t;
    }
}

int check_shape(const rdfc_dcn_shape *s, Geo &g) {
    RDFC_REQUIRE(s != nullptr, "shape is NULL");
    RDFC_REQUIRE(s->B > 0 && s->Cin > 0 && s->Cout > 0 && s->H > 0 && s->W > 0, "empty tensor dimension");
    RDFC_REQUIRE(s->kh > 0 && s->kw > 0 && s->sh > 0 && s->sw > 0 && s->dh > 0 && s->dw > 0 && s->ph >= 0 &&
                     s->pw >= 0,
                 "bad kernel/stride/dilation/padding");
    RDFC_REQUIRE(s->group > 0 && s->deformable_group > 0, "group and deformable_group must be positive");
    // modulated_deform_conv_cuda.cu:56-63
    const int step = s->im2col_step < s->B ? s->im2col_step : s->B;
    RDFC_REQUIRE(step > 0 && s->B % step == 0, "batch(%d) must divide im2col_step(%d)", s->B, step);
    RDFC_REQUIRE(s->Cin % s->group == 0 && s->Cout % s->group == 0,
                 "channels(%d) and channels_out(%d) must divide group(%d)", s->Cin, s->Cout, s->group);
    RDFC_REQUIRE(s->Cin % s->deformable_group == 0, "channels(%d) must divide deformable_group(%d)", s->Cin,
                 s->deformable_group);
    g = Geo{s->B, s->Cin, s->H, s->W, s->Cout, s->kh, s->kw, s->sh, s->sw, s->ph, s->pw, s->dh, s->dw,
            s->group, s->deformable_group, 0, 0};
    g.Ho = (s->H + 2 * s->ph - (s->dh * (s->kh - 1) + 1)) / s->sh + 1;
    g.Wo = (s->W + 2 * s->pw - (s->dw * (s->kw - 1) + 1)) / s->sw + 1;
    RDFC_REQUIRE(g.Ho > 0 && g.Wo > 0, "empty output (%d x %d)", g.Ho, g.Wo);
    RDFC_REQUIRE(s->B <= 65535 && s->group <= 65535, "batch / group exceed grid limits");
    return 0;
}

template <typename T>
int fwd(const void *input, const void *weight, const void *bias, const void *offset, const void *mask, void *output,
        const Geo &g, cudaStream_t st) {
    dim3 grid(cdiv(g.Ho * g.Wo, TP), g.B, g.group);
    if (mask)
        dcn_fwd_kernel<T, true><<<grid, NT, 0, st>>>((const T *)input, (const T *)weight, (const T *)bias,
                                                     (const T *)offset, (const T *)mask, (T *)output, g);
    else
        dcn_fwd_kernel<T, false><<<grid, NT, 0, st>>>((const T *)input, (const T *)weight, (const T *)bias,
                                                      (const T *)offset, nullptr, (T *)output, g);
    RDFC_CHECK_LAUNCH("dcn_fwd_kernel");
    return 0;
}

// ---------------------------------------------------------------- forward on the tensor cores ------------------
// out = W . (mask * deform_im2col(x, offset)) + b as the reference factors it (modulated_deform_conv_cuda.cu:78-118): the sampled
// columns are materialised -- here as fp16 halves [hi | lo] per (pixel, group), so that the contraction can run on tcgen05 with
// split operands at fp32 fidelity (conv_umma.cu, Params::split_c) -- then ONE 1x1 implicit GEMM per group contracts them with
// the filter bank packed [W_hi ; W_lo ; W_hi], and a transposition returns the NCHW layout of the DCN boundary.
// cols[pixel][group][2 * Kg] with Kg = (Cin / group) * kh * kw, TAP-MAJOR: k = tap * (Cin / group) + ci_local (the filter pack below
// follows), so that a chunk of 64 rows is one tap over 64 channels and the sampling position, the four bilinear weights (corner
// zeroing folded in, modulated_deform_im2col_cuda.cuh:25-54) and the mask are computed once per (pixel, tap, deformable group)
// instead of once per sample.  grid (ceil(P / 32), B), 8 warps.  Sampling runs with one lane per PIXEL (offset / mask planes and
// the image rows are read coalesced, as in the reference's im2col), the values go through a shared-memory tile, and the write-out
// runs with one warp per pixel and the lanes along the channels, so that every pixel's column block leaves as 128-byte rows.
// Split-precision operands are fp16 halves, and fp16 has a narrow exponent range: every tensor that gets split is first scaled by a
// power of two chosen from its largest magnitude (hi < 2048, so lo = x - hi keeps 11 significant bits down to ~3e-5 of the largest
// element), and the GEMM epilogue multiplies the exact inverse back.  The maxima live on the device (no host synchronisation):
// am[0] = max |input|, am[1] = max |mask| (1 when there is none), am[2] = max |weight|, am[3] = max |grad_output|, as the bit
// patterns of non-negative floats (which order like unsigned integers).
struct AmaxArgs { const float *p[4]; long long n[4]; };
__global__ void __launch_bounds__(NT) dcn_amax_kernel(AmaxArgs a, unsigned *am) {
    const int seg = blockIdx.y;
    const float *x = a.p[seg];
    if (!x) return;
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < a.n[seg]; i += (long long)gridDim.x * NT) m = fmaxf(m, fabsf(__ldg(x + i)));
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, sft));
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(am + seg, __float_as_uint(m));
}
__device__ __forceinline__ float scale_cols(const unsigned *am) { return pow2_scale(__uint_as_float(am[0]) * (am[1] ? __uint_as_float(am[1]) : 1.f)); }
__device__ __forceinline__ float scale_w(const unsigned *am) { return pow2_scale(__uint_as_float(am[2])); }
__device__ __forceinline__ float scale_g(const unsigned *am) { return pow2_scale(__uint_as_float(am[3])); }

template <bool kMask>
__global__ void __launch_bounds__(NT) dcn_im2col_split_kernel(const float *__restrict__ input, const float *__restrict__ offset,
                                                              const float *__restrict__ mask, __half *__restrict__ cols, Geo g,
                                                              const unsigned *__restrict__ am) {
    __shared__ float tile[64][33];
    const float sx = scale_cols(am);
    const int K = g.kh * g.kw, P = g.Ho * g.Wo, Cg = g.Cin / g.group, Kg = Cg * K, cpd = g.Cin / g.dg;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, b = blockIdx.y, p0 = blockIdx.x * 32;
    const int p = p0 + lane, ho = p / g.Wo, wo = p - ho * g.Wo;
    const long long HW = (long long)g.H * g.W;
    const float *img = input + (long long)b * g.Cin * HW;
    for (int grp = 0; grp < g.group; ++grp)
        for (int tap = 0; tap < K; ++tap) {
            const int ky = tap / g.kw, kx = tap - ky * g.kw;
            for (int c0 = 0; c0 < Cg; c0 += 64) {
                int cur_dg = -1, i1 = 0, i2 = 0, i3 = 0, i4 = 0;
                float w1 = 0.f, w2 = 0.f, w3 = 0.f, w4 = 0.f, mk = 1.f;
#pragma unroll 1
                for (int r = warp * 8; r < warp * 8 + 8; ++r) {
                    const int cl = c0 + r;
                    float v = 0.f;
                    if (cl < Cg && p < P) {
                        const int ci = grp * Cg + cl, dgi = ci / cpd;
                        if (dgi != cur_dg) {
                            cur_dg = dgi;
                            const float *offp = offset + ((long long)b * g.dg * 2 * K + (long long)dgi * 2 * K + 2 * tap) * P + p;
                            const float y = (float)(ho * g.sh - g.ph + ky * g.dh) + __ldg(offp), x = (float)(wo * g.sw - g.pw + kx * g.dw) + __ldg(offp + P);
                            if (kMask) mk = __ldg(mask + ((long long)b * g.dg * K + (long long)dgi * K + tap) * P + p);
                            w1 = w2 = w3 = w4 = 0.f; i1 = i2 = i3 = i4 = 0;
                            if (y > -1.f && x > -1.f && y < (float)g.H && x < (float)g.W) {
                                const int yl = (int)floorf(y), xl = (int)floorf(x), yh = yl + 1, xh = xl + 1;
                                const float ly = y - yl, lx = x - xl, hy = 1.f - ly, hx = 1.f - lx;
                                if (yl >= 0 && xl >= 0) { w1 = hy * hx; i1 = yl * g.W + xl; }
                                if (yl >= 0 && xh <= g.W - 1) { w2 = hy * lx; i2 = yl * g.W + xh; }
                                if (yh <= g.H - 1 && xl >= 0) { w3 = ly * hx; i3 = yh * g.W + xl; }
                                if (yh <= g.H - 1 && xh <= g.W - 1) { w4 = ly * lx; i4 = yh * g.W + xh; }
                            }
                        }
                        const float *im = img + (long long)ci * HW;
                        v = w1 * __ldg(im + i1) + w2 * __ldg(im + i2) + w3 * __ldg(im + i3) + w4 * __ldg(im + i4);
                        if (kMask) v *= mk;
                    }
                    tile[r][lane] = v;
                }
                __syncthreads();
                for (int px = warp; px < 32; px += NT / 32) {
                    const int pp = p0 + px, cl = c0 + 2 * lane;              // two consecutive channels per lane (Cg even)
                    if (pp < P && cl < Cg) {
                        const float v0 = tile[2 * lane][px] * sx, v1 = tile[2 * lane + 1][px] * sx;
                        __half *row = cols + (((long long)b * P + pp) * g.group + grp) * (2 * Kg) + tap * Cg + cl;
                        const __half2 hi = __floats2half2_rn(v0, v1);
                        const float2 hf = __half22float2(hi);
                        *reinterpret_cast<__half2 *>(row) = hi;
                        *reinterpret_cast<__half2 *>(row + Kg) = __floats2half2_rn(v0 - hf.x, v1 - hf.y);
                    }
                }
                __syncthreads();
            }
        }
}

// filter bank of one group -> UMMA packing [1 tap][3 Kg / 8][CoutP][8] of [W_hi ; W_lo ; W_hi] (fp16), rows tap-major as the columns
// vec[co] = 1 / (scale of the columns * scale of the filters): the GEMM epilogue's per-channel factor
__global__ void __launch_bounds__(NT) dcn_pack_x3_kernel(const float *__restrict__ w, __half *__restrict__ packed, int Cog, int CoutP, int Cg, int K,
                                                         const unsigned *__restrict__ am, float *__restrict__ vec) {
    const int Kg = Cg * K, total = 3 * Kg * CoutP;
    const float sw = scale_w(am);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < CoutP; i += gridDim.x * blockDim.x) vec[i] = 1.f / (sw * scale_cols(am));
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7, co = (i >> 3) % CoutP, ch = i / (8 * CoutP);
        const int kk = ch * 8 + e, k = kk % Kg, part = kk / Kg, tap = k / Cg, cl = k - tap * Cg;
        float v = 0.f;
        if (co < Cog) {
            const float x = __ldg(w + (long long)co * Kg + cl * K + tap) * sw;
            const float hi = __half2float(__float2half_rn(x));
            v = part == 1 ? x - hi : hi;
        }
        packed[i] = __float2half_rn(v);
    }
}

__global__ void __launch_bounds__(NT) nhwc_to_nchw_kernel(const float *__restrict__ x, float *__restrict__ out, int B, int C, int P) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += NT / 32)
        if (p0 + r < P && c0 + tx < C) tile[r][tx] = x[((long long)b * P + p0 + r) * C + c0 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += NT / 32)
        if (c0 + r < C && p0 + tx < P) out[((long long)b * C + c0 + r) * P + p0 + tx] = tile[tx][r];
}

bool fwd_tc_ok(const Geo &g) {
    const int Kg = (g.Cin / g.group) * g.kh * g.kw, Cog = g.Cout / g.group;
    return Kg % 32 == 0 && (g.Cin / g.group) % 2 == 0 && Cog >= 16 && Cog % 8 == 0 && knob("RDFC_DCN_TC", 1) != 0;
}

// device scratch of one call: am[4] (maxima), then the epilogue vector
struct Aux { unsigned *am; float *vec; };
int aux_alloc(Aux *a, int nvec, cudaStream_t st) {
    void *p = nullptr;
    RDFC_CUDA(cudaMallocAsync(&p, 16 + sizeof(float) * (size_t)nvec, st));
    RDFC_CUDA(cudaMemsetAsync(p, 0, 16, st));
    a->am = (unsigned *)p; a->vec = (float *)((char *)p + 16);
    return 0;
}
int amax_launch(const Aux &a, const float *x, long long nx, const float *mask, long long nm, const float *w, long long nw, const float *go, long long ng,
                cudaStream_t st) {
    AmaxArgs args{{x, mask, w, go}, {nx, nm, nw, ng}};
    long long nmax = nx > ng ? nx : ng;
    const int blocks = (int)min((long long)cdiv(nmax, NT * 8), (long long)sm_count() * 4);
    dcn_amax_kernel<<<dim3(blocks, 4), NT, 0, st>>>(args, a.am);
    RDFC_CHECK_LAUNCH("dcn_amax_kernel");
    return 0;
}

int fwd_tc(const float *input, const float *weight, const float *bias, const float *offset, const float *mask, float *output,
           const Geo &g, cudaStream_t st) {
    const int K = g.kh * g.kw, P = g.Ho * g.Wo, Kg = (g.Cin / g.group) * K, Cog = g.Cout / g.group, CoutP = (Cog + 15) / 16 * 16;
    const long long npix = (long long)g.B * P;
    __half *cols = nullptr, *packed = nullptr;
    float *tmp = nullptr;
    Aux aux{};
    const size_t cols_bytes = (size_t)npix * g.group * 2 * Kg * sizeof(__half), pk_bytes = (size_t)3 * Kg * CoutP * sizeof(__half);
    RDFC_CUDA(cudaMallocAsync((void **)&cols, cols_bytes, st));
    RDFC_CUDA(cudaMallocAsync((void **)&packed, pk_bytes * g.group, st));
    RDFC_CUDA(cudaMallocAsync((void **)&tmp, (size_t)npix * g.Cout * sizeof(float), st));
    int rc = aux_alloc(&aux, CoutP, st);
    if (rc == 0)
        rc = amax_launch(aux, input, (long long)g.B * g.Cin * g.H * g.W, mask, mask ? (long long)g.B * g.dg * K * P : 0, weight,
                         (long long)g.Cout * Kg, nullptr, 0, st);
    if (rc == 0) {
        const dim3 grid(cdiv(P, 32), g.B);
        if (mask) dcn_im2col_split_kernel<true><<<grid, NT, 0, st>>>(input, offset, mask, cols, g, aux.am);
        else dcn_im2col_split_kernel<false><<<grid, NT, 0, st>>>(input, offset, nullptr, cols, g, aux.am);
        count_launch();
    }
    for (int grp = 0; grp < g.group && rc == 0; ++grp) {
        __half *pk = packed + (size_t)grp * 3 * Kg * CoutP;
        dcn_pack_x3_kernel<<<cdiv(3 * Kg * CoutP, NT), NT, 0, st>>>(weight + (long long)grp * Cog * Kg, pk, Cog, CoutP, g.Cin / g.group, K, aux.am, aux.vec);
        count_launch();
        rdfc_conv_desc d{};
        d.B = g.B; d.Hi = d.Ho = g.Ho; d.Wi = d.Wo = g.Wo;
        d.kh = d.kw = 1; d.stride = 1; d.pad = 0; d.act = RDFC_ACT_NONE; d.path = RDFC_PATH_UMMA_BF16;
        d.in.ptr = cols + (size_t)grp * 2 * Kg; d.in.dtype = RDFC_BF16; d.in.C = 2 * Kg; d.in.pix_stride = g.group * 2 * Kg;
        d.out.ptr = tmp + (size_t)grp * Cog; d.out.dtype = RDFC_F32; d.out.C = Cog; d.out.pix_stride = g.Cout;
        d.weight = pk; d.scale = aux.vec; d.shift = bias ? bias + (size_t)grp * Cog : nullptr;
        rc = conv_umma_forward(&d, st, nullptr, nullptr, nullptr, Kg);
    }
    if (rc == 0) {
        nhwc_to_nchw_kernel<<<dim3(cdiv(P, 32), cdiv(g.Cout, 32), g.B), NT, 0, st>>>(tmp, output, g.B, g.Cout, P);
        count_launch();
        if (cudaGetLastError() != cudaSuccess) rc = fail(RDFC_ERR_CUDA, "dcn forward (tensor cores): kernel launch failed");
    }
    cudaFreeAsync(cols, st); cudaFreeAsync(packed, st); cudaFreeAsync(tmp, st);
    if (aux.am) cudaFreeAsync(aux.am, st);
    return rc;
}

// ---------------------------------------------------------------- backward on the tensor cores -----------------
// The reference's backward (modulated_deform_conv_cuda.cu:124-280) is: columns' gradient = W^T . grad_output (GEMM), col2im_coord /
// col2im over it, and grad_weight = grad_output . columns^T (GEMM with K = pixels).  Here both GEMMs run on tcgen05 at fp32 fidelity:
//   gsplit  = grad_output as fp16 halves [hi | lo] per (pixel, group)                              (dcn_gout_split_kernel)
//   gcols   = 1x1 implicit GEMM of gsplit with the filter bank transposed, fp32 [pixel][group][tap-major k]   (conv_umma, split operands)
//   grad_input / grad_offset / grad_mask from gcols in one pass                                    (dcn_col2im_coord_kernel)
//   grad_weight = sum over pixels gsplit^T . cols: the filter-gradient kernel of wgrad_umma.cu (K = pixels, MN-major operands) run for
//   the three split products hi.hi + hi.lo + lo.hi into consecutive chunk ranges of one workspace    (dcn_wgrad_reduce_kernel)

// grad_output NCHW fp32 -> [pixel][group][hi (Cog) | lo (Cog)] fp16, scaled
__global__ void __launch_bounds__(NT) dcn_gout_split_kernel(const float *__restrict__ gout, __half *__restrict__ gs, int Cout, int Cog, int P,
                                                            const unsigned *__restrict__ am) {
    __shared__ float tile[32][33];
    const float sg = scale_g(am);
    const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += NT / 32)
        if (c0 + r < Cout && p0 + tx < P) tile[r][tx] = __ldg(gout + ((long long)b * Cout + c0 + r) * P + p0 + tx) * sg;
    __syncthreads();
    for (int r = ty; r < 32; r += NT / 32) {
        const int c = c0 + tx, pp = p0 + r;
        if (c < Cout && pp < P) {
            const int grp = c / Cog, cl = c - grp * Cog;
            const float v = tile[tx][r];
            const __half hi = __float2half_rn(v);
            __half *row = gs + (((long long)b * P + pp) * (Cout / Cog) + grp) * (2 * Cog);
            row[cl] = hi;
            row[Cog + cl] = __float2half_rn(v - __half2float(hi));
        }
    }
}

// filter bank of one group, transposed -> UMMA packing [3 Cog / 8][KgP][8] of [W_hi ; W_lo ; W_hi] along the OUTPUT channels of the layer
// (the GEMM's input channels); GEMM column k = tap * Cg + ci_local.  vec[k] = 1 / (scale of grad_output * scale of the filters).
__global__ void __launch_bounds__(NT) dcn_pack_t_x3_kernel(const float *__restrict__ w, __half *__restrict__ packed, int Cog, int KgP, int Cg, int K,
                                                           const unsigned *__restrict__ am, float *__restrict__ vec) {
    const int Kg = Cg * K, total = 3 * Cog * KgP;
    const float sw = scale_w(am);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < KgP; i += gridDim.x * blockDim.x) vec[i] = 1.f / (sw * scale_g(am));
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7, k = (i >> 3) % KgP, ch = i / (8 * KgP);
        const int kk = ch * 8 + e, c = kk % Cog, part = kk / Cog, tap = k / Cg, cl = k - tap * Cg;
        float v = 0.f;
        if (k < Kg) {
            const float x = __ldg(w + (long long)c * Kg + cl * K + tap) * sw;
            const float hi = __half2float(__float2half_rn(x));
            v = part == 1 ? x - hi : hi;
        }
        packed[i] = __float2half_rn(v);
    }
}

// grad_input (col2im, modulated_deform_im2col_cuda.cuh:197-254), grad_offset / grad_mask (col2im_coord, cuh:257-328) from the columns'
// gradient gcols[pixel][group][tap * Cg + ci_local] (fp32).  grid (ceil(P / 32), B), 8 warps; the mirror image of the im2col kernel: a chunk
// of 64 channels of one tap is read with the lanes along the channels, goes through a shared-memory tile, and is consumed with one lane per
// PIXEL (coalesced image reads and atomics), the position / bilinear weights computed once per (pixel, tap, deformable group); the per-pixel
// sums over the channels of a deformable group are combined through shared memory in a fixed order.
// kDet (RDFC_DETERMINISTIC): grad_input goes to gacc in fixed point, bounded per destination by K * P contributions of at most
// am[0] = max |gcols| x am[1] = max |mask|.
constexpr int MAXDG = 16;
template <bool kMask, bool kDet>
__global__ void __launch_bounds__(NT) dcn_col2im_coord_kernel(const float *__restrict__ input, const float *__restrict__ offset, const float *__restrict__ mask,
                                                              const float *__restrict__ gcols, float *__restrict__ gin, float *__restrict__ goff,
                                                              float *__restrict__ gmask, Geo g, long long *__restrict__ gacc,
                                                              const unsigned long long *__restrict__ am) {
    __shared__ float tile[64][33];
    __shared__ float part[NT / 32][3][32];
    __shared__ float acc[MAXDG][3][32];
    __shared__ int part_dg[NT / 32];
    const int K = g.kh * g.kw, P = g.Ho * g.Wo, Cg = g.Cin / g.group, Kg = Cg * K, cpd = g.Cin / g.dg;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, b = blockIdx.y, p0 = blockIdx.x * 32;
    const int p = p0 + lane, ho = p / g.Wo, wo = p - ho * g.Wo;
    const long long HW = (long long)g.H * g.W;
    const float *img = input + (long long)b * g.Cin * HW;
    float *gimg = gin ? gin + (long long)b * g.Cin * HW : nullptr;
    long long *gacc_img = kDet && gacc ? gacc + (long long)b * g.Cin * HW : nullptr;
    const Fx<float> fx(kDet ? (double)K * P : 1.0, am, kDet ? (kMask ? 2 : 1) : 0);
    for (int tap = 0; tap < K; ++tap) {
        const int ky = tap / g.kw, kx = tap - ky * g.kw;
        for (int i = threadIdx.x; i < g.dg * 96; i += NT) (&acc[0][0][0])[i] = 0.f;
        for (int grp = 0; grp < g.group; ++grp)
            for (int c0 = 0; c0 < Cg; c0 += 64) {
                __syncthreads();                                           // previous chunk's tile / part consumed, acc zeroed
                for (int px = warp; px < 32; px += NT / 32) {
                    const int pp = p0 + px, cl = c0 + 2 * lane;
                    float2 v = make_float2(0.f, 0.f);
                    if (pp < P && cl < Cg) v = __ldg(reinterpret_cast<const float2 *>(gcols + ((long long)b * P + pp) * ((long long)g.group * Kg) + (long long)grp * Kg + tap * Cg + cl));
                    tile[2 * lane][px] = v.x;
                    tile[2 * lane + 1][px] = v.y;
                }
                __syncthreads();
                float sm = 0.f, sy = 0.f, sx = 0.f;
                const int cfirst = c0 + warp * 8;
                const int dgi = (grp * Cg + (cfirst < Cg ? cfirst : 0)) / cpd;
                if (cfirst < Cg && p < P) {
                    const float *offp = offset + ((long long)b * g.dg * 2 * K + (long long)dgi * 2 * K + 2 * tap) * P + p;
                    const float y = (float)(ho * g.sh - g.ph + ky * g.dh) + __ldg(offp), x = (float)(wo * g.sw - g.pw + kx * g.dw) + __ldg(offp + P);
                    const float mk = kMask ? __ldg(mask + ((long long)b * g.dg * K + (long long)dgi * K + tap) * P + p) : 1.f;
                    if (y > -1.f && x > -1.f && y < (float)g.H && x < (float)g.W) {
                        const int yl = (int)floorf(y), xl = (int)floorf(x), yh = yl + 1, xh = xl + 1;
                        const float ly = y - yl, lx = x - xl, hy = 1.f - ly, hx = 1.f - lx;
                        const bool f1 = yl >= 0 && xl >= 0, f2 = yl >= 0 && xh <= g.W - 1, f3 = yh <= g.H - 1 && xl >= 0, f4 = yh <= g.H - 1 && xh <= g.W - 1;
                        const int i1 = f1 ? yl * g.W + xl : 0, i2 = f2 ? yl * g.W + xh : 0, i3 = f3 ? yh * g.W + xl : 0, i4 = f4 ? yh * g.W + xh : 0;
#pragma unroll 1
                        for (int r = warp * 8; r < warp * 8 + 8; ++r) {
                            const int cl = c0 + r;
                            if (cl >= Cg) break;
                            const long long pl = (long long)(grp * Cg + cl) * HW;
                            const float *im = img + pl;
                            const float gcol = tile[r][lane];
                            const float v1 = f1 ? __ldg(im + i1) : 0.f, v2 = f2 ? __ldg(im + i2) : 0.f, v3 = f3 ? __ldg(im + i3) : 0.f, v4 = f4 ? __ldg(im + i4) : 0.f;
                            const float val = hy * hx * v1 + hy * lx * v2 + ly * hx * v3 + ly * lx * v4;
                            sm += gcol * val;
                            sy += gcol * mk * (hx * (v3 - v1) + lx * (v4 - v2));
                            sx += gcol * mk * (hy * (v2 - v1) + ly * (v4 - v3));
                            if (kDet && gacc_img) {
                                const float top = gcol * mk;
                                long long *ga = gacc_img + pl;
                                if (f1) fx_add(ga + i1, fx.to_fixed(hy * hx * top));
                                if (f2) fx_add(ga + i2, fx.to_fixed(hy * lx * top));
                                if (f3) fx_add(ga + i3, fx.to_fixed(ly * hx * top));
                                if (f4) fx_add(ga + i4, fx.to_fixed(ly * lx * top));
                            } else if (!kDet && gimg) {
                                const float top = gcol * mk;
                                float *gi = gimg + pl;
                                if (f1) atomicAdd(gi + i1, hy * hx * top);
                                if (f2) atomicAdd(gi + i2, hy * lx * top);
                                if (f3) atomicAdd(gi + i3, ly * hx * top);
                                if (f4) atomicAdd(gi + i4, ly * lx * top);
                            }
                        }
                    }
                }
                part[warp][0][lane] = sm; part[warp][1][lane] = sy; part[warp][2][lane] = sx;
                if (lane == 0) part_dg[warp] = cfirst < Cg ? dgi : -1;
                __syncthreads();
                if (threadIdx.x < 96) {
                    const int comp = threadIdx.x >> 5, ln = threadIdx.x & 31;
                    for (int w = 0; w < NT / 32; ++w)
                        if (part_dg[w] >= 0) acc[part_dg[w]][comp][ln] += part[w][comp][ln];
                }
            }
        __syncthreads();
        for (int i = threadIdx.x; i < g.dg * 96; i += NT) {
            const int dgi = i / 96, comp = (i / 32) % 3, ln = i & 31, pp = p0 + ln;
            if (pp >= P) continue;
            const float v = acc[dgi][comp][ln];
            if (comp == 0) { if (kMask && gmask) gmask[((long long)b * g.dg * K + (long long)dgi * K + tap) * P + pp] = v; }
            else if (goff) goff[((long long)b * g.dg * 2 * K + (long long)dgi * 2 * K + 2 * tap + (comp - 1)) * P + pp] = v;
        }
        __syncthreads();
    }
}

// grad_weight[co][ci_local][tap] = inv * sum over the (3 * nchunk) partial blocks [Cog][Kg] (tap-major k) of one group
__global__ void __launch_bounds__(NT) dcn_wgrad_reduce_kernel(const float *__restrict__ partial, float *__restrict__ gw, int Cog, int Cg, int K, int nblocks,
                                                              const unsigned *__restrict__ am) {
    const int Kg = Cg * K;
    const long long total = (long long)Cog * Kg;
    const float inv = 1.f / (scale_g(am) * scale_cols(am));
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int o = (int)(e / Kg), k = (int)(e - (long long)o * Kg), tap = k / Cg, cl = k - tap * Cg;
        float s = 0.f;
        for (int c = 0; c < nblocks; ++c) s += __ldg(partial + (long long)c * total + e);
        gw[(long long)o * Kg + cl * K + tap] = s * inv;
    }
}

bool bwd_tc_ok(const Geo &g) {
    const int Cg = g.Cin / g.group, Kg = Cg * g.kh * g.kw, Cog = g.Cout / g.group, cpd = g.Cin / g.dg;
    return Kg % 32 == 0 && Cg % 8 == 0 && cpd % 8 == 0 && Cog % 32 == 0 && g.dg <= MAXDG && knob("RDFC_DCN_TC", 1) != 0;
}

// det: grad_input through dcn_col2im_coord_kernel<kMask, true> and a conversion (stream-ordered workspace: the maxima, the int64 image)
int bwd_tc(const float *input, const float *weight, const float *offset, const float *mask, const float *gout, float *gin, float *goff, float *gmask,
           float *gw, float *gb, const Geo &g, cudaStream_t st, bool det) {
    const int K = g.kh * g.kw, P = g.Ho * g.Wo, Cg = g.Cin / g.group, Kg = Cg * K, Cog = g.Cout / g.group, KgP = (Kg + 15) / 16 * 16;
    const long long npix = (long long)g.B * P;
    __half *gs = nullptr, *cols = nullptr, *packed = nullptr;
    float *gcols = nullptr, *ws = nullptr;
    unsigned long long *fx = nullptr;                                   // det: [am: 2][acc: B * Cin * H * W]
    const long long nin = (long long)g.B * g.Cin * g.H * g.W;
    Aux aux{};
    const bool need_data = gin || goff || gmask;
    int rc = aux_alloc(&aux, KgP, st);
    if (rc == 0)
        rc = amax_launch(aux, input, (long long)g.B * g.Cin * g.H * g.W, mask, mask ? (long long)g.B * g.dg * K * P : 0, weight, (long long)g.Cout * Kg, gout,
                         npix * g.Cout, st);
    if (rc) return rc;
    if (gin && det) {
        RDFC_CUDA(cudaMallocAsync((void **)&fx, 8 * (2 + (size_t)nin), st));
        RDFC_CUDA(cudaMemsetAsync(fx, 0, 8 * (2 + (size_t)nin), st));
    } else if (gin) {
        RDFC_CUDA(cudaMemsetAsync(gin, 0, sizeof(float) * (size_t)g.B * g.Cin * g.H * g.W, st));
    }
    RDFC_CUDA(cudaMallocAsync((void **)&gs, (size_t)npix * g.group * 2 * Cog * sizeof(__half), st));
    dcn_gout_split_kernel<<<dim3(cdiv(P, 32), cdiv(g.Cout, 32), g.B), NT, 0, st>>>(gout, gs, g.Cout, Cog, P, aux.am);
    count_launch();
    if (need_data) {
        RDFC_CUDA(cudaMallocAsync((void **)&gcols, (size_t)npix * g.group * Kg * sizeof(float), st));
        RDFC_CUDA(cudaMallocAsync((void **)&packed, (size_t)3 * Cog * KgP * sizeof(__half), st));
        for (int grp = 0; grp < g.group && rc == 0; ++grp) {
            dcn_pack_t_x3_kernel<<<cdiv(3 * Cog * KgP, NT), NT, 0, st>>>(weight + (long long)grp * Cog * Kg, packed, Cog, KgP, Cg, K, aux.am, aux.vec);
            count_launch();
            rdfc_conv_desc d{};
            d.B = g.B; d.Hi = d.Ho = g.Ho; d.Wi = d.Wo = g.Wo;
            d.kh = d.kw = 1; d.stride = 1; d.pad = 0; d.act = RDFC_ACT_NONE; d.path = RDFC_PATH_UMMA_BF16;
            d.in.ptr = gs + (size_t)grp * 2 * Cog; d.in.dtype = RDFC_BF16; d.in.C = 2 * Cog; d.in.pix_stride = g.group * 2 * Cog;
            d.out.ptr = gcols + (size_t)grp * Kg; d.out.dtype = RDFC_F32; d.out.C = Kg; d.out.pix_stride = g.group * Kg;
            d.weight = packed; d.scale = aux.vec; d.shift = nullptr;
            rc = conv_umma_forward(&d, st, nullptr, nullptr, nullptr, Cog);
        }
        if (rc == 0 && fx) {
            rc = fx_amax(gcols, npix * g.group * Kg, fx, st);
            if (rc == 0 && mask) rc = fx_amax(mask, (long long)g.B * g.dg * K * P, fx + 1, st);
            if (rc == 0) {
                const dim3 grid(cdiv(P, 32), g.B);
                if (mask) dcn_col2im_coord_kernel<true, true><<<grid, NT, 0, st>>>(input, offset, mask, gcols, nullptr, goff, gmask, g, (long long *)(fx + 2), fx);
                else dcn_col2im_coord_kernel<false, true><<<grid, NT, 0, st>>>(input, offset, nullptr, gcols, nullptr, goff, nullptr, g, (long long *)(fx + 2), fx);
                count_launch();
                rc = fx_convert((const long long *)(fx + 2), gin, nin, (double)K * P, fx, mask ? 2 : 1, st);
            }
        } else if (rc == 0) {
            const dim3 grid(cdiv(P, 32), g.B);
            if (mask) dcn_col2im_coord_kernel<true, false><<<grid, NT, 0, st>>>(input, offset, mask, gcols, gin, goff, gmask, g, nullptr, nullptr);
            else dcn_col2im_coord_kernel<false, false><<<grid, NT, 0, st>>>(input, offset, nullptr, gcols, gin, goff, nullptr, g, nullptr, nullptr);
            count_launch();
        }
    }
    if (gw && rc == 0) {
        RDFC_CUDA(cudaMallocAsync((void **)&cols, (size_t)npix * g.group * 2 * Kg * sizeof(__half), st));
        const dim3 grid(cdiv(P, 32), g.B);
        if (mask) dcn_im2col_split_kernel<true><<<grid, NT, 0, st>>>(input, offset, mask, cols, g, aux.am);
        else dcn_im2col_split_kernel<false><<<grid, NT, 0, st>>>(input, offset, nullptr, cols, g, aux.am);
        count_launch();
        rdfc_wgrad_desc wd{};
        wd.B = g.B; wd.Hg = wd.Hi = g.Ho; wd.Wg = wd.Wi = g.Wo; wd.k = 1; wd.stride = 1; wd.pad = 0;
        wd.grad_out.dtype = RDFC_BF16; wd.grad_out.C = Cog; wd.grad_out.pix_stride = g.group * 2 * Cog;
        wd.input.dtype = RDFC_BF16; wd.input.C = Kg; wd.input.pix_stride = g.group * 2 * Kg;
        wd.grad_out.ptr = gs; wd.input.ptr = cols;
        const long long per = wgrad_umma_workspace_floats(&wd);
        if (per < 0) rc = RDFC_ERR_INVALID;
        if (rc == 0) RDFC_CUDA(cudaMallocAsync((void **)&ws, (size_t)per * 3 * sizeof(float), st));
        for (int grp = 0; grp < g.group && rc == 0; ++grp) {
            int nchunk = 0, nc = 0;
            const long long blk = (long long)Cog * Kg;
            for (int t = 0; t < 3 && rc == 0; ++t) {                      // hi.hi, hi.lo, lo.hi
                wd.grad_out.ptr = gs + (size_t)grp * 2 * Cog + (t == 2 ? Cog : 0);
                wd.input.ptr = cols + (size_t)grp * 2 * Kg + (t == 1 ? Kg : 0);
                rc = wgrad_umma_partials(&wd, ws + (long long)nchunk * blk, 1, st, &nc);
                nchunk += nc;
            }
            if (rc == 0) {
                dcn_wgrad_reduce_kernel<<<(int)min((long long)cdiv(blk, NT), (long long)sm_count() * 8), NT, 0, st>>>(ws, gw + (long long)grp * blk, Cog, Cg, K, nchunk, aux.am);
                count_launch();
            }
        }
    }
    if (gb && rc == 0) {
        dcn_bwd_bias_kernel<float><<<g.Cout, NT, 0, st>>>(gout, gb, g.B, g.Cout, P);
        count_launch();
    }
    if (rc == 0 && cudaGetLastError() != cudaSuccess) rc = fail(RDFC_ERR_CUDA, "dcn backward (tensor cores): kernel launch failed");
    if (gs) cudaFreeAsync(gs, st);
    if (gcols) cudaFreeAsync(gcols, st);
    if (packed) cudaFreeAsync(packed, st);
    if (cols) cudaFreeAsync(cols, st);
    if (ws) cudaFreeAsync(ws, st);
    if (fx) cudaFreeAsync(fx, st);
    cudaFreeAsync(aux.am, st);
    return rc;
}

// det: grad_input through dcn_bwd_data_kernel<T, kMask, true> and a conversion (stream-ordered workspace: the maxima, the int64 image)
template <typename T>
int bwd_data_det(const T *input, const T *weight, const T *offset, const T *mask, const T *gout, T *gin, T *goff, T *gmask,
                 const Geo &g, cudaStream_t st) {
    const int K = g.kh * g.kw, P = g.Ho * g.Wo;
    const long long nin = (long long)g.B * g.Cin * g.H * g.W, total = (long long)g.B * g.dg * K * P;
    unsigned long long *fx = nullptr;                                   // [am: 3][acc: nin]
    RDFC_CUDA(cudaMallocAsync((void **)&fx, 8 * (3 + (size_t)nin), st));
    long long *acc = (long long *)(fx + 3);
    int rc = 0;
    if (cudaMemsetAsync(fx, 0, 8 * (3 + (size_t)nin), st) != cudaSuccess) rc = fail(RDFC_ERR_CUDA, "rdfc_dcn_backward_ex: memset failed");
    if (rc == 0) rc = fx_amax(gout, (long long)g.B * g.Cout * P, fx, st);
    if (rc == 0) {
        dcn_wsum_max_kernel<T><<<cdiv((long long)g.Cin * K, NT), NT, 0, st>>>(weight, g, fx + 1);
        count_launch();
    }
    if (rc == 0 && mask) rc = fx_amax(mask, (long long)g.B * g.dg * K * P, fx + 2, st);
    if (rc == 0) {
        const int blocks = (int)min((long long)cdiv(total, NT), (long long)sm_count() * 16);
        if (mask) dcn_bwd_data_kernel<T, true, true><<<blocks, NT, 0, st>>>(input, weight, offset, mask, gout, nullptr, goff, gmask, g, acc, fx);
        else dcn_bwd_data_kernel<T, false, true><<<blocks, NT, 0, st>>>(input, weight, offset, nullptr, gout, nullptr, goff, nullptr, g, acc, fx);
        count_launch();
        rc = fx_convert(acc, gin, nin, (double)K * P, fx, mask ? 3 : 2, st);
    }
    if (rc == 0 && cudaGetLastError() != cudaSuccess) rc = fail(RDFC_ERR_CUDA, "rdfc_dcn_backward_ex: kernel launch failed");
    cudaFreeAsync(fx, st);
    return rc;
}

template <typename T>
int bwd(const void *input, const void *weight, const void *offset, const void *mask, const void *gout, void *gin,
        void *goff, void *gmask, void *gw, void *gb, const Geo &g, cudaStream_t st, bool det) {
    const int K = g.kh * g.kw, P = g.Ho * g.Wo;
    if (gin && det) {
        if (int rc = bwd_data_det<T>((const T *)input, (const T *)weight, (const T *)offset, (const T *)mask, (const T *)gout, (T *)gin,
                                     (T *)goff, (T *)gmask, g, st))
            return rc;
    } else if (gin || goff || gmask) {
        if (gin) RDFC_CUDA(cudaMemsetAsync(gin, 0, sizeof(T) * (size_t)g.B * g.Cin * g.H * g.W, st));
        const long long total = (long long)g.B * g.dg * K * P;
        const int blocks = (int)min((long long)cdiv(total, NT), (long long)sm_count() * 16);
        if (mask)
            dcn_bwd_data_kernel<T, true, false><<<blocks, NT, 0, st>>>((const T *)input, (const T *)weight,
                                                                       (const T *)offset, (const T *)mask, (const T *)gout,
                                                                       (T *)gin, (T *)goff, (T *)gmask, g, nullptr, nullptr);
        else
            dcn_bwd_data_kernel<T, false, false><<<blocks, NT, 0, st>>>((const T *)input, (const T *)weight,
                                                                        (const T *)offset, nullptr, (const T *)gout,
                                                                        (T *)gin, (T *)goff, nullptr, g, nullptr, nullptr);
        RDFC_CHECK_LAUNCH("dcn_bwd_data_kernel");
    }
    if (gw) {
        const size_t smem = sizeof(T) * (NT + g.Cout / g.group);
        RDFC_REQUIRE(smem <= 48 * 1024, "Cout/group too large for the filter-gradient kernel");
        if (mask)
            dcn_bwd_weight_kernel<T, true><<<g.Cin * K, NT, smem, st>>>((const T *)input, (const T *)offset,
                                                                        (const T *)mask, (const T *)gout, (T *)gw, g);
        else
            dcn_bwd_weight_kernel<T, false><<<g.Cin * K, NT, smem, st>>>((const T *)input, (const T *)offset, nullptr,
                                                                         (const T *)gout, (T *)gw, g);
        RDFC_CHECK_LAUNCH("dcn_bwd_weight_kernel");
    }
    if (gb) {
        dcn_bwd_bias_kernel<T><<<g.Cout, NT, 0, st>>>((const T *)gout, (T *)gb, g.B, g.Cout, P);
        RDFC_CHECK_LAUNCH("dcn_bwd_bias_kernel");
    }
    return 0;
}

}  // namespace
}  // namespace rdfc

using namespace rdfc;

extern "C" int rdfc_dcn_out_size(const rdfc_dcn_shape *s, int *Ho, int *Wo) {
    Geo g;
    if (int rc = check_shape(s, g)) return rc;
    if (Ho) *Ho = g.Ho;
    if (Wo) *Wo = g.Wo;
    return 0;
}

extern "C" int rdfc_dcn_forward(const void *input, const void *weight, const void *bias, const void *offset,
                                const void *mask, void *output, const rdfc_dcn_shape *s, int dtype, void *stream) {
    Geo g;
    if (int rc = check_shape(s, g)) return rc;
    RDFC_REQUIRE(input && weight && offset && output, "input / weight / offset / output must not be NULL");
    cudaStream_t st = (cudaStream_t)stream;
    // GEMM-sized layers: sampled columns + tcgen05 contraction at fp32 fidelity (split fp16 operands); thin layers: the strip kernel
    if (dtype == RDFC_F32 && fwd_tc_ok(g))
        return fwd_tc((const float *)input, (const float *)weight, (const float *)bias, (const float *)offset, (const float *)mask,
                      (float *)output, g, st);
    if (dtype == RDFC_F32) return fwd<float>(input, weight, bias, offset, mask, output, g, st);
    if (dtype == RDFC_F64) return fwd<double>(input, weight, bias, offset, mask, output, g, st);
    return fail(RDFC_ERR_UNSUPPORTED, "rdfc_dcn_forward: dtype %d not supported (fp32 / fp64 only, as the reference)",
                dtype);
}

static int dcn_backward(const void *input, const void *weight, const void *offset, const void *mask, const void *grad_output,
                        void *grad_input, void *grad_offset, void *grad_mask, void *grad_weight, void *grad_bias,
                        const rdfc_dcn_shape *s, int dtype, void *stream, bool det) {
    Geo g;
    if (int rc = check_shape(s, g)) return rc;
    RDFC_REQUIRE(input && weight && offset && grad_output, "input / weight / offset / grad_output must not be NULL");
    RDFC_REQUIRE(mask || !grad_mask, "grad_mask requested without a mask (DCN v1 has none)");
    cudaStream_t st = (cudaStream_t)stream;
    // GEMM-sized layers: both contractions of the backward on tcgen05 at fp32 fidelity; thin layers / fp64: the CUDA-core kernels
    if (dtype == RDFC_F32 && bwd_tc_ok(g))
        return bwd_tc((const float *)input, (const float *)weight, (const float *)offset, (const float *)mask, (const float *)grad_output,
                      (float *)grad_input, (float *)grad_offset, (float *)grad_mask, (float *)grad_weight, (float *)grad_bias, g, st, det);
    if (dtype == RDFC_F32)
        return bwd<float>(input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask, grad_weight,
                          grad_bias, g, st, det);
    if (dtype == RDFC_F64)
        return bwd<double>(input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask, grad_weight,
                           grad_bias, g, st, det);
    return fail(RDFC_ERR_UNSUPPORTED, "rdfc_dcn_backward: dtype %d not supported", dtype);
}

extern "C" int rdfc_dcn_backward(const void *input, const void *weight, const void *offset, const void *mask,
                                 const void *grad_output, void *grad_input, void *grad_offset, void *grad_mask,
                                 void *grad_weight, void *grad_bias, const rdfc_dcn_shape *s, int dtype,
                                 void *stream) {
    return dcn_backward(input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask, grad_weight, grad_bias, s, dtype,
                        stream, false);
}

extern "C" int rdfc_dcn_backward_ex(const void *input, const void *weight, const void *offset, const void *mask,
                                    const void *grad_output, void *grad_input, void *grad_offset, void *grad_mask,
                                    void *grad_weight, void *grad_bias, const rdfc_dcn_shape *s, int dtype,
                                    void *stream, int flags) {
    RDFC_REQUIRE((flags & ~RDFC_DETERMINISTIC) == 0, "rdfc_dcn_backward_ex: unknown flags 0x%x", flags);
    return dcn_backward(input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask, grad_weight, grad_bias, s, dtype,
                        stream, (flags & RDFC_DETERMINISTIC) != 0);
}
