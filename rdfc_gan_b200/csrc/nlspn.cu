// NLSPN: fused offset/affinity stage and the propagation loop (fp32, NCHW, channels_f == 1, k_f == 3).
//
// Replaces nlspn/nlspn_model.py:68-138 (NLPSN._get_offset_affinity: a 3x3 conv, 8 ModulatedDeformConvFunction calls
// with a 1x1 kernel and ~25 small ATen kernels) by ONE kernel, and nlspn_model.py:140-144,166-173 (prop_time x
// {columns alloc, im2col, addmm(K=9,N=1), permute+contiguous}) by one gather kernel per iteration with no
// intermediate buffer.  The propagation is HBM / L2 bound: per pixel and iteration it streams 16 offsets + 9
// affinities (the centre tap's offsets are identically zero and are not read), gathers 36 feature corners from a
// shared-memory band, and writes one float.  One launch per iteration over the whole batch (walking the batch in L2-sized
// groups was measured slower: the launches get too small).
#include <stdlib.h>

#include <cuda_fp16.h>

#include "common.cuh"
#include "fixed_point.cuh"

namespace rdfc {
namespace {

constexpr int TX = 32, TY = 8;   // pixel tile of a CTA (one warp = one 32-pixel row segment -> coalesced planes)

// bilinear sample with the DCN validity rule and per-corner zeroing (deformconv/src/cuda/modulated_deform_im2col_cuda.cuh:25-54,180)
__device__ __forceinline__ float bilinear(const float *__restrict__ im, int H, int W, float y, float x) {
    if (!(y > -1.f && x > -1.f && y < (float)H && x < (float)W)) return 0.f;
    const float fy = floorf(y), fx = floorf(x);
    const int yl = (int)fy, xl = (int)fx;
    const float ly = y - fy, lx = x - fx, hy = 1.f - ly, hx = 1.f - lx;
    const bool y0 = yl >= 0, y1 = yl + 1 <= H - 1, x0 = xl >= 0, x1 = xl + 1 <= W - 1;
    const float *r0 = im + (long long)yl * W + xl;
    const float v1 = (y0 && x0) ? __ldg(r0) : 0.f;
    const float v2 = (y0 && x1) ? __ldg(r0 + 1) : 0.f;
    const float v3 = (y1 && x0) ? __ldg(r0 + W) : 0.f;
    const float v4 = (y1 && x1) ? __ldg(r0 + W + 1) : 0.f;
    return hy * hx * v1 + hy * lx * v2 + ly * hx * v3 + ly * lx * v4;
}

// ------------------------------------------------------------------------------------------------------------------
// Offset / affinity stage.  grid (ceil(W/TX), ceil(H/TY), B), block TX*TY.
//   1. conv_offset_aff: 8 -> 24 channels, 3x3, pad 1 (guidance tile + halo staged in shared memory, weights too)
//   2. offsets: tap j (of the 8 non-centre taps) takes conv channels (2j, 2j+1) as (dy, dx)   (nlspn_model.py:76)
//   3. affinity: AS/ASS raw, TC tanh/scale, TGASS tanh/(scale+1e-8)                           (:82-87)
//   4. conf_prop: aff_j *= bilinear(confidence, h + dy_j, w + dx_j)  (1x1 kernel, pad 0)       (:96-119)
//   5. normalise by max(sum|aff| + 1e-4, 1) (ASS/TGASS) or sum|aff| + 1e-4 (AS); aff_ref = 1 - sum  (:122-136)
//   6. output: fp32 planes offset (B,18,H,W) / aff (B,9,H,W) in the reference's layout, or (kPacked) the fp16 stream the
//      packed propagation kernel reads: 24 halves per pixel, see below
template <bool kPacked>
__global__ void __launch_bounds__(TX *TY) nlspn_affinity_kernel(const float *__restrict__ guidance,
                                                                const float *__restrict__ confidence,
                                                                const float *__restrict__ conv_w,
                                                                const float *__restrict__ conv_b,
                                                                const float *__restrict__ aff_scale, int affinity,
                                                                int conf_prop, float *__restrict__ offset,
                                                                float *__restrict__ aff, uint4 *__restrict__ packed, int H, int W) {
    __shared__ __align__(16) float s_w[72 * 24];     // [(ci*9 + tap)][24 outputs]: one LDS.128 feeds 4 FMAs
    __shared__ float s_b[24];
    __shared__ float s_g[8][TY + 2][TX + 2];
    const int tid = threadIdx.y * TX + threadIdx.x;
    const int b = blockIdx.z, x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;
    const long long P = (long long)H * W;
    for (int e = tid; e < 24 * 72; e += TX * TY) s_w[(e % 72) * 24 + e / 72] = conv_w[e];
    if (tid < 24) s_b[tid] = conv_b[tid];
    for (int e = tid; e < 8 * (TY + 2) * (TX + 2); e += TX * TY) {
        const int c = e / ((TY + 2) * (TX + 2)), r = e % ((TY + 2) * (TX + 2));
        const int yy = y0 + r / (TX + 2) - 1, xx = x0 + r % (TX + 2) - 1;
        s_g[c][r / (TX + 2)][r % (TX + 2)] =
            (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(guidance + ((long long)b * 8 + c) * P + (long long)yy * W + xx) : 0.f;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= W || y >= H) return;

    float o[24];
#pragma unroll
    for (int c = 0; c < 24; ++c) o[c] = s_b[c];
#pragma unroll
    for (int ci = 0; ci < 8; ++ci)
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const float g = s_g[ci][threadIdx.y + t / 3][threadIdx.x + t % 3];
            const float4 *w4 = reinterpret_cast<const float4 *>(s_w + (ci * 9 + t) * 24);
#pragma unroll
            for (int c4 = 0; c4 < 6; ++c4) {
                const float4 w = w4[c4];
                o[4 * c4 + 0] = fmaf(w.x, g, o[4 * c4 + 0]);
                o[4 * c4 + 1] = fmaf(w.y, g, o[4 * c4 + 1]);
                o[4 * c4 + 2] = fmaf(w.z, g, o[4 * c4 + 2]);
                o[4 * c4 + 3] = fmaf(w.w, g, o[4 * c4 + 3]);
            }
        }

    const float scale = __ldg(aff_scale);
    float a[8];
    float abs_sum = 0.f;
    const float *conf = confidence + (long long)b * P;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float v = o[16 + j];
        if (affinity == RDFC_AFF_TC) v = tanhf(v) / scale;
        else if (affinity == RDFC_AFF_TGASS) v = tanhf(v) / (scale + 1e-8f);
        if (conf_prop) v *= bilinear(conf, H, W, (float)y + o[2 * j], (float)x + o[2 * j + 1]);
        a[j] = v;
        abs_sum += fabsf(v);
    }
    abs_sum += 1e-4f;
    if (affinity == RDFC_AFF_ASS || affinity == RDFC_AFF_TGASS) abs_sum = abs_sum < 1.f ? 1.f : abs_sum;
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        if (affinity != RDFC_AFF_TC) a[j] = a[j] / abs_sum;
        sum += a[j];
    }
    const long long pix = (long long)y * W + x;
    if (kPacked) {
        // pixel g = b*P + pix lives in block g / 32 at lane g % 32: chunk 0 = (dy,dx) of neighbours 0..3, chunk 1 = neighbours
        // 4..7, chunk 2 = the 8 affinities; chunks of a block are 512 bytes apart
        const long long g = (long long)b * P + pix;
        uint4 *p = packed + (g >> 5) * 96 + (g & 31);
        auto h2 = [](float a_, float b_) { const __half2 h = __floats2half2_rn(a_, b_); return *reinterpret_cast<const uint32_t *>(&h); };
        p[0] = make_uint4(h2(o[0], o[1]), h2(o[2], o[3]), h2(o[4], o[5]), h2(o[6], o[7]));
        p[32] = make_uint4(h2(o[8], o[9]), h2(o[10], o[11]), h2(o[12], o[13]), h2(o[14], o[15]));
        p[64] = make_uint4(h2(a[0], a[1]), h2(a[2], a[3]), h2(a[4], a[5]), h2(a[6], a[7]));
        return;
    }
    float *offp = offset + (long long)b * 18 * P + pix;
    float *affp = aff + (long long)b * 9 * P + pix;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = j < 4 ? j : j + 1;   // centre tap inserted at index 4
        offp[(long long)(2 * k) * P] = o[2 * j];
        offp[(long long)(2 * k + 1) * P] = o[2 * j + 1];
        affp[(long long)k * P] = a[j];
    }
    offp[8 * P] = 0.f;
    offp[9 * P] = 0.f;
    affp[4 * P] = 1.f - sum;
}

// ------------------------------------------------------------------------------------------------------------------
// Propagation: out(h,w) = sum_k aff_k(h,w) * bilinear(in', h - 1 + k/3 + dy_k, w - 1 + k%3 + dx_k),  in' = in blended with
// the sparse input where preserve_input asks for it (nlspn_model.py:159-160,169).
//
// A CTA owns a contiguous run of image rows (rows are dealt evenly over one wave of CTAs; a run may span images) and
// walks it in sub-bands.  For a sub-band it first stages the feature rows its taps can reach (+- halo) in shared memory
// with a zero border, so that
//   * the 36 corner reads per pixel are LDS with NO bounds predicates: the DCN validity rule and per-corner zeroing
//     (modulated_deform_im2col_cuda.cuh:25-54,180) fall out of clamping the sample position to [-1, H] x [-1, W] and
//     reading zeros from the border;
//   * the preserve_input blend happens while staging (no separate pass over the feature map);
//   * the offset / affinity stream is read straight from HBM with 16- or 8-byte vectors (no L1 allocation);
//   * taps that leave the staged band (|offset| > halo) take the global-memory path (rare).
// Two stream formats:
//   fp32 planes  offset (B,18,H,W) + aff (B,9,H,W), the reference's layout (fp32 parity mode, the Module API): 25 planes
//                read per pixel (the centre tap's offsets are identically zero), two pixels per thread;
//   packed fp16  24 halves per pixel (16 offsets + 8 affinities; centre affinity = 1 - sum of the rounded others, so the
//                operator stays an exact affine combination), 48 B instead of 100 B per pixel and iteration, stored as
//                three 16-byte chunks per pixel, chunk-planar within blocks of 32 pixels (every warp load is one
//                contiguous 512-byte run), one pixel per thread (bf16 inference mode).
// The last iteration can apply the generator's output fusion (rdf_generator.py:401-406: clamp, 2-way confidence softmax,
// weighted sum) in its epilogue.
struct FuseOut { const float *d1, *c1, *c2; float *pred; };

// feature value at linear image index i, with the preserve_input blend
__device__ __forceinline__ float feat_at(const float *__restrict__ im, const float *__restrict__ fix, long long i) {
    float v = __ldg(im + i);
    if (fix) {
        const float f = __ldg(fix + i);
        v = f > 0.f ? f : v;
    }
    return v;
}

// bilinear sample from global memory (escape path and the fallback kernel), blend included
__device__ __forceinline__ float bilinear_fix(const float *__restrict__ im, const float *__restrict__ fix, int H, int W, float y, float x) {
    if (!(y > -1.f && x > -1.f && y < (float)H && x < (float)W)) return 0.f;
    const float fy = floorf(y), fx = floorf(x);
    const int yl = (int)fy, xl = (int)fx;
    const float ly = y - fy, lx = x - fx, hy = 1.f - ly, hx = 1.f - lx;
    const bool y0 = yl >= 0, y1 = yl + 1 <= H - 1, x0 = xl >= 0, x1 = xl + 1 <= W - 1;
    const long long i = (long long)yl * W + xl;
    const float v1 = (y0 && x0) ? feat_at(im, fix, i) : 0.f;
    const float v2 = (y0 && x1) ? feat_at(im, fix, i + 1) : 0.f;
    const float v3 = (y1 && x0) ? feat_at(im, fix, i + W) : 0.f;
    const float v4 = (y1 && x1) ? feat_at(im, fix, i + W + 1) : 0.f;
    return hy * hx * v1 + hy * lx * v2 + ly * hx * v3 + ly * lx * v4;
}

struct BandView {
    const float *tile;      // [nrows][pitch], tile row 0 = image row ty0, tile column tc = image column tc - 1
    const float *im, *fix;  // the image (and the sparse input, or NULL) in global memory: escape path
    int pitch, ty0, nrows, H, W;
    float Hf, Wf;
};

// Nine-tap gather from a staged band with the escape test hoisted out of the tap loop: the common case (no tap leaves
// the band) is straight-line code with 36 independent LDS.  dyf/dxf/af: the pixel's 9 offsets and affinities.
template <typename FDy, typename FDx, typename FA>
__device__ __forceinline__ float gather9(const BandView &v, FDy dyf, FDx dxf, FA af, int y, int x) {
    float ymin = 1e30f, ymax = -1e30f;            // rows only: columns are staged over the full width
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const float cy = fminf(fmaxf((float)(y - 1 + k / 3) + dyf(k), -1.f), v.Hf);
        ymin = fminf(ymin, cy);
        ymax = fmaxf(ymax, cy);
    }
    const bool esc = ((int)floorf(ymin) < v.ty0) | ((int)floorf(ymax) + 1 >= v.ty0 + v.nrows);
    float acc = 0.f;
    if (!esc) {
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            const float cy = fminf(fmaxf((float)(y - 1 + k / 3) + dyf(k), -1.f), v.Hf);
            const float cx = fminf(fmaxf((float)(x - 1 + k % 3) + dxf(k), -1.f), v.Wf);
            const float fy = floorf(cy), fx = floorf(cx);
            const float ly = cy - fy, lx = cx - fx, hy = 1.f - ly, hx = 1.f - lx;
            // tile index in float (exact: < 2^24), one conversion per tap instead of two plus an integer multiply-add
            const float *q = v.tile + (int)fmaf(fy - (float)v.ty0, (float)v.pitch, fx + 1.f);
            acc = fmaf(af(k), hy * hx * q[0] + hy * lx * q[1] + ly * hx * q[v.pitch] + ly * lx * q[v.pitch + 1], acc);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 9; ++k)
            acc = fmaf(af(k), bilinear_fix(v.im, v.fix, v.H, v.W, (float)(y - 1 + k / 3) + dyf(k), (float)(x - 1 + k % 3) + dxf(k)), acc);
    }
    return acc;
}

constexpr int BAND_THREADS = 256;

// stage image rows [ty0, ty0 + nrows) of `im` (blended with `fix`) into the tile, zero outside the image
__device__ __forceinline__ void stage_band(float *tile, const float *__restrict__ im, const float *__restrict__ fix, int ty0, int nrows,
                                           int pitch, int H, int W) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int tr = warp; tr < nrows; tr += BAND_THREADS / 32) {
        const int iy = ty0 + tr;
        const bool yok = iy >= 0 && iy < H;
        const long long base = (long long)iy * W - 1;
        float *dst = tile + tr * pitch;
        for (int tc = lane; tc < pitch; tc += 32) dst[tc] = (yok && tc >= 1 && tc <= W) ? feat_at(im, fix, base + tc) : 0.f;
    }
}

// epilogue of one output value at linear index o: store / clamp / fused output fusion
template <bool kFinal>
__device__ __forceinline__ float finish(float acc, int clamp, const FuseOut &fz, long long o) {
    if (kFinal) {
        if (clamp) acc = fminf(fmaxf(acc, -1.f), 1.f);
        if (fz.pred) {
            const float a = __ldg(fz.c1 + o), b = __ldg(fz.c2 + o), m = fmaxf(a, b);
            const float e1 = expf(a - m), e2 = expf(b - m), inv = 1.f / (e1 + e2);
            fz.pred[o] = __ldg(fz.d1 + o) * (e1 * inv) + acc * (e2 * inv);
        }
    }
    return acc;
}

__device__ __forceinline__ float ld_stream(const float *p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float2 ld_stream2(const float *p) {
    float2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_stream4(const uint4 *p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// ---- fp32 planes, kPix pixels per thread ------------------------------------------------------------------------------
template <bool kFinal, int kPix, int kMinBlocks>
__global__ void __launch_bounds__(BAND_THREADS, kMinBlocks)
nlspn_prop_band_kernel(const float *__restrict__ in, const float *__restrict__ offset, const float *__restrict__ aff,
                       const float *__restrict__ fixp, float *__restrict__ out, float *__restrict__ inter, FuseOut fz, int clamp,
                       int B, int H, int W, int rows_per_cta, int sub_rows, int halo, int pitch) {
    extern __shared__ float band_tile[];                 // rows of `pitch` floats; tile column tc <-> image column tc - 1 (-1 .. W + 2)
    const long long total = (long long)B * H, P = (long long)H * W;
    long long row = (long long)blockIdx.x * rows_per_cta;
    const long long row_end = row + rows_per_cta < total ? row + rows_per_cta : total;
    const int Wp = W / kPix;
    const float Hf = (float)H, Wf = (float)W;
    // Programmatic dependent launch: the next iteration's grid may take SM slots as this grid's CTAs retire (its CTAs then
    // sit in griddepcontrol.wait until this grid has completed and flushed), which removes the launch gap and the CTA
    // ramp-up between the launches.  Nothing of the previous iteration is read before the wait.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    while (row < row_end) {
        const int b = (int)(row / H), y_lo = (int)(row - (long long)b * H);
        long long nrl = row_end - row;
        if (nrl > H - y_lo) nrl = H - y_lo;          // rows of this image
        if (nrl > sub_rows) nrl = sub_rows;          // ... that fit the tile
        const int nr = (int)nrl;
        const int ty0 = y_lo - halo - 1;             // image row of tile row 0
        const int nrows = nr + 2 * halo + 3;
        const float *im = in + (long long)b * P;
        const float *fix = fixp ? fixp + (long long)b * P : nullptr;
        __syncthreads();                              // previous sub-band is done with the tile
        stage_band(band_tile, im, fix, ty0, nrows, pitch, H, W);
        __syncthreads();
        const BandView bv{band_tile, im, fix, pitch, ty0, nrows, H, W, Hf, Wf};
        const int nitems = nr * Wp;
        for (int idx = threadIdx.x; idx < nitems; idx += BAND_THREADS) {
            const int ry = idx / Wp, x = kPix * (idx - ry * Wp), y = y_lo + ry;
            const long long pix = (long long)y * W + x;
            const float *offp = offset + (long long)b * 18 * P + pix;
            const float *affp = aff + (long long)b * 9 * P + pix;
            const long long o = (long long)b * P + pix;
            if (kPix == 2) {
                float2 a[9], dy[9], dx[9];
#pragma unroll
                for (int k = 0; k < 9; ++k) {
                    a[k] = ld_stream2(affp + (long long)k * P);
                    if (k == 4) {
                        dy[k] = dx[k] = make_float2(0.f, 0.f);
                    } else {
                        dy[k] = ld_stream2(offp + (long long)(2 * k) * P);
                        dx[k] = ld_stream2(offp + (long long)(2 * k + 1) * P);
                    }
                }
                float acc0 = gather9(bv, [&](int k) { return dy[k].x; }, [&](int k) { return dx[k].x; }, [&](int k) { return a[k].x; }, y, x);
                float acc1 = gather9(bv, [&](int k) { return dy[k].y; }, [&](int k) { return dx[k].y; }, [&](int k) { return a[k].y; }, y, x + 1);
                acc0 = finish<kFinal>(acc0, clamp, fz, o);
                acc1 = finish<kFinal>(acc1, clamp, fz, o + 1);
                *reinterpret_cast<float2 *>(out + o) = make_float2(acc0, acc1);
                if (inter) *reinterpret_cast<float2 *>(inter + o) = make_float2(acc0, acc1);
            } else {
                float a[9], dy[9], dx[9];
#pragma unroll
                for (int k = 0; k < 9; ++k) {
                    a[k] = ld_stream(affp + (long long)k * P);
                    if (k == 4) {
                        dy[k] = dx[k] = 0.f;
                    } else {
                        dy[k] = ld_stream(offp + (long long)(2 * k) * P);
                        dx[k] = ld_stream(offp + (long long)(2 * k + 1) * P);
                    }
                }
                float acc = gather9(bv, [&](int k) { return dy[k]; }, [&](int k) { return dx[k]; }, [&](int k) { return a[k]; }, y, x);
                acc = finish<kFinal>(acc, clamp, fz, o);
                out[o] = acc;
                if (inter) inter[o] = acc;
            }
        }
        row += nr;
    }
}

// ---- packed fp16 stream, one pixel per thread -------------------------------------------------------------------------
__device__ __forceinline__ float2 h2f(uint32_t u) {
    const __half2 h = *reinterpret_cast<const __half2 *>(&u);
    return __half22float2(h);
}

template <bool kFinal>
__global__ void __launch_bounds__(BAND_THREADS, 4)
nlspn_prop_packed_kernel(const float *__restrict__ in, const uint4 *__restrict__ pk, const float *__restrict__ fixp,
                         float *__restrict__ out, FuseOut fz, int clamp, int B, int H, int W, int rows_per_cta, int sub_rows, int halo, int pitch) {
    extern __shared__ float band_tile[];
    const long long total = (long long)B * H, P = (long long)H * W;
    long long row = (long long)blockIdx.x * rows_per_cta;
    const long long row_end = row + rows_per_cta < total ? row + rows_per_cta : total;
    const float Hf = (float)H, Wf = (float)W;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    while (row < row_end) {
        const int b = (int)(row / H), y_lo = (int)(row - (long long)b * H);
        long long nrl = row_end - row;
        if (nrl > H - y_lo) nrl = H - y_lo;
        if (nrl > sub_rows) nrl = sub_rows;
        const int nr = (int)nrl;
        const int ty0 = y_lo - halo - 1;
        const int nrows = nr + 2 * halo + 3;
        const float *im = in + (long long)b * P;
        const float *fix = fixp ? fixp + (long long)b * P : nullptr;
        __syncthreads();
        stage_band(band_tile, im, fix, ty0, nrows, pitch, H, W);
        __syncthreads();
        const BandView bv{band_tile, im, fix, pitch, ty0, nrows, H, W, Hf, Wf};
        // linear pixel range of the sub-band; the walk starts at the enclosing 32-pixel block so that lane == g % 32
        const long long g0 = (long long)b * P + (long long)y_lo * W, g1 = g0 + (long long)nr * W;
        // software pipeline: the three 16-byte loads of the NEXT pixel are in flight while this one is gathered (one pixel per thread and
        // iteration made every iteration a serial load -> compute chain: ~2.9 us each, the kernel was latency-bound at 0.45 of the HBM peak)
        long long g = (g0 & ~31ll) + threadIdx.x;
        uint4 n0 = make_uint4(0, 0, 0, 0), n1 = n0, n2 = n0;
        if (g < g1) { const uint4 *p = pk + (g >> 5) * 96 + (g & 31); n0 = ld_stream4(p); n1 = ld_stream4(p + 32); n2 = ld_stream4(p + 64); }
        for (; g < g1; g += BAND_THREADS) {
            const uint4 c0 = n0, c1 = n1, c2 = n2;
            if (g + BAND_THREADS < g1) {
                const uint4 *p = pk + ((g + BAND_THREADS) >> 5) * 96 + ((g + BAND_THREADS) & 31);
                n0 = ld_stream4(p); n1 = ld_stream4(p + 32); n2 = ld_stream4(p + 64);
            }
            if (g < g0) continue;
            const int pix = (int)(g - (long long)b * P), y = pix / W, x = pix - y * W;
            float dy[9], dx[9], a[9];
            {
                float2 t;
                t = h2f(c0.x); dy[0] = t.x; dx[0] = t.y;
                t = h2f(c0.y); dy[1] = t.x; dx[1] = t.y;
                t = h2f(c0.z); dy[2] = t.x; dx[2] = t.y;
                t = h2f(c0.w); dy[3] = t.x; dx[3] = t.y;
                dy[4] = dx[4] = 0.f;
                t = h2f(c1.x); dy[5] = t.x; dx[5] = t.y;
                t = h2f(c1.y); dy[6] = t.x; dx[6] = t.y;
                t = h2f(c1.z); dy[7] = t.x; dx[7] = t.y;
                t = h2f(c1.w); dy[8] = t.x; dx[8] = t.y;
                t = h2f(c2.x); a[0] = t.x; a[1] = t.y;
                t = h2f(c2.y); a[2] = t.x; a[3] = t.y;
                t = h2f(c2.z); a[5] = t.x; a[6] = t.y;
                t = h2f(c2.w); a[7] = t.x; a[8] = t.y;
                a[4] = 1.f - (((a[0] + a[1]) + (a[2] + a[3])) + ((a[5] + a[6]) + (a[7] + a[8])));
            }
            float acc = gather9(bv, [&](int k) { return dy[k]; }, [&](int k) { return dx[k]; }, [&](int k) { return a[k]; }, y, x);
            acc = finish<kFinal>(acc, clamp, fz, g);
            out[g] = acc;
        }
        row += nr;
    }
}

// ---- fallback: one thread per pixel straight from global memory (images too wide for a shared-memory band) ---------
template <bool kFinal>
__global__ void __launch_bounds__(TX *TY) nlspn_prop_kernel(const float *__restrict__ in, const float *__restrict__ offset,
                                                            const float *__restrict__ aff, const float *__restrict__ fixp,
                                                            float *__restrict__ out, float *__restrict__ inter, FuseOut fz, int clamp,
                                                            int H, int W) {
    const int x = blockIdx.x * TX + threadIdx.x, y = blockIdx.y * TY + threadIdx.y, b = blockIdx.z;
    if (x >= W || y >= H) return;
    const long long P = (long long)H * W, pix = (long long)y * W + x;
    const float *offp = offset + (long long)b * 18 * P + pix;
    const float *affp = aff + (long long)b * 9 * P + pix;
    const float *im = in + (long long)b * P;
    const float *fix = fixp ? fixp + (long long)b * P : nullptr;
    float dy[9], dx[9], a[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        a[k] = ld_stream(affp + (long long)k * P);
        dy[k] = k == 4 ? 0.f : ld_stream(offp + (long long)(2 * k) * P);
        dx[k] = k == 4 ? 0.f : ld_stream(offp + (long long)(2 * k + 1) * P);
    }
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k)
        acc = fmaf(a[k], bilinear_fix(im, fix, H, W, (float)(y - 1 + k / 3) + dy[k], (float)(x - 1 + k % 3) + dx[k]), acc);
    acc = finish<kFinal>(acc, clamp, fz, (long long)b * P + pix);
    out[(long long)b * P + pix] = acc;
    if (inter) inter[(long long)b * P + pix] = acc;
}

// feat = (1 - m) * feat + m * fix, m = fix > 0 is folded into the band staging; this kernel only serves prop_time == 0 callers
__global__ void fuse_depth_kernel(const float *__restrict__ d1, const float *__restrict__ c1,
                                  const float *__restrict__ d2, const float *__restrict__ c2,
                                  float *__restrict__ d2c, float *__restrict__ pred, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v2 = fminf(fmaxf(d2[i], -1.f), 1.f);
        const float a = c1[i], b = c2[i], m = fmaxf(a, b);
        const float e1 = expf(a - m), e2 = expf(b - m), inv = 1.f / (e1 + e2);
        if (d2c) d2c[i] = v2;
        pred[i] = d1[i] * (e1 * inv) + v2 * (e2 * inv);
    }
}

// Row pitch of the staged band in floats: W + 4 columns, rounded up to a multiple of 32 so that a tap's shared-memory bank depends on
// its COLUMN only -- lanes are consecutive pixels, so taps whose rows differ from lane to lane (rough offset fields) collide only when two
// lanes land on the same column, not whenever (row x pitch + column) happens to coincide modulo 32.  RDFC_NLSPN_PITCH32 = 0: W + 4.
static int band_pitch(int W) { return knob("RDFC_NLSPN_PITCH32", 1) != 0 ? (W + 4 + 31) / 32 * 32 : W + 4; }

// launch geometry of the band kernels: CTAs per SM, rows per CTA, rows per sub-band (what fits the tile), shared memory
struct BandGeom { int per_sm, rows_per_cta, sub_rows, nctas; size_t smem; bool ok; };
static BandGeom band_geom(int B, int H, int W, int halo, int per_sm_max) {
    BandGeom g{};
    const long long total = (long long)B * H;
    const size_t row_bytes = (size_t)band_pitch(W) * sizeof(float);
    for (int per_sm = per_sm_max; per_sm >= 1; --per_sm) {
        const size_t cap = (size_t)(220 * 1024) / per_sm - 1024;
        int fit = (int)(cap / row_bytes) - 2 * halo - 3;                 // sub-band rows that fit beside the halo
        if (const long long sub = knob("RDFC_NLSPN_SUB", 0); sub > 0 && fit > sub && per_sm == per_sm_max) fit = (int)sub;   // tests: force sub-bands
        if (fit < (per_sm > 1 && knob("RDFC_NLSPN_SUB", 0) <= 0 ? 12 : 1)) continue;   // fewer CTAs per SM before tiny sub-bands
        long long ctas = (long long)sm_count() * per_sm;
        if (ctas > total) ctas = total;
        g.per_sm = per_sm;
        g.rows_per_cta = (int)((total + ctas - 1) / ctas);
        g.sub_rows = fit < g.rows_per_cta ? fit : g.rows_per_cta;
        if (g.sub_rows > H) g.sub_rows = H;
        g.nctas = (int)((total + g.rows_per_cta - 1) / g.rows_per_cta);
        g.smem = (size_t)(g.sub_rows + 2 * halo + 3) * row_bytes;
        g.ok = true;
        return g;
    }
    return g;
}

template <typename Kern, typename... Args>
static cudaError_t launch_pdl(Kern kern, int grid, int block, size_t smem, cudaStream_t st, int pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

static size_t packed_bytes(int B, int H, int W) { return (size_t)(((long long)B * H * W + 31) / 32) * 1536; }

}  // namespace
}  // namespace rdfc

using namespace rdfc;

static int affinity_check(const void *guidance, const void *confidence, const void *conv_w, const void *conv_b, const void *aff_scale,
                          int affinity, int conf_prop, int B, int H, int W) {
    RDFC_REQUIRE(guidance && conv_w && conv_b && aff_scale, "NULL pointer argument");
    RDFC_REQUIRE(!conf_prop || confidence, "conf_prop requires a confidence map (nlspn_model.py:150-151)");
    RDFC_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535, "bad shape (%d,%d,%d)", B, H, W);
    RDFC_REQUIRE(affinity >= RDFC_AFF_AS && affinity <= RDFC_AFF_TGASS, "unknown affinity mode %d", affinity);
    return 0;
}

extern "C" int rdfc_nlspn_affinity_forward(const float *guidance, const float *confidence, const float *conv_w,
                                           const float *conv_b, const float *aff_scale, int affinity, int conf_prop,
                                           float *offset, float *aff, int B, int H, int W, void *stream) {
    if (int rc = affinity_check(guidance, confidence, conv_w, conv_b, aff_scale, affinity, conf_prop, B, H, W)) return rc;
    RDFC_REQUIRE(offset && aff, "NULL output pointer");
    dim3 grid(cdiv(W, TX), cdiv(H, TY), B), block(TX, TY);
    nlspn_affinity_kernel<false><<<grid, block, 0, (cudaStream_t)stream>>>(guidance, confidence, conv_w, conv_b, aff_scale,
                                                                            affinity, conf_prop, offset, aff, nullptr, H, W);
    RDFC_CHECK_LAUNCH("nlspn_affinity_kernel");
    return 0;
}

extern "C" size_t rdfc_nlspn_packed_bytes(int B, int H, int W) { return (B > 0 && H > 0 && W > 0) ? packed_bytes(B, H, W) : 0; }

extern "C" int rdfc_nlspn_affinity_forward_packed(const float *guidance, const float *confidence, const float *conv_w,
                                                  const float *conv_b, const float *aff_scale, int affinity, int conf_prop,
                                                  void *packed, int B, int H, int W, void *stream) {
    if (int rc = affinity_check(guidance, confidence, conv_w, conv_b, aff_scale, affinity, conf_prop, B, H, W)) return rc;
    RDFC_REQUIRE(packed && ((uintptr_t)packed % 16) == 0, "packed stream must be a 16-byte aligned buffer of rdfc_nlspn_packed_bytes()");
    dim3 grid(cdiv(W, TX), cdiv(H, TY), B), block(TX, TY);
    nlspn_affinity_kernel<true><<<grid, block, 0, (cudaStream_t)stream>>>(guidance, confidence, conv_w, conv_b, aff_scale,
                                                                           affinity, conf_prop, nullptr, nullptr, (uint4 *)packed, H, W);
    RDFC_CHECK_LAUNCH("nlspn_affinity_kernel");
    return 0;
}

// shared body of the two propagate entry points: `packed` != NULL selects the fp16 stream
static int propagate(const float *feat_init, const float *offset, const float *aff, const void *packed, const float *feat_fix,
                     int preserve_input, float *out, float *scratch, float *inter, int B, int H, int W, int prop_time, int clamp_out,
                     const rdfc_fuse_out *fuse, cudaStream_t st) {
    RDFC_REQUIRE(feat_init && out && scratch, "NULL pointer argument");
    RDFC_REQUIRE(!preserve_input || feat_fix, "preserve_input requires feat_fix (nlspn_model.py:157-158)");
    RDFC_REQUIRE(B > 0 && H > 0 && W > 0 && prop_time >= 0, "bad shape (%d,%d,%d) x %d", B, H, W, prop_time);
    RDFC_REQUIRE(!fuse || (fuse->d1 && fuse->c1 && fuse->c2 && fuse->pred), "fuse: NULL pointer");
    const long long P = (long long)H * W;
    const FuseOut fz = fuse ? FuseOut{fuse->d1, fuse->c1, fuse->c2, fuse->pred} : FuseOut{nullptr, nullptr, nullptr, nullptr};
    const int clamp = (clamp_out || fuse) ? 1 : 0;          // the output fusion reads clamp(depth_map_2) (rdf_generator.py:401)
    if (prop_time == 0) {
        if (fuse) {
            const int nblk = (int)min((long long)cdiv(B * P, 256), (long long)sm_count() * 8);
            fuse_depth_kernel<<<nblk, 256, 0, st>>>(fuse->d1, fuse->c1, feat_init, fuse->c2, out, fuse->pred, (size_t)(B * P));
            RDFC_CHECK_LAUNCH("fuse_depth_kernel");
        } else {
            RDFC_CUDA(cudaMemcpyAsync(out, feat_init, sizeof(float) * B * P, cudaMemcpyDeviceToDevice, st));
        }
        return 0;
    }
    const float *fix = preserve_input ? feat_fix : nullptr;
    // band halo rows: taps beyond it take the global path (measured at sigma = 2.2 px offsets: 8 -> 49.5, 6 -> 47.8, 4 -> 47.2 us)
    const int halo = (int)knob("RDFC_NLSPN_HALO", 6);
    const int pdl = knob("RDFC_NLSPN_PDL", 1) != 0;         // programmatic dependent launch between the iterations
    const bool simple = knob("RDFC_NLSPN_SIMPLE", 0) != 0;
    // pixels per thread of the fp32-plane kernel: 2 -> 3 CTAs / SM (measured best), 1 (odd widths) -> 5 CTAs / SM
    const int pix = (!packed && W % 2 == 0 && P % 2 == 0 && ((uintptr_t)offset % 8) == 0 && ((uintptr_t)aff % 8) == 0 &&
                     ((uintptr_t)out % 8) == 0 && ((uintptr_t)scratch % 8) == 0 && (!inter || ((uintptr_t)inter % 8) == 0)) ? 2 : 1;
    const int per_sm_max = (int)knob("RDFC_NLSPN_PER_SM", packed ? 4 : (pix == 2 ? 3 : 5));
    const BandGeom g = band_geom(B, H, W, halo, per_sm_max);
    const bool band = g.ok && !simple;
    RDFC_REQUIRE(band || !packed, "packed NLSPN stream: image too wide for the band kernel (W = %d)", W);
    if (band) {
        if (packed) {
            RDFC_CUDA(cudaFuncSetAttribute(nlspn_prop_packed_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
            RDFC_CUDA(cudaFuncSetAttribute(nlspn_prop_packed_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        } else if (pix == 2) {
            RDFC_CUDA(cudaFuncSetAttribute(nlspn_prop_band_kernel<false, 2, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
            RDFC_CUDA(cudaFuncSetAttribute(nlspn_prop_band_kernel<true, 2, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        } else {
            RDFC_CUDA(cudaFuncSetAttribute(nlspn_prop_band_kernel<false, 1, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
            RDFC_CUDA(cudaFuncSetAttribute(nlspn_prop_band_kernel<true, 1, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        }
    }
    float *bufs[2] = {scratch, out};
    const float *cur = feat_init;
    for (int t = 0; t < prop_time; ++t) {
        float *dst = bufs[(prop_time - 1 - t) % 2 == 0 ? 1 : 0];      // ping-pong parity: the last iteration lands in `out`
        float *it = inter ? inter + (long long)t * B * P : nullptr;
        const bool last = t == prop_time - 1;
        const FuseOut none{nullptr, nullptr, nullptr, nullptr};
        if (band && packed) {
            if (last) RDFC_CUDA(launch_pdl(nlspn_prop_packed_kernel<true>, g.nctas, BAND_THREADS, g.smem, st, pdl, cur, (const uint4 *)packed, fix, dst, fz, clamp, B, H, W, g.rows_per_cta, g.sub_rows, halo, band_pitch(W)));
            else RDFC_CUDA(launch_pdl(nlspn_prop_packed_kernel<false>, g.nctas, BAND_THREADS, g.smem, st, pdl, cur, (const uint4 *)packed, fix, dst, none, 0, B, H, W, g.rows_per_cta, g.sub_rows, halo, band_pitch(W)));
            RDFC_CHECK_LAUNCH("nlspn_prop_packed_kernel");
        } else if (band) {
#define RDFC_BAND(FIN, PX, MB, FZ, CL)                                                                                            \
    RDFC_CUDA(launch_pdl(nlspn_prop_band_kernel<FIN, PX, MB>, g.nctas, BAND_THREADS, g.smem, st, pdl, cur, offset, aff, fix, dst, it, \
                         FZ, CL, B, H, W, g.rows_per_cta, g.sub_rows, halo, band_pitch(W)))
            if (pix == 2) { if (last) RDFC_BAND(true, 2, 3, fz, clamp); else RDFC_BAND(false, 2, 3, none, 0); }
            else { if (last) RDFC_BAND(true, 1, 5, fz, clamp); else RDFC_BAND(false, 1, 5, none, 0); }
#undef RDFC_BAND
            RDFC_CHECK_LAUNCH("nlspn_prop_band_kernel");
        } else {
            RDFC_REQUIRE(B <= 65535, "batch too large for the fallback kernel");
            dim3 grid(cdiv(W, TX), cdiv(H, TY), B), block(TX, TY);
            if (last) nlspn_prop_kernel<true><<<grid, block, 0, st>>>(cur, offset, aff, fix, dst, it, fz, clamp, H, W);
            else nlspn_prop_kernel<false><<<grid, block, 0, st>>>(cur, offset, aff, fix, dst, it, none, 0, H, W);
            RDFC_CHECK_LAUNCH("nlspn_prop_kernel");
        }
        cur = dst;
    }
    return 0;
}

extern "C" int rdfc_nlspn_propagate_forward(const float *feat_init, const float *offset, const float *aff,
                                            const float *feat_fix, int preserve_input, float *out, float *scratch,
                                            float *inter, int B, int H, int W, int prop_time, int clamp_out,
                                            const rdfc_fuse_out *fuse, void *stream) {
    RDFC_REQUIRE(offset && aff, "NULL pointer argument");
    return propagate(feat_init, offset, aff, nullptr, feat_fix, preserve_input, out, scratch, inter, B, H, W, prop_time, clamp_out,
                     fuse, (cudaStream_t)stream);
}

extern "C" int rdfc_nlspn_propagate_forward_packed(const float *feat_init, const void *packed, const float *feat_fix,
                                                   int preserve_input, float *out, float *scratch, int B, int H, int W,
                                                   int prop_time, int clamp_out, const rdfc_fuse_out *fuse, void *stream) {
    RDFC_REQUIRE(packed && ((uintptr_t)packed % 16) == 0, "packed stream must be 16-byte aligned");
    return propagate(feat_init, nullptr, nullptr, packed, feat_fix, preserve_input, out, scratch, nullptr, B, H, W, prop_time,
                     clamp_out, fuse, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------------------------
// Backward of the offset / affinity stage up to the conv output (training): given dL/d offset (B,18,H,W) and dL/d aff (B,9,H,W)
// it produces dL/d conv_offset_aff(guidance) (B,24,H,W), scatters dL/d confidence (the 1x1 DCN gathers of nlspn_model.py:96-119,
// offsets detached there) and accumulates dL/d aff_scale_const (TGASS).  The raw affinity channels are recomputed (8 of the 24
// conv outputs); the offsets are read back from the forward's output.  The conv's own backward (8 <-> 24 channels, 0.24 GFLOP per
// image) is left to the caller.
// kDet (RDFC_DETERMINISTIC): no atomics.  The confidence scatter's per-tap values go to g_tap (B,8,H,W) with their maximum in
// am[0], for nlspn_conf_scatter_det_kernel; the per-CTA sums of dL/d aff_scale go to g_scale[CTA index], for nlspn_sum_kernel.
template <bool kDet>
__global__ void __launch_bounds__(TX *TY) nlspn_affinity_bwd_kernel(const float *__restrict__ guidance, const float *__restrict__ confidence,
                                                                    const float *__restrict__ conv_w, const float *__restrict__ conv_b,
                                                                    const float *__restrict__ aff_scale, int affinity, int conf_prop,
                                                                    const float *__restrict__ offset, const float *__restrict__ g_offset,
                                                                    const float *__restrict__ g_aff, float *__restrict__ g_conv,
                                                                    float *__restrict__ g_conf, float *__restrict__ g_scale, int H, int W,
                                                                    float *__restrict__ g_tap, unsigned long long *__restrict__ am) {
    __shared__ __align__(16) float s_w[72 * 8];      // the 8 affinity channels: [(ci*9 + tap)][8]
    __shared__ float s_b[8];
    __shared__ float s_g[8][TY + 2][TX + 2];
    __shared__ float s_red[TX * TY / 32];
    const int tid = threadIdx.y * TX + threadIdx.x;
    const int b = blockIdx.z, x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;
    const long long P = (long long)H * W;
    for (int e = tid; e < 8 * 72; e += TX * TY) s_w[(e % 72) * 8 + e / 72] = conv_w[16 * 72 + e];
    if (tid < 8) s_b[tid] = conv_b[16 + tid];
    for (int e = tid; e < 8 * (TY + 2) * (TX + 2); e += TX * TY) {
        const int c = e / ((TY + 2) * (TX + 2)), r = e % ((TY + 2) * (TX + 2));
        const int yy = y0 + r / (TX + 2) - 1, xx = x0 + r % (TX + 2) - 1;
        s_g[c][r / (TX + 2)][r % (TX + 2)] =
            (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(guidance + ((long long)b * 8 + c) * P + (long long)yy * W + xx) : 0.f;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    const bool live = x < W && y < H;
    float gs = 0.f;                                  // this pixel's contribution to dL/d aff_scale_const
    unsigned long long tap_max = 0;                  // kDet: max |per-tap confidence gradient|
    if (live) {
        float r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = s_b[j];
#pragma unroll
        for (int ci = 0; ci < 8; ++ci)
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const float g = s_g[ci][threadIdx.y + t / 3][threadIdx.x + t % 3];
                const float4 *w4 = reinterpret_cast<const float4 *>(s_w + (ci * 9 + t) * 8);
                const float4 w0 = w4[0], w1 = w4[1];
                r[0] = fmaf(w0.x, g, r[0]); r[1] = fmaf(w0.y, g, r[1]); r[2] = fmaf(w0.z, g, r[2]); r[3] = fmaf(w0.w, g, r[3]);
                r[4] = fmaf(w1.x, g, r[4]); r[5] = fmaf(w1.y, g, r[5]); r[6] = fmaf(w1.z, g, r[6]); r[7] = fmaf(w1.w, g, r[7]);
            }
        const long long pix = (long long)y * W + x;
        const float *offp = offset + (long long)b * 18 * P + pix;
        const float *gop = g_offset + (long long)b * 18 * P + pix;
        const float *gap = g_aff + (long long)b * 9 * P + pix;
        float *gc = g_conv + (long long)b * 24 * P + pix;
        const float scale = __ldg(aff_scale);
        const float den = affinity == RDFC_AFF_TGASS ? scale + 1e-8f : scale;
        const float *conf = conf_prop ? confidence + (long long)b * P : nullptr;
        float t[8], v[8], c[8], u[8], dy[8], dx[8];
        float abs_sum = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = j < 4 ? j : j + 1;
            dy[j] = __ldg(offp + (long long)(2 * k) * P);
            dx[j] = __ldg(offp + (long long)(2 * k + 1) * P);
            t[j] = (affinity == RDFC_AFF_TC || affinity == RDFC_AFF_TGASS) ? tanhf(r[j]) : r[j];
            v[j] = (affinity == RDFC_AFF_TC || affinity == RDFC_AFF_TGASS) ? t[j] / den : r[j];
            c[j] = conf_prop ? bilinear(conf, H, W, (float)y + dy[j], (float)x + dx[j]) : 1.f;
            u[j] = v[j] * c[j];
            abs_sum += fabsf(u[j]);
        }
        abs_sum += 1e-4f;
        bool clamped = false;
        if ((affinity == RDFC_AFF_ASS || affinity == RDFC_AFF_TGASS) && abs_sum < 1.f) { abs_sum = 1.f; clamped = true; }
        const float g_ref = __ldg(gap + 4 * P);           // aff_ref = 1 - sum(aff)  (nlspn_model.py:132-136)
        float ga[8], dot = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = j < 4 ? j : j + 1;
            ga[j] = __ldg(gap + (long long)k * P) - g_ref;
            dot += ga[j] * u[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float gu = ga[j];
            if (affinity != RDFC_AFF_TC) {                // aff = u / S, S = sum|u| + 1e-4 (clamped from below: constant)
                const float sgn = u[j] > 0.f ? 1.f : (u[j] < 0.f ? -1.f : 0.f);
                gu = ga[j] / abs_sum - (clamped ? 0.f : dot / (abs_sum * abs_sum) * sgn);
            }
            const float gv = gu * c[j];
            if (conf_prop && kDet) {
                const float gcj = gu * v[j];
                g_tap[((long long)b * 8 + j) * P + pix] = gcj;
                const unsigned long long bits = fx_bits(gcj);
                tap_max = bits > tap_max ? bits : tap_max;
            } else if (conf_prop) {                       // dL/d confidence: transposed bilinear gather at (y + dy, x + dx)
                const float gcj = gu * v[j], sy = (float)y + dy[j], sx = (float)x + dx[j];
                if (gcj != 0.f && sy > -1.f && sx > -1.f && sy < (float)H && sx < (float)W) {
                    const float fy = floorf(sy), fx = floorf(sx);
                    const int yl = (int)fy, xl = (int)fx;
                    const float ly = sy - fy, lx = sx - fx;
                    float *gim = g_conf + (long long)b * P;
#pragma unroll
                    for (int aa = 0; aa < 2; ++aa)
#pragma unroll
                        for (int cc = 0; cc < 2; ++cc) {
                            const int yy = yl + aa, xx = xl + cc;
                            if (yy >= 0 && yy <= H - 1 && xx >= 0 && xx <= W - 1)
                                atomicAdd(gim + (long long)yy * W + xx, (aa ? ly : 1.f - ly) * (cc ? lx : 1.f - lx) * gcj);
                        }
                }
            }
            float gr = gv;
            if (affinity == RDFC_AFF_TC || affinity == RDFC_AFF_TGASS) {
                gr = gv * (1.f - t[j] * t[j]) / den;
                gs -= gv * t[j] / (den * den);
            }
            gc[(long long)(16 + j) * P] = gr;
            const int k = j < 4 ? j : j + 1;
            gc[(long long)(2 * j) * P] = __ldg(gop + (long long)(2 * k) * P);          // conv channel 2j / 2j+1 = (dy, dx) of neighbour j
            gc[(long long)(2 * j + 1) * P] = __ldg(gop + (long long)(2 * k + 1) * P);
        }
    }
    if (kDet && conf_prop) fx_warp_max(tap_max, am);
    if (g_scale) {                                    // block reduction, one atomic per CTA
        for (int o = 16; o > 0; o >>= 1) gs += __shfl_down_sync(0xffffffffu, gs, o);
        if ((tid & 31) == 0) s_red[tid >> 5] = gs;
        __syncthreads();
        if (tid == 0) {
            float tot = 0.f;
            for (int w = 0; w < TX * TY / 32; ++w) tot += s_red[w];
            if (kDet) g_scale[((long long)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = tot;
            else if (tot != 0.f) atomicAdd(g_scale, tot);
        }
    }
}

// kDet confidence scatter: g_tap (B,8,H,W) -> acc (B,H,W) in fixed point.  Destination bound: the 8 taps of every pixel of the
// image, each at most max |g_tap| (the four bilinear weights sum to 1).  grid (ceil(P / 256), B).
__global__ void __launch_bounds__(256) nlspn_conf_scatter_det_kernel(const float *__restrict__ g_tap, const float *__restrict__ offset,
                                                                     long long *__restrict__ acc, const unsigned long long *__restrict__ am,
                                                                     int H, int W) {
    const long long P = (long long)H * W;
    const int b = blockIdx.y;
    const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
    if (pix >= P) return;
    const Fx<float> fx(8.0 * (double)P, am, 1);
    const int y = (int)(pix / W), x = (int)(pix - (long long)y * W);
    const float *offp = offset + (long long)b * 18 * P + pix;
    long long *gim = acc + (long long)b * P;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = j < 4 ? j : j + 1;
        const float gcj = __ldg(g_tap + ((long long)b * 8 + j) * P + pix);
        const float sy = (float)y + __ldg(offp + (long long)(2 * k) * P), sx = (float)x + __ldg(offp + (long long)(2 * k + 1) * P);
        if (gcj != 0.f && sy > -1.f && sx > -1.f && sy < (float)H && sx < (float)W) {
            const float fy = floorf(sy), fxl = floorf(sx);
            const int yl = (int)fy, xl = (int)fxl;
            const float ly = sy - fy, lx = sx - fxl;
#pragma unroll
            for (int aa = 0; aa < 2; ++aa)
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) {
                    const int yy = yl + aa, xx = xl + cc;
                    if (yy >= 0 && yy <= H - 1 && xx >= 0 && xx <= W - 1)
                        fx_add(gim + (long long)yy * W + xx, fx.to_fixed((aa ? ly : 1.f - ly) * (cc ? lx : 1.f - lx) * gcj));
                }
        }
    }
}

// out[0] = sum of part[0..n) in a fixed order (one CTA: strided per-thread sums, then a fixed tree)
__global__ void __launch_bounds__(256) nlspn_sum_kernel(const float *__restrict__ part, int n, float *__restrict__ out) {
    __shared__ float red[256];
    float s = 0.f;
    for (int i = threadIdx.x; i < n; i += 256) s += part[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int h = 128; h > 0; h >>= 1) {
        if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = red[0];
}

// ------------------------------------------------------------------------------------------------------------------
// Backward of the propagation (training, SURVEY 8f rank 1).  One iteration is y = A x' with
//   (A x')[p] = sum_k aff_k[p] * bilinear(x', p + tap_k + offset_k[p]),   x' = preserve_input ? blend(x, fix) : x,
// the reference's 18 ModulatedDeformConvFunction calls with w = 1, b = 0 (nlspn_model.py:140-175).  Its backward
// (modulated_deform_conv_cuda.cu:124-280, kernels modulated_deform_im2col_cuda.cuh:197-328) is split in two phases:
//   1. g_{t-1} = A^T g_t for t = T..1: the col2im scatter (cuh:197-254); it needs no feature values, only offsets / affinities.
//   2. ONE pass over the pixels that accumulates, over all T iterations, grad_aff_k += g_t * bilinear(x'_{t-1}) and
//      grad_offset_k += g_t * aff_k * d bilinear / d(y, x) (col2im_coord, cuh:257-328) in registers and writes the 27 planes once,
//      instead of 18 read-modify-write rounds over them.
struct BwdPos { int yl, xl; float ly, lx; bool valid; };
__device__ __forceinline__ BwdPos bwd_pos(float y, float x, int H, int W) {
    BwdPos q;
    q.valid = y > -1.f && x > -1.f && y < (float)H && x < (float)W;      // cuh:180 / :228
    const float yf = floorf(y), xf = floorf(x);
    q.yl = (int)yf; q.xl = (int)xf; q.ly = y - yf; q.lx = x - xf;
    return q;
}

// g (raw) -> finalised in place: iterations below the last one add the gradient that arrived through list_feat and apply
// the (1 - mask_fix) factor of the blend (nlspn_model.py:169); then scattered into gprev (zero-initialised).
__global__ void __launch_bounds__(256) nlspn_bwd_scatter_kernel(float *__restrict__ g, const float *__restrict__ ginter,
                                                                const float *__restrict__ fix, const float *__restrict__ offset,
                                                                const float *__restrict__ aff, float *__restrict__ gprev,
                                                                int finalize, int H, int W) {
    const long long P = (long long)H * W;
    const int b = blockIdx.y;
    const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
    if (pix >= P) return;
    const long long o = (long long)b * P + pix;
    float gv = g[o];
    if (finalize) {
        if (fix && __ldg(fix + o) > 0.f) gv = 0.f;
        if (ginter) gv += __ldg(ginter + o);
        g[o] = gv;
    }
    if (gv == 0.f) return;
    const int y = (int)(pix / W), x = (int)(pix - (long long)y * W);
    const float *offp = offset + (long long)b * 18 * P + pix;
    const float *affp = aff + (long long)b * 9 * P + pix;
    float *gim = gprev + (long long)b * P;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const float sy = (float)(y - 1 + k / 3) + __ldg(offp + (long long)(2 * k) * P);
        const float sx = (float)(x - 1 + k % 3) + __ldg(offp + (long long)(2 * k + 1) * P);
        const BwdPos q = bwd_pos(sy, sx, H, W);
        if (!q.valid) continue;
        const float top = gv * __ldg(affp + (long long)k * P);
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int yy = q.yl + a, xx = q.xl + c;
                if (yy >= 0 && yy <= H - 1 && xx >= 0 && xx <= W - 1)
                    atomicAdd(gim + (long long)yy * W + xx, (a ? q.ly : 1.f - q.ly) * (c ? q.lx : 1.f - q.lx) * top);
            }
    }
}

// feats: x_0 = feat_init, x_t = inter[t-1]; G: finalised g_1..g_T at G + t * B * P.
template <bool kPreserve>
__global__ void __launch_bounds__(256) nlspn_bwd_coord_kernel(const float *__restrict__ feat_init, const float *__restrict__ inter,
                                                              const float *__restrict__ fix, const float *__restrict__ G,
                                                              const float *__restrict__ offset, const float *__restrict__ aff,
                                                              float *__restrict__ goff, float *__restrict__ gaff,
                                                              int B, int H, int W, int T) {
    const long long P = (long long)H * W, BP = (long long)B * P;
    const int b = blockIdx.y;
    const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
    if (pix >= P) return;
    const long long o = (long long)b * P + pix;
    const int y = (int)(pix / W), x = (int)(pix - (long long)y * W);
    const float *offp = offset + (long long)b * 18 * P + pix;
    const float *affp = aff + (long long)b * 9 * P + pix;
    const float *fx = kPreserve ? fix + (long long)b * P : nullptr;
#pragma unroll 1
    for (int k = 0; k < 9; ++k) {
        const float sy = (float)(y - 1 + k / 3) + __ldg(offp + (long long)(2 * k) * P);
        const float sx = (float)(x - 1 + k % 3) + __ldg(offp + (long long)(2 * k + 1) * P);
        const float m = __ldg(affp + (long long)k * P);
        float a_m = 0.f, a_y = 0.f, a_x = 0.f;
        // cuh:84-125 / :295-322: outside (-1, H) x (-1, W) every derivative is zero
        if (!(sy <= -1.f || sy >= (float)H || sx <= -1.f || sx >= (float)W)) {
            const BwdPos q = bwd_pos(sy, sx, H, W);
            const int yh = q.yl + 1, xh = q.xl + 1;
            const bool ok1 = q.yl >= 0 && q.xl >= 0, ok2 = q.yl >= 0 && xh <= W - 1, ok3 = yh <= H - 1 && q.xl >= 0,
                       ok4 = yh <= H - 1 && xh <= W - 1;
            const long long i1 = (long long)q.yl * W + q.xl, i2 = i1 + 1, i3 = i1 + W, i4 = i3 + 1;
            const float hy = 1.f - q.ly, hx = 1.f - q.lx;
            for (int t = 1; t <= T; ++t) {
                const float gv = __ldg(G + (long long)t * BP + o);
                if (gv == 0.f) continue;
                const float *im = (t == 1 ? feat_init : inter + (long long)(t - 2) * BP) + (long long)b * P;
                float v1 = ok1 ? __ldg(im + i1) : 0.f, v2 = ok2 ? __ldg(im + i2) : 0.f, v3 = ok3 ? __ldg(im + i3) : 0.f,
                      v4 = ok4 ? __ldg(im + i4) : 0.f;
                if (kPreserve) {        // x' = fix where fix > 0 (nlspn_model.py:159-160,169)
                    const float f1 = ok1 ? __ldg(fx + i1) : 0.f, f2 = ok2 ? __ldg(fx + i2) : 0.f, f3 = ok3 ? __ldg(fx + i3) : 0.f,
                                f4 = ok4 ? __ldg(fx + i4) : 0.f;
                    v1 = f1 > 0.f ? f1 : v1; v2 = f2 > 0.f ? f2 : v2; v3 = f3 > 0.f ? f3 : v3; v4 = f4 > 0.f ? f4 : v4;
                }
                const float val = hy * hx * v1 + hy * q.lx * v2 + q.ly * hx * v3 + q.ly * q.lx * v4;
                a_m += gv * val;
                a_y += gv * (hx * (v3 - v1) + q.lx * (v4 - v2));
                a_x += gv * (hy * (v2 - v1) + q.ly * (v4 - v3));
            }
        }
        gaff[(long long)b * 9 * P + (long long)k * P + pix] = a_m;
        goff[(long long)b * 18 * P + (long long)(2 * k) * P + pix] = a_y * m;
        goff[(long long)b * 18 * P + (long long)(2 * k + 1) * P + pix] = a_x * m;
    }
}

__global__ void nlspn_bwd_final_kernel(const float *__restrict__ g0, const float *__restrict__ fix, float *__restrict__ out, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = (fix && __ldg(fix + i) > 0.f) ? 0.f : g0[i];
}

// Deterministic propagation backward (RDFC_DETERMINISTIC), per iteration t = T..1:
//   nlspn_bwd_det_scatter_kernel   acc += fixed(A^T g_t) with 2^k from the bound P * max_p sum_k |aff_k[p]| * max |g_t|
//                                  (no tap crosses an image boundary, the four bilinear weights of a tap sum to 1)
//   nlspn_bwd_det_finalize_kernel  g_{t-1} = float(acc), then for t-1 >= 1 the finalisation of nlspn_bwd_scatter_kernel
//                                  ((1 - mask_fix), + grad_inter), acc = 0 for the next iteration, max |g_{t-1}|
// am[0] = max_p sum_k |aff_k[p]|, am[t] = max |g_t| after its finalisation.
__global__ void __launch_bounds__(256) nlspn_bwd_det_scatter_kernel(const float *__restrict__ g, const float *__restrict__ offset,
                                                                    const float *__restrict__ aff, long long *__restrict__ acc,
                                                                    const unsigned long long *__restrict__ am_aff,
                                                                    const unsigned long long *__restrict__ am_g, int H, int W) {
    const long long P = (long long)H * W;
    const int b = blockIdx.y;
    const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
    if (pix >= P) return;
    const float gv = g[(long long)b * P + pix];
    if (gv == 0.f) return;
    const unsigned long long am[2] = {*am_aff, *am_g};
    const Fx<float> fx((double)P, am, 2);
    const int y = (int)(pix / W), x = (int)(pix - (long long)y * W);
    const float *offp = offset + (long long)b * 18 * P + pix;
    const float *affp = aff + (long long)b * 9 * P + pix;
    long long *gim = acc + (long long)b * P;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const float sy = (float)(y - 1 + k / 3) + __ldg(offp + (long long)(2 * k) * P);
        const float sx = (float)(x - 1 + k % 3) + __ldg(offp + (long long)(2 * k + 1) * P);
        const BwdPos q = bwd_pos(sy, sx, H, W);
        if (!q.valid) continue;
        const float top = gv * __ldg(affp + (long long)k * P);
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int yy = q.yl + a, xx = q.xl + c;
                if (yy >= 0 && yy <= H - 1 && xx >= 0 && xx <= W - 1)
                    fx_add(gim + (long long)yy * W + xx, fx.to_fixed((a ? q.ly : 1.f - q.ly) * (c ? q.lx : 1.f - q.lx) * top));
            }
    }
}

// acc == NULL: g already holds the raw values (t = T).  src_aff, src_g: the two maxima of the scatter that filled acc.  fix / ginter as in
// nlspn_bwd_scatter_kernel's finalisation (NULL: not applied).  am_out: max |result| (NULL: not needed).  aff != NULL: also
// am_aff = max_p sum_k |aff_k[p]|.  Grid-stride over the B*P pixels (whole warps, for the maxima).
__global__ void __launch_bounds__(256) nlspn_bwd_det_finalize_kernel(long long *__restrict__ acc, const unsigned long long *__restrict__ src_aff,
                                                                     const unsigned long long *__restrict__ src_g,
                                                                     float *__restrict__ g, const float *__restrict__ fix,
                                                                     const float *__restrict__ ginter, unsigned long long *__restrict__ am_out,
                                                                     const float *__restrict__ aff, unsigned long long *__restrict__ am_aff,
                                                                     long long P, long long BP) {
    unsigned long long m = 0, ma = 0;
    float dn1 = 1.f, dn2 = 1.f;
    bool ok = true;
    if (acc) {
        const unsigned long long src[2] = {*src_aff, *src_g};
        const Fx<float> fx((double)P, src, 2);
        dn1 = fx.dn1; dn2 = fx.dn2; ok = fx.ok;
    }
    for (long long o = (long long)blockIdx.x * 256 + threadIdx.x; o < BP; o += (long long)gridDim.x * 256) {
        float gv;
        if (acc) {
            gv = ok ? __ll2float_rn(acc[o]) * dn1 * dn2 : __int_as_float(0x7fffffff);
            acc[o] = 0;
        } else {
            gv = g[o];
        }
        if (fix && __ldg(fix + o) > 0.f) gv = 0.f;
        if (ginter) gv += __ldg(ginter + o);
        g[o] = gv;
        const unsigned long long bits = fx_bits(gv);
        m = bits > m ? bits : m;
        if (aff) {
            const long long b = o / P, pix = o - b * P;
            float sa = 0.f;
#pragma unroll
            for (int k = 0; k < 9; ++k) sa += fabsf(__ldg(aff + (b * 9 + k) * P + pix));
            const unsigned long long ab = fx_bits(sa);
            ma = ab > ma ? ab : ma;
        }
    }
    if (am_out) fx_warp_max(m, am_out);
    if (aff) fx_warp_max(ma, am_aff);
}

extern "C" int rdfc_nlspn_affinity_backward(const float *guidance, const float *confidence, const float *conv_w, const float *conv_b,
                                            const float *aff_scale, int affinity, int conf_prop, const float *offset,
                                            const float *grad_offset, const float *grad_aff, float *grad_conv, float *grad_confidence,
                                            float *grad_aff_scale, int B, int H, int W, void *stream) {
    RDFC_REQUIRE(guidance && conv_w && conv_b && aff_scale && offset && grad_offset && grad_aff && grad_conv, "NULL pointer argument");
    RDFC_REQUIRE(!conf_prop || (confidence && grad_confidence), "conf_prop requires confidence and grad_confidence");
    RDFC_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535, "bad shape (%d,%d,%d)", B, H, W);
    RDFC_REQUIRE(affinity >= RDFC_AFF_AS && affinity <= RDFC_AFF_TGASS, "unknown affinity mode %d", affinity);
    cudaStream_t st = (cudaStream_t)stream;
    if (conf_prop) RDFC_CUDA(cudaMemsetAsync(grad_confidence, 0, sizeof(float) * (size_t)B * H * W, st));
    if (grad_aff_scale) RDFC_CUDA(cudaMemsetAsync(grad_aff_scale, 0, sizeof(float), st));
    dim3 grid(cdiv(W, TX), cdiv(H, TY), B), block(TX, TY);
    nlspn_affinity_bwd_kernel<false><<<grid, block, 0, st>>>(guidance, confidence, conv_w, conv_b, aff_scale, affinity, conf_prop, offset,
                                                             grad_offset, grad_aff, grad_conv, grad_confidence, grad_aff_scale, H, W,
                                                             nullptr, nullptr);
    RDFC_CHECK_LAUNCH("nlspn_affinity_bwd_kernel");
    return 0;
}

// RDFC_DETERMINISTIC: the confidence scatter in fixed point (per-tap values, their maximum, then the scatter and the conversion),
// dL/d aff_scale as per-CTA partials summed in a fixed order.  Workspace: stream-ordered, freed before returning.
static int affinity_backward_det(const float *guidance, const float *confidence, const float *conv_w, const float *conv_b,
                                 const float *aff_scale, int affinity, int conf_prop, const float *offset, const float *grad_offset,
                                 const float *grad_aff, float *grad_conv, float *grad_confidence, float *grad_aff_scale, int B, int H,
                                 int W, cudaStream_t st) {
    const long long P = (long long)H * W, BP = (long long)B * P;
    dim3 grid(cdiv(W, TX), cdiv(H, TY), B), block(TX, TY);
    const long long nctas = (long long)grid.x * grid.y * grid.z;
    // [am: 1 u64][acc: B*P i64][g_tap: 8*B*P f32][partials: nctas f32]
    const size_t acc_off = 8, tap_off = acc_off + 8 * (size_t)(conf_prop ? BP : 0), part_off = tap_off + 4 * (size_t)(conf_prop ? 8 * BP : 0);
    char *ws = nullptr;
    RDFC_CUDA(cudaMallocAsync((void **)&ws, part_off + 4 * (size_t)nctas, st));
    unsigned long long *am = (unsigned long long *)ws;
    long long *acc = (long long *)(ws + acc_off);
    float *g_tap = (float *)(ws + tap_off), *part = (float *)(ws + part_off);
    int rc = 0;
    if (cudaMemsetAsync(ws, 0, tap_off, st) != cudaSuccess) rc = fail(RDFC_ERR_CUDA, "rdfc_nlspn_affinity_backward_ex: memset failed");
    if (rc == 0) {
        nlspn_affinity_bwd_kernel<true><<<grid, block, 0, st>>>(guidance, confidence, conv_w, conv_b, aff_scale, affinity, conf_prop, offset,
                                                                grad_offset, grad_aff, grad_conv, nullptr, grad_aff_scale ? part : nullptr,
                                                                H, W, g_tap, am);
        count_launch();
    }
    if (rc == 0 && conf_prop) {
        nlspn_conf_scatter_det_kernel<<<dim3((unsigned)cdiv(P, 256), (unsigned)B), 256, 0, st>>>(g_tap, offset, acc, am, H, W);
        count_launch();
        rc = fx_convert<float>(acc, grad_confidence, BP, 8.0 * (double)P, am, 1, st);
    }
    if (rc == 0 && grad_aff_scale) {
        nlspn_sum_kernel<<<1, 256, 0, st>>>(part, (int)nctas, grad_aff_scale);
        count_launch();
    }
    if (rc == 0 && cudaGetLastError() != cudaSuccess) rc = fail(RDFC_ERR_CUDA, "rdfc_nlspn_affinity_backward_ex: kernel launch failed");
    cudaFreeAsync(ws, st);
    return rc;
}

extern "C" int rdfc_nlspn_affinity_backward_ex(const float *guidance, const float *confidence, const float *conv_w, const float *conv_b,
                                               const float *aff_scale, int affinity, int conf_prop, const float *offset,
                                               const float *grad_offset, const float *grad_aff, float *grad_conv, float *grad_confidence,
                                               float *grad_aff_scale, int B, int H, int W, void *stream, int flags) {
    RDFC_REQUIRE((flags & ~RDFC_DETERMINISTIC) == 0, "rdfc_nlspn_affinity_backward_ex: unknown flags 0x%x", flags);
    if (!(flags & RDFC_DETERMINISTIC))
        return rdfc_nlspn_affinity_backward(guidance, confidence, conv_w, conv_b, aff_scale, affinity, conf_prop, offset, grad_offset,
                                            grad_aff, grad_conv, grad_confidence, grad_aff_scale, B, H, W, stream);
    RDFC_REQUIRE(guidance && conv_w && conv_b && aff_scale && offset && grad_offset && grad_aff && grad_conv, "NULL pointer argument");
    RDFC_REQUIRE(!conf_prop || (confidence && grad_confidence), "conf_prop requires confidence and grad_confidence");
    RDFC_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535, "bad shape (%d,%d,%d)", B, H, W);
    RDFC_REQUIRE(affinity >= RDFC_AFF_AS && affinity <= RDFC_AFF_TGASS, "unknown affinity mode %d", affinity);
    return affinity_backward_det(guidance, confidence, conv_w, conv_b, aff_scale, affinity, conf_prop, offset, grad_offset, grad_aff,
                                 grad_conv, grad_confidence, grad_aff_scale, B, H, W, (cudaStream_t)stream);
}

extern "C" int rdfc_nlspn_propagate_backward(const float *grad_out, const float *grad_inter, const float *feat_init,
                                             const float *inter, const float *offset, const float *aff, const float *feat_fix,
                                             int preserve_input, float *grad_feat_init, float *grad_offset, float *grad_aff,
                                             float *scratch, int B, int H, int W, int prop_time, void *stream) {
    RDFC_REQUIRE(grad_out && feat_init && offset && aff && grad_feat_init && grad_offset && grad_aff && scratch, "NULL pointer argument");
    RDFC_REQUIRE(!preserve_input || feat_fix, "preserve_input requires feat_fix (nlspn_model.py:157-158)");
    RDFC_REQUIRE(B > 0 && H > 0 && W > 0 && prop_time >= 0 && B <= 65535, "bad shape (%d,%d,%d) x %d", B, H, W, prop_time);
    RDFC_REQUIRE(prop_time <= 1 || inter, "the backward needs the forward's intermediate results (inter)");
    cudaStream_t st = (cudaStream_t)stream;
    const long long P = (long long)H * W, BP = (long long)B * P;
    const int T = prop_time;
    const float *fix = preserve_input ? feat_fix : nullptr;
    if (T == 0) {
        RDFC_CUDA(cudaMemcpyAsync(grad_feat_init, grad_out, sizeof(float) * BP, cudaMemcpyDeviceToDevice, st));
        RDFC_CUDA(cudaMemsetAsync(grad_offset, 0, sizeof(float) * 18 * BP, st));
        RDFC_CUDA(cudaMemsetAsync(grad_aff, 0, sizeof(float) * 9 * BP, st));
        return 0;
    }
    // scratch = G[0..T]: G[T] = grad_out (the caller's grad_inter[T-1], if any, is added by the first scatter), the rest zero
    float *G = scratch;
    RDFC_CUDA(cudaMemsetAsync(G, 0, sizeof(float) * T * BP, st));
    RDFC_CUDA(cudaMemcpyAsync(G + (long long)T * BP, grad_out, sizeof(float) * BP, cudaMemcpyDeviceToDevice, st));
    dim3 grid((unsigned)cdiv(P, 256), (unsigned)B);
    for (int t = T; t >= 1; --t) {
        const float *gi = grad_inter ? grad_inter + (long long)(t - 1) * BP : nullptr;
        // the last iteration's output is not blended: only list_feat's gradient is added there
        nlspn_bwd_scatter_kernel<<<grid, 256, 0, st>>>(G + (long long)t * BP, gi, t < T ? fix : nullptr, offset, aff,
                                                       G + (long long)(t - 1) * BP, (t < T || gi) ? 1 : 0, H, W);
        RDFC_CHECK_LAUNCH("nlspn_bwd_scatter_kernel");
    }
    const int nblk = (int)min((long long)cdiv(BP, 256), (long long)sm_count() * 8);
    nlspn_bwd_final_kernel<<<nblk, 256, 0, st>>>(G, fix, grad_feat_init, BP);
    RDFC_CHECK_LAUNCH("nlspn_bwd_final_kernel");
    if (fix)
        nlspn_bwd_coord_kernel<true><<<grid, 256, 0, st>>>(feat_init, inter, fix, G, offset, aff, grad_offset, grad_aff, B, H, W, T);
    else
        nlspn_bwd_coord_kernel<false><<<grid, 256, 0, st>>>(feat_init, inter, fix, G, offset, aff, grad_offset, grad_aff, B, H, W, T);
    RDFC_CHECK_LAUNCH("nlspn_bwd_coord_kernel");
    return 0;
}

// RDFC_DETERMINISTIC: phase 1 as fixed-point scatters into one int64 plane, converted and finalised per iteration; phase 2 and the
// final kernel as in rdfc_nlspn_propagate_backward.  Workspace: stream-ordered, freed before returning.
static int propagate_backward_det(const float *grad_out, const float *grad_inter, const float *feat_init, const float *inter,
                                  const float *offset, const float *aff, const float *fix, float *grad_feat_init, float *grad_offset,
                                  float *grad_aff, float *G, int B, int H, int W, int T, cudaStream_t st) {
    const long long P = (long long)H * W, BP = (long long)B * P;
    // [am: T + 1 u64][acc: B*P i64]
    char *ws = nullptr;
    RDFC_CUDA(cudaMallocAsync((void **)&ws, 8 * ((size_t)T + 1 + (size_t)BP), st));
    unsigned long long *am = (unsigned long long *)ws;
    long long *acc = (long long *)(ws + 8 * ((size_t)T + 1));
    int rc = 0;
    if (cudaMemsetAsync(ws, 0, 8 * ((size_t)T + 1 + (size_t)BP), st) != cudaSuccess ||
        cudaMemcpyAsync(G + (long long)T * BP, grad_out, sizeof(float) * BP, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
        rc = fail(RDFC_ERR_CUDA, "rdfc_nlspn_propagate_backward_ex: memset / copy failed");
    const int nblk = fx_blocks(BP);
    const dim3 grid((unsigned)cdiv(P, 256), (unsigned)B);
    if (rc == 0) {          // g_T: the last iteration's output is not blended, only list_feat's gradient is added; + max sum |aff|
        nlspn_bwd_det_finalize_kernel<<<nblk, 256, 0, st>>>(nullptr, nullptr, nullptr, G + (long long)T * BP, nullptr,
                                                            grad_inter ? grad_inter + (long long)(T - 1) * BP : nullptr, am + T, aff, am, P, BP);
        count_launch();
    }
    for (int t = T; t >= 1 && rc == 0; --t) {
        nlspn_bwd_det_scatter_kernel<<<grid, 256, 0, st>>>(G + (long long)t * BP, offset, aff, acc, am, am + t, H, W);
        const bool fin = t - 1 >= 1;
        nlspn_bwd_det_finalize_kernel<<<nblk, 256, 0, st>>>(acc, am, am + t, G + (long long)(t - 1) * BP, fin ? fix : nullptr,
                                                            (fin && grad_inter) ? grad_inter + (long long)(t - 2) * BP : nullptr,
                                                            fin ? am + t - 1 : nullptr, nullptr, nullptr, P, BP);
        count_launch(2);
    }
    if (rc == 0) {
        nlspn_bwd_final_kernel<<<nblk, 256, 0, st>>>(G, fix, grad_feat_init, BP);
        if (fix)
            nlspn_bwd_coord_kernel<true><<<grid, 256, 0, st>>>(feat_init, inter, fix, G, offset, aff, grad_offset, grad_aff, B, H, W, T);
        else
            nlspn_bwd_coord_kernel<false><<<grid, 256, 0, st>>>(feat_init, inter, fix, G, offset, aff, grad_offset, grad_aff, B, H, W, T);
        count_launch(2);
    }
    if (rc == 0 && cudaGetLastError() != cudaSuccess) rc = fail(RDFC_ERR_CUDA, "rdfc_nlspn_propagate_backward_ex: kernel launch failed");
    cudaFreeAsync(ws, st);
    return rc;
}

extern "C" int rdfc_nlspn_propagate_backward_ex(const float *grad_out, const float *grad_inter, const float *feat_init,
                                                const float *inter, const float *offset, const float *aff, const float *feat_fix,
                                                int preserve_input, float *grad_feat_init, float *grad_offset, float *grad_aff,
                                                float *scratch, int B, int H, int W, int prop_time, void *stream, int flags) {
    RDFC_REQUIRE((flags & ~RDFC_DETERMINISTIC) == 0, "rdfc_nlspn_propagate_backward_ex: unknown flags 0x%x", flags);
    // T == 0 copies and zero-fills: nothing to scatter
    if (!(flags & RDFC_DETERMINISTIC) || prop_time == 0)
        return rdfc_nlspn_propagate_backward(grad_out, grad_inter, feat_init, inter, offset, aff, feat_fix, preserve_input, grad_feat_init,
                                             grad_offset, grad_aff, scratch, B, H, W, prop_time, stream);
    RDFC_REQUIRE(grad_out && feat_init && offset && aff && grad_feat_init && grad_offset && grad_aff && scratch, "NULL pointer argument");
    RDFC_REQUIRE(!preserve_input || feat_fix, "preserve_input requires feat_fix (nlspn_model.py:157-158)");
    RDFC_REQUIRE(B > 0 && H > 0 && W > 0 && prop_time > 0 && B <= 65535, "bad shape (%d,%d,%d) x %d", B, H, W, prop_time);
    RDFC_REQUIRE(prop_time <= 1 || inter, "the backward needs the forward's intermediate results (inter)");
    return propagate_backward_det(grad_out, grad_inter, feat_init, inter, offset, aff, preserve_input ? feat_fix : nullptr, grad_feat_init,
                                  grad_offset, grad_aff, scratch, B, H, W, prop_time, (cudaStream_t)stream);
}

extern "C" int rdfc_fuse_depth_forward(const float *d1, const float *c1, const float *d2, const float *c2,
                                       float *d2_clamped, float *pred, size_t n, void *stream) {
    RDFC_REQUIRE(d1 && c1 && d2 && c2 && pred, "NULL pointer argument");
    if (n == 0) return 0;
    const int nblk = (int)min((long long)cdiv((long long)n, 256), (long long)sm_count() * 8);
    fuse_depth_kernel<<<nblk, 256, 0, (cudaStream_t)stream>>>(d1, c1, d2, c2, d2_clamped, pred, n);
    RDFC_CHECK_LAUNCH("fuse_depth_kernel");
    return 0;
}
