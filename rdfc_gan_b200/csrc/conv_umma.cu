// Implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM), bf16 x bf16 -> fp32.
// Persistent, warp-specialised, double-buffered in TMEM.
//
// One kernel covers every GEMM-shaped layer of the generator (encoder_decoder/common.py:29-61, the torchvision
// BasicBlock convs, the decode heads rdf_generator.py:68-102 and the per-pixel EqualLinear of W-AdaIN
// model_utils.py:72-75): 3x3 / 1x1, stride 1 / 2, and ConvTranspose2d(k3,s2,p1,op1) as four sub-pixel phases.
//
// GEMM view of one tile:  D[128*NACC pixels, BN couts] += A[pixels, 32 cin] * B[couts, 32 cin]^T  over (cin block, tap)
//   * a tile is NACC accumulators of 16 x 8 output pixels (128 TMEM lanes x BN fp32 columns each, MMA row m = 8*r + c),
//     arranged nax across x (NACC / nax) down so that the padded tile grid wastes the fewest pixels.
//   * CTAs are persistent (grid = min(#tiles, #SMs)), 16 warps (4 per scheduler = 128 registers per thread), and walk
//     tiles round-robin.  The roles run decoupled through mbarrier rings that continue across tiles, so the loads of
//     tile t+1 and the epilogue of tile t-1 overlap the MMAs of tile t:
//       warp 0      A loader (one thread): per 32-channel block and plane ONE cp.async.bulk.tensor.4d of the tile's
//                   input HALO (every pixel any tap can touch) through a tensor map over the NHWC input: box = 32
//                   channels x plane columns x plane rows, SWIZZLE_64B into [pixel][64 B], out-of-bounds zero fill =
//                   the conv padding.  A core-matrix group is 8 consecutive pixels of a row, SBO = the plane's row
//                   pitch, and every filter tap is just a different descriptor start address into the same staged
//                   plane (input leaves L2 ~1.2x, not 9x).  Stride-2 layers load the four input-parity planes with
//                   element stride 2; a transposed conv enumerates its four output phases as separate tiles, each a
//                   1/2/2/4-tap conv over the input grid.
//                   (warps 0-5 are the im2col builders of the fused input stems, which stage a no-swizzle
//                   [cin/8][pixel][16 B] layout.)
//       warp 7      B loader: one stage = the pre-packed (32-cin, BN) filter blocks of all nine taps of a k-block (3x3 convs
//                   with N <= 128; one filter row = 3 taps when two such stages do not fit), cp.async.bulk (TMA 1-D) issued
//                   by all lanes.
//       warp 6      MMA issuer: convergent loop, one elected lane issues tcgen05.mma (M=128, N=BN, K=16) and frees
//                   stages with tcgen05.commit.  In TMA mode warp 5 is a second issuer for tiles of >= 2 accumulators
//                   (each issuer owns half of them; both commit on the same barriers).
//       warps 8-15  epilogue: tcgen05.ld 32x32b.x16 -> y = act(acc*scale + shift + residual) -> bf16 NHWC channel
//                   slice (this is how every torch.cat of the reference disappears); mode 2 applies W-AdaIN, mode 3
//                   turns the 9 * ncols head columns into fp32 planes by a shift-add through shared memory.  TMEM holds
//                   two accumulator sets (when 2*NACC*BN <= 512), so the MMA warp fills set (t+1)&1 while the epilogue
//                   drains set t&1.
#include <cuda.h>
#include <limits.h>
#include <stdlib.h>

#include "common.cuh"

namespace rdfc {
namespace {

constexpr int BK = 32;            // input channels per A stage (2 MMAs of K=16)
constexpr int KCH = BK / 8;       // 16-byte cin chunks per stage
constexpr int TH = 16;            // tile rows (= 8-row groups of one M=128 MMA)
// 16 warps: the register file is split per scheduler (16K registers each), so 4 warps per scheduler leave 128
// registers per thread; 18 warps (5 on two schedulers) would cap every thread at 96 and spill the epilogue.
constexpr int NPROD_WARPS = 6, NPROD = NPROD_WARPS * 32;   // A producer threads of the stems (warps 0-5)
constexpr int PIXPASS = NPROD / 4;                         // pixels staged per pass of the producer threads (48)
constexpr int MMA_WARP = 6, BLOAD_WARP = 7, EPI_WARP0 = 8, NEPI_WARPS = 8;
constexpr int MMA2_WARP = 5;       // second MMA issuer (TMA mode only, where warps 1-5 have no staging work); another scheduler than MMA_WARP
constexpr int NTHREADS = 16 * 32;
constexpr int MAX_PLANES = 4, MAX_TAPS = 9;
// mbarriers for <= 8 A stages, <= 16 B stages, 2+2 accumulator sets, 4 residual slabs; TMEM slot.  The last 192 bytes are
// unused: they keep `fixed` in the tile planner, and with it the stage counts every layer was tuned with, as they are.
constexpr int BAR_BYTES = (2 * 8 + 2 * 16 + 4 + 4) * 8 + 16 + 192;
constexpr int EPI_SLAB_BYTES = 128 * 64;      // one staged epilogue slab: 128 pixels x 32 bf16 channels

struct Plane {
    int ystep, yoff, xstep, xoff;  // input pixel = (ystep*(ty0+r) + yoff, xstep*(tx0+c) + xoff)
    int rows, cols, base;          // extent and first pixel slot of the plane inside a stage
};
struct Tap {
    int plane, sy, sx, wtap;       // staged plane, shift inside it, index of the filter tap in the packed weights
};
struct Phase {                     // one sub-pixel phase of a transposed conv (or the single phase of a conv)
    int ntaps;
    Tap taps[MAX_TAPS];
    int oyo, oxo;                  // output pixel = (oys*(ty0+r) + oyo, oxs*(tx0+c) + oxo)
};
struct Params {
    // A operand through TMA (a_tma != 0): one 4-D tensor map (C, W, H, B) over the NHWC input view; box = 32 channels x
    // plane columns x plane rows, SWIZZLE_64B, zero fill outside the image = the conv padding
    alignas(64) CUtensorMap tmap_a;
    // Epilogue through TMA (tma_out != 0, MODE_STD only): 4-D tensor maps (C, W, H, B) over the NHWC output view and the
    // residual view; box = 32 channels x 8 x 16 pixels (one accumulator's 128 MMA rows), SWIZZLE_64B.  The epilogue stages
    // 32-channel slabs [pixel][64 B] in shared memory and writes them with cp.async.bulk.tensor stores (out-of-range pixels and
    // channels are clipped by the TMA unit); residual slabs arrive the same way through tensor loads.
    alignas(64) CUtensorMap tmap_out;
    alignas(64) CUtensorMap tmap_res;
    int tma_out;
    // fp32-faithful contraction on the 16-bit tensor cores ("3 x fp16"): the input is a split tensor [hi(C) | lo(C)] per pixel
    // (hi = fp16(x), lo = fp16(x - hi): 22 mantissa bits together) and the filter bank is packed as [W_hi ; W_lo ; W_hi] along
    // Cin, so that the K loop computes x_hi W_hi + x_hi W_lo + x_lo W_hi with fp32 accumulation (the dropped x_lo W_lo term is
    // 2^-22 relative).  A bf16 split (8 + 8 bits) was measured first: 1.3e-4 max-abs on the O(1)-activation goldens, not enough.
    // k-block i reads input channels split_ch(i); out_f32: fp32 NHWC output / residual (MODE_GENERAL).
    int split_c;                   // C (input channels of the layer) when split, else 0
    int out_f32;
    int dual;                      // two MMA issuer warps (MMA_WARP and MMA2_WARP), each owning a subset of the accumulators
    int fast9;                     // nacc == 1, gtaps == 9, TMA operands, one phase: the MMA warp issues a stage as one statement (RDFC_UMMA_FAST9)
    int epi_split;                 // one-accumulator tiles: the two epilogue groups share the accumulator's column steps (RDFC_UMMA_EPISPLIT)
    int kbs;                       // 1x1 convs: 32-channel k-blocks per A stage (plane j = channels 32 j.. of the same pixels, tap j = its filter block)
    // a_tma: the A operand arrives through tmap_a (every layer but the stems, whose producers build it);
    // a_tx_bytes: bytes the TMA loads of one stage deliver (planes x rows x cols x 64)
    int a_tma, px16, a_plane_bytes, a_tx_bytes;
    int _pad_tma;   // px16: 16-byte units per staged pixel (4 with TMA: [pixel][64 B]; 1 in the stems: [cin/8][pixel][16 B])
    const __nv_bfloat16 *in;
    int in_stride, B, Hi, Wi;
    int Ht, Wt, tiles_y, tiles_x, n_tiles_n, nphases, ntiles;   // tile space
    const __nv_bfloat16 *w;
    int CoutP, cin_chunks, nkb;    // padded Cout, Cin/8, Cin/BK
    __nv_bfloat16 *out;
    int out_stride, Cout, Ho, Wo, oys, oxs;
    const __nv_bfloat16 *res;
    int res_stride;
    const float *scale, *shift;
    int act, nacc, nax, bn, sa, sb, npix, npix_pad, nplanes, tmem_cols, nsets;   // nacc accumulators = nax across x (nacc / nax) down
    int ncols;                     // fused decode heads: fp32 output planes, one per output column
    int tstep_y, tstep_x, torg;    // tile origin = index * step + torg (shift-add heads: overlapping 16x16 regions, step 14, origin -1)
    float *plane[16];
    long long plane_bstride[16];
    int act_col[16];
    Plane planes[MAX_PLANES];
    // per (phase, tap), precomputed on the host so the MMA / filter-loader threads only add:
    //   tap_alo / tap_ahi : A-operand shared-memory descriptor of the tap's shifted view, without the stage base
    //   tap_w             : element offset of the tap's filter block in the packed weights
    int ntaps[4], oyo[4], oxo[4];
    uint32_t tap_alo[4][MAX_TAPS], tap_ahi[4][MAX_TAPS];
    long long tap_w[4][MAX_TAPS];
    int dbg_flags;                 // development aid (RDFC_UMMA_SKIP): 1 = no output stores, 2 = no TMEM loads
    long long *dbg;                // development aid: per-CTA role timers (RDFC_UMMA_DBG=1), else nullptr
    long long w_kb_stride;         // elements between consecutive 32-cin blocks of one tap
    // fused input stems (rdfc_stem_forward): the producers build im2col rows from fp32 NCHW inputs instead of copying
    const float *stem_in0, *stem_in1;
    int stem_c0, stem_k;           // channels of in0; im2col rows in use (9 * channels), the rest of the 64 are zero
    __nv_bfloat16 *out2;           // second destination for output columns >= split (NULL: none)
    int out2_stride, split;
    // fused W-AdaIN epilogue (rdfc_wadain_conv_forward): tile columns = [gamma half | beta half]
    const __nv_bfloat16 *wad_x;    // normalised tensor (NULL: not a W-AdaIN launch)
    int wad_x_stride, wad_C;
    const float *wad_mean, *wad_rstd;
    const __nv_bfloat16 *wad_w;    // optional [gamma weight | beta weight] tensor (2C channels), `weighting=True`
    int wad_w_stride;
    int gtaps;                     // filter taps per B stage (3 for 3x3 convs: one wait / commit per filter row)
    int vec32;                     // output (and residual) slices are 32-byte aligned: 256-bit stores / loads
    int b_contig;                  // the 4 cin chunks of a stage are contiguous in the packed weights (one Cout tile)
    // split_factor (with split_c): the device factor s of an input scaled by a power of two before its split (rdfc_conv_forward /
    // rdfc_heads_forward on fp32 data), else NULL.  Its exact inverse is folded into s_scale when staged (convs) or applied to each
    // tap sum (heads).
    const float *split_factor;
};

struct Tile {
    int b, ty0, tx0, n0, z;
};
__device__ __forceinline__ Tile decode_tile(const Params &P, int tile) {
    Tile t;
    const int nt = tile % P.n_tiles_n; tile /= P.n_tiles_n;      // Cout tile fastest: the A halo stays hot in L2
    const int txi = tile % P.tiles_x; tile /= P.tiles_x;
    const int tyi = tile % P.tiles_y; tile /= P.tiles_y;
    t.z = tile % P.nphases; tile /= P.nphases;
    t.b = tile;
    t.ty0 = tyi * P.tstep_y + P.torg; t.tx0 = txi * P.tstep_x + P.torg; t.n0 = nt * P.bn;
    return t;
}

// ---- PTX wrappers ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug traps after ~4 s instead of hanging the GPU.
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
template <bool kBackoff = false>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;  // fast path: no clock read, no loop
    const long long t0 = clock64();
    for (;;) {
        if (mbar_try_wait(bar, parity)) return;
        if (kBackoff) __nanosleep(128);      // long waits: do not steal issue slots from the MMA / producer warps
        if (clock64() - t0 > 8000000000ll) {
            printf("rdfc conv_umma: mbarrier timeout (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x,
                   bar, parity);
            __trap();
        }
    }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// descriptors passed as (lo, hi) words: advancing an operand is one 32-bit add on the start-address field
__device__ __forceinline__ void tc_mma2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                        uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc)
        : "memory");
}
// A whole 9-tap stage of a one-accumulator tile (18 MMAs) as ONE asm statement: no table loads, loops, predicates or dispatch between the MMAs.
// tlo[t] = tap t's A descriptor low word (without the stage base); filters of tap t sit t * b_tap16 after b_lo.
__device__ __forceinline__ void tc_mma_stage9(uint32_t d_tmem, const uint32_t (&tlo)[9], uint32_t a_stage_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t acc0, uint32_t b_tap16, uint32_t aks, uint32_t bks) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t.reg .b32 ta, tb;\n\t"
        "setp.ne.b32 p, %15, 0;\n\tsetp.eq.b32 q, 0, 0;\n\t"
        "add.u32 ta, %1, %10;\n\t"
        "mov.b32 tb, %12;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, p;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %2, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %3, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %4, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %5, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %6, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %7, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %8, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "add.u32 ta, %9, %10;\n\t"
        "add.u32 tb, tb, %16;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "add.u32 ta, ta, %17;\n\tadd.u32 tb, tb, %18;\n\t"
        "mov.b64 da, {ta, %11};\n\tmov.b64 db, {tb, %13};\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %14, q;\n\t"
        "sub.u32 tb, tb, %18;\n\t"
        "}"
        ::"r"(d_tmem), "r"(tlo[0]), "r"(tlo[1]), "r"(tlo[2]), "r"(tlo[3]), "r"(tlo[4]), "r"(tlo[5]), "r"(tlo[6]), "r"(tlo[7]), "r"(tlo[8]), "r"(a_stage_lo),
          "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc0), "r"(b_tap16), "r"(aks), "r"(bks)
        : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// all MMAs of one (k-block, tap): BK/16 k-steps x NACC accumulators, fully unrolled
// accumulator j = (jy, jx) covers the 16 x 8 pixel block at rows 16 jy, columns 8 jx of the tile: its A view starts
// jy * 16 plane rows + jx * 8 pixels further (jx_step = 8, jy_step = 16 * plane pitch, in 16-byte units)
template <int NACC>
__device__ __forceinline__ void issue_tap(uint32_t d_base, uint32_t bn, uint32_t a_lo, uint32_t a_hi, uint32_t a_kstep,
                                          uint32_t b_lo, uint32_t b_hi, uint32_t b_kstep, uint32_t idesc, uint32_t acc0,
                                          const uint32_t (&jy16)[4], const uint32_t (&jx8)[4]) {
    const uint32_t pitch = a_hi & 0x3fffu;           // plane row pitch in 16-byte units (the descriptor's SBO)
    uint32_t joff[NACC];
#pragma unroll
    for (int j = 0; j < NACC; ++j) joff[j] = jy16[j] * pitch + jx8[j];
#pragma unroll
    for (int k2 = 0; k2 < BK / 16; ++k2)
#pragma unroll
        for (int j = 0; j < NACC; ++j)      // consecutive MMAs target different accumulators
            tc_mma2(d_base + (uint32_t)j * bn, a_lo + joff[j] + (uint32_t)k2 * a_kstep, a_hi, b_lo + (uint32_t)k2 * b_kstep, b_hi,
                    idesc, k2 ? 1u : acc0);
}
// issue only; the registers are valid after tc_wait_ld(v)
__device__ __forceinline__ void tc_ld16_issue(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
// the "+r" operands tie every later use of v to this wait (the compiler may not hoist them above it)
__device__ __forceinline__ void tc_wait_ld(uint32_t (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                   "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :
                 : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// opaque register copy: stops ptxas from re-reading a kernel parameter from the constant bank inside hot loops (with a
// ~200 KB shared-memory carve-out an LDC / local-memory access costs hundreds of cycles there)
// An empty asm() does not do it: it vanishes in the PTX and ptxas re-materialises the ld.param as LDC at every use.  Adding
// a zero ptxas cannot prove to be zero (%smid >> 31, read once per thread) makes the value a computed one that stays in a
// register.
__device__ __forceinline__ uint32_t opaque_zero() { uint32_t s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); return s >> 31; }
__device__ __forceinline__ int keep_(int x, uint32_t kz) { return x + (int)kz; }
__device__ __forceinline__ uint32_t keep_(uint32_t x, uint32_t kz) { return x + kz; }
#define keep(x) keep_((x), kz)
__device__ __forceinline__ void st_global_v8(void *p, const uint32_t (&o)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]),
                 "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7])
                 : "memory");
}
__device__ __forceinline__ void ld_global_v8(const void *p, uint32_t (&o)[8]) {
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(o[0]), "=r"(o[1]), "=r"(o[2]), "=r"(o[3]), "=r"(o[4]), "=r"(o[5]), "=r"(o[6]), "=r"(o[7])
                 : "l"(p));
}

// role timers (development aid): accumulate clock64() deltas only when P.dbg is set
#ifdef RDFC_UMMA_TIMERS       // compile-time: the 64-bit accumulators cost registers in every role
#define DBG_ON (P.dbg != nullptr)
#else
#define DBG_ON false
#endif
#define DBG_T0() const long long _t0 = DBG_ON ? clock64() : 0
#define DBG_ACC(var) if (DBG_ON) var += clock64() - _t0

// kGeneral = false: the hot variant (bf16 NHWC output, act in {none, ReLU, LeakyReLU}); true adds tanh / sigmoid, partial
// channel steps, unaligned slices and fp32 output, whose code would otherwise cost the hot epilogue registers.
// kMode = MODE_WADAIN: W-AdaIN epilogue over [gamma | beta] column tiles.  kMode = MODE_HEADS: the decode heads as ONE
// 1x1 GEMM to 9 * ncols columns (tap-major) over overlapping 16x16 pixel regions + a shift-add through shared memory.
enum { MODE_STD = 0, MODE_GENERAL = 1, MODE_WADAIN = 2, MODE_HEADS = 3 };
template <int kMode>
__global__ void __launch_bounds__(NTHREADS, 1) conv_umma_kernel(const __grid_constant__ Params P) {
    constexpr bool kGeneral = kMode == MODE_GENERAL;
    extern __shared__ __align__(1024) unsigned char smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Programmatic dependent launch (host: cudaLaunchAttributeProgrammaticStreamSerialization): the next kernel of the stream
    // may take this CTA's SM as soon as it exits and run its own setup / filter loads; every role that touches activations
    // (A producers, epilogue) executes griddepcontrol.wait first, i.e. waits for the preceding grid to complete and flush.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const long long t_kernel0 = DBG_ON ? clock64() : 0;
    if (DBG_ON && threadIdx.x == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); P.dbg[blockIdx.x * 16 + 15] = (long long)gt; }
    const int a_stage_bytes = P.a_tma ? P.nplanes * P.a_plane_bytes : KCH * P.npix_pad * 16;
    const int b_tap_bytes = KCH * P.bn * 16, b_stage_bytes = P.gtaps * b_tap_bytes;
    const int tile0 = blockIdx.x, tile_step = gridDim.x;
    // stages start on a 1 KB boundary (the SWIZZLE_64B pattern the TMA writes repeats every 1 KB; the host adds the slack)
    unsigned char *sA = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);
    unsigned char *sB = sA + (size_t)P.sa * a_stage_bytes;
    // epilogue staging (tma_out): [2 groups][2 buffers] output slabs, then [2 groups][2 buffers] residual slabs; 1 KB aligned
    // because every stage size is a multiple of 1 KB
    unsigned char *sE = sB + (size_t)P.sb * b_stage_bytes;
    const int epi_bytes = P.tma_out ? (P.res ? 8 : 4) * EPI_SLAB_BYTES : 0;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sE + epi_bytes);
    // barrier map: a_full[sa] a_empty[sa] b_full[sb] b_empty[sb] acc_full[2] acc_empty[2]
    const uint32_t bar0 = smem_u32(bars);
    auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
    const uint32_t kz = opaque_zero();
    const int sa_k = keep(P.sa), sb_k = keep(P.sb);
    const int A_FULL = 0, A_EMPTY = sa_k, B_FULL = 2 * sa_k, B_EMPTY = B_FULL + sb_k, ACC_FULL = B_EMPTY + sb_k,
              ACC_EMPTY = ACC_FULL + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + ACC_EMPTY + 2);
    const int RES_FULL = ACC_EMPTY + 3;               // [group][buffer]: a residual slab has landed
    // per-channel epilogue vectors, padded to CoutP with (1, 0): 16-byte aligned after the barrier block
    float *s_scale = reinterpret_cast<float *>(sE + epi_bytes + BAR_BYTES);
    float *s_shift = s_scale + P.CoutP;
    uint2 *s_tap = reinterpret_cast<uint2 *>(s_shift + P.CoutP);      // [phase][tap] A-descriptor words (lo, hi)
    float *s_stat = reinterpret_cast<float *>(s_tap + 4 * MAX_TAPS);   // W-AdaIN: mean[C], rstd[C] of the current image; stem: input patch;
                                                                       // shift-add heads: Y[256 region pixels][bn + 1] fp32
    if (threadIdx.x < 4 * MAX_TAPS)
        s_tap[threadIdx.x] = make_uint2(P.tap_alo[threadIdx.x / MAX_TAPS][threadIdx.x % MAX_TAPS],
                                        P.tap_ahi[threadIdx.x / MAX_TAPS][threadIdx.x % MAX_TAPS]);
    for (int i = threadIdx.x; i < P.CoutP; i += NTHREADS) {
        // times the exact inverse of a scaled split's factor (a power of two)
        s_scale[i] = ((P.scale && i < P.Cout) ? P.scale[i] : 1.f) * (P.split_factor ? __frcp_rn(__ldg(P.split_factor)) : 1.f);
        s_shift[i] = (P.shift && i < P.Cout) ? P.shift[i] : 0.f;
    }

    // ---- one-time setup
    if (threadIdx.x == 0) {
        const int nissue = P.dual ? 2 : 1;           // every issuer commits on the "empty" / "accumulator full" barriers
        for (int i = 0; i < P.sa; ++i) { mbar_init(BAR(A_FULL + i), P.a_tma ? 1 : NPROD); mbar_init(BAR(A_EMPTY + i), nissue); }
        for (int i = 0; i < P.sb; ++i) { mbar_init(BAR(B_FULL + i), 1); mbar_init(BAR(B_EMPTY + i), nissue); }
        for (int i = 0; i < 2; ++i) { mbar_init(BAR(ACC_FULL + i), nissue); mbar_init(BAR(ACC_EMPTY + i), NEPI_WARPS); }
        for (int i = 0; i < 4; ++i) mbar_init(BAR(RES_FULL + i), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)P.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int set_cols = P.nacc * P.bn;

    const bool mma_role = warp == MMA_WARP || (warp == MMA2_WARP && P.dual);
    if (mma_role) {
        // ================= MMA issuer =================
        // Measured (RDFC_UMMA_SKIP=4, every MMA issued with N = 16): the loop costs ~80 cycles per MMA in the issuing warp
        // whatever N is -- R2UR moves of the descriptor words and the UTCHMMA issue itself -- so one issuer caps every
        // layer with N <= 128.  With P.dual two warps on different schedulers issue disjoint halves of the accumulators of a
        // tile (MMAs into different TMEM columns are independent); both commit on the same barriers (count 2).
        // The whole warp walks the loop convergently (barrier waits, ring bookkeeping); one elected lane issues.  Per
        // MMA the issue cost is one 32-bit add on a descriptor word; the per-tap descriptor words come from the
        // shared-memory table and are fetched before the wait on the filter stage.
        // instruction descriptor: bf16 x bf16 -> fp32, N = bn, M = 128
#ifdef RDFC_UMMA_TIMERS
        // RDFC_UMMA_SKIP & 4: issue every MMA with N = 16 (wrong results): is the loop bound by issue or by the tensor pipe?
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(((P.dbg_flags & 4) ? 16 : P.bn) >> 3) << 17) | (8u << 24);
#else
        // operand format: bf16 (1), or fp16 (0) for the split fp32-faithful mode (11 + 11 mantissa bits per operand)
        const uint32_t fmt = P.split_c ? 0u : 1u;
        const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(P.bn >> 3) << 17) | (8u << 24);
#endif
        // one k-step = 16 channels: two chunk planes further in the [cin/8][pixel][16 B] layout, 32 bytes in [pixel][64 B]
        const uint32_t a_kstep = keep(P.a_tma ? 2u : 2u * (uint32_t)P.npix_pad), b_kstep = keep(2u * (uint32_t)P.bn);
        const uint32_t b_hi = (128u >> 4) | (1u << 14);                                     // SBO = 128 B, version bit 46
        const uint32_t b_lo0 = keep(((smem_u32(sB) & 0x3FFFFu) >> 4) | ((uint32_t)P.bn << 16));    // LBO = staged rows * 16 B
        const uint32_t a_lo0 = keep((smem_u32(sA) & 0x3FFFFu) >> 4);
        const uint32_t a_stage16 = keep((uint32_t)a_stage_bytes >> 4), b_stage16 = keep((uint32_t)b_stage_bytes >> 4);
        const uint32_t b_tap16 = keep((uint32_t)b_tap_bytes >> 4);
        const uint32_t bn = keep((uint32_t)P.bn);
        const int nax = keep(P.nax), sa_n = keep(P.sa), sb_n = keep(P.sb), nkb = keep(P.nkb), gtaps = keep(P.gtaps);
        const int nsets = keep(P.nsets), gt3 = keep(P.gtaps < 3 ? P.gtaps : 3);
        // this issuer's accumulators: [jb, jb + nacc) of the tile's P.nacc
        const int jb = keep(warp == MMA_WARP ? 0 : (P.nacc + 1) / 2);
        const int nacc = keep(P.dual ? (warp == MMA_WARP ? (P.nacc + 1) / 2 : P.nacc / 2) : P.nacc);
        uint32_t jy16[4], jx8[4];                  // accumulator j: 16 * (rows down) and 8 * (blocks across), decoded once
#pragma unroll
        for (int j = 0; j < 4; ++j) { jy16[j] = keep(16u * (uint32_t)((j + jb) / nax)); jx8[j] = keep(8u * (uint32_t)P.px16 * (uint32_t)((j + jb) % nax)); }
        // one accumulator, 9-tap stages, TMA operands: the stage is one asm statement over register-resident tap words
        const bool fast9 = keep(P.fast9) != 0;
        uint32_t tlo9[9], thi9 = 0;
#pragma unroll
        for (int q = 0; q < 9; ++q) tlo9[q] = 0;
        if (fast9) {
#pragma unroll
            for (int q = 0; q < 9; ++q) tlo9[q] = keep(P.tap_alo[0][q]);
            thi9 = keep(P.tap_ahi[0][0]);
        }
        int s = 0, sb = 0, it = 0;
        uint32_t a_par = 0, b_par = 0;
        long long t_acc = 0, t_a = 0, t_b = 0, t_mma = 0, t_commit = 0;
        const long long t_start = DBG_ON ? clock64() : 0;
        for (int tile = tile0; tile < P.ntiles; tile += tile_step, ++it) {
            const Tile t = decode_tile(P, tile);
            const int z = t.z, ngroups = P.ntaps[z] / gtaps;
            const uint2 *ztap = s_tap + z * MAX_TAPS;
            const int set = nsets == 2 ? (it & 1) : 0;
            const int use = nsets == 2 ? (it >> 1) : it;          // how often this set has been used before
            { DBG_T0(); mbar_wait(BAR(ACC_EMPTY + set), (use & 1) ^ 1); DBG_ACC(t_acc); }   // epilogue has drained this set
            tc_fence_after();
            const uint32_t d_base = tmem_base + (uint32_t)(set * set_cols) + (uint32_t)jb * bn;
            for (int i = 0; i < nkb; ++i) {
                { DBG_T0(); mbar_wait(BAR(A_FULL + s), a_par); DBG_ACC(t_a); }
                const uint32_t a_stage_lo = a_lo0 + (uint32_t)s * a_stage16;
                for (int gi = 0; gi < ngroups; ++gi) {
                    const uint32_t b_lo = b_lo0 + (uint32_t)sb * b_stage16;
                    { DBG_T0(); mbar_wait(BAR(B_FULL + sb), b_par); DBG_ACC(t_b); }
                    tc_fence_after();
                    if (elect_one()) {
                        const long long _tm0 = DBG_ON ? clock64() : 0;
                        if (fast9) {
                            tc_mma_stage9(d_base, tlo9, a_stage_lo, thi9, b_lo, b_hi, idesc, (i | gi) ? 1u : 0u, b_tap16, a_kstep, b_kstep);
                        } else
                        for (int r3 = 0; r3 < gtaps; r3 += 3) {        // a stage holds 1, 2, 3 or 9 taps: up to three at a time
                        uint2 td[3];
#pragma unroll
                        for (int tg = 0; tg < 3; ++tg) td[tg] = ztap[gi * gtaps + r3 + (tg < gt3 ? tg : 0)];
#pragma unroll
                        for (int tg = 0; tg < 3; ++tg) {
                            if (tg < gt3) {
                                const uint32_t acc0 = (i | gi | r3 | tg) ? 1u : 0u;
                                const uint32_t a_lo = td[tg].x + a_stage_lo, a_hi = td[tg].y, bl = b_lo + (uint32_t)(r3 + tg) * b_tap16;
                                switch (nacc) {
                                    case 1:
                                        issue_tap<1>(d_base, bn, a_lo, a_hi, a_kstep, bl, b_hi, b_kstep, idesc, acc0, jy16, jx8);
                                        break;
                                    case 2:
                                        issue_tap<2>(d_base, bn, a_lo, a_hi, a_kstep, bl, b_hi, b_kstep, idesc, acc0, jy16, jx8);
                                        break;
                                    case 3:
                                        issue_tap<3>(d_base, bn, a_lo, a_hi, a_kstep, bl, b_hi, b_kstep, idesc, acc0, jy16, jx8);
                                        break;
                                    default:
                                        issue_tap<4>(d_base, bn, a_lo, a_hi, a_kstep, bl, b_hi, b_kstep, idesc, acc0, jy16, jx8);
                                        break;
                                }
                            }
                        }
                        }
                        const long long _tm1 = DBG_ON ? clock64() : 0;
                        tc_commit(BAR(B_EMPTY + sb));
                        if (gi == ngroups - 1) {
                            tc_commit(BAR(A_EMPTY + s));
                            if (i == nkb - 1) tc_commit(BAR(ACC_FULL + set));
                        }
                        if (DBG_ON) { const long long _tm2 = clock64(); t_mma += _tm1 - _tm0; t_commit += _tm2 - _tm1; }
                    }
                    __syncwarp();
                    if (++sb == sb_n) { sb = 0; b_par ^= 1u; }
                }
                if (++s == sa_n) { s = 0; a_par ^= 1u; }
            }
        }
        if (DBG_ON && lane == 0 && warp == MMA_WARP) {
            long long *o = P.dbg + blockIdx.x * 16;
            o[0] = clock64() - t_start; o[1] = t_acc; o[2] = t_a; o[3] = t_b;
        }
        if (DBG_ON && warp == MMA_WARP) {            // the elected lane's own counters (it is not necessarily lane 0)
            const long long m = t_mma, c = t_commit;
            if (m | c) { P.dbg[blockIdx.x * 16 + 11] = m; P.dbg[blockIdx.x * 16 + 12] = c; }
        }
    } else if (warp < NPROD_WARPS && P.a_tma) {
        // ================= A producer, TMA mode: one elected thread =================
        // Per k-block and plane ONE cp.async.bulk.tensor: box = 32 channels x plane columns x plane rows of the NHWC
        // input, SWIZZLE_64B into [pixel][64 B]; coordinates outside the image are zero-filled (= the conv padding).
        // cp.async staging tops out at ~6 B/cycle/SM (L1 miss tracking x L2 latency); the TMA engine does not.
        if (threadIdx.x == 0) {
            asm volatile("griddepcontrol.wait;" ::: "memory");
            const int nkb = P.nkb, sa_n = P.sa, npl = P.nplanes;
            const uint32_t sA0 = smem_u32(sA), plane_b = (uint32_t)P.a_plane_bytes;
            int s = 0;
            uint32_t par = 1;
            for (int tile = tile0; tile < P.ntiles; tile += tile_step) {
                const Tile t = decode_tile(P, tile);
                for (int i = 0; i < nkb; ++i) {
                    mbar_wait(BAR(A_EMPTY + s), par);
                    const uint32_t full = BAR(A_FULL + s);
#ifdef RDFC_UMMA_TIMERS
                    // RDFC_UMMA_SKIP & 8: stage nothing (wrong results): what do the TMA writes cost the tensor pipe?
                    if (P.dbg_flags & 8) { mbar_arrive(full); if (++s == sa_n) { s = 0; par ^= 1u; } continue; }
#endif
                    mbar_expect_tx(full, (uint32_t)P.a_tx_bytes);
                    // input channel of k-block i: plain convs walk the channels; split inputs walk hi, hi again, then lo
                    int a_ch = i * BK * P.kbs;
                    if (P.split_c) a_ch = a_ch < P.split_c ? a_ch : (a_ch < 2 * P.split_c ? a_ch - P.split_c : a_ch - P.split_c);
                    for (int pl = 0; pl < npl; ++pl) {
                        const Plane &q = P.planes[pl];
                        asm volatile(
                            "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
                                sA0 + (uint32_t)s * (uint32_t)a_stage_bytes + (uint32_t)pl * plane_b),
                            "l"(&P.tmap_a), "r"(a_ch + (P.kbs > 1 ? pl * BK : 0)), "r"(q.xstep * t.tx0 + q.xoff), "r"(q.ystep * t.ty0 + q.yoff), "r"(t.b), "r"(full)
                            : "memory");
                    }
                    if (++s == sa_n) { s = 0; par ^= 1u; }
                }
            }
        }
    } else if (warp < NPROD_WARPS) {
        // ================= A producers, stem mode =================
        // The "input" of the 1x1 GEMM is the im2col matrix of the 3x3 stems, built on the fly: slot (pixel p, chunk ch)
        // of k-block i holds rows k = 32 i + 8 ch .. + 8, row k = (channel k / 9, tap k % 9).  Per tile the producers
        // first stage the fp32 input patch (all channels, tile + 1-pixel halo, zeros outside the image) in shared
        // memory, so a row is one LDS at a per-thread constant offset: no bounds tests, no L2 round trip per slot.
        asm volatile("griddepcontrol.wait;" ::: "memory");
        const int ch = threadIdx.x & 3, p0 = threadIdx.x >> 2;
        const int Hi = P.Hi, Wi = P.Wi, TWs = 8 * P.nax, THs = TH * (P.nacc / P.nax), nj = (P.npix + PIXPASS - 1) / PIXPASS;
        const int PW = TWs + 2, PH = THs + 2, nch = P.stem_k / 9, plane_sz = PH * PW, tw_shift = 31 - __clz(TWs);
        const long long HW = (long long)Hi * Wi;
        float *patch = s_stat + 2 * P.wad_C;                     // [nch][PH][PW] + one zero cell
        const int zero_cell = nch * plane_sz;
        int delta[2][8];            // patch offset of row k relative to the slot's centre cell (r + 1, c + 1) of plane 0
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int k = 32 * i + 8 * ch + e;
                if (k < P.stem_k) {
                    const int ci = k / 9, tp = k - 9 * ci;
                    delta[i][e] = ci * plane_sz + (tp / 3 - 1) * PW + (tp % 3 - 1);
                } else {
                    delta[i][e] = INT_MIN;
                }
            }
        const uint32_t dst_thread = smem_u32(sA) + (uint32_t)(ch * P.npix_pad + p0) * 16u;
        // The patch is double-buffered: the 4-byte cp.asyncs of tile n+1 (zero-fill outside the image; every cell of a thread
        // in flight at once) are issued before tile n's slots are built, so the L2 round trip of the fill -- ~2000 cycles,
        // as long as building a whole tile -- is off the critical path.
        const int patch_stride = nch * plane_sz + 4;               // floats per buffer: cells, the zero cell, padding
        auto fill_patch = [&](int tile, int buf) {
            const Tile t = decode_tile(P, tile);
            const float *b0 = P.stem_in0 + (long long)t.b * P.stem_c0 * HW;
            const float *b1 = P.stem_in1 ? P.stem_in1 + (long long)t.b * HW : b0;
            const uint32_t patch_s = smem_u32(patch + buf * patch_stride);
            int pr = threadIdx.x / PW, pc = threadIdx.x - pr * PW;       // flat cell index = pr * PW + pc, pr over nch * PH rows
            const int dr = NPROD / PW, dc = NPROD - dr * PW;
            for (int e = threadIdx.x; e < nch * plane_sz; e += NPROD) {
                const int ci = pr >= 3 * PH ? 3 : (pr >= 2 * PH ? 2 : (pr >= PH ? 1 : 0));    // nch <= 4 here (asserted on the host)
                const int iy = t.ty0 + (pr - ci * PH) - 1, ix = t.tx0 + pc - 1;
                const bool ok = iy >= 0 && iy < Hi && ix >= 0 && ix < Wi;
                const float *src = ok ? (ci < P.stem_c0 ? b0 + (long long)ci * HW : b1) + (long long)iy * Wi + ix : b0;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(patch_s + 4u * (uint32_t)e), "l"(src), "r"(ok ? 4u : 0u) : "memory");
                pr += dr; pc += dc;
                if (pc >= PW) { pc -= PW; ++pr; }
            }
        };
        if (tile0 < P.ntiles) fill_patch(tile0, 0);
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (threadIdx.x == 0) patch[zero_cell] = patch[patch_stride + zero_cell] = 0.f;      // never touched by the fills
        int s = 0, it = 0;
        uint32_t par = 1;
        for (int tile = tile0; tile < P.ntiles; tile += tile_step, ++it) {
            asm volatile("bar.sync 3, %0;" ::"n"(NPROD) : "memory");          // the previous tile's slots are built: its buffer is free
            if (tile + tile_step < P.ntiles) fill_patch(tile + tile_step, (it + 1) & 1);
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 1;" ::: "memory");               // this tile's patch has landed (my cells) ...
            asm volatile("bar.sync 3, %0;" ::"n"(NPROD) : "memory");          // ... and everyone else's
            const float *pb = patch + (it & 1) * patch_stride;
            for (int i = 0; i < P.nkb; ++i) {
                mbar_wait(BAR(A_EMPTY + s), par);
                const uint32_t dst = dst_thread + (uint32_t)s * (uint32_t)a_stage_bytes;
                for (int j = 0; j < nj; ++j) {
                    const int p = j * PIXPASS + p0;
                    if (p >= P.npix) break;
                    const int centre = ((p >> tw_shift) + 1) * PW + (p & (TWs - 1)) + 1;      // TWs is 8, 16 or 32
                    float v[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int dl = i == 0 ? delta[0][e] : delta[1][e];
                        v[e] = pb[dl == INT_MIN ? zero_cell : centre + dl];
                    }
                    uint32_t w[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
                        w[e] = *reinterpret_cast<const uint32_t *>(&h2);
                    }
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + (uint32_t)j * (uint32_t)(PIXPASS * 16)),
                                 "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3])
                                 : "memory");
                }
                fence_proxy_async();              // generic-proxy stores -> visible to the tensor core (async proxy)
                mbar_arrive(BAR(A_FULL + s));
                if (++s == P.sa) { s = 0; par ^= 1u; }
            }
        }
    } else if (warp == BLOAD_WARP) {
        // ================= B loader (TMA 1-D bulk copies of pre-packed filter blocks) =================
        // The warp walks the ring convergently; lane 0 posts the byte count, then every lane issues its share of the stage's
        // copies.  A 9-tap stage of a filter view that is not contiguous over the k-block is 36 copies of ~1 KB; issued by one
        // thread they took as long as the MMAs of the stage (measured with CTA pairs).
        {
            const uint32_t piece = keep((uint32_t)P.bn * 16u);            // one cin chunk of the tile's filter rows
            const long long chunk_stride = (long long)P.CoutP * 8;
            const uint32_t sB0 = smem_u32(sB);
            const int sb_n = keep(P.sb), nkb = keep(P.nkb), gtaps = keep(P.gtaps), b_contig = keep(P.b_contig);
            int sb = 0;
            uint32_t par = 1;
            long long t_be = 0;
            for (int tile = tile0; tile < P.ntiles; tile += tile_step) {
                const Tile t = decode_tile(P, tile);
                const int z = t.z, ngroups = P.ntaps[z] / gtaps;
                const __nv_bfloat16 *w_n0 = P.w + (long long)t.n0 * 8;
                for (int i = 0; i < nkb; ++i, w_n0 += P.w_kb_stride)
                    for (int gi = 0; gi < ngroups; ++gi) {
                        const uint32_t dst = sB0 + (uint32_t)sb * (uint32_t)b_stage_bytes;
                        { DBG_T0(); mbar_wait(BAR(B_EMPTY + sb), par); DBG_ACC(t_be); }
                        const uint32_t full = BAR(B_FULL + sb);
#ifdef RDFC_UMMA_TIMERS
                        if (P.dbg_flags & 16) { if (lane == 0) mbar_arrive(full); if (++sb == sb_n) { sb = 0; par ^= 1u; } continue; }   // no filter loads
#endif
                        if (lane == 0) mbar_expect_tx(full, (uint32_t)b_stage_bytes);
                        __syncwarp();
                        if (b_contig) {
                            for (int tg = lane; tg < gtaps; tg += 32)
                                bulk_g2s(dst + (uint32_t)tg * (uint32_t)b_tap_bytes, w_n0 + P.tap_w[z][gi * gtaps + tg], piece * KCH, full);
                        } else {
                            for (int q = lane; q < gtaps * KCH; q += 32) {
                                const int tg = q / KCH, ch = q - tg * KCH;
                                bulk_g2s(dst + (uint32_t)tg * (uint32_t)b_tap_bytes + (uint32_t)ch * piece,
                                         w_n0 + P.tap_w[z][gi * gtaps + tg] + ch * chunk_stride, piece, full);
                            }
                        }
                        if (++sb == sb_n) { sb = 0; par ^= 1u; }
                    }
            }
            if (DBG_ON && lane == 0) P.dbg[blockIdx.x * 16 + 5] = t_be;
        }
        __syncwarp();
    } else {
        // ================= epilogue (warps 8..15): warp w reads TMEM lanes 32*(w%4).., group (w-8)/4 takes every
        // other accumulator.  y = act(acc*scale + shift + residual) -> bf16 NHWC slice, or fp32 planes (heads).
        // 16 columns per step, software-pipelined: the tcgen05.ld and the residual load of step g+1 are in flight
        // while step g is computed and stored; (scale, shift) come from shared memory (the L1 left beside a 200 KB
        // carve-out is too small to keep them: every __ldg was an L2 round trip).
        asm volatile("griddepcontrol.wait;" ::: "memory");       // before the first residual / statistics read and the first store
        const int wq = warp & 3, grp = (warp - EPI_WARP0) >> 2;
        const int r = 4 * wq + (lane >> 3), c = lane & 7;     // MMA row m = 32*wq + lane = 8*r + c
        const int bn = P.bn, Cout = P.Cout, out_stride = P.out_stride, res_stride = P.res_stride;
        // bit 1 vec32, bits 2.. development skip flags: one register for the inner-loop switches
        const int flags = (P.vec32 ? 2 : 0) | (P.dbg_flags << 2);
        const int act = P.act, nacc = P.nacc, nax = P.nax, nsets = P.nsets;
        const int Ht = P.Ht, Wt = P.Wt, Ho = P.Ho, Wo = P.Wo, oys = P.oys, oxs = P.oxs;
#define vec32 (kMode == MODE_STD || (flags & 2))      // MODE_STD: the host guarantees 32-byte aligned slices and Cout % 16 == 0
#define skip (flags >> 2)
        const float slope = act == RDFC_ACT_RELU ? 0.f : (act == RDFC_ACT_LEAKY02 ? 0.2f : 1.f);
        const __nv_bfloat16 *res = (kGeneral && P.out_f32) ? nullptr : P.res;            // fp32 mode: the residual is read as floats below
        const float *res32 = (kGeneral && P.out_f32) ? reinterpret_cast<const float *>(P.res) : nullptr;
        __nv_bfloat16 *const outp = P.out;
        const int G = bn >> 4;
        int it = 0, wad_b = -1;
        long long t_accfull = 0, t_epi = 0;
        // TMA epilogue (P.tma_out): per group of 4 warps (= one accumulator of 128 pixels at a time) two output slab buffers
        // and two residual slab buffers, indexed by a slab counter that runs across accumulators and tiles.  My pixel's row in
        // a slab is m = 32 wq + lane ([m][64 B]); SWIZZLE_64B puts 16-byte chunk k at position k ^ ((m >> 1) & 3), which also
        // makes the 16-byte shared-memory accesses of a quarter warp conflict-free.
        const bool tma_epi = kMode == MODE_STD && P.tma_out;
        const uint32_t ebuf = smem_u32(sE) + (uint32_t)grp * 2u * EPI_SLAB_BYTES;
        const uint32_t rbuf = smem_u32(sE) + 4u * EPI_SLAB_BYTES + (uint32_t)grp * 2u * EPI_SLAB_BYTES;
        const bool leader = wq == 0 && lane == 0;
        const uint32_t row_off = (uint32_t)(32 * wq + lane) * 64u, swz = (uint32_t)(((32 * wq + lane) >> 1) & 3);
        uint32_t ctr = 0;
        if (tma_epi) {
            for (int tile = tile0; tile < P.ntiles; tile += tile_step, ++it) {
                const Tile t = decode_tile(P, tile);
                const int oyo = P.oyo[t.z], oxo = P.oxo[t.z];
                const int set = nsets == 2 ? (it & 1) : 0;
                const int use = nsets == 2 ? (it >> 1) : it;
                const long long _te = DBG_ON ? clock64() : 0;
                // ---- epilogue through shared memory + TMA: per 32-channel slab of an accumulator
                //   TMEM -> registers -> y = act(acc*scale + shift + residual slab) -> bf16 slab in shared memory -> one
                //   cp.async.bulk.tensor store of the 8 x 16 pixel box (the TMA unit clips pixels / channels outside the tensor).
                // Slab `ctr` uses buffers ctr & 1.  Before the group barrier of slab ctr the leader has waited until the store of
                // slab ctr - 1 has read its buffer, so after the barrier buffer (ctr + 1) & 1 is free for the next slab; the
                // residual slab of ctr + 2 is requested after the barrier (everybody has read slab ctr's residual by then).
                const int nslab = bn >> 5, nitems = ((nacc - grp + 1) >> 1) * nslab;
                auto coords = [&](int q, int &c0, int &x, int &y) {
                    const int j = grp + 2 * (q / nslab), sl = q - (q / nslab) * nslab;
                    c0 = t.n0 + 32 * sl; x = oxs * (t.tx0 + 8 * (j % nax)) + oxo; y = oys * (t.ty0 + 16 * (j / nax)) + oyo;
                };
                auto issue_res = [&](int q, uint32_t cq) {           // leader only
                    int c0, x, y;
                    coords(q, c0, x, y);
                    const uint32_t bar = BAR(RES_FULL + 2 * grp + (int)(cq & 1u));
                    mbar_expect_tx(bar, (uint32_t)EPI_SLAB_BYTES);
                    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
                                     rbuf + (cq & 1u) * (uint32_t)EPI_SLAB_BYTES),
                                 "l"(&P.tmap_res), "r"(c0), "r"(x), "r"(y), "r"(t.b), "r"(bar)
                                 : "memory");
                };
                // this tile's first two residual slabs do not depend on the MMAs: request them before waiting for the accumulators
                // (every lane of the group is past the previous tile's last barrier, i.e. done reading the residual buffers)
                if (res && leader) {
                    if (nitems > 0) issue_res(0, ctr);
                    if (nitems > 1) issue_res(1, ctr + 1);
                }
                { DBG_T0(); mbar_wait<true>(BAR(ACC_FULL + set), use & 1); DBG_ACC(t_accfull); }
                tc_fence_after();
                for (int q = 0; q < nitems; ++q, ++ctr) {
                    const int j = grp + 2 * (q / nslab), sl = q - (q / nslab) * nslab;
                    const uint32_t trow = tmem_base + ((uint32_t)(32 * wq) << 16) + (uint32_t)(set * set_cols + j * bn + 32 * sl);
                    uint32_t va[16], vb[16];
                    tc_ld16_issue(trow, va);
                    tc_ld16_issue(trow + 16u, vb);
                    const uint32_t eb = ebuf + (ctr & 1u) * (uint32_t)EPI_SLAB_BYTES + row_off;
                    const uint32_t rb = rbuf + (ctr & 1u) * (uint32_t)EPI_SLAB_BYTES + row_off;
                    if (res) mbar_wait(BAR(RES_FULL + 2 * grp + (int)(ctr & 1u)), (ctr >> 1) & 1u);
                    tc_wait_ld(va);
                    tc_wait_ld(vb);
                    const int nb = t.n0 + 32 * sl;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {                    // 16 channels = two 16-byte chunks
                        const uint32_t (&v)[16] = h ? vb : va;
                        float f[16];
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) {
                            const float4 sc = *reinterpret_cast<const float4 *>(s_scale + nb + 16 * h + 4 * q4);
                            const float4 sh = *reinterpret_cast<const float4 *>(s_shift + nb + 16 * h + 4 * q4);
                            f[4 * q4 + 0] = fmaf(__uint_as_float(v[4 * q4 + 0]), sc.x, sh.x);
                            f[4 * q4 + 1] = fmaf(__uint_as_float(v[4 * q4 + 1]), sc.y, sh.y);
                            f[4 * q4 + 2] = fmaf(__uint_as_float(v[4 * q4 + 2]), sc.z, sh.z);
                            f[4 * q4 + 3] = fmaf(__uint_as_float(v[4 * q4 + 3]), sc.w, sh.w);
                        }
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            const uint32_t chunk = ((uint32_t)(2 * h + k) ^ swz) << 4;
                            if (res) {
                                uint32_t rr[4];
                                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rr[0]), "=r"(rr[1]), "=r"(rr[2]), "=r"(rr[3]) : "r"(rb + chunk));
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const float2 p2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&rr[e]));
                                    f[8 * k + 2 * e] += p2.x;
                                    f[8 * k + 2 * e + 1] += p2.y;
                                }
                            }
                            uint32_t o[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const float y0 = f[8 * k + 2 * e], y1 = f[8 * k + 2 * e + 1];
                                const __nv_bfloat162 h2 = __floats2bfloat162_rn(fmaxf(y0, slope * y0), fmaxf(y1, slope * y1));
                                o[e] = *reinterpret_cast<const uint32_t *>(&h2);
                            }
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(eb + chunk), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
                        }
                    }
                    fence_proxy_async();                              // my slab rows -> visible to the TMA unit
                    if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");       // store ctr - 1 has read its buffer
                    if (grp == 0) asm volatile("bar.sync 4, 128;" ::: "memory"); else asm volatile("bar.sync 5, 128;" ::: "memory");
                    if (leader) {
                        int c0, x, y;
                        coords(q, c0, x, y);
                        asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4}], [%5];" ::"l"(&P.tmap_out),
                                     "r"(c0), "r"(x), "r"(y), "r"(t.b), "r"(ebuf + (ctr & 1u) * (uint32_t)EPI_SLAB_BYTES)
                                     : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        if (res && q + 2 < nitems) issue_res(q + 2, ctr + 2);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + set));
                if (DBG_ON) t_epi += clock64() - _te;
            }
            if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // my stores have been written
        } else
        for (int tile = tile0; tile < P.ntiles; tile += tile_step, ++it) {
            const Tile t = decode_tile(P, tile);
            const int oyo = P.oyo[t.z], oxo = P.oxo[t.z];
            const int set = nsets == 2 ? (it & 1) : 0;
            const int use = nsets == 2 ? (it >> 1) : it;
            const long long _te = DBG_ON ? clock64() : 0;
            { DBG_T0(); mbar_wait<true>(BAR(ACC_FULL + set), use & 1); DBG_ACC(t_accfull); }
            tc_fence_after();
            if (kMode == MODE_HEADS) {
                // ---- decode heads (rdf_generator.py:372-398), shift-add form.  The GEMM gave Y[p, t * ncols + q] =
                // W_t[q, :] . X[p, :] for the 16 x 16 pixel region; head q at pixel p is act(bias_q + sum_t Y[p + d_t, t, q]).
                // Regions overlap by 2 pixels: a region produces its inner 14 x 14 outputs (zero padding = Y of the
                // zero-filled pixels outside the image).
                float *Ys = s_stat;
                const int pitch = bn + 1, ncols = P.ncols;
                const int prow = (4 * wq + (lane >> 3)) * 16 + 8 * grp + (lane & 7);        // nacc == 2, nax == 2: j = grp
                const uint32_t trow = tmem_base + ((uint32_t)(32 * wq) << 16) + (uint32_t)(set * set_cols + grp * bn);
                asm volatile("bar.sync 2, %0;" ::"n"(NEPI_WARPS * 32) : "memory");          // previous region's sums are done with Ys
                for (int g = 0; g < G; ++g) {
                    uint32_t v[16];
                    tc_ld16(trow + (uint32_t)(16 * g), v);
                    float *yp = Ys + prow * pitch + 16 * g;
#pragma unroll
                    for (int q = 0; q < 16; ++q) yp[q] = __uint_as_float(v[q]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + set));
                asm volatile("bar.sync 2, %0;" ::"n"(NEPI_WARPS * 32) : "memory");
                // a scaled split input (factor s): the taps are s times the output's, so the bias enters as bias * s and the sum
                // is multiplied by 1 / s.  Both are exact: this is bias + taps / s rounded step by step.  Without a split both are 1.
                const float fac = P.split_factor ? __ldg(P.split_factor) : 1.f, inv = __frcp_rn(fac);
                for (int item = threadIdx.x - EPI_WARP0 * 32; item < 196 * ncols; item += NEPI_WARPS * 32) {
                    const int q = item / 196, pi = item - q * 196, iy = pi / 14, ix = pi - iy * 14;
                    const int oy = t.ty0 + 1 + iy, ox = t.tx0 + 1 + ix;
                    if (oy >= Ho || ox >= Wo) continue;
                    const float *yq = Ys + (iy * 16 + ix) * pitch + q;
                    float acc = s_shift[q] * fac;
#pragma unroll
                    for (int t9 = 0; t9 < 9; ++t9) acc += yq[((t9 / 3) * 16 + (t9 % 3)) * pitch + t9 * ncols];
                    acc *= inv;
                    const int a = P.act_col[q];
                    if (a == RDFC_ACT_TANH) acc = tanhf(acc);
                    else if (a == RDFC_ACT_SIGMOID) acc = 1.f / (1.f + expf(-acc));
                    P.plane[q][(long long)t.b * P.plane_bstride[q] + (long long)oy * Wo + ox] = acc;
                }
                continue;
            }
            if (kMode == MODE_WADAIN) {
                // ---- W-AdaIN: out = (acc_g + bias_g) * (x - mean) * rstd + (acc_b + bias_b), 16 channels per step
                const int C = P.wad_C, half = bn >> 1, c0 = (t.n0 / bn) * half;
                if (t.b != wad_b) {                       // (mean, rstd) of this image -> shared memory
                    asm volatile("bar.sync 2, %0;" ::"n"(NEPI_WARPS * 32) : "memory");
                    for (int e = threadIdx.x - EPI_WARP0 * 32; e < C; e += NEPI_WARPS * 32) {
                        s_stat[e] = P.wad_mean[(long long)t.b * C + e];
                        s_stat[C + e] = P.wad_rstd[(long long)t.b * C + e];
                    }
                    asm volatile("bar.sync 2, %0;" ::"n"(NEPI_WARPS * 32) : "memory");
                    wad_b = t.b;
                }
                for (int j = grp; j < nacc; j += 2) {
                    const int yy = t.ty0 + 16 * (j / nax) + r, xx = t.tx0 + 8 * (j % nax) + c;
                    const bool ok = yy < Ht && xx < Wt;
                    const long long opix = ok ? ((long long)t.b * Ho + yy) * Wo + xx : 0;
                    const uint32_t trow = tmem_base + ((uint32_t)(32 * wq) << 16) + (uint32_t)(set * set_cols + j * bn);
                    const __nv_bfloat16 *xrow = P.wad_x + opix * P.wad_x_stride + c0;
                    const __nv_bfloat16 *wrow = P.wad_w ? P.wad_w + opix * P.wad_w_stride + c0 : nullptr;
                    __nv_bfloat16 *orow = outp + opix * out_stride + c0;
                    for (int g = 0; g < (half >> 4); ++g) {
                        uint32_t vg[16], vb[16], xr[8], gw[8], bw[8];
                        tc_ld16_issue(trow + (uint32_t)(16 * g), vg);
                        tc_ld16_issue(trow + (uint32_t)(half + 16 * g), vb);
                        if (ok) ld_global_v8(xrow + 16 * g, xr);
                        if (ok && wrow) { ld_global_v8(wrow + 16 * g, gw); ld_global_v8(wrow + C + 16 * g, bw); }
                        tc_wait_ld(vg);
                        tc_wait_ld(vb);
                        if (!ok) continue;
                        uint32_t o[8];
                        // the step's 16 means / rstds / gamma biases / beta biases as 16-byte shared-memory loads (64 scalar loads before)
                        float mu[16], rs[16], sg[16], sb[16];
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) {
                            const float4 a = *reinterpret_cast<const float4 *>(s_stat + c0 + 16 * g + 4 * q4);
                            const float4 b4 = *reinterpret_cast<const float4 *>(s_stat + C + c0 + 16 * g + 4 * q4);
                            const float4 c4 = *reinterpret_cast<const float4 *>(s_shift + t.n0 + 16 * g + 4 * q4);
                            const float4 d4 = *reinterpret_cast<const float4 *>(s_shift + t.n0 + half + 16 * g + 4 * q4);
                            mu[4 * q4] = a.x; mu[4 * q4 + 1] = a.y; mu[4 * q4 + 2] = a.z; mu[4 * q4 + 3] = a.w;
                            rs[4 * q4] = b4.x; rs[4 * q4 + 1] = b4.y; rs[4 * q4 + 2] = b4.z; rs[4 * q4 + 3] = b4.w;
                            sg[4 * q4] = c4.x; sg[4 * q4 + 1] = c4.y; sg[4 * q4 + 2] = c4.z; sg[4 * q4 + 3] = c4.w;
                            sb[4 * q4] = d4.x; sb[4 * q4 + 1] = d4.y; sb[4 * q4 + 2] = d4.z; sb[4 * q4 + 3] = d4.w;
                        }
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float2 xv = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&xr[q]));
                            const float n0v = (xv.x - mu[2 * q]) * rs[2 * q], n1v = (xv.y - mu[2 * q + 1]) * rs[2 * q + 1];
                            float g0 = __uint_as_float(vg[2 * q]) + sg[2 * q], g1 = __uint_as_float(vg[2 * q + 1]) + sg[2 * q + 1];
                            float b0 = __uint_as_float(vb[2 * q]) + sb[2 * q], b1 = __uint_as_float(vb[2 * q + 1]) + sb[2 * q + 1];
                            if (wrow) {
                                const float2 gwv = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&gw[q]));
                                const float2 bwv = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&bw[q]));
                                g0 *= gwv.x; g1 *= gwv.y; b0 *= bwv.x; b1 *= bwv.y;
                            }
                            const float y0 = fmaf(g0, n0v, b0);
                            const float y1 = fmaf(g1, n1v, b1);
                            const __nv_bfloat162 h2 = __floats2bfloat162_rn(y0, y1);
                            o[q] = *reinterpret_cast<const uint32_t *>(&h2);
                        }
                        st_global_v8(orow + 16 * g, o);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + set));
                continue;
            }
            const int n0 = t.n0;
            // one accumulator per tile: both groups of epilogue warps share it, taking alternate 16-column steps (the second group used to
            // idle).  Measured: 705 -> 697 us on the 128 -> 160 head conv -- its epilogue is busy 95 % of the time but does not bound it.
            const bool split_cols = nacc == 1 && P.epi_split;
            const int gfirst = split_cols ? grp : 0, gs = split_cols ? 2 : 1;
            for (int j = split_cols ? 0 : grp; j < nacc; j += 2) {
                const int yy = t.ty0 + 16 * (j / nax) + r, xx = t.tx0 + 8 * (j % nax) + c;
                const int oy = oys * yy + oyo, ox = oxs * xx + oxo;
                const bool ok = yy < Ht && xx < Wt && oy < Ho && ox < Wo;
                const long long opix = ok ? ((long long)t.b * Ho + oy) * Wo + ox : 0;
                const uint32_t trow = tmem_base + ((uint32_t)(32 * wq) << 16) + (uint32_t)(set * set_cols + j * bn);
                const __nv_bfloat16 *rrow = res ? res + opix * res_stride + n0 : nullptr;
                __nv_bfloat16 *orow = outp + opix * out_stride + n0;
                __nv_bfloat16 *orow2 = P.out2 ? P.out2 + opix * P.out2_stride + n0 - P.split : nullptr;

                auto load_res = [&](int g, uint4 &r0, uint4 &r1) {
                    if (rrow && ok && (kMode == MODE_STD || n0 + 16 * g + 16 <= Cout)) {
                        if (vec32) {
                            uint32_t rr[8];
                            ld_global_v8(rrow + 16 * g, rr);
                            r0 = make_uint4(rr[0], rr[1], rr[2], rr[3]); r1 = make_uint4(rr[4], rr[5], rr[6], rr[7]);
                        } else {
                            const uint4 *rp = reinterpret_cast<const uint4 *>(rrow + 16 * g);
                            r0 = rp[0]; r1 = rp[1];
                        }
                    } else {
                        r0 = r1 = make_uint4(0u, 0u, 0u, 0u);
                    }
                };
                auto process = [&](const uint32_t (&v)[16], const uint4 &r0, const uint4 &r1, int g) {
                    const int n = 16 * g;
                    if (!ok || (kMode != MODE_STD && n0 + n >= Cout)) return;
                    float f[16];
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        const float4 sc = *reinterpret_cast<const float4 *>(s_scale + n0 + n + 4 * q4);
                        const float4 sh = *reinterpret_cast<const float4 *>(s_shift + n0 + n + 4 * q4);
                        f[4 * q4 + 0] = fmaf(__uint_as_float(v[4 * q4 + 0]), sc.x, sh.x);
                        f[4 * q4 + 1] = fmaf(__uint_as_float(v[4 * q4 + 1]), sc.y, sh.y);
                        f[4 * q4 + 2] = fmaf(__uint_as_float(v[4 * q4 + 2]), sc.z, sh.z);
                        f[4 * q4 + 3] = fmaf(__uint_as_float(v[4 * q4 + 3]), sc.w, sh.w);
                    }
                    if (kGeneral && P.out_f32) {
                        // fp32-faithful mode: fp32 NHWC output (and residual), 16 channels = 64 bytes per lane
                        float *op = reinterpret_cast<float *>(P.out) + opix * out_stride + n0 + n;
                        const float *rp = res32 ? res32 + opix * res_stride + n0 + n : nullptr;
                        const int nvalid = Cout - n0 - n;
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) {
                            if (4 * q4 + 4 <= nvalid) {
                                float4 y = make_float4(f[4 * q4], f[4 * q4 + 1], f[4 * q4 + 2], f[4 * q4 + 3]);
                                if (rp) {
                                    const float4 r4 = __ldg(reinterpret_cast<const float4 *>(rp) + q4);
                                    y.x += r4.x; y.y += r4.y; y.z += r4.z; y.w += r4.w;
                                }
                                if (act <= RDFC_ACT_LEAKY02) {
                                    y.x = fmaxf(y.x, slope * y.x); y.y = fmaxf(y.y, slope * y.y); y.z = fmaxf(y.z, slope * y.z); y.w = fmaxf(y.w, slope * y.w);
                                } else {
                                    y.x = apply_act(y.x, act); y.y = apply_act(y.y, act); y.z = apply_act(y.z, act); y.w = apply_act(y.w, act);
                                }
                                reinterpret_cast<float4 *>(op)[q4] = y;
                            } else {
#pragma unroll
                                for (int e = 0; e < 4; ++e)
                                    if (4 * q4 + e < nvalid) {
                                        float y = f[4 * q4 + e] + (rp ? __ldg(rp + 4 * q4 + e) : 0.f);
                                        op[4 * q4 + e] = act <= RDFC_ACT_LEAKY02 ? fmaxf(y, slope * y) : apply_act(y, act);
                                    }
                            }
                        }
                        return;
                    }
                    const bool full = kMode == MODE_STD || n0 + n + 16 <= Cout;
                    if (res && full) {
                        const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float2 p2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&rr[q]));
                            f[2 * q] += p2.x;
                            f[2 * q + 1] += p2.y;
                        }
                    } else if (res) {
#pragma unroll
                        for (int q = 0; q < 16; ++q)
                            if (q < Cout - n0 - n) f[q] += __bfloat162float(rrow[n + q]);
                    }
                    if (!kGeneral || act <= RDFC_ACT_LEAKY02) {         // none / relu / leaky, branch-free: max(v, slope*v)
#pragma unroll
                        for (int q = 0; q < 16; ++q) f[q] = fmaxf(f[q], slope * f[q]);
                    } else {
#pragma unroll
                        for (int q = 0; q < 16; ++q) f[q] = act == RDFC_ACT_TANH ? tanhf(f[q]) : 1.f / (1.f + expf(-f[q]));
                    }
                    __nv_bfloat16 *op = (orow2 && n0 + n >= P.split ? orow2 : orow) + n;
                    if (skip & 1) return;
                    if (full) {
                        uint32_t o[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * q], f[2 * q + 1]);
                            o[q] = *reinterpret_cast<const uint32_t *>(&h2);
                        }
                        if (vec32) {
                            st_global_v8(op, o);          // one full 32-byte sector per lane and instruction
                        } else {
                            uint4 *o4 = reinterpret_cast<uint4 *>(op);
                            o4[0] = make_uint4(o[0], o[1], o[2], o[3]);
                            o4[1] = make_uint4(o[4], o[5], o[6], o[7]);
                        }
                    } else {
                        const int nvalid = Cout - n0 - n;
#pragma unroll
                        for (int q = 0; q < 16; ++q)
                            if (q < nvalid) op[q] = __float2bfloat16_rn(f[q]);
                    }
                };

                // column steps of this warp: all of them, or -- one-accumulator tiles, where the second group of epilogue warps would idle --
                // every other one (gs = 2, first step = the group)
                uint32_t va[16], vb[16];
                uint4 ra0, ra1, rb0, rb1;
                if (gfirst < G) {
                    if (!(skip & 2))
                    tc_ld16_issue(trow + (uint32_t)(16 * gfirst), va);                 // warp-collective: never under a lane-dependent branch
                    load_res(gfirst, ra0, ra1);
                }
                for (int g = gfirst; g < G; g += 2 * gs) {
                    const int g1 = g + gs, g2 = g1 + gs;
                    tc_wait_ld(va);
                    if (g1 < G) { if (!(skip & 2)) tc_ld16_issue(trow + (uint32_t)(16 * g1), vb); load_res(g1, rb0, rb1); }
                    process(va, ra0, ra1, g);
                    if (g1 < G) {
                        tc_wait_ld(vb);
                        if (g2 < G) { if (!(skip & 2)) tc_ld16_issue(trow + (uint32_t)(16 * g2), va); load_res(g2, ra0, ra1); }
                        process(vb, rb0, rb1, g1);
                    }
                }
            }
            // this warp is done reading the accumulator set: hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + set));
            if (DBG_ON) t_epi += clock64() - _te;
        }
        if (DBG_ON && warp == EPI_WARP0 && lane == 0) { P.dbg[blockIdx.x * 16 + 9] = t_accfull; P.dbg[blockIdx.x * 16 + 10] = t_epi; }
#undef vec32
#undef skip
    }
    tc_fence_before();
    __syncthreads();
    if (DBG_ON && threadIdx.x == 0) {
        P.dbg[blockIdx.x * 16 + 13] = clock64() - t_kernel0;
        unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        P.dbg[blockIdx.x * 16 + 14] = (long long)gt;
    }
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)P.tmem_cols) : "memory");
    }
}

long long *g_dbg_buf = nullptr;

int next_pow2_cols(int c) {
    int p = 32;
    while (p < c) p <<= 1;
    return p;
}

}  // namespace

// Host-side planning: planes, taps, tile shape, stage counts.
int wadain_tile(int C) { return (2 * C) % 256 == 0 ? 256 : 128; }

// split_c != 0: `d->in` is a split bf16 tensor [hi(split_c) | lo(split_c)] (see Params::split_c) and the filter bank holds
// 3 * split_c input channels; the output (and residual) may then be fp32 NHWC.  split_factor: see Params::split_factor.
int conv_umma_forward(const rdfc_conv_desc *d, cudaStream_t st, const rdfc_heads_desc *heads, const rdfc_stem_desc *stem,
                      const rdfc_wadain_conv_desc *wad, int split_c, const float *split_factor) {
    RDFC_REQUIRE((stem || d->in.dtype == RDFC_BF16) && (heads || d->out.dtype == RDFC_BF16 || (split_c && d->out.dtype == RDFC_F32)),
                 "UMMA conv: bf16 in/out only");
    RDFC_REQUIRE(!d->in.nchw && !d->out.nchw && !d->in2.ptr, "UMMA conv: single NHWC source / NHWC output only");
    RDFC_REQUIRE(d->in.C % BK == 0, "UMMA conv: Cin (%d) must be a multiple of %d", d->in.C, BK);
    RDFC_REQUIRE((stem || (d->in.pix_stride % 8 == 0 && ((uintptr_t)d->in.ptr % 16) == 0)) && ((uintptr_t)d->weight % 16) == 0 &&
                     (heads || (d->out.pix_stride % 8 == 0 && ((uintptr_t)d->out.ptr % 16) == 0)),
                 "UMMA conv: views must be 16-byte aligned with pixel strides that are multiples of 8 elements");
    RDFC_REQUIRE(!d->residual.ptr || (d->residual.dtype == d->out.dtype && d->residual.pix_stride % 8 == 0 &&
                                      ((uintptr_t)d->residual.ptr % 16) == 0),
                 "UMMA conv: residual must be an aligned NHWC view of the output's dtype");
    RDFC_REQUIRE(!split_c || (!stem && !wad && d->in.C == 2 * split_c && split_c % BK == 0),
                 "UMMA conv (split input): [hi | lo] view with 2 x %d channels expected", split_c);
    RDFC_REQUIRE((!d->scale || ((uintptr_t)d->scale % 16) == 0) && (!d->shift || ((uintptr_t)d->shift % 16) == 0),
                 "UMMA conv: scale / shift vectors must be 16-byte aligned");
    const bool k3 = d->kh == 3 && d->kw == 3, k1 = d->kh == 1 && d->kw == 1;
    RDFC_REQUIRE(k3 || k1, "UMMA conv: 3x3 or 1x1 kernels only");
    RDFC_REQUIRE(d->stride == 1 || d->stride == 2, "UMMA conv: stride 1 or 2");
    RDFC_REQUIRE(!d->transposed || (k3 && d->stride == 2 && d->pad == 1), "UMMA conv: transposed = k3 s2 p1 op1 only");
    RDFC_REQUIRE(d->transposed || d->pad == (k3 ? 1 : 0), "UMMA conv: padding must be (k-1)/2");

    Params P{};
    P.in = (const __nv_bfloat16 *)d->in.ptr; P.in_stride = d->in.pix_stride;
    P.B = d->B; P.Hi = d->Hi; P.Wi = d->Wi;
    P.w = (const __nv_bfloat16 *)d->weight;
    P.Cout = d->out.C; P.CoutP = (P.Cout + 15) / 16 * 16;
    P.cin_chunks = d->in.C / 8; P.nkb = d->in.C / BK;
    if (split_c) { P.split_c = split_c; P.cin_chunks = 3 * split_c / 8; P.nkb = 3 * split_c / BK; P.out_f32 = d->out.dtype == RDFC_F32; }
    P.split_factor = split_factor;
    P.out = (__nv_bfloat16 *)d->out.ptr; P.out_stride = d->out.pix_stride; P.Ho = d->Ho; P.Wo = d->Wo;
    P.res = (const __nv_bfloat16 *)d->residual.ptr; P.res_stride = d->residual.pix_stride;
    P.scale = d->scale; P.shift = d->shift; P.act = d->act;
    if (wad) {
        P.wad_x = (const __nv_bfloat16 *)wad->x.ptr; P.wad_x_stride = wad->x.pix_stride; P.wad_C = wad->x.C;
        P.wad_mean = wad->mean; P.wad_rstd = wad->rstd;
        P.wad_w = (const __nv_bfloat16 *)wad->gwbw.ptr; P.wad_w_stride = wad->gwbw.pix_stride;
        P.Cout = 2 * wad->x.C; P.CoutP = P.Cout;              // GEMM columns; the output view has C channels
    }
    if (stem) {
        RDFC_REQUIRE(stem->C0 + (stem->in1 ? 1 : 0) <= 4, "stem: at most 4 input planes in total");
        P.stem_in0 = stem->in0; P.stem_in1 = stem->in1; P.stem_c0 = stem->C0;
        P.stem_k = 9 * (stem->C0 + (stem->in1 ? 1 : 0));
        if (stem->out2.ptr) {
            P.out2 = (__nv_bfloat16 *)stem->out2.ptr; P.out2_stride = stem->out2.pix_stride; P.split = stem->out.C;
            P.Cout = stem->out.C + stem->out2.C; P.CoutP = (P.Cout + 15) / 16 * 16;
        }
    }
    if (heads) {
        P.ncols = heads->ncols;
        for (int q = 0; q < 16; ++q) {
            P.plane[q] = heads->out[q]; P.plane_bstride[q] = heads->out_bstride[q]; P.act_col[q] = heads->act[q];
        }
    }

    // tile space: output grid for convs, input grid for the sub-pixel phases of a transposed conv
    P.Ht = d->transposed ? d->Hi : d->Ho;
    P.Wt = d->transposed ? d->Wi : d->Wo;
    P.oys = P.oxs = d->transposed ? 2 : 1;
    P.nphases = d->transposed ? 4 : 1;
    // Cout tile.  One tcgen05.mma (M=128, K=16) costs max(~76, N/2) cycles (measured, scripts/umma_rate.cu), so N
    // should be >= 128; N = 128 rather than 256 leaves room for two accumulator sets of two accumulators in TMEM.
    int bn_max = 128;
    if (P.CoutP > 128 && P.CoutP % 128 != 0) bn_max = 256;               // e.g. 160: one tile beats 2 x 80
    // measured (B = 32, profiles/): N = 256 wins for 256- and 512-wide 3x3 stride-1 convs (+10..13 %) and the 512 -> 256
    // transposed conv (+29 %); stride-2 convs prefer N = 128 with two accumulator sets unless the output is tiny (en6)
    if (k3 && P.CoutP % 256 == 0) {
        if (d->stride == 1 || d->transposed) bn_max = 256;
        else if ((long long)d->B * d->Ho * d->Wo < 128ll * sm_count()) bn_max = 256;
    }
    if (k1 && P.CoutP % 256 == 0) bn_max = 256;                          // 1x1: the A stage feeds one tap only, so widen N
    if (wad) bn_max = wadain_tile(wad->x.C);
    if (const long long e = knob("RDFC_UMMA_BN", KNOB_UNSET); e != KNOB_UNSET) bn_max = (int)e;        // development knob
    P.bn = P.CoutP < bn_max ? P.CoutP : bn_max;
    while (P.CoutP % P.bn) P.bn -= 16;   // largest multiple of 16 <= bn_max dividing the padded Cout
    P.n_tiles_n = P.CoutP / P.bn;
    // accumulators per tile: wide tiles amortise the filter stream (B bytes per MMA ~ 1/NACC); double-buffer TMEM
    // whenever two sets of >= 2 accumulators fit; small problems need more tiles than SMs.
    const long long pixels = (long long)P.B * P.Ht * P.Wt * P.nphases;
    if (2 * 2 * P.bn <= 512) {            // N <= 128: two accumulator sets of 2..4 accumulators
        P.nsets = 2;
        P.nacc = 512 / (2 * P.bn) < 4 ? 512 / (2 * P.bn) : 4;
    } else {                              // wide N (e.g. 160, 256): one set
        P.nsets = 1;
        P.nacc = 512 / P.bn < 4 ? 512 / P.bn : 4;
        // measured (B = 32): a 256-wide 3x3 stride-1 conv with ONE N tile (en4, 57x76) is 12-22 % faster with one accumulator
        // and two TMEM sets (9 rounds of 128-pixel tiles instead of 5 rounds of 256, and the epilogue overlaps); with two N
        // tiles (en5: 512 wide, 29x38) the filter stream of one-accumulator tiles (64 B/clk/SM) saturates L2: -17 %
        if (k3 && d->stride == 1 && !d->transposed && P.n_tiles_n == 1 && 2 * P.bn <= 512) { P.nacc = 1; P.nsets = 2; }
    }
    while (P.nacc > 1 && (P.Wt <= 8 * (P.nacc - 1) || pixels / (128 * P.nacc) * P.n_tiles_n < sm_count())) --P.nacc;
    if (d->stride == 2 && !d->transposed && k3 && P.nacc > 2) P.nacc = 2;   // four parity planes: keep the stage small
    if (const long long e = knob("RDFC_UMMA_NACC", KNOB_UNSET); e != KNOB_UNSET) P.nacc = (int)e;      // development knob
    if (heads) P.nacc = 2;                                               // 16 x 16 pixel regions (see MODE_HEADS)
    if (const long long e = knob("RDFC_UMMA_NSETS", KNOB_UNSET); e != KNOB_UNSET) P.nsets = (int)e;    // development knob
    if (P.nsets * P.nacc * P.bn > 512) P.nsets = 1;
    // arrange the accumulators nax across x nay down so that the padded tile grid wastes the fewest pixels
    {
        long long best = -1;
        for (int nax = 1; nax <= P.nacc; ++nax) {
            if (P.nacc % nax) continue;
            const int nay = P.nacc / nax;
            const long long area = (long long)cdiv(P.Ht, 16 * nay) * 16 * nay * cdiv(P.Wt, 8 * nax) * 8 * nax;
            // measured (64 -> 64 at 228x304): the 2 x 2 arrangement beats 4 x 1 by 7 % at equal area, so it wins ties within 3 %
            const long long score = area * 100 + (nax == nay ? 0 : area * 3);
            if (best < 0 || score < best) { best = score; P.nax = nax; }
        }
        if (const long long e = knob("RDFC_UMMA_NAX", KNOB_UNSET); e != KNOB_UNSET) P.nax = (int)e;    // development knob
        if (heads) P.nax = 2;
    }
    const int TW = 8 * P.nax, TH = rdfc::TH * (P.nacc / P.nax);
    P.tstep_y = TH; P.tstep_x = TW; P.torg = 0;
    if (heads) {                              // overlapping 16 x 16 regions, each producing its inner 14 x 14 outputs
        RDFC_REQUIRE(P.nacc == 2 && P.nax == 2 && TH == 16 && TW == 16, "heads: internal tile shape");
        P.tstep_y = P.tstep_x = 14; P.torg = -1;
    }
    P.tiles_y = cdiv(P.Ht, P.tstep_y); P.tiles_x = cdiv(P.Wt, P.tstep_x);

    // A operand through TMA tensor-map loads unless the producers have to build it (stem mode)
    P.a_tma = !stem;
    RDFC_REQUIRE(!P.a_tma || tmap_encoder() != nullptr, "UMMA conv: the CUDA driver does not provide cuTensorMapEncodeTiled");
    P.px16 = P.a_tma ? 4 : 1;
    P.dual = P.a_tma && P.nacc >= 2;
    if (const long long e = knob("RDFC_UMMA_DUAL", KNOB_UNSET); e != KNOB_UNSET) P.dual = P.dual && (int)e != 0;      // development knob
    P.ntiles = P.tiles_x * P.tiles_y * P.B * P.nphases * P.n_tiles_n;
    // 1x1 convs: one tap per A stage means 2 * nacc MMAs per stage against ~500 cycles of barrier / commit / ring overhead in the issuing
    // warp (role timers, DESIGN 8.10).  Stage `kbs` consecutive 32-channel k-blocks at once: k-block j of a stage is "plane" j (the same
    // pixels, channel coordinate + 32 j) and "tap" j (its block of the packed filters), so the kernel's tap loop walks them inside one stage.
    P.kbs = 1;
    if (k1 && P.a_tma && !heads && !split_c) {
        const int nkb_total = P.nkb;
        for (int cand = 3; cand >= 2; --cand)
            if (nkb_total % cand == 0) { P.kbs = cand; break; }
        if (const long long e = knob("RDFC_UMMA_KBS", KNOB_UNSET); e != KNOB_UNSET) P.kbs = (e >= 1 && e <= 3 && nkb_total % (int)e == 0) ? (int)e : 1;
        P.nkb = nkb_total / P.kbs;
    }
    Phase phases[4] = {};
    int base = 0;
    auto add_plane = [&](int ystep, int yoff, int xstep, int xoff, int rows, int cols) {
        P.planes[P.nplanes] = Plane{ystep, yoff, xstep, xoff, rows, cols, base};
        base += rows * cols;
        return P.nplanes++;
    };
    if (d->transposed) {
        // oy = 2*iy - 1 + ky: even rows take ky = 1 (iy = y); odd rows take ky = 0 (iy = y + 1) and ky = 2 (iy = y)
        const int pl = add_plane(1, 0, 1, 0, TH + 1, TW + 1);
        for (int a = 0; a < 2; ++a)
            for (int bq = 0; bq < 2; ++bq) {
                Phase &ph = phases[a * 2 + bq];
                ph.oyo = a; ph.oxo = bq; ph.ntaps = 0;
                for (int ky = 0; ky < 3; ++ky)
                    for (int kx = 0; kx < 3; ++kx) {
                        if ((ky % 2 == 1) != (a == 0) || (kx % 2 == 1) != (bq == 0)) continue;
                        ph.taps[ph.ntaps++] = Tap{pl, ky == 0 ? 1 : 0, kx == 0 ? 1 : 0, ky * 3 + kx};
                    }
            }
    } else if (d->stride == 1 && P.kbs > 1) {
        for (int j = 0; j < P.kbs; ++j) {
            const int pl = add_plane(1, 0, 1, 0, TH, TW);
            phases[0].taps[phases[0].ntaps++] = Tap{pl, 0, 0, j};
        }
    } else if (d->stride == 1) {
        const int pl = add_plane(1, -d->pad, 1, -d->pad, TH + d->kh - 1, TW + d->kw - 1);
        Phase &ph = phases[0];
        for (int ky = 0; ky < d->kh; ++ky)
            for (int kx = 0; kx < d->kw; ++kx) ph.taps[ph.ntaps++] = Tap{pl, ky, kx, ky * d->kw + kx};
    } else if (k1) {
        for (int j = 0; j < P.kbs; ++j) {
            const int pl = add_plane(2, 0, 2, 0, TH, TW);
            phases[0].taps[phases[0].ntaps++] = Tap{pl, 0, 0, j};
        }
    } else {
        // iy = 2*oy - 1 + ky: ky = 1 reads the even-row plane; ky = 0 / 2 read the odd-row plane (rows oy-1 / oy)
        int pl[2][2];
        for (int py = 0; py < 2; ++py)
            for (int px = 0; px < 2; ++px)
                pl[py][px] = add_plane(2, py ? -1 : 0, 2, px ? -1 : 0, TH + 1, TW + 1);   // one TMA box shape
        Phase &ph = phases[0];
        for (int ky = 0; ky < 3; ++ky)
            for (int kx = 0; kx < 3; ++kx)
                ph.taps[ph.ntaps++] = Tap{pl[ky != 1][kx != 1], ky == 2 ? 1 : 0, kx == 2 ? 1 : 0, ky * 3 + kx};
    }
    P.npix = base;
    P.npix_pad = (base + 7) / 8 * 8;
    if (P.a_tma) {
        // every plane of a layer has the same box; a plane occupies rows * cols * 64 B rounded up to the 1 KB swizzle period
        const Plane &q0 = P.planes[0];
        for (int pl = 1; pl < P.nplanes; ++pl)
            RDFC_REQUIRE(P.planes[pl].rows == q0.rows && P.planes[pl].cols == q0.cols, "UMMA conv: TMA planes must share a box");
        P.a_plane_bytes = (q0.rows * q0.cols * 64 + 1023) / 1024 * 1024;
        P.a_tx_bytes = P.nplanes * q0.rows * q0.cols * 64;
        const cuuint64_t gdim[4] = {(cuuint64_t)d->in.C, (cuuint64_t)P.Wi, (cuuint64_t)P.Hi, (cuuint64_t)P.B};
        const cuuint64_t gstr[3] = {(cuuint64_t)P.in_stride * 2, (cuuint64_t)P.Wi * P.in_stride * 2, (cuuint64_t)P.Hi * P.Wi * P.in_stride * 2};
        const cuuint32_t box[4] = {(cuuint32_t)BK, (cuuint32_t)(q0.xstep * (q0.cols - 1) + 1), (cuuint32_t)(q0.ystep * (q0.rows - 1) + 1), 1};
        const cuuint32_t estr[4] = {1, (cuuint32_t)q0.xstep, (cuuint32_t)q0.ystep, 1};
        RDFC_REQUIRE(box[1] <= 256 && box[2] <= 256, "UMMA conv: TMA box too large");
        const CUresult r = tmap_encoder()(&P.tmap_a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void *)d->in.ptr, gdim, gstr, box, estr,
                                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        RDFC_REQUIRE(r == CUDA_SUCCESS, "UMMA conv: cuTensorMapEncodeTiled failed (%d)", (int)r);
    } else {
        RDFC_REQUIRE(P.npix_pad < (1 << 14), "UMMA conv: staged halo too large for the descriptor LBO field");
    }
    P.w_kb_stride = (long long)KCH * P.CoutP * 8 * P.kbs;
    P.b_contig = P.n_tiles_n == 1;
    for (int z = 0; z < P.nphases; ++z) {
        const Phase &ph = phases[z];
        P.ntaps[z] = ph.ntaps; P.oyo[z] = ph.oyo; P.oxo[z] = ph.oxo;
        for (int tp = 0; tp < ph.ntaps; ++tp) {
            const Tap &tap = ph.taps[tp];
            const Plane &q = P.planes[tap.plane];
            // no-swizzle K-major descriptor: start = tap's shifted view (16-byte units), LBO = cin-chunk pitch,
            // SBO = plane row pitch (8 pixels of a row form one core matrix), bit 46 = descriptor version
            if (P.a_tma) {
                // SWIZZLE_64B K-major ([pixel][64 B], written by TMA): start = plane + shifted pixel, SBO = plane row pitch,
                // LBO unused (K = 16 < the swizzle width), layout type 4 in bits 61-63; the swizzle is a function of the
                // absolute shared-memory address, so an arbitrary pixel shift of the start address stays consistent
                // (scripts/tma_swz_test.cu)
                P.tap_alo[z][tp] = (uint32_t)(tap.plane * (P.a_plane_bytes >> 4) + (tap.sy * q.cols + tap.sx) * 4) | (1u << 16);
                P.tap_ahi[z][tp] = (uint32_t)(q.cols * 4) | (1u << 14) | (4u << 29);
            } else {
                P.tap_alo[z][tp] = (uint32_t)(q.base + tap.sy * q.cols + tap.sx) | ((uint32_t)P.npix_pad << 16);
                P.tap_ahi[z][tp] = (uint32_t)q.cols | (1u << 14);
            }
            P.tap_w[z][tp] = P.kbs > 1 ? (long long)tap.wtap * KCH * P.CoutP * 8          // "tap" j of a 1x1 stage = the j-th k-block's filter block
                                       : (long long)tap.wtap * P.cin_chunks * P.CoutP * 8;
        }
    }
    P.epi_split = knob("RDFC_UMMA_EPISPLIT", 1) != 0;
    P.tmem_cols = next_pow2_cols(P.nsets * P.nacc * P.bn);
    RDFC_REQUIRE(P.tmem_cols <= 512, "UMMA conv: accumulators exceed TMEM");

    // filter taps per B stage: one wait / commit per filter row of a 3x3 conv; the 1/2/2/4-tap phases of a transposed
    // conv and 1x1 convs stream tap by tap
    P.gtaps = (k3 && !d->transposed) ? 3 : (P.kbs > 1 ? P.kbs : 1);
    P.vec32 = !heads && ((uintptr_t)d->out.ptr % 32) == 0 && d->out.pix_stride % 16 == 0 &&
              (!P.out2 || (((uintptr_t)P.out2 % 32) == 0 && P.out2_stride % 16 == 0 && P.split % 16 == 0)) &&
              (!d->residual.ptr || (((uintptr_t)d->residual.ptr % 32) == 0 && d->residual.pix_stride % 16 == 0));
    if (P.out_f32) P.vec32 = 0;                    // fp32 output: the general epilogue variant
    const int a_stage = P.a_tma ? P.nplanes * P.a_plane_bytes : (KCH * P.npix_pad * 16 + 1023) / 1024 * 1024;
    const int stem_patch = stem ? 2 * ((P.stem_k / 9) * (TH + 2) * (TW + 2) + 4) * 4 : 0;  // two fp32 input patches of a tile (stem mode)
    const int heads_y = heads ? 256 * (P.bn + 1) * 4 : 0;                                   // shift-add heads: Y of a region
    // Epilogue through TMA stores (and TMA residual loads): hot variant only (bf16 NHWC, 32-byte aligned slices, whole
    // 32-channel slabs), single-CTA tiles.  Measured per layer at B = 32 (gpurun_out/r2_plan_tmaout*.txt): it pays where the
    // per-lane 32-byte residual loads + stores were the bottleneck -- stride-1 residual layers with N <= 128 (64 -> 64 + residual
    // @228x304: 269 -> 230 us, 230 -> 218 us; 128 -> 128 + residual: 154 -> 150 us) -- and costs elsewhere (the slabs take 32-64 KB
    // from the operand stages: stride-2 convs 121 -> 138 us, 256-wide + residual 144 -> 168 us, 128 -> 160 719 -> 769 us), so it
    // is selected per layer.  RDFC_UMMA_TMAOUT: 0 = never, 1 = where it pays (default), 2 = every eligible layer, transposed convs
    // (element-strided store boxes) included -- the tests run all three.
    const int mode_std = !heads && !wad && !(P.act > RDFC_ACT_LEAKY02 || !P.vec32 || P.Cout % 16 != 0);
    const long long tmaout_knob = knob("RDFC_UMMA_TMAOUT", 1);
    const bool tmaout_pays = d->residual.ptr && P.bn <= 128 && !d->transposed && d->stride == 1;
    P.tma_out = mode_std && P.a_tma && !P.out2 && P.bn % 32 == 0 &&
                (tmaout_knob >= 2 || (tmaout_knob == 1 && tmaout_pays));
    if (P.tma_out) {
        const int es = d->transposed ? 2 : 1;
        const cuuint32_t box[4] = {32, (cuuint32_t)(es * 7 + 1), (cuuint32_t)(es * 15 + 1), 1};
        const cuuint32_t estr[4] = {1, (cuuint32_t)es, (cuuint32_t)es, 1};
        auto encode = [&](CUtensorMap *tm, const void *ptr, int C, int stride) {
            const cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)P.Wo, (cuuint64_t)P.Ho, (cuuint64_t)P.B};
            const cuuint64_t gstr[3] = {(cuuint64_t)stride * 2, (cuuint64_t)P.Wo * stride * 2, (cuuint64_t)P.Ho * P.Wo * stride * 2};
            return tmap_encoder()(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void *)ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                  CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        };
        CUresult r = encode(&P.tmap_out, d->out.ptr, d->out.C, d->out.pix_stride);
        if (r == CUDA_SUCCESS && d->residual.ptr) r = encode(&P.tmap_res, d->residual.ptr, d->residual.C, d->residual.pix_stride);
        RDFC_REQUIRE(r == CUDA_SUCCESS, "UMMA conv: cuTensorMapEncodeTiled (epilogue) failed (%d)", (int)r);
    }
    const int epi_stage = P.tma_out ? (d->residual.ptr ? 8 : 4) * EPI_SLAB_BYTES : 0;
    const int fixed = BAR_BYTES + 2 * P.CoutP * 4 + 4 * MAX_TAPS * 8 + 2 * P.wad_C * 4 + stem_patch + heads_y + 256 + epi_stage;   // barriers, (scale, shift) and tap tables, slack, epilogue slabs
    const int budget = 219 * 1024;
    // The issuing warp pays ~1000 cycles per filter stage (barrier wait, commits, ring bookkeeping) that the tensor pipe does
    // not overlap (role timers: issue is blocking at the pipe's rate), so a 3x3 conv stages all nine taps of a k-block at once
    // when two such stages and two A stages fit.
    if (k3 && !d->transposed && !stem && 2 * a_stage + 2 * 9 * KCH * P.bn * 16 + fixed <= budget) P.gtaps = 9;
    if (const long long e = knob("RDFC_UMMA_GTAPS", KNOB_UNSET); e != KNOB_UNSET) P.gtaps = (int)e;    // development knob (1, 3 or 9)
    // joff of accumulator 0 is 0 (jb = 0): the fast path needs nothing but the tap table
    P.fast9 = P.gtaps == 9 && P.nacc == 1 && P.a_tma && P.nphases == 1 && !P.dual && knob("RDFC_UMMA_FAST9", 1) != 0;
    const int b_stage = P.gtaps * KCH * P.bn * 16;
    // A ring first (>= 2 stages: the producers publish k-block i while k-block i+1 is in flight), then B stages (2..6)
    // the filter stream is latency-bound: bytes in flight per SM = bandwidth x L2 latency (~2000 cycles), so keep
    // >= 64 KB of filter stages in flight when the tile allows it
    // filter ring: enough stages to cover ~2500 cycles of L2 latency at the rate the tensor core drains them
    {
        const int mma_cycles = P.bn / 2 > 54 ? P.bn / 2 : 54;                 // measured: max(N/2, ~54) per M=128, K=16 MMA
        const int stage_cycles = P.gtaps * P.nacc * (BK / 16) * mma_cycles;
        P.sb = 2500 / stage_cycles + 2;
        if (P.sb < 3) P.sb = P.gtaps == 9 ? 2 : 3;
        if (P.sb > 16) P.sb = 16;
    }
    if (const long long e = knob("RDFC_UMMA_SB", KNOB_UNSET); e != KNOB_UNSET) P.sb = (int)e;          // development knob (<= 16)
    while (P.sb > 3 && 3 * a_stage + P.sb * b_stage + fixed > budget) --P.sb;     // prefer >= 3 A stages (2 in flight)
    while (P.sb > 2 && 2 * a_stage + P.sb * b_stage + fixed > budget) --P.sb;
    P.sa = (budget - fixed - P.sb * b_stage) / a_stage;
    if (P.sa > 6) P.sa = 6;
    if (const long long e = knob("RDFC_UMMA_SA", KNOB_UNSET); e != KNOB_UNSET) P.sa = (int)e < P.sa ? (int)e : P.sa;
    RDFC_REQUIRE(P.sa >= 1 && P.sa <= 8 && P.sb >= 1 && P.sb <= 16, "UMMA conv: tile does not fit shared memory");
    const size_t smem = (size_t)P.sa * a_stage + (size_t)P.sb * b_stage + fixed + 1024;
    void (*const kernels[4])(Params) = {conv_umma_kernel<MODE_STD>, conv_umma_kernel<MODE_GENERAL>, conv_umma_kernel<MODE_WADAIN>,
                                        conv_umma_kernel<MODE_HEADS>};   // indexed by mode
    static bool attr_set[64] = {};                 // per device: the attribute belongs to the function ON a device
    int dev_id = 0;
    RDFC_CUDA(cudaGetDevice(&dev_id));
    if (!attr_set[dev_id & 63]) {
        for (auto k : kernels) RDFC_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr_set[dev_id & 63] = true;
    }
    if (const long long e = knob("RDFC_UMMA_SKIP", KNOB_UNSET); e != KNOB_UNSET) P.dbg_flags = (int)e;
    static long long *dbg_buf = nullptr;
    if (knob("RDFC_UMMA_DBG", 0)) {
        if (!dbg_buf) RDFC_CUDA(cudaMalloc(&dbg_buf, 148 * 16 * sizeof(long long)));
        RDFC_CUDA(cudaMemsetAsync(dbg_buf, 0, 148 * 16 * sizeof(long long), st));
        P.dbg = dbg_buf;
        g_dbg_buf = dbg_buf;
    }
    int grid = P.ntiles < sm_count() ? P.ntiles : sm_count();
    if (const long long e = knob("RDFC_UMMA_GRID", KNOB_UNSET); e != KNOB_UNSET) grid = (int)e < P.ntiles ? (int)e : P.ntiles;   // development knob
    const int mode = heads ? MODE_HEADS : wad ? MODE_WADAIN
                     : (P.act > RDFC_ACT_LEAKY02 || !P.vec32 || P.Cout % 16 != 0) ? MODE_GENERAL : MODE_STD;
    // measured with the two-lane graph: early launch of the next conv takes SMs the other lane's CTAs would have used, and the
    // step does not get faster (10.61 / 10.63 ms with, 10.58 / 10.47 ms without), so it is off by default
    static int pdl = -1;
    if (pdl < 0) pdl = knob("RDFC_UMMA_PDL", 0) != 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl;
    cfg.attrs = attr; cfg.numAttrs = 1;
    RDFC_CUDA(cudaLaunchKernelEx(&cfg, kernels[mode], P));
    RDFC_CHECK_LAUNCH("conv_umma_kernel");
    return 0;
}

// development aid: copies the role timers of the last RDFC_UMMA_DBG=1 launch (148 CTAs x 16 slots) to the host
int conv_umma_read_dbg(long long *host, int n) {
    if (!g_dbg_buf) return -1;
    RDFC_CUDA(cudaDeviceSynchronize());
    RDFC_CUDA(cudaMemcpy(host, g_dbg_buf, sizeof(long long) * (n < 148 * 16 ? n : 148 * 16), cudaMemcpyDeviceToHost));
    return 0;
}

}  // namespace rdfc
