// Filter gradient of the 3x3 (and 1x1: one tap, the input box is the pixels themselves) convolutions on tcgen05 (the training step's largest kernel; reference: autograd of nn.Conv2d /
// nn.ConvTranspose2d in RDFC-GAN/lib/models/generator/rdf_generator/encoder_decoder/common.py:29-61 -> cuDNN wgrad).
//
//   dW[o][i][ky][kx] = sum over (b, py, px) of  G[b, py, px, o] * I[b, s*py - 1 + ky, s*px - 1 + kx, i]
//
// is a GEMM whose K dimension is the PIXEL index, so with NHWC tensors both operands are "MN-major": the channel (M / N) index is
// the contiguous one.  tcgen05 takes such operands straight from shared memory: a TMA box [pixels][64 channels] with SWIZZLE_128B is
// exactly the canonical MN-major SW128 layout (one pixel = one 128-byte row, 8 pixels = one swizzle atom, SBO = 1024 B between
// groups of 8 pixels, LBO = the distance between blocks of 64 channels), and -- the swizzle being a function of the absolute
// shared-memory address -- a filter tap is a start-address shift by whole pixels into the staged input patch
// (scripts/umma_mn_test.cu pins all of this against a CPU sum).
//
// Tile: one CTA owns a (64 input channels) x (NB <= 96 output channels) block of ALL nine taps over a chunk of pixel rows (split K):
//   A = the input patch, M = 128 = [64 channels under tap a ; the same 64 channels under tap b]: the second block of 64 rows sits LBO
//       bytes after the first, and LBO may be ANY multiple of 16 bytes -- here the address distance of two taps, so one MMA feeds two
//       taps (an M = 64 MMA is no faster than an M = 128 one: 47.4 vs 48.2 cycles at N = 64, measured);
//   B = the output gradient, N = NB (two 64-channel boxes when NB > 64; N = 96 costs what N = 64 costs, 48 cycles);
//   D = five accumulators of 128 lanes x NB columns in TMEM (tap pairs (0,1) (2,3) (4,5) (6,7) (8,8)), 5 * 96 <= 512 columns.
// Per K = 16 pixels that is 5 MMAs = 240 cycles for 64 x NB x 9 taps (the MMAs are shared-memory-bandwidth bound: 4 KB of A + up to
// 3 KB of B per MMA at 128 B / cycle).  Stride-2 convolutions stage the four parity planes of the patch (TMA element strides 2), a tap
// then addresses (plane, shift) and a pair's LBO is the distance between the two planes' pixels.
// Roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warps 2-5 = epilogue (TMEM -> fp32 partials [chunk][tap][O][I],
// coalesced along i); wgrad_umma_reduce_kernel sums the chunks in a fixed order (bit-reproducible) into torch's (O, I, 3, 3).
#include <cuda.h>

#include "common.cuh"

namespace rdfc {
namespace {

constexpr int WU_MAXST = 6;

struct WuParams {
    alignas(64) CUtensorMap tmG;
    alignas(64) CUtensorMap tmI;
    int B, Hg, Wg, s, pad, ntap, npair, TR, TW, NB, nob, nib, O, Ich;
    int fp16;                   // operands are fp16 (the DCN path's split halves) instead of bf16
    int groups_per_img, total_groups, tiles_per_cta, total_tiles, nst;
    int dbg;                    // development knob RDFC_WGRAD_DBG: 1 = stage nothing, 2 = issue no MMAs (wrong results; what bounds the kernel?)
    uint32_t g_box_bytes, g_boxes, i_plane_bytes, i_planes, i_off, stage_bytes, tx_bytes, rpitch, ncol;
    uint32_t toff[9];           // byte offset of tap t's pixel (row 0, column 0 of the tile) inside the staged input region
    int pa[5], pb[5];           // tap pairs, toff[pa] <= toff[pb]
    float *partial;             // [chunk][tap][O][Ich]
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// bounded wait: traps after ~4 s instead of hanging the GPU
__device__ __forceinline__ void wait_bar(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0,1,0,p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) break;
        if (clock64() - t0 > 8000000000ll) __trap();
    }
}
__device__ __forceinline__ void tma4d(uint32_t dst, const CUtensorMap *tm, int c0, int c1, int c2, int c3, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst), "l"(tm), "r"(c0),
                 "r"(c1), "r"(c2), "r"(c3), "r"(bar)
                 : "memory");
}

__global__ void __launch_bounds__(192, 1) wgrad_umma_kernel(const __grid_constant__ WuParams P) {
    extern __shared__ __align__(1024) unsigned char wu_smem[];
    __shared__ __align__(8) uint64_t full[WU_MAXST], empty[WU_MAXST], done;
    __shared__ uint32_t tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t sbase = (smem_u32(wu_smem) + 1023u) & ~1023u;
    if (threadIdx.x == 0) {
        for (int s = 0; s < P.nst; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&full[s])));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&empty[s])));
        }
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&done)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_slot;
    const int ob = blockIdx.x / P.nib, ib = blockIdx.x - ob * P.nib, chunk = blockIdx.y;
    // split K by TILES (row group x column tile), a contiguous run per CTA
    const int xtiles = (P.Wg + P.TW - 1) / P.TW;
    const int t_begin = chunk * P.tiles_per_cta, ntiles = min(t_begin + P.tiles_per_cta, P.total_tiles) - t_begin;

    if (warp == 0) {
        if (elect_one()) {
            int grp = t_begin / xtiles, xt = t_begin - grp * xtiles;
            for (int t = 0; t < ntiles; ++t) {
                const int s = t % P.nst;
                if (t >= P.nst) wait_bar(smem_u32(&empty[s]), (uint32_t)((t / P.nst - 1) & 1));
                const int b = grp / P.groups_per_img, gy0 = (grp - b * P.groups_per_img) * P.TR, gx0 = xt * P.TW;
                const uint32_t st = sbase + (uint32_t)s * P.stage_bytes, fb = smem_u32(&full[s]);
                if (P.dbg & 1) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(fb) : "memory"); if (++xt == xtiles) { xt = 0; ++grp; } continue; }
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fb), "r"(P.tx_bytes) : "memory");
                for (uint32_t bx = 0; bx < P.g_boxes; ++bx) tma4d(st + bx * P.g_box_bytes, &P.tmG, ob * P.NB + 64 * (int)bx, gx0, gy0, b, fb);
                if (P.i_planes == 1) {
                    tma4d(st + P.i_off, &P.tmI, ib * 64, P.s * gx0 - P.pad, P.s * gy0 - P.pad, b, fb);
                } else {
                    for (int py = 0; py < 2; ++py)
                        for (int px = 0; px < 2; ++px)
                            tma4d(st + P.i_off + (uint32_t)(py * 2 + px) * P.i_plane_bytes, &P.tmI, ib * 64, 2 * gx0 - 1 + px, 2 * gy0 - 1 + py, b, fb);
                }
                if (++xt == xtiles) { xt = 0; ++grp; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // One lane issues; what it costs per MMA bounds the kernel once the operands are staged (a first version recomputed the
        // descriptors from kernel parameters -- re-read from the constant bank after every asm volatile -- and ran at 88 cycles per MMA
        // against the pipe's 48): everything the loop needs sits in registers (an opaque zero keeps ptxas from re-materialising the
        // parameters), descriptors advance by one 32-bit add, the pair loop is unrolled for the 9-tap and the 1-tap case.
        uint32_t kz;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(kz));
        kz >>= 31;
        // instruction descriptor: fp32 accumulate, bf16 (or fp16) operands, both MN-major, M = 128, N = NB
        const uint32_t idesc = ((1u << 4) | (P.fp16 ? 0u : (1u << 7) | (1u << 10)) | (1u << 15) | (1u << 16) | ((uint32_t)(P.NB >> 3) << 17) | (8u << 24)) + kz;
        const uint32_t desc_hi = ((uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29)) + kz;      // SBO = 1024, version 1, SWIZZLE_128B
        uint32_t a_lo[5], d_col[5];                                                         // per pair: tap a's offset (16-byte units) | LBO; accumulator
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            a_lo[j] = (j < P.npair ? (P.toff[P.pa[j]] >> 4) | (((P.toff[P.pb[j]] - P.toff[P.pa[j]]) >> 4) << 16) : 0u) + kz;
            d_col[j] = tmem + (uint32_t)j * P.ncol + kz;
        }
        const uint32_t b_lbo = ((P.g_box_bytes >> 4) << 16) + kz;
        const int hsteps = P.TW / 16 + (int)kz, TR = P.TR + (int)kz, nst = P.nst + (int)kz, nine = (P.npair == 5) + (int)kz, dbg2 = (P.dbg & 2) + (int)kz;
        const uint32_t rstep_i = (P.rpitch >> 4) + kz, rstep_g = ((uint32_t)(P.TW * 128) >> 4) + kz, stage16 = (P.stage_bytes >> 4) + kz;
        const uint32_t i_off16 = (P.i_off >> 4) + kz, base16 = ((sbase & 0x3FFFFu) >> 4) + kz;
        const uint32_t full0 = smem_u32(&full[0]) + kz, empty0 = smem_u32(&empty[0]) + kz, done_b = smem_u32(&done) + kz;
        int s = 0;
        uint32_t par = 0;
        for (int t = 0; t < ntiles; ++t) {
            wait_bar(full0 + 8u * (uint32_t)s, par);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (elect_one()) {
                const uint32_t gG = base16 + (uint32_t)s * stage16;
                uint32_t ia_r = gG + i_off16, ga_r = gG | b_lbo;
                uint32_t acc = t ? 1u : 0u;
                for (int r = 0; r < (dbg2 ? (t == 0) : TR); ++r) {
                    uint32_t ia = ia_r, ga = ga_r;
                    for (int h = 0; h < hsteps; ++h) {
                        if (nine) {
#pragma unroll
                            for (int j = 0; j < 5; ++j) {
                                asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\tmov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
                                             "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(d_col[j]),
                                             "r"(a_lo[j] + ia), "r"(ga), "r"(desc_hi), "r"(idesc), "r"(acc)
                                             : "memory");
                            }
                        } else {
                            asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\tmov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
                                         "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(d_col[0]),
                                         "r"(a_lo[0] + ia), "r"(ga), "r"(desc_hi), "r"(idesc), "r"(acc)
                                         : "memory");
                        }
                        acc = 1u;
                        ia += 128u; ga += 128u;                              // 16 pixels = 2048 bytes
                    }
                    ia_r += rstep_i; ga_r += rstep_g;
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(empty0 + 8u * (uint32_t)s) : "memory");
                if (t == ntiles - 1) asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(done_b) : "memory");
            }
            __syncwarp();
            if (++s == nst) { s = 0; par ^= 1u; }
        }
    } else {
        wait_bar(smem_u32(&done), 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp & 3, m = 32 * q + lane, second = m >> 6, i = ib * 64 + (m & 63);
        const bool i_ok = i < P.Ich;
        for (int j = 0; j < P.npair; ++j) {
            if (second && P.pb[j] == P.pa[j]) break;                       // warp-uniform: the last pair is one tap twice
            const int tap = second ? P.pb[j] : P.pa[j];
            float *dst = P.partial + (((long long)chunk * P.ntap + tap) * P.O) * P.Ich + i;
            for (int c0 = 0; c0 < P.NB; c0 += 16) {
                uint32_t v[16];
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                             : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                               "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                             : "r"(tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)j * P.ncol + (uint32_t)c0));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const int o = ob * P.NB + c0 + c;
                    if (i_ok && o < P.O && c0 + c < P.NB) dst[(long long)o * P.Ich] = __uint_as_float(v[c]);
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u));
}

// dW[o][i][tap] (torch's (O, I, 3, 3)) = sum over chunks of partial[chunk][tap][o][i], in chunk order
__global__ void __launch_bounds__(256) wgrad_umma_reduce_kernel(const float *__restrict__ partial, float *__restrict__ dw, int O, int Ich, int nchunk,
                                                                int ntap) {
    const long long per = (long long)O * Ich, total = ntap * per;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int tap = (int)(e / per);
        const long long oi = e - (long long)tap * per;
        float s = 0.f;
        for (int c = 0; c < nchunk; ++c) s += __ldg(partial + (long long)c * total + e);
        dw[oi * ntap + tap] = s;
    }
}

}  // namespace

struct WuGeom { WuParams P; int nchunk; size_t smem; long long ws_floats; };

static int wgrad_umma_geom(const rdfc_wgrad_desc *d, WuGeom *g) {
    WuParams &P = g->P;
    P.B = d->B; P.Hg = d->Hg; P.Wg = d->Wg; P.s = d->stride; P.pad = d->pad; P.O = d->grad_out.C; P.Ich = d->input.C;
    P.ntap = d->k * d->k; P.npair = (P.ntap + 1) / 2;
    // tile: 32-pixel rows unless 16-pixel rows waste fewer columns; rows per tile so that a stage stays near 45-60 KB
    const int w32 = cdiv(P.Wg, 32) * 32, w16 = cdiv(P.Wg, 16) * 16;
    P.TW = (int)knob("RDFC_WGRAD_TW", w16 < w32 ? 16 : 32);
    P.TR = (P.s == 1 || d->k == 1) ? (P.TW == 32 ? 4 : 8) : (P.TW == 32 ? 2 : 4);
    if (P.TR > P.Hg) P.TR = P.Hg;
    P.nob = cdiv(P.O, 96);
    P.NB = cdiv(cdiv(P.O, P.nob), 16) * 16;          // the MMA's N; channels past O (O % 16 == 8) are TMA zero fill, masked in the epilogue
    P.nib = cdiv(P.Ich, 64);
    P.ncol = (uint32_t)P.NB;
    P.g_boxes = P.NB > 64 ? 2 : 1;
    P.g_box_bytes = (uint32_t)(P.TR * P.TW * 128);
    P.i_off = P.g_boxes * P.g_box_bytes;
    int prow, pcol;                                   // rows / columns of one staged input plane
    if (d->k == 1) { P.i_planes = 1; prow = P.TR; pcol = P.TW; }                           // 1x1: the pixels themselves (every s-th)
    else if (P.s == 1) { P.i_planes = 1; prow = P.TR + 2; pcol = P.TW + 2; }
    else { P.i_planes = 4; prow = P.TR + 1; pcol = P.TW + 1; }
    P.i_plane_bytes = (uint32_t)((prow * pcol * 128 + 1023) / 1024 * 1024);
    P.rpitch = (uint32_t)pcol * 128u;
    P.stage_bytes = P.i_off + P.i_planes * P.i_plane_bytes;
    P.tx_bytes = P.g_boxes * P.g_box_bytes + P.i_planes * (uint32_t)(prow * pcol * 128);
    for (int t = 0; t < 9; ++t) P.toff[t] = 0;
    for (int ky = 0; ky < d->k; ++ky)
        for (int kx = 0; kx < d->k; ++kx) {
            if (d->k == 1) {
                P.toff[0] = 0;
            } else if (P.s == 1) {
                P.toff[ky * 3 + kx] = (uint32_t)(ky * pcol + kx) * 128u;
            } else {    // row 2 gy - 1 + ky: ky = 0 -> plane 0 (rows -1, 1, ..) row gy; ky = 1 -> plane 1 (rows 0, 2, ..) row gy; ky = 2 -> plane 0 row gy + 1
                const int py = ky == 1, dy = ky == 2, px = kx == 1, dx = kx == 2;
                P.toff[ky * 3 + kx] = (uint32_t)(py * 2 + px) * P.i_plane_bytes + (uint32_t)(dy * pcol + dx) * 128u;
            }
        }
    for (int j = 0; j < 5; ++j) { P.pa[j] = P.pb[j] = 0; }
    for (int j = 0; j < P.npair; ++j) {
        int a = 2 * j, b = 2 * j + 1 < P.ntap ? 2 * j + 1 : 2 * j;
        if (P.toff[a] > P.toff[b]) { const int t = a; a = b; b = t; }
        P.pa[j] = a; P.pb[j] = b;
        RDFC_REQUIRE(P.toff[b] - P.toff[a] < (1u << 18), "wgrad (tcgen05): tap distance exceeds the descriptor's LBO field");
    }
    P.nst = (int)((220u * 1024u) / P.stage_bytes);
    if (P.nst > WU_MAXST) P.nst = WU_MAXST;
    RDFC_REQUIRE(P.nst >= 2, "wgrad (tcgen05): stage of %u bytes does not fit twice", P.stage_bytes);
    g->smem = (size_t)P.nst * P.stage_bytes + 1024;
    P.groups_per_img = cdiv(P.Hg, P.TR);
    P.total_groups = P.B * P.groups_per_img;
    const int nblk = P.nob * P.nib;
    int want = sm_count() / nblk;                      // one CTA per SM (each allocates all of TMEM): about one wave in total
    if (want < 1) want = 1;
    P.total_tiles = P.total_groups * cdiv(P.Wg, P.TW);
    P.tiles_per_cta = cdiv(P.total_tiles, want);
    g->nchunk = cdiv(P.total_tiles, P.tiles_per_cta);
    P.dbg = (int)knob("RDFC_WGRAD_DBG", 0);
    g->ws_floats = (long long)g->nchunk * P.ntap * P.O * P.Ich;
    return 0;
}

long long wgrad_umma_workspace_floats(const rdfc_wgrad_desc *d) {
    WuGeom g;
    return wgrad_umma_geom(d, &g) == 0 ? g.ws_floats : -1;
}

// the split-K partials only: workspace[chunk][tap][O][Ich] for chunk < *nchunk (callers that combine several products -- the DCN
// filter gradient's split-precision terms -- reduce them themselves); fp16 != 0: the views hold fp16 values
int wgrad_umma_partials(const rdfc_wgrad_desc *d, float *workspace, int fp16, cudaStream_t st, int *nchunk) {
    WuGeom g;
    if (int rc = wgrad_umma_geom(d, &g)) return rc;
    WuParams &P = g.P;
    P.partial = workspace;
    P.fp16 = fp16;
    RDFC_REQUIRE(((uintptr_t)d->grad_out.ptr % 16) == 0 && ((uintptr_t)d->input.ptr % 16) == 0, "wgrad (tcgen05): 16-byte aligned tensors");
    RDFC_REQUIRE(tmap_encoder() != nullptr, "wgrad (tcgen05): the CUDA driver does not provide cuTensorMapEncodeTiled");
    {
        const cuuint64_t gdim[4] = {(cuuint64_t)P.O, (cuuint64_t)d->Wg, (cuuint64_t)d->Hg, (cuuint64_t)d->B};
        const cuuint64_t ps = (cuuint64_t)d->grad_out.pix_stride * 2;
        const cuuint64_t gstr[3] = {ps, ps * d->Wg, ps * d->Wg * d->Hg};
        const cuuint32_t box[4] = {64, (cuuint32_t)P.TW, (cuuint32_t)P.TR, 1}, estr[4] = {1, 1, 1, 1};
        const CUresult r = tmap_encoder()(&P.tmG, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void *)d->grad_out.ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        RDFC_REQUIRE(r == CUDA_SUCCESS, "wgrad (tcgen05): cuTensorMapEncodeTiled (grad_out) failed (%d)", (int)r);
    }
    {
        const cuuint64_t gdim[4] = {(cuuint64_t)P.Ich, (cuuint64_t)d->Wi, (cuuint64_t)d->Hi, (cuuint64_t)d->B};
        const cuuint64_t ps = (cuuint64_t)d->input.pix_stride * 2;
        const cuuint64_t gstr[3] = {ps, ps * d->Wi, ps * d->Wi * d->Hi};
        const int prow = d->k == 1 ? P.TR : (P.s == 1 ? P.TR + 2 : P.TR + 1), pcol = d->k == 1 ? P.TW : (P.s == 1 ? P.TW + 2 : P.TW + 1);
        const cuuint32_t box[4] = {64, (cuuint32_t)(P.s * (pcol - 1) + 1), (cuuint32_t)(P.s * (prow - 1) + 1), 1};
        const cuuint32_t estr[4] = {1, (cuuint32_t)P.s, (cuuint32_t)P.s, 1};
        const CUresult r = tmap_encoder()(&P.tmI, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void *)d->input.ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        RDFC_REQUIRE(r == CUDA_SUCCESS, "wgrad (tcgen05): cuTensorMapEncodeTiled (input) failed (%d)", (int)r);
    }
    static bool attr[64] = {};
    int dev = 0;
    RDFC_CUDA(cudaGetDevice(&dev));
    if (!attr[dev & 63]) {
        RDFC_CUDA(cudaFuncSetAttribute(wgrad_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        attr[dev & 63] = true;
    }
    wgrad_umma_kernel<<<dim3(P.nob * P.nib, g.nchunk), 192, g.smem, st>>>(P);
    RDFC_CHECK_LAUNCH("wgrad_umma_kernel");
    *nchunk = g.nchunk;
    return 0;
}

int wgrad_umma(const rdfc_wgrad_desc *d, float *grad_weight, float *workspace, cudaStream_t st) {
    int nchunk = 0;
    if (int rc = wgrad_umma_partials(d, workspace, 0, st, &nchunk)) return rc;
    const int ntap = d->k * d->k;
    const long long total = (long long)ntap * d->grad_out.C * d->input.C;
    const int nblk = (int)min((long long)cdiv(total, 256), (long long)sm_count() * 8);
    wgrad_umma_reduce_kernel<<<nblk, 256, 0, st>>>(workspace, grad_weight, d->grad_out.C, d->input.C, nchunk, ntap);
    RDFC_CHECK_LAUNCH("wgrad_umma_reduce_kernel");
    return 0;
}

}  // namespace rdfc
