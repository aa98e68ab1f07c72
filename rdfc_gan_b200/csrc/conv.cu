// rdfc_conv_forward: validates the descriptor and dispatches to the tcgen05 (bf16) or CUDA-core (fp32) kernel.
#include "common.cuh"

namespace rdfc {
int conv_simt_forward(const rdfc_conv_desc *d, cudaStream_t st);
int conv_umma_forward(const rdfc_conv_desc *d, cudaStream_t st, const rdfc_heads_desc *heads, const rdfc_stem_desc *stem,
                      const rdfc_wadain_conv_desc *wad, int split_c);
int split_f32_forward(const rdfc_view *x, void *out_bf16, long long npix, cudaStream_t st);
int wadain_tile(int C);
int conv_umma_read_dbg(long long *host, int n);
}  // namespace rdfc

using namespace rdfc;

static int check_conv_geometry(const rdfc_conv_desc *d) {
    RDFC_REQUIRE(d != nullptr, "descriptor is NULL");
    RDFC_REQUIRE(d->in.ptr && d->out.ptr && d->weight, "conv: input / output / weight must not be NULL");
    RDFC_REQUIRE(d->B > 0 && d->Hi > 0 && d->Wi > 0 && d->Ho > 0 && d->Wo > 0 && d->in.C > 0 && d->out.C > 0,
                 "conv: empty dimension");
    RDFC_REQUIRE(d->kh > 0 && d->kw > 0 && d->kh * d->kw <= 9 && d->stride > 0 && d->pad >= 0, "conv: bad kernel geometry");
    if (d->transposed) {
        RDFC_REQUIRE(d->Ho <= 2 * d->Hi && d->Wo <= 2 * d->Wi, "conv: transposed output larger than 2x input");
    } else {
        const int ho = (d->Hi + 2 * d->pad - d->kh) / d->stride + 1, wo = (d->Wi + 2 * d->pad - d->kw) / d->stride + 1;
        RDFC_REQUIRE(d->Ho == ho && d->Wo == wo, "conv: output size (%d,%d) != expected (%d,%d)", d->Ho, d->Wo, ho, wo);
    }
    RDFC_REQUIRE(d->in.nchw || d->in.pix_stride >= d->in.C, "conv: input pixel stride smaller than its channel count");
    RDFC_REQUIRE(d->out.nchw || d->out.pix_stride >= d->out.C, "conv: output pixel stride smaller than its channel count");
    return 0;
}

extern "C" int rdfc_conv_forward(const rdfc_conv_desc *d, void *stream) {
    if (int rc = check_conv_geometry(d)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (d->path == RDFC_PATH_UMMA_BF16) return conv_umma_forward(d, st, nullptr, nullptr, nullptr, 0);
    if (d->path == RDFC_PATH_SIMT_F32) return conv_simt_forward(d, st);
    if (d->path == RDFC_PATH_UMMA_F32X3) {
        // fp32-faithful contraction on the bf16 tensor cores: split the fp32 input into [hi | lo] bf16 halves (one HBM pass into the
        // caller's workspace), then the tcgen05 kernel walks x_hi W_hi + x_hi W_lo + x_lo W_hi and writes fp32
        RDFC_REQUIRE(d->in.dtype == RDFC_F32 && d->out.dtype == RDFC_F32 && !d->in.nchw && !d->out.nchw && !d->in2.ptr,
                     "conv (fp32 on tensor cores): single fp32 NHWC source and fp32 NHWC output");
        RDFC_REQUIRE(d->in.C % 32 == 0, "conv (fp32 on tensor cores): Cin (%d) must be a multiple of 32", d->in.C);
        const long long npix = (long long)d->B * d->Hi * d->Wi;
        RDFC_REQUIRE(d->workspace && d->workspace_bytes >= (size_t)npix * d->in.C * 4 && ((uintptr_t)d->workspace % 128) == 0,
                     "conv (fp32 on tensor cores): workspace of B*Hi*Wi*Cin*4 bytes (128-byte aligned) required");
        if (int rc = split_f32_forward(&d->in, d->workspace, npix, st)) return rc;
        rdfc_conv_desc e = *d;
        e.in.ptr = d->workspace; e.in.dtype = RDFC_BF16; e.in.C = 2 * d->in.C; e.in.pix_stride = 2 * d->in.C;
        e.path = RDFC_PATH_UMMA_BF16;
        return conv_umma_forward(&e, st, nullptr, nullptr, nullptr, d->in.C);
    }
    return fail(RDFC_ERR_INVALID, "conv: unknown path %d", d->path);
}

extern "C" int rdfc_conv_forward_split(const rdfc_conv_desc *d, void *stream) {
    if (int rc = check_conv_geometry(d)) return rc;
    RDFC_REQUIRE(d->path == RDFC_PATH_UMMA_F32X3, "conv (split input): path must be RDFC_PATH_UMMA_F32X3");
    RDFC_REQUIRE(d->in.dtype == RDFC_F16 && !d->in.nchw && d->in.C % 64 == 0,
                 "conv (split input): an fp16 [hi | lo] view with 2 x Cin channels, Cin %% 32 == 0, expected (got %d channels)", d->in.C);
    RDFC_REQUIRE(d->out.dtype == RDFC_F32 && !d->out.nchw && !d->in2.ptr && !d->residual.ptr,
                 "conv (split input): fp32 NHWC output, no second source, no residual");
    RDFC_REQUIRE(d->scale != nullptr, "conv (split input): the per-Cout inverse scale vector is required");
    rdfc_conv_desc e = *d;
    e.in.dtype = RDFC_BF16;                 // 16-bit operands: the split path of the kernel reads them as fp16
    e.path = RDFC_PATH_UMMA_BF16;
    return conv_umma_forward(&e, (cudaStream_t)stream, nullptr, nullptr, nullptr, d->in.C / 2);
}

extern "C" int rdfc_heads_forward(const rdfc_heads_desc *h, void *stream) {
    RDFC_REQUIRE(h != nullptr && h->in.ptr && h->weight && h->shift, "heads: NULL argument");
    RDFC_REQUIRE(h->ncols >= 1 && h->ncols <= 16, "heads: ncols must be 1..16");
    RDFC_REQUIRE(h->B > 0 && h->H > 0 && h->W > 0, "heads: empty dimension");
    for (int q = 0; q < h->ncols; ++q) RDFC_REQUIRE(h->out[q] != nullptr, "heads: output plane %d is NULL", q);
    rdfc_conv_desc d{};
    d.B = h->B; d.Hi = d.Ho = h->H; d.Wi = d.Wo = h->W;
    d.kh = d.kw = 1; d.stride = 1; d.pad = 0; d.act = RDFC_ACT_NONE; d.path = RDFC_PATH_UMMA_BF16;    // the GEMM part: 1x1
    d.in = h->in;
    d.out.ptr = h->out[0]; d.out.dtype = RDFC_F32; d.out.C = (9 * h->ncols + 15) / 16 * 16; d.out.pix_stride = d.out.C;
    d.weight = h->weight; d.scale = nullptr; d.shift = h->shift;
    int split_c = 0;
    if (h->in.dtype == RDFC_F32) {
        // fp32 input (the tensor-core fp32 mode): split it into [hi | lo] fp16 halves first; the filter bank then holds 3 x C channels
        const long long npix = (long long)h->B * h->H * h->W;
        RDFC_REQUIRE(!h->in.nchw && h->in.C % 32 == 0, "heads (fp32 input): NHWC view with C %% 32 == 0");
        RDFC_REQUIRE(h->workspace && h->workspace_bytes >= (size_t)npix * h->in.C * 4 && ((uintptr_t)h->workspace % 128) == 0,
                     "heads (fp32 input): workspace of B*H*W*C*4 bytes (128-byte aligned) required");
        if (int rc = split_f32_forward(&h->in, h->workspace, npix, (cudaStream_t)stream)) return rc;
        split_c = h->in.C;
        d.in.ptr = h->workspace; d.in.dtype = RDFC_BF16; d.in.C = 2 * split_c; d.in.pix_stride = 2 * split_c;
    }
    return conv_umma_forward(&d, (cudaStream_t)stream, h, nullptr, nullptr, split_c);
}

extern "C" int rdfc_stem_forward(const rdfc_stem_desc *m, void *stream) {
    RDFC_REQUIRE(m != nullptr && m->in0 && m->out.ptr && m->weight, "stem: NULL argument");
    RDFC_REQUIRE(m->B > 0 && m->H > 0 && m->W > 0, "stem: empty dimension");
    RDFC_REQUIRE(m->C0 >= 1 && m->C0 + (m->in1 ? 1 : 0) <= 4, "stem: at most 4 input planes in total");
    RDFC_REQUIRE(m->act == RDFC_ACT_NONE || m->act == RDFC_ACT_RELU || m->act == RDFC_ACT_LEAKY02, "stem: unsupported activation");
    RDFC_REQUIRE(m->out.dtype == RDFC_BF16 && !m->out.nchw && (!m->out2.ptr || (m->out2.dtype == RDFC_BF16 && !m->out2.nchw)),
                 "stem: bf16 NHWC destinations only");
    RDFC_REQUIRE(!m->out2.ptr || (m->out.C % 16 == 0 && m->out2.pix_stride % 8 == 0 && ((uintptr_t)m->out2.ptr % 16) == 0),
                 "stem: the first destination must take a multiple of 16 columns; the second must be 16-byte aligned");
    rdfc_conv_desc d{};
    d.B = m->B; d.Hi = d.Ho = m->H; d.Wi = d.Wo = m->W;
    d.kh = d.kw = 1; d.stride = 1; d.pad = 0; d.act = m->act; d.path = RDFC_PATH_UMMA_BF16;
    d.in.ptr = (void *)m->in0; d.in.dtype = RDFC_F32; d.in.C = 64; d.in.pix_stride = 64;      // the virtual im2col matrix
    d.out = m->out;
    d.weight = m->weight; d.scale = m->scale; d.shift = m->shift;
    return conv_umma_forward(&d, (cudaStream_t)stream, nullptr, m, nullptr, 0);
}

extern "C" int rdfc_wadain_tile(int C) { return wadain_tile(C); }

extern "C" int rdfc_wadain_conv_forward(const rdfc_wadain_conv_desc *w, void *stream) {
    RDFC_REQUIRE(w != nullptr && w->style.ptr && w->x.ptr && w->out.ptr && w->weight && w->bias && w->mean && w->rstd,
                 "wadain conv: NULL argument");
    RDFC_REQUIRE(w->B > 0 && w->H > 0 && w->W > 0, "wadain conv: empty dimension");
    RDFC_REQUIRE(w->x.C % 64 == 0 && w->out.C == w->x.C, "wadain conv: C (%d) must be a multiple of 64 and match the output", w->x.C);
    RDFC_REQUIRE(w->x.dtype == RDFC_BF16 && w->out.dtype == RDFC_BF16 && w->style.dtype == RDFC_BF16 && !w->x.nchw && !w->out.nchw,
                 "wadain conv: bf16 NHWC views only");
    RDFC_REQUIRE(((uintptr_t)w->x.ptr % 32) == 0 && w->x.pix_stride % 16 == 0 && ((uintptr_t)w->out.ptr % 32) == 0 &&
                     w->out.pix_stride % 16 == 0,
                 "wadain conv: x / out slices must be 32-byte aligned");
    RDFC_REQUIRE(!w->gwbw.ptr || (w->gwbw.dtype == RDFC_BF16 && !w->gwbw.nchw && w->gwbw.C == 2 * w->x.C &&
                                  ((uintptr_t)w->gwbw.ptr % 32) == 0 && w->gwbw.pix_stride % 16 == 0),
                 "wadain conv: gwbw must be a 32-byte aligned bf16 NHWC view with 2C channels");
    rdfc_conv_desc d{};
    d.B = w->B; d.Hi = d.Ho = w->H; d.Wi = d.Wo = w->W;
    d.kh = d.kw = 1; d.stride = 1; d.pad = 0; d.act = RDFC_ACT_NONE; d.path = RDFC_PATH_UMMA_BF16;
    d.in = w->style; d.out = w->out;
    d.weight = w->weight; d.scale = nullptr; d.shift = w->bias;
    return conv_umma_forward(&d, (cudaStream_t)stream, nullptr, nullptr, w, 0);
}

// development aid (not part of the public ABI): role timers of the last conv_umma launch under RDFC_UMMA_DBG=1
extern "C" int rdfc_dev_umma_timers(long long *host, int n) { return conv_umma_read_dbg(host, n); }
