"""Execution engine of the generator forward pass (rdf_generator.py:280-414) on the sm_100a kernels.

The engine turns the module tree (parameter containers) into
  * packed weights: filters in GEMM form ([tap][cin][cout] fp32 for the CUDA-core path, [tap][cin/8][cout][8] bf16
    for the tcgen05 path), eval-mode BatchNorm folded into a per-channel (scale, shift) epilogue, EqualLR applied;
  * a Plan per input shape: NHWC activation buffers laid out so that every ``torch.cat`` of the reference is a
    channel slice of a preallocated buffer, and a flat list of C-ABI calls with fixed pointers, captured in a CUDA
    graph and replayed.

HBM layout (per image, C channels innermost; bf16 in 'bf16' mode, fp32 in 'fp32' mode):
    head_r  (H, W, 160)  = [rgb_pred_dec1 64 | rgb_conf_dec1 32 | rgb_fe1 64]
    head_d  (H, W, 224)  = [id_dec1 64 | cf_dec1 32 | gd_dec1 64 | depth_fe1 64]
    cat2_x  (H, W, 128)  = [de2 64 | fe2 64]          cat3_x (H/2, W/2, 192) = [de3 64 | fe3 128]
    cat4_x  (H/4,W/4,384)= [de4 128 | fe4 256]        cat5_x (H/8, W/8, 768) = [de5 256 | fe5 512]     fe6_x (H/16, W/16, 512)
NLSPN tensors stay fp32 NCHW as in the reference (guide (B,8,H,W), offset (B,18,H,W), aff (B,9,H,W)).
"""
import ctypes
import os
import math

import torch

from . import _cabi as C


def _down(n):
    return (n - 1) // 2 + 1      # conv k3 s2 p1 (and 1x1 s2 p0)


def pack_weight(w, umma, x3=False):
    """(Cout, Cin, kh, kw) fp32 filters -> the layout rdfc_conv_forward reads for the conv path:
    RDFC_PATH_SIMT_F32    (umma False)     [tap][cin][cout] fp32;
    RDFC_PATH_UMMA_BF16   (umma, not x3)   [tap][cin/8][CoutP][8] bf16, Cout zero-padded to CoutP = a multiple of 16;
    RDFC_PATH_UMMA_F32X3  (umma and x3)    the same layout in fp16 over [W_hi ; W_lo ; W_hi] along Cin (3 Cin channels)."""
    if x3:       # [W_hi ; W_lo ; W_hi] along Cin, fp16 halves (11 + 11 mantissa bits): the kernel pairs them with x_hi, x_hi, x_lo
        w_hi = w.to(torch.float16).float()
        w = torch.cat([w_hi, (w - w_hi).to(torch.float16).float(), w_hi], 1)
    Cout, Cin, kh, kw = w.shape
    g = w.permute(0, 2, 3, 1).reshape(Cout, kh * kw, Cin)          # [cout][tap][cin]
    if not umma:
        return g.permute(1, 2, 0).contiguous()                      # [tap][cin][cout] fp32
    CoutP = (Cout + 15) // 16 * 16
    if CoutP != Cout:
        g = torch.cat([g, g.new_zeros(CoutP - Cout, kh * kw, Cin)], 0)
    return g.reshape(CoutP, kh * kw, Cin // 8, 8).permute(1, 2, 0, 3).contiguous().to(torch.float16 if x3 else torch.bfloat16)


class _Packed:
    """Persistent device storage for one (possibly fused) conv layer's packed filters and epilogue vectors."""

    def __init__(self):
        self.weight = self.scale = self.shift = None

    def store(self, weight, scale, shift):
        for name, val in (("weight", weight), ("scale", scale), ("shift", shift)):
            cur = getattr(self, name)
            if val is None:
                setattr(self, name, None)
            elif cur is None or cur.shape != val.shape or cur.dtype != val.dtype or cur.device != val.device:
                setattr(self, name, val.contiguous().clone())
            else:
                cur.copy_(val)


class Plan:
    def __init__(self):
        self.steps = []          # callables taking the stream pointer
        self.names = []          # debug: one label per step
        self.keep = []           # ctypes structs / tensors that must outlive the plan
        self.graph = None
        self.n_launch = 0
        # Two lanes: the RGB and the depth branch are independent between their fusion points (rdf_generator.py:295-368), so
        # the captured graph runs them on two streams.  Every conv is a persistent kernel of <= 148 CTAs; while the last
        # round of one launch leaves SMs idle (29x38 layers: 2.2 rounds of tiles) the other lane's CTAs take them.
        self.cur_lane = 0
        self.marks = []          # (step index, lane): steps from that index on run on `lane` (0 = main, 1 = side)
        self.sync = {}           # step index -> ['fork' | 'join', ...] applied before that step

    def lane(self, lane):
        self.cur_lane = lane
        self.marks.append((len(self.steps), lane))

    def fork(self):
        self.sync.setdefault(len(self.steps), []).append('fork')

    def join(self):
        self.sync.setdefault(len(self.steps), []).append('join')
        self.lane(0)

    def lanes(self):
        out, cur, marks = [], 0, sorted(self.marks, key=lambda m: m[0])
        mi = 0
        for i in range(len(self.steps)):
            while mi < len(marks) and marks[mi][0] <= i:
                cur = marks[mi][1]
                mi += 1
            out.append(cur)
        return out

    def run_eager(self):
        """All steps in list order on the current stream (list order respects every dependency)."""
        s = C.stream_ptr()
        for f in self.steps:
            f(s)

    def run_lanes(self, side):
        """Lane-1 steps on `side`, the rest on the current stream, with the recorded fork / join edges (used under capture)."""
        main = torch.cuda.current_stream()
        lanes = self.lanes()
        for i, f in enumerate(self.steps):
            for op in self.sync.get(i, ()):
                if op == 'fork':
                    side.wait_stream(main)
                else:
                    main.wait_stream(side)
            f((side if lanes[i] else main).cuda_stream)
        for op in self.sync.get(len(self.steps), ()):
            if op == 'join':
                main.wait_stream(side)
        main.wait_stream(side)

    def run(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self.run_eager()


class GeneratorEngine:
    def __init__(self, gen):
        self.gen = gen
        # 'fp32'    every contraction on the CUDA cores in fp32: the strict parity mode (<= 5e-5 on every golden)
        # 'fp32_tc' fp32 tensors, GEMM-shaped convs (Cin % 32 == 0, Cout >= 16) and the decode heads on the 16-bit tensor cores with
        #           split operands (RDFC_PATH_UMMA_F32X3: x_hi W_hi + x_hi W_lo + x_lo W_hi, fp16 halves, fp32 accumulation):
        #           <= 1e-5 on the bench recipe, <= 2e-4 on the O(1)-activation stress goldens (the tensor cores' fp32 accumulation
        #           is not IEEE round-to-nearest), ~6-10x faster than 'fp32'
        # 'bf16'    the throughput mode
        self.precision = 'fp32'
        self.use_cuda_graph = True
        self.max_plans = 4       # plans (activation buffers + a captured graph each) kept per engine, least recently used first out
        self._plans = {}         # (B, H, W, Cs, device, precision) -> Plan, in LRU order
        self._packed = {}        # (precision, layer name) -> _Packed
        self._wver = {}          # precision -> parameter version stamp
        self._recipes = {}       # (precision, layer name) -> (sources, umma, transposed) for in-place re-packing
        self._device = None      # packed weights and plans live on ONE device; moving the module drops them

    def clear_plans(self, precision=None):
        """Drop cached plans (their activation buffers, descriptors and CUDA graphs) -- all of them, or one precision's.
        Plans are also evicted least-recently-used beyond `max_plans`.  A plan's fixed I/O buffers are shared by every call
        that hits it: calls must be issued from one stream / thread at a time (the reference's modules have the same
        single-stream contract through cuDNN workspaces)."""
        for key in [k for k in self._plans if precision is None or k[5] == precision]:
            del self._plans[key]

    # ------------------------------------------------------------------------------------------- weights --------
    def _stamp(self):
        g = self.gen
        return tuple((t.data_ptr(), t._version) for t in list(g.parameters()) + list(g.buffers()))

    @staticmethod
    def _bn_fold(bn):
        scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
        return scale, bn.bias.detach().float() - bn.running_mean.detach().float() * scale

    def _pack(self, name, sources, precision, umma, transposed=False, x3=False):
        """sources: list of (weight (Cout,Cin,kh,kw) or ConvT (Cin,Cout,kh,kw), bn module or None, bias or None),
        fused along Cout."""
        self._recipes[(precision, name)] = (sources, umma, transposed, x3)
        ws, scs, shs = [], [], []
        for w, bn, bias in sources:
            w = (w() if callable(w) else w).detach().float()
            if transposed:
                w = w.permute(1, 0, 2, 3)                # -> (Cout, Cin, kh, kw), scatter-form taps kept
            ws.append(w)
            if bn is not None:
                sc, sh = self._bn_fold(bn)
            else:
                sc = torch.ones(w.shape[0], device=w.device)
                bias = bias() if callable(bias) else bias
                sh = bias.detach().float() if bias is not None else torch.zeros(w.shape[0], device=w.device)
            scs.append(sc)
            shs.append(sh)
        packed = pack_weight(torch.cat(ws, 0), umma, x3)
        p = self._packed.setdefault((precision, name), _Packed())
        p.store(packed, torch.cat(scs).contiguous(), torch.cat(shs).contiguous())
        return p

    def _pack_nlspn(self, precision):
        pl = self.gen.nlspn_refine_module.prop_layer
        pw = self._packed.setdefault((precision, 'nlspn'), _Packed())
        pw.store(pl.conv_offset_aff.weight.detach().float(), pl.aff_scale_const.detach().float(),
                 pl.conv_offset_aff.bias.detach().float())
        return pw

    def _repack(self, precision):
        """Refresh every packed tensor of this precision in place (pointers, plans and CUDA graphs stay valid)."""
        for (prec, name), (sources, umma, transposed, x3) in list(self._recipes.items()):
            if prec == precision:
                self._pack(name, sources, precision, umma, transposed, x3)
        if (precision, 'nlspn') in self._packed:
            self._pack_nlspn(precision)

    # ------------------------------------------------------------------------------------------- plan -----------
    def _build_plan(self, B, H, W, Cs, device, precision):
        g = self.gen
        bf16 = precision == 'bf16'
        tc32 = precision == 'fp32_tc'
        adt = torch.bfloat16 if bf16 else torch.float32
        plan = Plan()
        plan.precision = precision
        def new(*shape, dtype=None):
            t = torch.empty(shape, dtype=dtype or adt, device=device)
            plan.keep.append(t)          # descriptors hold raw pointers: every buffer must live as long as the plan
            return t

        def f32(*shape):
            return new(*shape, dtype=torch.float32)

        Hs = [None, H, H, _down(H)]
        Ws = [None, W, W, _down(W)]
        for _ in range(3):
            Hs.append(_down(Hs[-1]))
            Ws.append(_down(Ws[-1]))            # index = encoder level 1..6
        chan = {2: 64, 3: 128, 4: 256, 5: 512}
        dchan = {5: 256, 4: 128, 3: 64, 2: 64}
        has_gd = g.use_nlspn_refine
        if has_gd and g.nlspn_refine_module.prop_layer.k_f != 3:
            raise NotImplementedError("the fused NLSPN kernels support prop_kernel == 3 (the reference's only setting)")

        plan.stem_in = f32(B, Cs, H, W)
        plan.depth = f32(B, 1, H, W)
        head = {'r': new(B, H, W, 160), 'd': new(B, H, W, 224 if has_gd else 160)}
        fe1 = {'r': (head['r'], 96, 64), 'd': (head['d'], 160 if has_gd else 96, 64)}
        cat = {x: {l: new(B, Hs[l], Ws[l], dchan[l] + chan[l]) for l in (2, 3, 4, 5)} for x in 'rd'}
        fe6 = {x: new(B, Hs[6], Ws[6], 512) for x in 'rd'}
        tmp = {x: {l: [new(B, Hs[l], Ws[l], chan[l]) for _ in range(4)] for l in (2, 3, 4, 5)} for x in 'rd'}   # t1, ya, yb, downsample

        def conv(name, sources, inp, out, k, stride=1, pad=None, act=C.ACT_NONE, transposed=False, residual=None,
                 in2=None, hin=None, hout=None, out_nchw=False, in_nchw=False):
            """inp/out/residual/in2: (tensor, c0, C) NHWC slices, or NCHW tensors when *_nchw."""
            pad = (k - 1) // 2 if pad is None else pad
            vin = C.view(inp, nchw=True) if in_nchw else C.view(inp[0], inp[2], inp[1])
            vin2 = C.view(None) if in2 is None else C.view(in2[0], in2[2], in2[1])
            vout = C.view(out, nchw=True) if out_nchw else C.view(out[0], out[2], out[1])
            vres = C.view(None) if residual is None else C.view(residual[0], residual[2], residual[1])
            cin = vin.C + (vin2.C if in2 is not None else 0)
            umma = (bf16 and not in_nchw and not out_nchw and in2 is None and cin % 32 == 0 and vout.C >= 16 and
                    vin.dtype == C.BF16 and vout.dtype == C.BF16)
            x3 = (tc32 and not in_nchw and not out_nchw and in2 is None and cin % 32 == 0 and
                  vout.C >= 16 and vin.dtype == C.F32 and vout.dtype == C.F32)
            pk = self._pack(name, sources, precision, umma or x3, transposed, x3)
            d = C.ConvDesc()
            d.B, (d.Hi, d.Wi), (d.Ho, d.Wo) = B, hin, hout
            d.kh = d.kw = k
            d.stride, d.pad, d.transposed, d.act = stride, pad, int(transposed), act
            d.path = C.PATH_UMMA_BF16 if umma else (C.PATH_UMMA_F32X3 if x3 else C.PATH_SIMT_F32)
            d.inp, d.in2, d.out, d.residual = vin, vin2, vout, vres
            if x3:       # the split [hi | lo] copy of the input: one scratch buffer per lane (the two lanes run concurrently)
                ws = x3_scratch[plan.cur_lane]
                assert ws.numel() >= B * hin[0] * hin[1] * cin * 4, (name, cin, hin)
                d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
            d.weight, d.scale, d.shift = pk.weight.data_ptr(), pk.scale.data_ptr(), pk.shift.data_ptr()
            plan.keep.append((d, pk))
            plan.names.append(f"conv {name} k{k} s{stride} T{int(transposed)} {vin.C}->{vout.C} {hin}->{hout} {'umma' if umma else ('umma_x3' if x3 else 'simt')}")
            if x3:
                plan.n_launch += 1
            plan.steps.append(lambda s, d=d: C.check(C.lib.rdfc_conv_forward(ctypes.byref(d), s)))
            plan.n_launch += 1

        x3_scratch = None
        if tc32:
            # largest split input: the 224-channel full-resolution head buffer (4 bytes per element, like the fp32 tensor itself)
            x3_scratch = [new(B * H * W * 224 * 4, dtype=torch.uint8) for _ in range(2)]

        def seq_src(mod):           # conv_bn_relu / convt_bn_relu Sequential -> (weight, bn, bias)
            bn = mod[1] if len(mod) > 1 and isinstance(mod[1], torch.nn.BatchNorm2d) else None
            return (mod[0].weight, bn, mod[0].bias)

        # ---- stems (rdf_generator.py:286-292): NCHW fp32 in, NHWC slice out
        L = C.ACT_LEAKY02
        full = (H, W)
        if bf16 and Cs + 1 <= 4:
            # all three stems as ONE tensor-core launch: im2col rows built by the producer warps from the fp32 NCHW inputs
            self._plan_stem(plan, B, H, W, Cs, fe1)
        elif bf16 and Cs + 1 <= 128:
            # many-channel stem input (RDF-GAN's 40-channel guidance): pack [stem | depth | 0] to bf16 NHWC once, then the
            # stems are two tensor-core 3x3 convs over it (block-sparse filters: the depth column only feeds the 1 -> 16 stem)
            Cpad = (Cs + 1 + 31) // 32 * 32
            xin = new(B, H, W, Cpad)
            plan.names.append(f'pack_stem_input {Cs}+1 -> {Cpad}')
            plan.steps.append(lambda s: C.check(C.lib.rdfc_pack_stem_input(C.ptr(plan.stem_in), Cs, C.ptr(plan.depth), C.ptr(xin),
                                                                         Cpad, B, H, W, s)))
            plan.n_launch += 1

            def padded(mod, c0):
                def f():
                    w = mod[0].weight.detach().float()
                    out = w.new_zeros(w.shape[0], Cpad, 3, 3)
                    out[:, c0:c0 + w.shape[1]] = w
                    return out
                return f

            def src(mod, c0):
                bn = mod[1] if len(mod) > 1 and isinstance(mod[1], torch.nn.BatchNorm2d) else None
                return (padded(mod, c0), bn, mod[0].bias)

            conv('rgb_branch_en1', [src(g.rgb_branch_en1, 0)], (xin, 0, Cpad), fe1['r'], 3, act=L, hin=full, hout=full)
            conv('depth_branch_en1', [src(g.depth_branch_en1_rgb, 0), src(g.depth_branch_en1_depth, Cs)], (xin, 0, Cpad), fe1['d'], 3,
                 act=L, hin=full, hout=full)
        else:
            conv('rgb_branch_en1', [seq_src(g.rgb_branch_en1)], plan.stem_in, fe1['r'], 3, act=L, in_nchw=True, hin=full, hout=full)
            conv('depth_branch_en1_rgb', [seq_src(g.depth_branch_en1_rgb)], plan.stem_in, (fe1['d'][0], fe1['d'][1], 48), 3,
                 act=L, in_nchw=True, hin=full, hout=full)
            conv('depth_branch_en1_depth', [seq_src(g.depth_branch_en1_depth)], plan.depth,
                 (fe1['d'][0], fe1['d'][1] + 48, 16), 3, act=L, in_nchw=True, hin=full, hout=full)

        # ---- encoders (rdf_generator.py:295-312)
        feat = {}
        plan.fork()
        for x, ed in (('r', g.rgb_branch_encoder_decoder), ('d', g.depth_branch_encoder_decoder)):
            plan.lane(0 if x == 'r' else 1)
            cur, hw_cur = fe1[x], full
            for l in (2, 3, 4, 5):
                layer = getattr(ed, f'en{l}')
                hw = (Hs[l], Ws[l])
                t1, ya, yb, ds = tmp[x][l]
                for bi, blk in enumerate(layer):
                    last = bi == len(layer) - 1
                    dst = (cat[x][l], dchan[l], chan[l]) if last else ((ya if bi % 2 == 0 else yb), 0, chan[l])
                    nm = f'{x}.en{l}.{bi}'
                    stride = blk.stride
                    if blk.downsample is not None:
                        conv(nm + '.ds', [(blk.downsample[0].weight, blk.downsample[1], None)], cur, (ds, 0, chan[l]), 1,
                             stride=stride, hin=hw_cur, hout=hw)
                        ident = (ds, 0, chan[l])
                    else:
                        ident = cur
                    conv(nm + '.c1', [(blk.conv1.weight, blk.bn1, None)], cur, (t1, 0, chan[l]), 3, stride=stride,
                         act=C.ACT_RELU, hin=hw_cur, hout=hw)
                    conv(nm + '.c2', [(blk.conv2.weight, blk.bn2, None)], (t1, 0, chan[l]), dst, 3, act=C.ACT_RELU,
                         residual=ident, hin=hw, hout=hw)
                    cur, hw_cur = dst, hw
                feat[(x, l)] = cur
            conv(f'{x}.en6', [seq_src(ed.en6)], cur, (fe6[x], 0, 512), 3, stride=2, act=L, hin=hw_cur, hout=(Hs[6], Ws[6]))

        plan.join()
        # ---- decoders with RGB<-depth fusion (rdf_generator.py:315-368)
        xr, xd = (fe6['r'], 0, 512), (fe6['d'], 0, 512)
        lvl_in = 6
        for n, l in enumerate((5, 4, 3, 2), start=1):
            hw_in, hw_out = (Hs[lvl_in], Ws[lvl_in]), (Hs[l], Ws[l])      # ConvT output cropped to the skip's size
            plan.fork()                  # the depth branch's ConvT only reads xd: it runs beside the fusion + RGB ConvT
            fz = self._plan_fuse(plan, conv, new, f32, getattr(g, f'fuse_layer{n}'), n, xr, xd, B, hw_in, precision)
            conv(f'r.de{l}', [seq_src(getattr(g.rgb_branch_encoder_decoder, f'de{l}'))], fz, (cat['r'][l], 0, dchan[l]), 3,
                 stride=2, pad=1, act=L, transposed=True, hin=hw_in, hout=hw_out)
            plan.lane(1)
            conv(f'd.de{l}', [seq_src(getattr(g.depth_branch_encoder_decoder, f'de{l}'))], xd, (cat['d'][l], 0, dchan[l]), 3,
                 stride=2, pad=1, act=L, transposed=True, hin=hw_in, hout=hw_out)
            plan.join()
            xr, xd = (cat['r'][l], 0, dchan[l] + chan[l]), (cat['d'][l], 0, dchan[l] + chan[l])
            lvl_in = l

        # ---- decode heads (rdf_generator.py:372-398); the *_dec1 convs that share an input run as ONE conv
        # the RGB branch's heads (lane 1) run beside the depth branch's heads and the NLSPN refinement (lane 0)
        plan.fork()
        plan.lane(1)
        conv('r.dec1', [seq_src(g.rgb_pred_dec1), seq_src(g.rgb_conf_dec1)], xr, (head['r'], 0, 96), 3, act=L, hin=full, hout=full)
        plan.lane(0)
        d_srcs = [seq_src(g.id_dec1), seq_src(g.cf_dec1)] + ([seq_src(g.gd_dec1)] if has_gd else [])
        conv('d.dec1', d_srcs, xd, (head['d'], 0, 160 if has_gd else 96), 3, act=L, hin=full, hout=full)
        plan.d1, plan.c1, plan.pred_init, plan.conf = f32(B, 1, H, W), f32(B, 1, H, W), f32(B, 1, H, W), f32(B, 1, H, W)
        if has_gd:
            plan.guide = f32(B, 8, H, W)
        P_ = H * W
        if bf16 or tc32:
            # all *_dec0 heads of a branch as ONE tensor-core conv over the whole head buffer (block-sparse filters)
            plan.lane(1)
            self._plan_heads(plan, 'r.dec0', head['r'], B, H, W, [
                dict(mod=g.rgb_pred_dec0[0], act=C.ACT_TANH, segs=[(0, 64, 0), (64, 64, 96)], out=[(plan.d1, 0, P_)]),
                dict(mod=g.rgb_conf_dec0[0], act=C.ACT_SIGMOID, segs=[(0, 32, 64), (32, 64, 96)], out=[(plan.c1, 0, P_)])],
                precision, x3_scratch)
            plan.lane(0)
            fe = 160 if has_gd else 96
            cols = [dict(mod=g.id_dec0[0], act=C.ACT_TANH, segs=[(0, 64, 0), (64, 64, fe)], out=[(plan.pred_init, 0, P_)]),
                    dict(mod=g.cf_dec0[0], act=C.ACT_SIGMOID, segs=[(0, 32, 64), (32, 64, fe)], out=[(plan.conf, 0, P_)])]
            if has_gd:
                cols.append(dict(mod=g.gd_dec0[0], act=C.ACT_NONE, segs=[(0, 64, 96), (64, 64, fe)],
                                 out=[(plan.guide, k * P_, 8 * P_) for k in range(8)]))
            self._plan_heads(plan, 'd.dec0', head['d'], B, H, W, cols, precision, x3_scratch)
        else:
            plan.lane(1)
            conv('rgb_pred_dec0', [seq_src(g.rgb_pred_dec0)], (head['r'], 0, 64), plan.d1, 3, act=C.ACT_TANH, in2=fe1['r'],
                 out_nchw=True, hin=full, hout=full)
            conv('rgb_conf_dec0', [(g.rgb_conf_dec0[0].weight, None, g.rgb_conf_dec0[0].bias)], (head['r'], 64, 96), plan.c1, 3,
                 act=C.ACT_SIGMOID, out_nchw=True, hin=full, hout=full)
            plan.lane(0)
            conv('id_dec0', [seq_src(g.id_dec0)], (head['d'], 0, 64), plan.pred_init, 3, act=C.ACT_TANH, in2=fe1['d'],
                 out_nchw=True, hin=full, hout=full)
            conv('cf_dec0', [(g.cf_dec0[0].weight, None, g.cf_dec0[0].bias)], (head['d'], 64, 32), plan.conf, 3,
                 act=C.ACT_SIGMOID, in2=fe1['d'], out_nchw=True, hin=full, hout=full)
            if has_gd:
                conv('gd_dec0', [seq_src(g.gd_dec0)], (head['d'], 96, 128), plan.guide, 3, out_nchw=True, hin=full, hout=full)

        # ---- NLSPN + output fusion (rdf_generator.py:400-406)
        plan.d2, plan.pred = f32(B, 1, H, W), f32(B, 1, H, W)
        n = B * H * W
        if has_gd:
            pl = g.nlspn_refine_module.prop_layer
            plan.scratch, plan.d2raw = f32(B, 1, H, W), f32(B, 1, H, W)
            pw = self._pack_nlspn(precision)
            plan.keep.append(pw)
            aff_mode, conf_prop, preserve, T = C.AFFINITY[pl.affinity], int(bool(pl.conf_prop)), int(bool(pl.preserve_input)), pl.prop_time
            fix = C.ptr(plan.depth) if preserve else None
            fz = C.FuseOut(plan.d1.data_ptr(), plan.c1.data_ptr(), plan.conf.data_ptr(), plan.pred.data_ptr())
            plan.keep.append(fz)
            plan.names.append('nlspn_affinity')
            if bf16:
                # bf16 mode: offsets / affinities as a packed fp16 stream (48 B instead of 100 B per pixel and iteration)
                plan.packed = new(C.lib.rdfc_nlspn_packed_bytes(B, H, W), dtype=torch.uint8)
                plan.steps.append(lambda s: C.check(C.lib.rdfc_nlspn_affinity_forward_packed(
                    C.ptr(plan.guide), C.ptr(plan.conf), C.ptr(pw.weight), C.ptr(pw.shift), C.ptr(pw.scale), aff_mode, conf_prop,
                    C.ptr(plan.packed), B, H, W, s)))

                def prop(src, dst, iters, fuse):
                    return lambda s: C.check(C.lib.rdfc_nlspn_propagate_forward_packed(
                        C.ptr(src), C.ptr(plan.packed), fix, preserve, C.ptr(dst), C.ptr(plan.scratch), B, H, W, iters, 0,
                        ctypes.byref(fz) if fuse else None, s))
            else:
                plan.offset, plan.aff = f32(B, 18, H, W), f32(B, 9, H, W)
                plan.steps.append(lambda s: C.check(C.lib.rdfc_nlspn_affinity_forward(
                    C.ptr(plan.guide), C.ptr(plan.conf), C.ptr(pw.weight), C.ptr(pw.shift), C.ptr(pw.scale), aff_mode, conf_prop,
                    C.ptr(plan.offset), C.ptr(plan.aff), B, H, W, s)))

                def prop(src, dst, iters, fuse):
                    return lambda s: C.check(C.lib.rdfc_nlspn_propagate_forward(
                        C.ptr(src), C.ptr(plan.offset), C.ptr(plan.aff), fix, preserve, C.ptr(dst), C.ptr(plan.scratch), None,
                        B, H, W, iters, 0, ctypes.byref(fz) if fuse else None, s))
            # iterations 1..T-1 beside the RGB heads; the last one applies the output fusion (clamp, confidence softmax, weighted
            # sum) in its epilogue and therefore waits for the RGB heads' d1 / c1
            src = plan.pred_init
            if T > 1:
                plan.names.append(f'nlspn_propagate x{T - 1}')
                plan.steps.append(prop(src, plan.d2raw, T - 1, False))
                src = plan.d2raw
            plan.join()
            plan.names.append('nlspn_propagate (last) + fuse_depth' if T > 0 else 'fuse_depth')
            plan.steps.append(prop(src, plan.d2, min(T, 1), True))
            plan.n_launch += 1 + max(T, 1)
        else:
            plan.join()
            plan.names.append('fuse_depth')
            plan.steps.append(lambda s: C.check(C.lib.rdfc_fuse_depth_forward(
                C.ptr(plan.d1), C.ptr(plan.c1), C.ptr(plan.pred_init), C.ptr(plan.conf), C.ptr(plan.d2), C.ptr(plan.pred), n, s)))
            plan.n_launch += 1
        plan.outputs = (plan.d1, plan.c1, plan.d2, plan.conf, plan.pred)
        return plan

    def _plan_stem(self, plan, B, H, W, Cs, fe1):
        """rgb_branch_en1 | depth_branch_en1_rgb | depth_branch_en1_depth (rdf_generator.py:286-292) as one 64 -> 128
        GEMM over im2col rows k = ci*9 + ky*3 + kx (stem input channels first, then the depth map's nine taps)."""
        g = self.gen
        K = 64

        def padded(mod, k0):
            def f():
                w = mod[0].weight.detach().float()                     # (Cout, Cin, 3, 3)
                out = w.new_zeros(w.shape[0], K, 1, 1)
                out[:, k0:k0 + w.shape[1] * 9, 0, 0] = w.reshape(w.shape[0], -1)
                return out
            return f

        def src(mod, k0):
            bn = mod[1] if len(mod) > 1 and isinstance(mod[1], torch.nn.BatchNorm2d) else None
            return (padded(mod, k0), bn, mod[0].bias)

        srcs = [src(g.rgb_branch_en1, 0), src(g.depth_branch_en1_rgb, 0), src(g.depth_branch_en1_depth, 9 * Cs)]
        pk = self._pack('stems', srcs, 'bf16', True)
        d = C.StemDesc()
        d.B, d.H, d.W = B, H, W
        d.in0, d.C0, d.in1 = plan.stem_in.data_ptr(), Cs, plan.depth.data_ptr()
        d.out = C.view(fe1['r'][0], fe1['r'][2], fe1['r'][1])
        d.out2 = C.view(fe1['d'][0], fe1['d'][2], fe1['d'][1])
        d.weight, d.scale, d.shift, d.act = pk.weight.data_ptr(), pk.scale.data_ptr(), pk.shift.data_ptr(), C.ACT_LEAKY02
        plan.keep.append((d, pk))
        plan.names.append(f'stems {Cs}+1 -> 64|64 ({H}, {W}) umma')
        plan.steps.append(lambda s, d=d: C.check(C.lib.rdfc_stem_forward(ctypes.byref(d), s)))
        plan.n_launch += 1

    def _plan_heads(self, plan, name, buf, B, H, W, cols, precision='bf16', x3_scratch=None):
        """One rdfc_heads_forward over the NHWC head buffer `buf`.  cols: dicts with the head's conv module, activation,
        channel segments (src_c0, n, dst_c0) mapping the conv's input channels onto buffer channels, and output planes
        (tensor, element offset, batch stride)."""
        Ctot = buf.shape[3]

        nc = sum(c['mod'].weight.shape[0] for c in cols)
        NP = (9 * nc + 15) // 16 * 16

        def fused_weight():
            """(NP, Ctot, 1, 1): row t * nc + q = tap t (= ky * 3 + kx) of output column q, mapped onto buffer channels."""
            wq = torch.zeros(nc, Ctot, 3, 3, device=buf.device)
            q = 0
            for c in cols:
                w = c['mod'].weight.detach().float()
                for s0, n, d0 in c['segs']:
                    wq[q:q + w.shape[0], d0:d0 + n] = w[:, s0:s0 + n]
                q += w.shape[0]
            out = torch.zeros(NP, Ctot, 1, 1, device=buf.device)
            out[:9 * nc, :, 0, 0] = wq.permute(2, 3, 0, 1).reshape(9 * nc, Ctot)
            return out

        def fused_bias():
            return torch.cat([c['mod'].bias.detach().float() for c in cols] + [torch.zeros(NP - nc, device=buf.device)])

        tc32 = precision == 'fp32_tc'
        pk = self._pack(name, [(fused_weight, None, fused_bias)], precision, True, x3=tc32)
        d = C.HeadsDesc()
        d.B, d.H, d.W = B, H, W
        d.inp = C.view(buf)
        if tc32:         # fp32 head buffer: split into fp16 halves inside the call (this lane's scratch)
            ws = x3_scratch[plan.cur_lane]
            assert ws.numel() >= B * H * W * Ctot * 4
            d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
            plan.n_launch += 1
        d.weight, d.shift = pk.weight.data_ptr(), pk.shift.data_ptr()
        q = 0
        for c in cols:
            for t, off, bstride in c['out']:
                d.act[q] = c['act']
                d.out[q] = t.data_ptr() + 4 * off
                d.out_bstride[q] = bstride
                q += 1
        d.ncols = q
        plan.keep.append((d, pk))
        plan.names.append(f'heads {name} {Ctot}->{q}')
        plan.steps.append(lambda s, d=d: C.check(C.lib.rdfc_heads_forward(ctypes.byref(d), s)))
        plan.n_launch += 1

    def _plan_fuse(self, plan, conv, new, f32, layer, n, xr, xd, B, hw, precision):
        """fuse_layer{n}(rgb feature xr, depth feature xd) -> NHWC slice (tensor, 0, C).  model_utils.py:53-129."""
        from .model_utils import IN, AdaIN, AdaptiveInstanceNorm
        Hh, Ww = hw
        Cx, Cd = xr[2], xd[2]
        nchunk = C.lib.rdfc_instnorm_nchunk(Hh * Ww)
        out = new(B, Hh, Ww, Cx)
        vx, vd, vout = C.view(xr[0], xr[2], xr[1]), C.view(xd[0], xd[2], xd[1]), C.view(out)
        plan.keep += [vx, vd, vout]

        def stats(v, Cc, unbiased, want_std):
            part, mean, rstd = f32(B, nchunk, Cc, 2), f32(B, Cc), f32(B, Cc)
            plan.keep += [part, mean, rstd]
            plan.names.append(f'instnorm_stats {Cc}ch {Hh}x{Ww}')
            plan.steps.append(lambda s: C.check(C.lib.rdfc_instnorm_stats(
                ctypes.byref(v), B, Hh, Ww, 1e-5, unbiased, want_std, C.ptr(part), C.ptr(mean), C.ptr(rstd), s)))
            plan.n_launch += 2
            return mean, rstd

        if isinstance(layer, AdaptiveInstanceNorm) and precision == 'bf16' and Cx % 64 == 0 and Cd % 32 == 0:
            # style projection + W-AdaIN apply as ONE tensor-core launch: the (B,H,W,2C) gamma/beta tensor never exists
            lin = layer.style.linear
            tile = C.lib.rdfc_wadain_tile(Cx)
            half = tile // 2
            perm = torch.cat([torch.cat([torch.arange(t * half, (t + 1) * half), Cx + torch.arange(t * half, (t + 1) * half)])
                              for t in range(2 * Cx // tile)])
            w = lambda lin=lin, perm=perm: lin.effective_weight().detach()[perm.to(lin.bias.device)].reshape(2 * Cx, Cd, 1, 1)
            bias = lambda lin=lin, perm=perm: lin.bias.detach()[perm.to(lin.bias.device)]
            pk = self._pack(f'fuse{n}.style_wadain', [(w, None, bias)], 'bf16', True)
            mean, rstd = stats(vx, Cx, 0, 0)
            d = C.WadainConvDesc()
            d.B, d.H, d.W = B, Hh, Ww
            d.style, d.x, d.out = vd, vx, vout
            d.gwbw = C.view(None)
            if layer.weighting:         # model_utils.py:84-88: per-pixel weights of gamma / beta, two 1x1 convs of x fused into one
                gwbw = new(B, Hh, Ww, 2 * Cx)
                conv(f'fuse{n}.weighting', [(layer.gamma_weight_layer.weight, None, layer.gamma_weight_layer.bias),
                                            (layer.beta_weight_layer.weight, None, layer.beta_weight_layer.bias)],
                     xr, (gwbw, 0, 2 * Cx), 1, hin=hw, hout=hw)
                d.gwbw = C.view(gwbw)
                plan.keep.append(gwbw)
            d.weight, d.bias, d.mean, d.rstd = pk.weight.data_ptr(), pk.shift.data_ptr(), mean.data_ptr(), rstd.data_ptr()
            plan.keep.append((d, pk, mean, rstd))
            plan.names.append(f'wadain_conv fuse{n} {Cd}->2x{Cx} {Hh}x{Ww}')
            plan.steps.append(lambda s, d=d: C.check(C.lib.rdfc_wadain_conv_forward(ctypes.byref(d), s)))
            plan.n_launch += 1
        elif isinstance(layer, AdaptiveInstanceNorm):
            lin = layer.style.linear
            gb = new(B, Hh, Ww, 2 * Cx)
            w = lambda lin=lin: lin.effective_weight().detach().reshape(lin.out_features, lin.in_features, 1, 1)
            conv(f'fuse{n}.style', [(w, None, lin.bias)], xd, (gb, 0, 2 * Cx), 1, hin=hw, hout=hw)
            mean, rstd = stats(vx, Cx, 0, 0)
            vgb = C.view(gb)
            vgw = vbw = None
            if layer.weighting:
                gwbw = new(B, Hh, Ww, 2 * Cx)
                conv(f'fuse{n}.weighting', [(layer.gamma_weight_layer.weight, None, layer.gamma_weight_layer.bias),
                                            (layer.beta_weight_layer.weight, None, layer.beta_weight_layer.bias)],
                     xr, (gwbw, 0, 2 * Cx), 1, hin=hw, hout=hw)
                vgw, vbw = C.view(gwbw, Cx, 0), C.view(gwbw, Cx, Cx)
            plan.keep += [vgb, vgw, vbw, gb]
            plan.names.append(f'wadain_apply {Cx}ch {Hh}x{Ww}')
            plan.steps.append(lambda s: C.check(C.lib.rdfc_wadain_apply(
                ctypes.byref(vx), ctypes.byref(vgb), ctypes.byref(vgw) if vgw is not None else None,
                ctypes.byref(vbw) if vbw is not None else None, C.ptr(mean), C.ptr(rstd), ctypes.byref(vout), B, Hh, Ww, s)))
            plan.n_launch += 1
        elif isinstance(layer, AdaIN):
            assert Cx == Cd, "AdaIN needs equal channel counts (model_utils.py:107)"
            cm, cs = stats(vx, Cx, 1, 1)
            sm, ss = stats(vd, Cd, 1, 1)
            plan.names.append(f'adain_apply {Cx}ch {Hh}x{Ww}')
            plan.steps.append(lambda s: C.check(C.lib.rdfc_adain_apply(
                ctypes.byref(vx), C.ptr(cm), C.ptr(cs), C.ptr(sm), C.ptr(ss), ctypes.byref(vout), B, Hh, Ww, s)))
            plan.n_launch += 1
        elif isinstance(layer, IN):
            both = new(B, Hh, Ww, Cx + Cd)
            for v, c0, Cc in ((vx, 0, Cx), (vd, Cx, Cd)):
                mean, rstd = stats(v, Cc, 0, 0)
                vo = C.view(both, Cc, c0)
                plan.keep.append(vo)
                plan.names.append(f'norm_apply {Cc}ch {Hh}x{Ww}')
                plan.steps.append(lambda s, v=v, mean=mean, rstd=rstd, vo=vo: C.check(C.lib.rdfc_norm_apply(
                    ctypes.byref(v), C.ptr(mean), C.ptr(rstd), ctypes.byref(vo), B, Hh, Ww, s)))
                plan.n_launch += 1
            conv(f'fuse{n}.down', [(layer.down_channel.weight, None, layer.down_channel.bias)], (both, 0, Cx + Cd),
                 (out, 0, Cx), 1, hin=hw, hout=hw)
        else:
            raise NotImplementedError(type(layer))
        return (out, 0, Cx)

    # ------------------------------------------------------------------------------------------- run ------------
    def forward(self, stem_in, depth, clone=True):
        g = self.gen
        B, Cs, H, W = stem_in.shape
        if Cs != g.semantic_channels_in:
            raise RuntimeError(f"stem input has {Cs} channels, the generator was built for {g.semantic_channels_in}")
        if tuple(depth.shape) != (B, 1, H, W):
            raise RuntimeError(f"depth must be ({B},1,{H},{W}), got {tuple(depth.shape)}")
        if H < 16 or W < 16:
            raise RuntimeError("inputs smaller than 16x16 do not survive the four stride-2 stages")
        dev = stem_in.device
        pdev = next(g.parameters()).device
        if pdev != dev or depth.device != dev:
            raise RuntimeError(f"generator parameters are on {pdev}, inputs on {dev} / {depth.device}: move the module with .to(device)")
        if self._device != dev:          # first use, or the module moved: packed weights / plans of the old device are stale
            self._plans.clear()
            self._packed.clear()
            self._recipes.clear()
            self._wver.clear()
            self._device = dev
        key = (B, H, W, Cs, dev, self.precision)
        with torch.cuda.device(dev), torch.no_grad():
            stamp = self._stamp()
            plan = self._plans.pop(key, None)
            if plan is not None:
                self._plans[key] = plan                     # most recently used last
            if plan is None:
                while len(self._plans) >= self.max_plans:
                    del self._plans[next(iter(self._plans))]
                plan = self._plans[key] = self._build_plan(B, H, W, Cs, dev, self.precision)   # packs the weights too
                self._wver[self.precision] = stamp
                plan.stem_in.copy_(stem_in)
                plan.depth.copy_(depth)
                if self.use_cuda_graph:
                    self._capture(plan)
            elif self._wver.get(self.precision) != stamp:
                self._repack(self.precision)
                self._wver[self.precision] = stamp
            plan.stem_in.copy_(stem_in)
            plan.depth.copy_(depth)
            plan.run()
            return tuple(t.clone() for t in plan.outputs) if clone else plan.outputs

    def forward_stream(self, batches, device, want=(0, 1, 2, 3, 4), pre=None):
        """Pipelined inference over an iterable of HOST batches (stem_in, depth), pinned or not.  Yields, in order, a
        tuple of pinned CPU tensors (the outputs selected by `want`, indices into (d1, c1, d2, c2, pred)).

        Three streams keep the copy engines and the SMs busy at the same time: the H2D copy of batch i+1 and the D2H
        copy of batch i-1 run while batch i is computed.  Inputs land in ping-pong staging buffers and are moved into
        the plan's fixed input buffers by a device copy just before the graph replay; outputs are moved out of the plan
        into ping-pong buffers right after it, so neither copy engine ever touches memory a running graph uses."""
        cur = torch.cuda.current_stream(device)
        h2d, d2h = torch.cuda.Stream(device), torch.cuda.Stream(device)
        slots = [dict() for _ in range(2)]
        pending = []                                       # (slot index, d2h event)
        with torch.cuda.device(device), torch.no_grad():
            for i, (stem_h, depth_h) in enumerate(batches):
                sl = slots[i % 2]
                if 'stem' not in sl or sl['stem'].shape != stem_h.shape:
                    sl['stem'] = torch.empty(stem_h.shape, dtype=torch.float32, device=device)
                    sl['depth'] = torch.empty(depth_h.shape, dtype=torch.float32, device=device)
                    sl['consumed'] = torch.cuda.Event()
                    sl['consumed'].record(cur)
                    sl['out_d'] = sl['out_h'] = None
                with torch.cuda.stream(h2d):
                    h2d.wait_event(sl['consumed'])             # the device copy of batch i-2 out of this slot is done
                    sl['stem'].copy_(stem_h, non_blocking=True)
                    sl['depth'].copy_(depth_h, non_blocking=True)
                    ev_in = torch.cuda.Event()
                    ev_in.record(h2d)
                # results of batch i-2 (same slot) must have left the slot's output buffers before we overwrite them
                while pending and pending[0][0] == i % 2:
                    _, ev, outs = pending.pop(0)
                    ev.synchronize()
                    yield outs
                cur.wait_event(ev_in)
                # `pre` (a guidance network) maps the staged first tensor to the stem input on the compute stream; forward() copies its
                # result into the plan's own input buffer right away, so the network may reuse its output buffer for the next batch
                outs_dev = self.forward(sl['stem'] if pre is None else pre(sl['stem']), sl['depth'], clone=False)
                sl['consumed'].record(cur)                     # forward() copied the staging buffers into the plan first
                if sl['out_d'] is None:
                    sl['out_d'] = [torch.empty_like(outs_dev[k]) for k in want]
                    sl['out_h'] = [torch.empty(outs_dev[k].shape, dtype=outs_dev[k].dtype).pin_memory() for k in want]
                for dst, k in zip(sl['out_d'], want):
                    dst.copy_(outs_dev[k], non_blocking=True)
                ev_out = torch.cuda.Event()
                ev_out.record(cur)
                with torch.cuda.stream(d2h):
                    d2h.wait_event(ev_out)
                    for dst, src in zip(sl['out_h'], sl['out_d']):
                        dst.copy_(src, non_blocking=True)
                    ev_done = torch.cuda.Event()
                    ev_done.record(d2h)
                pending.append((i % 2, ev_done, tuple(sl['out_h'])))
            for _, ev, outs in pending:
                ev.synchronize()
                yield outs

    @staticmethod
    def _capture(plan):
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            plan.run_eager()            # warm-up: lazy cudaFuncSetAttribute calls happen outside the capture
        cur.wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        lane1 = torch.cuda.Stream()
        with torch.cuda.graph(graph):
            if os.environ.get('RDFC_LANES', '1') == '0':      # development knob: one stream
                plan.run_eager()
            else:
                plan.run_lanes(lane1)
        plan.graph = graph
        plan.keep.append(lane1)
