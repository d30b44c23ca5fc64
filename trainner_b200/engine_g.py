"""Fused forward/backward engine of the RRDBNet generator (reference: RRDBNet_arch.py:14-163).

HBM layout: every RDB owns ONE zero-bordered ("flat") NHWC bf16 buffer [N, h+2, w+2, nf + 4*gc]
(conv_flat.cu: with the border stored, a conv tap is a row shift of the flattened matrix and one
haloed smem tile feeds all 9 taps); conv_k reads channels
[0, nf+(k-1)gc) and writes its LeakyReLU'd output into channels [nf+(k-1)gc, nf+k*gc) -- the
reference's four torch.cat copies per RDB do not exist.  conv5's epilogue writes
0.2*conv5 + x (and, for the third RDB of an RRDB, the RRDB residual too) straight into channels
[0, nf) of the NEXT RDB's buffer.  The buffers double as the saved activations for backward; the
LeakyReLU masks are recomputed from the sign of the stored outputs.

Backward keeps one gradient buffer per RDB (ring of 4): dgrad of conv_k accumulates into channels
[0, nf+(k-1)gc) in the epilogue (read-modify-write), and the LAST writer of a slice applies that
slice's LeakyReLU mask, so the slice is directly conv_{k-1}'s pre-activation gradient.
"""
import ctypes as CT
import os

import torch

from . import _lib
from ._lib import ChainDesc, ChainStage, ColsumEntry, PackCatEntry, WgradRdbEntry, lib
from .runtime import sm_count_hint
from .runtime import (ConvLayer, ContextPool, pool_for, FlatGrads, Lease, LRELU_SLOPE, P, Plan, WeightPacker,
                      add_flat, add_igemm, add_wgrad, make_conv_desc, make_flat_desc, require_device, taps_conv,
                      taps_dgrad_s1)

BF16 = torch.bfloat16


class _GContext:
    pass


class RRDBNetEngine:
    def __init__(self, net):
        self.net = net
        self.device = None
        self.pools = {}

    # ------------------------------------------------------------------ setup
    def _setup(self, device):
        net = self.net
        self.device = device
        k = net._conv_index()
        self.fea = k["fea"]
        self.hr1 = k["hr1"]
        self.rdbs = [[ConvLayer(c, "rdb%d.conv%d" % (i, j + 1)) for j, c in enumerate(convs)]
                     for i, convs in enumerate(k["rdbs"])]
        self.lr = ConvLayer(k["lr"], "LR_conv")
        self.ups = [ConvLayer(c, "upconv%d" % i) for i, c in enumerate(k["ups"])]
        self.hr0 = ConvLayer(k["hr0"], "HR_conv0")
        self.tc_layers = [l for r in self.rdbs for l in r] + [self.lr] + self.ups + [self.hr0]
        # RDB input gradients use the GATHER form: for each channel slice s of the block's buffer
        # (x, x1..x4) ONE conv over the concatenated pre-activation gradients of all later convs,
        # instead of 5 read-modify-write dgrads (profiles/r01_flat_v0_timeline.txt: the RMW epilogue
        # dominated).  Wcat[r][s] : [9 taps][N_s rows = slice channels][K = dY_{s+1..4} | dO] bf16.
        nf, gc = net.nf, net.gc
        cat_entries = []
        self.wcat = []
        for r, convs in enumerate(self.rdbs):
            for l in convs:
                l.need_dgrad = False
            a = 0.04 if r % 3 == 2 else 0.2
            per_slice = []
            for sl in range(5):
                n_s = nf if sl == 0 else gc
                lo = 0 if sl == 0 else nf + (sl - 1) * gc
                k1 = (4 - sl) * gc
                k1p = (k1 + 63) // 64 * 64
                cols = k1p + nf
                wt = torch.zeros(9, n_s, cols, dtype=BF16, device=device)
                for kk in range(sl, 4):       # convs sl+1..4 (index kk), dY at G channels [nf+kk*gc, +gc)
                    cv = convs[kk]
                    cat_entries.append(PackCatEntry(cv.weight.data_ptr(), wt.data_ptr(), gc, cv.cin, 9, lo, n_s, n_s,
                                                    cols, (kk - sl) * gc, 1.0, 0, 1, 0))
                cv = convs[4]
                cat_entries.append(PackCatEntry(cv.weight.data_ptr(), wt.data_ptr(), nf, cv.cin, 9, lo, n_s, n_s, cols,
                                                k1p, a, 0, 1, 0))
                per_slice.append((wt, n_s, lo, k1, cols))
            self.wcat.append(per_slice)
        # Whole-trunk chain (csrc/rdb_chain.cu): stage-merged dense blocks with the slices kept in shared memory
        # and ONE launch per image group for all dense blocks -- the default trunk path (B200_TRUNK_CHAIN=0: the
        # per-conv flat kernels).  Shapes it does not cover (w > 125, nf != 64, gc != 32) use the flat kernels.
        #   forward  stage j: rows = outputs of conv_{j+1}..conv5 (192-32j), cols = the stage's input slice
        #   backward stage j: rows = slices x_{4-j}..x (TMEM column order), cols = dY of conv_{5-j}
        self.chain = os.environ.get("B200_TRUNK_CHAIN", "1") == "1" and nf == 64 and gc == 32
        nrdb_ = len(self.rdbs)
        if self.chain:
            # stage weights of all blocks, contiguous per stage: WF[j][r], WB[j][nrdb-1-r] (chain order of the backward)
            self.WF = [torch.zeros(nrdb_, 9, 192 - 32 * j, nf if j == 0 else gc, dtype=BF16, device=device) for j in range(5)]
            self.WB = [torch.zeros(nrdb_, 9, 192 - 32 * j, nf if j == 0 else gc, dtype=BF16, device=device) for j in range(5)]
            for r, convs in enumerate(self.rdbs):
                a = 0.04 if r % 3 == 2 else 0.2
                for j in range(5):
                    n_j = 192 - 32 * j
                    kc = nf if j == 0 else gc   # stage input channels = packed K width (64 or 32)
                    tf = self.WF[j][r]
                    tb = self.WB[j][nrdb_ - 1 - r]
                    ci_off, n_ci = (0, nf) if j == 0 else (nf + (j - 1) * gc, gc)
                    for kk in range(j, 5):
                        cv = convs[kk]
                        cat_entries.append(PackCatEntry(cv.weight.data_ptr(), tf.data_ptr(), cv.cout, cv.cin, 9, ci_off,
                                                        n_ci, n_j, kc, 0, 1.0, gc * (kk - j), 0, 0))
                    cv = convs[4 - j]   # the conv whose dY is this backward stage's input
                    for sp in range(j, 5):
                        so, sn = (nf + (3 - sp) * gc, gc) if sp < 4 else (0, nf)
                        cat_entries.append(PackCatEntry(cv.weight.data_ptr(), tb.data_ptr(), cv.cout, cv.cin, 9, so, sn,
                                                        n_j, kc, 0, a if j == 0 else 1.0, gc * (sp - j), 1, 0))
        self.packer = WeightPacker(self.tc_layers, device, cat_entries)
        self.grads = FlatGrads(list(net.parameters()), device)
        self.pools = {}

    def _ensure(self, x):
        require_device(x, "RRDBNet")
        if self.device != x.device or self.packer.stale_pointers():
            self._setup(x.device)

    @staticmethod
    def _chain_geometry(n, h, w):
        """(CTAs, exchange-buffer bytes, supported) of one rdb_chain launch over n images"""
        n_cta, ll = CT.c_int32(0), CT.c_int64(0)
        rc = lib.b200_rdb_chain_geometry(n, h, w, CT.byref(n_cta), CT.byref(ll))
        return n_cta.value, ll.value, rc == 0

    def _chain_groups(self, N, h, w):
        """image groups of one rdb_chain launch: as many images as give <= #SM 256-position super-tiles (one per CTA,
        all co-resident); None when the geometry is not supported (image too wide for the shared-memory regions)"""
        if not self._chain_geometry(1, h, w)[2]:
            return None
        g = (sm_count_hint() * 256) // ((h + 2) * (w + 2))
        if g < 1:
            return None
        return [(i, min(g, N - i)) for i in range(0, N, g)]

    # ------------------------------------------------------------------ plans
    def _make_context(self, N, h, w):
        net = self.net
        nf, gc, S = net.nf, net.gc, net.upscale
        C = nf + 4 * gc
        dev = self.device
        nrdb = len(self.rdbs)
        ctx = _GContext()
        ctx.shape = (N, h, w)
        e = lambda *s: torch.empty(*s, dtype=BF16, device=dev)
        ctx.x = torch.empty(N, net.in_nc, h, w, dtype=torch.float32, device=dev)
        z = lambda *s: torch.zeros(*s, dtype=BF16, device=dev)
        ctx.B = [z(N, h + 2, w + 2, C) for _ in range(nrdb)] + [z(N, h + 2, w + 2, nf)]   # flat, zero border
        Bc = [C] * nrdb + [nf]
        ctx.F0 = e(N, h, w, nf)
        # upsampler chain.  upconv: U[i] is the (already nearest-upsampled) input of upconv i.
        # pixelshuffle (block.py:374-387): U[i] is the input of conv i at ITS resolution and Z[i] the
        # 4*nf-channel pre-shuffle conv output.
        self.shuffle = (net.upsample_mode == "pixelshuffle")
        ctx.U, ctx.Z = [], []
        hh, ww = h, w
        for _ in self.ups:
            if self.shuffle:
                ctx.U.append(e(N, hh, ww, nf))
                ctx.Z.append(e(N, hh, ww, 4 * nf))
            hh, ww = hh * 2, ww * 2
            if not self.shuffle:
                ctx.U.append(e(N, hh, ww, nf))
        H, W = hh, ww
        ctx.V = e(N, H, W, nf)    # output of the last upconv (or of LR_conv when there is none)
        ctx.Wt = e(N, H, W, nf)   # output of HR_conv0
        ctx.out = torch.empty(N, net.out_nc, H, W, dtype=torch.float32, device=dev)
        ctx.HW = (H, W)

        # ---------------- forward plan
        f = Plan()
        f.add(lib.b200_conv3x3_thin_to_wide, P(ctx.x), P(self.fea.weight), P(self.fea.bias), P(ctx.F0),
              N, h, w, net.in_nc, nf, nf, 0, 0, None, None, 0, 0.0, None, 0, 0, 0.0)
        f.add(lib.b200_pad_copy, P(ctx.B[0]), Bc[0], 0, P(ctx.F0), nf, 0, N, h, w, nf)
        ctx.chain_groups = self._chain_groups(N, h, w) if self.chain else None
        use_chain = ctx.chain_groups is not None
        if use_chain:
            ll_bytes = max(self._chain_geometry(gn, h, w)[1] for _, gn in ctx.chain_groups)
            ctx.ll = torch.zeros(ll_bytes, dtype=torch.uint8, device=dev)
            ctx.epoch = torch.zeros(1, dtype=torch.int32, device=dev)
            entries = []
            for r, convs in enumerate(self.rdbs):
                Bi, Bo = ctx.B[r], ctx.B[r + 1]
                last_of_rrdb = (r % 3 == 2)
                for j in range(5):
                    e = ChainStage()
                    e.bias = convs[j].bias.data_ptr()
                    e.alpha, e.slope = 1.0, LRELU_SLOPE
                    if j < 4:
                        e.out, e.out_c, e.out_coff, e.act = Bi.data_ptr(), C, nf + j * gc, 1
                    else:
                        e.out, e.out_c, e.out_coff, e.act = Bo.data_ptr(), Bc[r + 1], 0, 0
                        e.alpha = 0.04 if last_of_rrdb else 0.2
                        e.res1, e.res1_c, e.res1_coff, e.beta1 = Bi.data_ptr(), C, 0, (0.2 if last_of_rrdb else 1.0)
                        if last_of_rrdb:
                            e.res2, e.res2_c, e.res2_coff, e.beta2 = ctx.B[r - 2].data_ptr(), C, 0, 1.0
                    entries.append(e)
            ctx.chain_tab_f = torch.frombuffer(bytearray(bytes((ChainStage * len(entries))(*entries))),
                                               dtype=torch.uint8).to(dev)
            ctx.chain_wf = (CT.c_void_p * 5)(*[t.data_ptr() for t in self.WF])
            rdb_flops = 2.0 * h * w * 9 * (nf * gc + (nf + gc) * gc + (nf + 2 * gc) * gc + (nf + 3 * gc) * gc + C * nf)
            for (g0, gn) in ctx.chain_groups:
                d = ChainDesc(N, g0, gn, h, w, C, 0, nrdb, 0)
                f.keep(d)
                f.add(lib.b200_rdb_chain, CT.byref(d), P(ctx.B[0]), ctx.chain_wf, P(ctx.chain_tab_f), P(ctx.ll), ll_bytes,
                      P(ctx.epoch), flops=rdb_flops * gn * nrdb, tag="rdb_chain", info="fwd %d img x %d blocks" % (gn, nrdb))
        for r, convs in enumerate([] if use_chain else self.rdbs):
            Bi, Bo = ctx.B[r], ctx.B[r + 1]
            last_of_rrdb = (r % 3 == 2)
            a = 0.04 if last_of_rrdb else 0.2
            b1 = 0.2 if last_of_rrdb else 1.0
            for kk in range(4):
                L = convs[kk]
                cin = nf + kk * gc
                d = make_flat_desc(N, h, w, C, 0, cin, C, cin, gc, taps_conv(3, 1), L.taps, L.fwd_rows, L.fwd_cols,
                                   act=1, slope=LRELU_SLOPE)
                add_flat(f, d, Bi, L.w_fwd, L.bias, y=Bi)
            L = convs[4]
            d = make_flat_desc(N, h, w, C, 0, C, Bc[r + 1], 0, nf, taps_conv(3, 1), L.taps, L.fwd_rows, L.fwd_cols,
                               alpha=a, beta1=b1, res_nch=nf, res1_c=C, res1_coff=0,
                               beta2=1.0 if last_of_rrdb else 0.0, res2_c=C, res2_coff=0)
            add_flat(f, d, Bi, L.w_fwd, L.bias, res1=Bi, res2=ctx.B[r - 2] if last_of_rrdb else None, y=Bo)
        # LR_conv + shortcut (+ nearest x2 folded into the store when an upconv follows); dense output
        L = self.lr
        first_dst = ctx.U[0] if self.ups else ctx.V
        d = make_flat_desc(N, h, w, nf, 0, nf, nf, 0, nf, taps_conv(3, 1), L.taps, L.fwd_rows, L.fwd_cols,
                           out_mode=2 if (self.ups and not self.shuffle) else 1, beta1=1.0, res_nch=nf,
                           res1_c=Bc[0], res1_coff=0)
        add_flat(f, d, ctx.B[nrdb], L.w_fwd, L.bias, res1=ctx.B[0], y=first_dst)
        hh, ww = h, w
        for i, L in enumerate(self.ups if self.shuffle else []):
            # conv nf -> 4 nf at (hh, ww), then PixelShuffle(2) + LeakyReLU into the next stage's input
            lastu = (i == len(self.ups) - 1)
            d = make_conv_desc(N, hh, ww, nf, 0, nf, hh, ww, hh, ww, 4 * nf, 0, 4 * nf, taps_conv(3, 1), L.taps,
                               L.fwd_rows, L.fwd_cols)
            add_igemm(f, d, ctx.U[i], L.w_fwd, L.bias, y=ctx.Z[i])
            f.add(lib.b200_pixel_shuffle2, P(ctx.Z[i]), P(ctx.V if lastu else ctx.U[i + 1]), N, hh, ww, nf, 1,
                  LRELU_SLOPE)
            hh, ww = hh * 2, ww * 2
        for i, L in enumerate([] if self.shuffle else self.ups):
            hh, ww = hh * 2, ww * 2
            lastu = (i == len(self.ups) - 1)
            dst = ctx.V if lastu else ctx.U[i + 1]
            d = make_conv_desc(N, hh, ww, nf, 0, nf, hh, ww, hh if lastu else 2 * hh, ww if lastu else 2 * ww,
                               nf, 0, nf, taps_conv(3, 1), L.taps, L.fwd_rows, L.fwd_cols,
                               upsample=0 if lastu else 1, act=1, slope=LRELU_SLOPE)
            add_igemm(f, d, ctx.U[i], L.w_fwd, L.bias, y=dst)
        L = self.hr0
        d = make_conv_desc(N, H, W, nf, 0, nf, H, W, H, W, nf, 0, nf, taps_conv(3, 1), L.taps, L.fwd_rows,
                           L.fwd_cols, act=1, slope=LRELU_SLOPE)
        add_igemm(f, d, ctx.V, L.w_fwd, L.bias, y=ctx.Wt)
        f.add(lib.b200_conv3x3_wide_to_thin, P(ctx.Wt), P(self.hr1.weight), P(self.hr1.bias), P(ctx.out),
              N, H, W, nf, nf, 0, net.out_nc, 0, None, 1.0)
        ctx.fwd = f
        ctx.bwd = None
        return ctx

    def _make_backward(self, ctx):
        net = self.net
        nf, gc = net.nf, net.gc
        CC = nf + 4 * gc
        N, h, w = ctx.shape
        H, W = ctx.HW
        dev = self.device
        nrdb = len(self.rdbs)
        g = self.grads.view
        e = lambda *s: torch.empty(*s, dtype=BF16, device=dev)
        ctx.dout = torch.empty(N, net.out_nc, H, W, dtype=torch.float32, device=dev)
        ctx.dWt = e(N, H, W, nf)
        ctx.dV = e(N, H, W, nf)
        ctx.dU = [e(*u.shape) for u in ctx.U]
        ctx.dP = [] if self.shuffle else [e(u.shape[0], u.shape[1] // 2, u.shape[2] // 2, nf) for u in ctx.U]
        ctx.dZ = [e(*z_.shape) for z_ in ctx.Z]
        # one flat gradient buffer per RDB (kept until the batched weight-gradient kernel has run:
        # 70 x 27 MB at config 2 -- HBM is 180 GB, launch count and atomics are the scarce resource)
        ctx.G = [torch.zeros(N, h + 2, w + 2, CC, dtype=BF16, device=dev) for _ in range(nrdb + 1)]
        ctx.dFea = e(N, h, w, nf)
        Hp, Wp = h + 2, w + 2
        b = Plan()
        SL = LRELU_SLOPE
        # HR_conv1 (wide->thin) backward
        b.add(lib.b200_conv3x3_thin_to_wide, P(ctx.dout), P(self.hr1.weight), None, P(ctx.dWt), N, H, W,
              net.out_nc, nf, nf, 0, 1, None, None, 0, 0.0, P(ctx.Wt), nf, 0, SL)
        b.add(lib.b200_conv3x3_thin_wgrad, P(ctx.dout), P(ctx.Wt), P(g(self.hr1.weight)), None,
              P(g(self.hr1.bias)), N, H, W, net.out_nc, nf, nf, 0, 0, None, None)
        # HR_conv0
        L = self.hr0
        d = make_conv_desc(N, H, W, nf, 0, nf, H, W, H, W, nf, 0, nf, taps_dgrad_s1(3, 1), L.taps, L.dgr_rows,
                           L.dgr_cols, mask_c=nf, mask_coff=0, mask_lo=0, mask_hi=nf, mask_slope=SL)
        add_igemm(b, d, ctx.dWt, L.w_dgr, mask=ctx.V, y=ctx.dV)
        add_wgrad(b, N, H, W, nf, 0, nf, H, W, nf, 0, nf, 3, 1, 1, 1.0, ctx.V, ctx.dWt, g(L.weight), g(L.bias))
        # upconvs, last to first.  dcur = gradient wrt the pre-activation of upconv i's conv output
        dcur = ctx.dV
        hh, ww = H, W
        for i in range(len(self.ups) - 1, -1, -1) if self.shuffle else []:
            # dcur = gradient wrt shuffle(Z[i]) (the LeakyReLU mask was applied by the consumer's dgrad)
            L = self.ups[i]
            hh, ww = hh // 2, ww // 2
            b.add(lib.b200_pixel_unshuffle2, P(dcur), P(ctx.dZ[i]), N, hh, ww, nf)
            add_wgrad(b, N, hh, ww, nf, 0, nf, hh, ww, 4 * nf, 0, 4 * nf, 3, 1, 1, 1.0, ctx.U[i], ctx.dZ[i],
                      g(L.weight), g(L.bias))
            if i > 0:   # U[i] = lrelu(shuffle(Z[i-1])) carries the mask of the previous stage
                d = make_conv_desc(N, hh, ww, 4 * nf, 0, 4 * nf, hh, ww, hh, ww, nf, 0, nf, taps_dgrad_s1(3, 1),
                                   L.taps, L.dgr_rows, L.dgr_cols, mask_c=nf, mask_coff=0, mask_lo=0, mask_hi=nf,
                                   mask_slope=SL)
                add_igemm(b, d, ctx.dZ[i], L.w_dgr, mask=ctx.U[i], y=ctx.dU[i])
            else:
                d = make_conv_desc(N, hh, ww, 4 * nf, 0, 4 * nf, hh, ww, hh, ww, nf, 0, nf, taps_dgrad_s1(3, 1),
                                   L.taps, L.dgr_rows, L.dgr_cols)
                add_igemm(b, d, ctx.dZ[i], L.w_dgr, y=ctx.dU[i])
            dcur = ctx.dU[i]
        for i in range(len(self.ups) - 1, -1, -1) if not self.shuffle else []:
            L = self.ups[i]
            d = make_conv_desc(N, hh, ww, nf, 0, nf, hh, ww, hh, ww, nf, 0, nf, taps_dgrad_s1(3, 1), L.taps,
                               L.dgr_rows, L.dgr_cols)
            add_igemm(b, d, dcur, L.w_dgr, y=ctx.dU[i])
            add_wgrad(b, N, hh, ww, nf, 0, nf, hh, ww, nf, 0, nf, 3, 1, 1, 1.0, ctx.U[i], dcur, g(L.weight),
                      g(L.bias))
            hh, ww = hh // 2, ww // 2
            # undo the nearest upsample; U[i] = up(lrelu(conv_{i-1})) for i > 0 carries the mask
            b.add(lib.b200_sumpool2x2_mask, P(ctx.dU[i]), P(ctx.U[i]) if i > 0 else None, P(ctx.dP[i]), N, hh,
                  ww, nf, SL)
            dcur = ctx.dP[i]
        dT = dcur  # gradient wrt (fea + LR_conv(trunk)) at LR resolution
        slot = lambda r: ctx.G[r]
        L = self.lr
        # dT is dense [N,h,w,nf]; its dgrad lands in the interior of the flat gradient buffer
        d = make_conv_desc(N, h, w, nf, 0, nf, h, w, Hp, Wp, CC, 0, nf, taps_dgrad_s1(3, 1), L.taps, L.dgr_rows,
                           L.dgr_cols, out_off=(1, 1))
        add_igemm(b, d, dT, L.w_dgr, y=slot(nrdb))
        # x flat (its own border is the conv's zero padding -> pad 0 on the flat grid), dy dense
        add_wgrad(b, N, Hp, Wp, nf, 0, nf, h, w, nf, 0, nf, 3, 1, 0, 1.0, ctx.B[nrdb], dT, g(L.weight), g(L.bias))
        use_chain = ctx.chain_groups is not None
        if use_chain:
            entries = []
            for r in range(nrdb - 1, -1, -1):
                Gr, dO, Br = slot(r), slot(r + 1), ctx.B[r]
                last_of_rrdb, first_of_rrdb = (r % 3 == 2), (r % 3 == 0)
                for j in range(5):
                    e = ChainStage()
                    e.alpha, e.mask_slope = 1.0, SL
                    e.out, e.out_c = Gr.data_ptr(), CC
                    if j < 4:
                        e.out_coff = nf + (3 - j) * gc
                        e.mask, e.mask_c, e.mask_coff = Br.data_ptr(), CC, nf + (3 - j) * gc
                    else:
                        e.out_coff = 0
                        e.res1, e.res1_c, e.res1_coff, e.beta1 = dO.data_ptr(), CC, 0, (0.2 if last_of_rrdb else 1.0)
                        if first_of_rrdb:
                            e.res2, e.res2_c, e.res2_coff, e.beta2 = slot(r + 3).data_ptr(), CC, 0, 1.0
                    entries.append(e)
            ctx.chain_tab_b = torch.frombuffer(bytearray(bytes((ChainStage * len(entries))(*entries))),
                                               dtype=torch.uint8).to(dev)
            ctx.chain_wb = (CT.c_void_p * 5)(*[t.data_ptr() for t in self.WB])
            rdb_flops = 2.0 * h * w * 9 * (nf * gc + (nf + gc) * gc + (nf + 2 * gc) * gc + (nf + 3 * gc) * gc + CC * nf)
            for (g0, gn) in ctx.chain_groups:
                d = ChainDesc(N, g0, gn, h, w, CC, 0, nrdb, 1)
                b.keep(d)
                b.add(lib.b200_rdb_chain, CT.byref(d), P(slot(nrdb)), ctx.chain_wb, P(ctx.chain_tab_b), P(ctx.ll),
                      ctx.ll.numel(), P(ctx.epoch), flops=rdb_flops * gn * nrdb, tag="rdb_chain",
                      info="bwd %d img x %d blocks" % (gn, nrdb))
        for r in range(nrdb - 1, -1, -1) if not use_chain else []:
            convs = self.rdbs[r]
            Gr, dO, Br = slot(r), slot(r + 1), ctx.B[r]
            last_of_rrdb = (r % 3 == 2)
            first_of_rrdb = (r % 3 == 0)
            a = 0.04 if last_of_rrdb else 0.2
            b1 = 0.2 if last_of_rrdb else 1.0
            for sl in range(4, -1, -1):
                wt, n_s, lo, k1, cols = self.wcat[r][sl]
                kw = dict(cx2=CC, cin2_off=0, cin2=nf)
                if sl == 0:
                    kw.update(beta1=b1, res_nch=nf, res1_c=CC, res1_coff=0, beta2=1.0 if first_of_rrdb else 0.0,
                              res2_c=CC, res2_coff=0)
                else:
                    kw.update(mask_c=CC, mask_coff=lo, mask_lo=0, mask_hi=n_s, mask_slope=SL)
                d = make_flat_desc(N, h, w, CC, nf + sl * gc, k1, CC, lo, n_s, taps_dgrad_s1(3, 1), 9, n_s, cols, **kw)
                add_flat(b, d, Gr if k1 else None, wt, x2=dO,
                         res1=dO if sl == 0 else None,
                         res2=slot(r + 3) if (sl == 0 and first_of_rrdb) else None,
                         mask=Br if sl > 0 else None, y=Gr)
        # ---- weight / bias gradients of all RDB convs: ONE batched tcgen05 kernel + one column-sum kernel
        P_pos = N * Hp * Wp
        tmb = lib.b200_tensor_map_bytes()
        maps_host = torch.empty(3 * nrdb * tmb + 64, dtype=torch.uint8)
        base = (maps_host.data_ptr() + 63) // 64 * 64
        vp = lambda xs: (CT.c_void_p * len(xs))(*xs)
        pitches = (CT.c_int32 * nrdb)(*([CC] * nrdb))
        _lib.check(lib.b200_wgrad_rdb_make_maps(base, nrdb, vp([ctx.B[r].data_ptr() for r in range(nrdb)]),
                                                vp([ctx.G[r].data_ptr() for r in range(nrdb)]),
                                                vp([ctx.G[r + 1].data_ptr() for r in range(nrdb)]), pitches,
                                                N, h, w, CC), "wgrad_rdb_make_maps")
        off = base - maps_host.data_ptr()
        ctx.wg_maps = maps_host[off:off + 3 * nrdb * tmb].clone().to(dev)
        entries, sums = [], []
        for r, convs in enumerate(self.rdbs):
            a = 0.04 if r % 3 == 2 else 0.2
            e = WgradRdbEntry()
            for kk in range(5):
                e.dw[kk] = g(convs[kk].weight).data_ptr()
            e.scale5 = a
            entries.append(e)
            for kk in range(4):
                sums.append(ColsumEntry(ctx.G[r].data_ptr(), g(convs[kk].bias).data_ptr(), P_pos, CC, nf + kk * gc, gc, 1.0))
            sums.append(ColsumEntry(ctx.G[r + 1].data_ptr(), g(convs[4].bias).data_ptr(), P_pos, CC, 0, nf, a))
        to_dev = lambda arr: torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
        ctx.wg_entries = to_dev((WgradRdbEntry * len(entries))(*entries))
        ctx.wg_sums = to_dev((ColsumEntry * len(sums))(*sums))
        ws_bytes = int(lib.b200_wgrad_rdb_ws_bytes(nrdb, N, h, w))
        ctx.wg_ws = torch.empty(max(ws_bytes, 4) // 4, dtype=torch.float32, device=dev)
        b.add(lib.b200_wgrad_rdb, P(ctx.wg_maps), P(ctx.wg_entries), nrdb, N, h, w, nf, gc, P(ctx.wg_ws), ws_bytes,
              flops=2.0 * N * h * w * 9 * nrdb * (nf * gc + (nf + gc) * gc + (nf + 2 * gc) * gc + (nf + 3 * gc) * gc + CC * nf),
              tag="wgrad_rdb", info="%d RDBs" % nrdb)
        b.add(lib.b200_colsum_multi, P(ctx.wg_sums), len(sums))
        # shortcut: d(fea) = interior(G[0][0:nf]) + dT  (dense), then the thin conv's weight gradient
        G0 = slot(0)
        b.add(lib.b200_unpad_add, P(ctx.dFea), nf, P(G0), CC, 0, P(dT), nf, N, h, w, nf)
        b.add(lib.b200_conv3x3_thin_wgrad, P(ctx.x), P(ctx.dFea), P(g(self.fea.weight)), P(g(self.fea.bias)), None,
              N, h, w, net.in_nc, nf, nf, 0, 1, None, None)
        ctx.bwd = b

    # ------------------------------------------------------------------ run
    def forward(self, x, need_backward):
        self._ensure(x)
        N, _, h, w = x.shape
        key = (N, h, w)
        pool = pool_for(self.pools, key, lambda: self._make_context(N, h, w))
        ctx = pool.acquire()
        self.packer.ensure()
        ctx.x.copy_(x)
        ctx.fwd.run()
        out = ctx.out.clone()
        if need_backward:
            return out, Lease(pool, ctx)
        pool.release(ctx)
        return out, None

    def backward(self, lease, dout):
        ctx = lease.ctx
        if ctx.bwd is None:
            self._make_backward(ctx)
        self.grads.attach()
        ctx.dout.copy_(dout)
        ctx.bwd.run()
        lease.release()
