"""Fused forward/backward engine of the VGG-style discriminator feature stack
(reference: architectures/discriminators.py:16-51, block.py:113-133 BatchNorm2d, block.py:91 LeakyReLU).

Per layer: tcgen05 implicit-GEMM conv (+bias) -> bf16 pre-BN tensor Z; warp/shared-memory
reduction of per-channel sum / sum-of-squares in fp32; one fused BN-apply + LeakyReLU pass.
Only Z is kept for backward (the activation and its LeakyReLU mask are recomputed from Z and the
batch statistics).  Every train-mode forward updates running_mean / running_var /
num_batches_tracked exactly like nn.BatchNorm2d (4 updates per training iteration, SURVEY 7.5).
"""
import weakref

import torch

from ._lib import BnFinalizeEntry, lib
from .runtime import (ConvLayer, ContextPool, pool_for, FlatGrads, Lease, LRELU_SLOPE, P, Plan, WeightPacker,
                      add_igemm, add_igemm_stats, igemm_stat_rows, add_wgrad, make_conv_desc, require_device, taps_conv, taps_dgrad_s1,
                      taps_dgrad_s2_k4)

BF16 = torch.bfloat16


class _DContext:
    pass


class DiscriminatorEngine:
    def __init__(self, net):
        self.net = net
        self.device = None
        self.pools = {}
        # Forward reuse: within one generation of the weights, D(x) of the SAME input tensor is
        # value-identical, so the second call (D-step after G-step: losses.py:400-403 vs :475-476)
        # only repeats the BatchNorm running-stat update.  Off by default; the owner of the
        # optimizer (models/sr_model.py) switches it on.
        self.reuse = False
        self._cache = {}

    def _setup(self, device):
        net = self.net
        self.device = device
        feats = list(net.features)
        self.conv0 = feats[0]
        self.layers = []  # (ConvLayer, bn)
        i = 2
        while i < len(feats):
            conv, bn = feats[i], feats[i + 1]
            assert isinstance(conv, torch.nn.Conv2d) and isinstance(bn, torch.nn.BatchNorm2d)
            self.layers.append((ConvLayer(conv, "features.%d" % i), bn))
            i += 3
        self.packer = WeightPacker([l for l, _ in self.layers], device)
        self.grads = FlatGrads(list(net.features.parameters()), device)
        self.pools = {}

    def _ensure(self, x):
        require_device(x, "Discriminator_VGG")
        if self.device != x.device or self.packer.stale_pointers():
            self._setup(x.device)

    # ------------------------------------------------------------------ plans
    def _make_context(self, N, S):
        net = self.net
        dev = self.device
        ctx = _DContext()
        ctx.N, ctx.S = N, S
        e = lambda *s: torch.empty(*s, dtype=BF16, device=dev)
        c0 = self.conv0.out_channels
        ctx.x = torch.empty(N, net.in_nc, S, S, dtype=torch.float32, device=dev)
        ctx.A = [e(N, S, S, c0)]
        ctx.Z, ctx.stats, ctx.mi, ctx.dims = [], [], [], []
        ctx.stat_part = [None] * len(self.layers)
        h = S
        for L, bn in self.layers:
            ho = (h + 2 * L.pad - L.kh) // L.stride + 1
            ctx.Z.append(e(N, ho, ho, L.cout))
            ctx.A.append(e(N, ho, ho, L.cout))
            ctx.stats.append(torch.empty(2 * L.cout, dtype=torch.float32, device=dev))
            ctx.mi.append(torch.empty(2 * L.cout, dtype=torch.float32, device=dev))
            ctx.dims.append((h, ho))
            h = ho
        ctx.hf = h
        cl = self.layers[-1][0].cout if self.layers else c0
        ctx.feat = torch.empty(N, cl, h, h, dtype=torch.float32, device=dev)
        SL = LRELU_SLOPE

        def fwd_plan(train):
            f = Plan()
            f.add(lib.b200_conv3x3_thin_to_wide, P(ctx.x), P(self.conv0.weight), P(self.conv0.bias), P(ctx.A[0]),
                  N, S, S, net.in_nc, c0, c0, 0, 0, None, None, 1, SL, None, 0, 0, 0.0)
            for i, (L, bn) in enumerate(self.layers):
                hi, ho = ctx.dims[i]
                d = make_conv_desc(N, hi, hi, L.cin, 0, L.cin, ho, ho, ho, ho, L.cout, 0, L.cout,
                                   taps_conv(L.kh, L.pad), L.taps, L.fwd_rows, L.fwd_cols, in_stride=L.stride)
                npix = N * ho * ho
                rows = igemm_stat_rows(d) if train else 0
                if rows:
                    # batch statistics from the conv epilogue (per-tile partial sums) where the conv kernel offers it,
                    # instead of a pass over Z
                    if ctx.stat_part[i] is None:
                        ctx.stat_part[i] = torch.empty(2 * L.cout * rows, dtype=torch.float32, device=dev)
                    add_igemm_stats(f, d, ctx.A[i], L.w_fwd, L.bias, ctx.Z[i], ctx.stat_part[i])
                    f.add(lib.b200_bn_partials_finalize, P(ctx.stat_part[i]), rows, P(ctx.stats[i]), P(ctx.mi[i]),
                          P(bn.running_mean), P(bn.running_var), npix, L.cout, float(bn.momentum), float(bn.eps))
                else:
                    add_igemm(f, d, ctx.A[i], L.w_fwd, L.bias, y=ctx.Z[i])
                if train and not rows:
                    f.add(lib.b200_bn_stats_finalize, P(ctx.Z[i]), P(ctx.stats[i]), P(ctx.mi[i]),
                          P(bn.running_mean), P(bn.running_var), npix, L.cout, float(bn.momentum), float(bn.eps))
                f.add(lib.b200_bn_apply_lrelu, P(ctx.Z[i]), P(ctx.mi[i]), P(bn.weight), P(bn.bias),
                      P(ctx.A[i + 1]), npix, L.cout, SL)
            f.add(lib.b200_nhwc_bf16_to_nchw_f32, P(ctx.A[-1]), P(ctx.feat), N, cl, ctx.hf, ctx.hf, cl, 0)
            return f

        ctx.fwd_train = fwd_plan(True)
        ctx.fwd_eval = fwd_plan(False)
        rf = Plan()   # the running-stat side effect of a train-mode forward, replayed on forward reuse: ONE launch
        ents = [BnFinalizeEntry(ctx.stats[i].data_ptr(), ctx.mi[i].data_ptr(), bn.running_mean.data_ptr(),
                                bn.running_var.data_ptr(), N * ctx.dims[i][1] * ctx.dims[i][1], L.cout,
                                float(bn.momentum), float(bn.eps), 0) for i, (L, bn) in enumerate(self.layers)]
        ctx.refinalize_table = torch.frombuffer(bytearray(bytes((BnFinalizeEntry * len(ents))(*ents))),
                                                dtype=torch.uint8).to(dev)
        rf.add(lib.b200_bn_finalize_multi, P(ctx.refinalize_table), len(ents), max(L.cout for L, _ in self.layers))
        ctx.refinalize = rf
        ctx.bwd = {}
        return ctx

    def _make_backward(self, ctx, wgrad, xgrad, train=True):
        net = self.net
        dev = self.device
        N, S = ctx.N, ctx.S
        SL = LRELU_SLOPE
        g = self.grads.view
        e = lambda *s: torch.empty(*s, dtype=BF16, device=dev)
        if not hasattr(ctx, "dA"):
            ctx.dfeat = torch.empty_like(ctx.feat)
            ctx.dA = [e(*a.shape) for a in ctx.A]
            ctx.dZ = [e(*z.shape) for z in ctx.Z]
            ctx.sums = [torch.empty_like(s) for s in ctx.stats]
            ctx.dx = torch.empty_like(ctx.x)
        b = Plan()
        cl = ctx.feat.shape[1]
        b.add(lib.b200_nchw_f32_to_nhwc_bf16, P(ctx.dfeat), P(ctx.dA[-1]), N, cl, ctx.hf, ctx.hf, cl, 0)
        c0 = self.conv0.out_channels
        for i in range(len(self.layers) - 1, -1, -1):
            L, bn = self.layers[i]
            hi, ho = ctx.dims[i]
            npix = N * ho * ho
            b.add(lib.b200_bn_bwd_reduce, P(ctx.Z[i]), P(ctx.dA[i + 1]), P(ctx.mi[i]), P(bn.weight), P(bn.bias),
                  P(ctx.sums[i]), P(g(bn.weight)) if wgrad else None, P(g(bn.bias)) if wgrad else None, npix, L.cout,
                  SL)
            b.add(lib.b200_bn_bwd_apply, P(ctx.Z[i]), P(ctx.dA[i + 1]), P(ctx.mi[i]), P(bn.weight), P(bn.bias),
                  P(ctx.sums[i]), P(ctx.dZ[i]), npix, L.cout, SL, 1 if train else 0)
            if wgrad:
                add_wgrad(b, N, hi, hi, L.cin, 0, L.cin, ho, ho, L.cout, 0, L.cout, L.kh, L.stride, L.pad, 1.0,
                          ctx.A[i], ctx.dZ[i], g(L.weight), g(L.bias))
            if i == 0 and not (wgrad or xgrad):
                break
            mask_kw = dict(mask_c=c0, mask_coff=0, mask_lo=0, mask_hi=c0, mask_slope=SL) if i == 0 else {}
            mask_t = ctx.A[0] if i == 0 else None
            if L.stride == 1:
                d = make_conv_desc(N, ho, ho, L.cout, 0, L.cout, hi, hi, hi, hi, L.cin, 0, L.cin,
                                   taps_dgrad_s1(L.kh, L.pad), L.taps, L.dgr_rows, L.dgr_cols, **mask_kw)
                add_igemm(b, d, ctx.dZ[i], L.w_dgr, mask=mask_t, y=ctx.dA[i])
            else:
                assert L.stride == 2 and L.kh == 4 and L.pad == 1
                # the four output-parity classes (each a 2x2-tap conv at half resolution) in ONE launch: the
                # small late layers are launch-bound, 4 launches of a few CTAs each wasted most of the GPU
                taps4 = [t for py in (0, 1) for px in (0, 1) for t in taps_dgrad_s2_k4(py, px)]
                d = make_conv_desc(N, ho, ho, L.cout, 0, L.cout, hi // 2, hi // 2, hi, hi, L.cin, 0, L.cin,
                                   taps4, L.taps, L.dgr_rows, L.dgr_cols, out_mul=(2, 2), out_off=(0, 0),
                                   parity_classes=4, **mask_kw)
                add_igemm(b, d, ctx.dZ[i], L.w_dgr, mask=mask_t, y=ctx.dA[i])
        # conv0 (thin -> wide, LeakyReLU): dA[0] now holds the pre-activation gradient
        if wgrad:
            b.add(lib.b200_conv3x3_thin_wgrad, P(ctx.x), P(ctx.dA[0]), P(g(self.conv0.weight)),
                  P(g(self.conv0.bias)), None, N, S, S, net.in_nc, c0, c0, 0, 1, None, None)
        if xgrad:
            b.add(lib.b200_conv3x3_wide_to_thin, P(ctx.dA[0]), P(self.conv0.weight), None, P(ctx.dx), N, S, S, c0,
                  c0, 0, net.in_nc, 1, None, 1.0)
        ctx.bwd[(wgrad, xgrad, train)] = b

    # ------------------------------------------------------------------ run
    def forward(self, x, need_backward, training):
        self._ensure(x)
        N, _, S, S2 = x.shape
        if S != S2:
            raise RuntimeError("Discriminator_VGG expects square inputs, got %dx%d" % (S, S2))
        key = (N, S)
        pool = pool_for(self.pools, key, lambda: self._make_context(N, S))
        self.packer.ensure()
        # Cache key: address + version counter + shape identify the VALUES only while the tensor that was
        # cached is still alive (the caching allocator hands a freed address to new tensors with version 0),
        # so the entry also holds a weak reference to that tensor: a dead reference is a miss.  A detach()ed
        # alias (D-step: netD(fake.detach())) shares storage and version counter with the live original.
        ckey = (x.data_ptr(), x._version, tuple(x.shape))
        if self.reuse and training:
            hit = self._cache.get(ckey)
            if hit is not None and hit[1] == self.packer.pack_count and hit[0] in pool.free \
                    and hit[2]() is not None:
                ctx = hit[0]
                pool.free.remove(ctx)
                ctx.refinalize.run()
                for _, bn in self.layers:
                    bn.num_batches_tracked.add_(1)
                feat = ctx.feat.clone()
                if need_backward:
                    return feat, Lease(pool, ctx)
                pool.release(ctx)
                return feat, None
        ctx = pool.acquire()
        for k in [k for k, v in self._cache.items() if v[0] is ctx]:
            del self._cache[k]
        if self.reuse and training:
            self._cache[ckey] = (ctx, self.packer.pack_count, weakref.ref(x))
        ctx.x.copy_(x)
        ctx.trained = bool(training)
        if training:
            ctx.fwd_train.run()
            for _, bn in self.layers:
                bn.num_batches_tracked.add_(1)
        else:
            for i, (L, bn) in enumerate(self.layers):
                ctx.mi[i][:L.cout].copy_(bn.running_mean)
                ctx.mi[i][L.cout:].copy_(torch.rsqrt(bn.running_var + bn.eps))
            ctx.fwd_eval.run()
        feat = ctx.feat.clone()
        if need_backward:
            return feat, Lease(pool, ctx)
        pool.release(ctx)
        return feat, None

    def backward(self, lease, dfeat, xgrad):
        ctx = lease.ctx
        wgrad = any(p.requires_grad for p in self.net.features.parameters())
        # eval()-mode forward (running statistics, ctx.mi filled from them): the same plan with the batch-mean
        # terms of the BatchNorm gradient switched off
        key = (wgrad, xgrad, bool(ctx.trained))
        if key not in ctx.bwd:
            self._make_backward(ctx, wgrad, xgrad, train=bool(ctx.trained))
        if wgrad:
            self.grads.attach()
        ctx.dfeat.copy_(dfeat)
        ctx.bwd[key].run()
        dx = ctx.dx.clone() if xgrad else None
        lease.release()
        return dx
