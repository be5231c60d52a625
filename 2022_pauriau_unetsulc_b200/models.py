"""B200-native ``UNet3D`` — drop-in for ``deepsulci.deeptools.models.UNet3D`` as the reference uses it.

Reference call sites (relative to /root/reference): ctor ``training.py:65-67``, ``pattern_class.py:352-356``,
``transfer_learning/transfer_learning.py:155-157``; ``model(inputs)`` ``training.py:206``, ``pattern_class.py:266``;
post-construction ``model.final_conv = nn.Conv3d(...)`` ``pattern_class.py:364``; prefix freezing by
``named_parameters`` ``transfer_learning/transfer_learning.py:330-335``; ``state_dict`` / ``.mdsm``
``pattern_class.py:304,366``.

The module holds ordinary fp32 ``nn.Parameter`` s under the upstream names (so ``state_dict``, ``deepcopy``,
``optim.SGD(model.parameters())`` and ``requires_grad`` masks keep working), but ``forward`` / ``backward`` never call
``nn.Conv3d`` / ``nn.GroupNorm``: they read the parameters and enqueue the hand-written sm_100a kernels of
``libunetsulc_b200.so`` (NDHWC bf16 activations, fp32 accumulation and statistics).  There is no CPU fallback.
"""
import os

import torch
import torch.nn as nn

from . import ops
from .ops import ActView

GN_EPS = 1e-5
# Weight-gradient split reduction: 13 short, latency-bound launches per step = 0.23 ms on the critical path (A/B with the
# reductions skipped, round 2, 1 x B200).  Three placements were measured on the same box (40-step graph replays):
#   "inline" (default): on the main stream right after each wgrad kernel ............................ 6.74 ms/step
#   "defer"  (B2_WGRAD_REDUCE=defer): ONE launch per step / per data-parallel bucket ................. 6.74-6.84 ms/step
#            (13 private workspaces = 455 MB go through HBM; the inline reduce finds its ~35 MB of partials in L2)
#   side stream, overlapping the following dgrad / GroupNorm kernels ................................ 6.91 ms/step
#            (its blocks delay CTAs of the persistent 148-CTA convolution grids; removed)
_WGRAD_REDUCE = os.environ.get("B2_WGRAD_REDUCE", "inline")

def _double_conv(in_ch, out_ch, encoder, order, num_groups):
    if encoder:
        c1 = (in_ch, max(out_ch // 2, in_ch))
        c2 = (c1[1], out_ch)
    else:
        c1 = (in_ch, out_ch)
        c2 = (out_ch, out_ch)
    seq = nn.Sequential()
    for pos, (ci, co) in ((1, c1), (2, c2)):
        seq.add_module("conv%d" % pos, nn.Conv3d(ci, co, 3, padding=1, bias=False))
        seq.add_module("relu%d" % pos, nn.ReLU())
        seq.add_module("norm%d" % pos, nn.GroupNorm(num_groups, co, eps=GN_EPS))
    return seq


class _Block(nn.Module):
    """Parameter holder for one encoder / decoder level (names match upstream: ``double_conv.conv1`` ...)."""

    def __init__(self, in_ch, out_ch, encoder, order, num_groups, is_max_pool=False):
        super().__init__()
        self.is_max_pool = is_max_pool
        self.double_conv = _double_conv(in_ch, out_ch, encoder, order, num_groups)

    def forward(self, *a, **k):  # never used: the network is executed by UNet3D as a whole
        raise RuntimeError("unetsulc_b200 blocks are parameter holders; call UNet3D.forward")


class _ConvLayer(object):
    """One (conv, norm) pair with its packed bf16 weights (re-packed when the fp32 master changes)."""

    def __init__(self, conv, norm):
        self.conv, self.norm = conv, norm
        self.cin, self.cout = conv.in_channels, conv.out_channels
        self._key = None
        self.wf = self.wd = None

    def key(self):
        w = self.conv.weight
        return (w._version, w.data_ptr(), str(w.device))

    def stale(self):
        return self.cin != 1 and self.key() != self._key

    def packs(self):
        if self.stale():
            self.wf, self.wd = ops.pack_conv_weights(self.conv.weight)
            self._key = self.key()
        return self.wf, self.wd


class _Saved(object):
    """Activations kept between forward and backward (all bf16 NDHWC)."""
    pass


class UNet3D(nn.Module):
    def __init__(self, in_channels, out_channels, final_sigmoid=False, interpolate=True, dropout=0.,
                 conv_layer_order='crg', init_channel_number=64):
        super().__init__()
        if in_channels != 1:
            raise ValueError("unetsulc_b200.UNet3D: in_channels=%r unsupported (skeleton volumes have 1)" % in_channels)
        if conv_layer_order != 'crg':
            raise ValueError("unetsulc_b200.UNet3D: conv_layer_order=%r unsupported ('crg' only)" % conv_layer_order)
        if not interpolate:
            raise ValueError("unetsulc_b200.UNet3D: interpolate=False (transposed conv) unsupported")
        if final_sigmoid:
            raise ValueError("unetsulc_b200.UNet3D: final_sigmoid=True unsupported (softmax head)")
        if dropout not in (0, 0., None):
            raise ValueError("unetsulc_b200.UNet3D: dropout=%r unsupported (reference passes 0.)" % dropout)
        f = init_channel_number
        if f not in (32, 64):
            raise ValueError("unetsulc_b200.UNet3D: init_channel_number=%r unsupported (32 or 64: the tcgen05 conv "
                             "kernels take 16-channel operands at the narrowest, and the statistics accumulators at "
                             "most 512 channels)" % (f,))
        g = min(f // 2, 32)
        self.num_groups = g
        self.init_channel_number = f
        o = conv_layer_order
        self.encoders = nn.ModuleList([
            _Block(in_channels, f, True, o, g, False),
            _Block(f, 2 * f, True, o, g, True),
            _Block(2 * f, 4 * f, True, o, g, True),
            _Block(4 * f, 8 * f, True, o, g, True)])
        self.decoders = nn.ModuleList([
            _Block(4 * f + 8 * f, 4 * f, False, o, g),
            _Block(2 * f + 4 * f, 2 * f, False, o, g),
            _Block(f + 2 * f, f, False, o, g)])
        self.final_conv = nn.Conv3d(f, out_channels, 1)
        self.final_activation = nn.Softmax(dim=1)
        self._layers_cache = None
        # data-parallel hook: called as hook(name_prefix, [grad tensors]) when a level's gradients are ready
        self.grad_ready_hook = None
        self.post_head_hook = None
        # data parallel: layer indices after which the pending weight-gradient reductions must be flushed (set by
        # BucketedGradReducer.begin(): the layers that close a gradient bucket); None = after every layer
        self.grad_flush_at = None
        # CUDA-graph capture: re-pack the bf16 weights of every trainable layer even when the packs are fresh, so that
        # the recorded step always contains the re-pack its replays need after each SGD update
        self.force_repack = False

    # ------------------------------------------------------------------------------------------ plumbing
    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k in ("_layers_cache", "_stat_pool"):
                new.__dict__[k] = None
            else:
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    def _layers(self):
        if self._layers_cache is None:
            L = []
            for blk in list(self.encoders) + list(self.decoders):
                dc = blk.double_conv
                L.append(_ConvLayer(dc.conv1, dc.norm1))
                L.append(_ConvLayer(dc.conv2, dc.norm2))
            self._layers_cache = L
        return self._layers_cache

    def _head(self):
        """final_conv as a list of 1x1x1 nn.Conv3d: one module, or the reference's chain for num_conv > 1
        (nn.Sequential of 1x1x1 convs WITHOUT activations, pattern_class.py:357-363)."""
        fc = self.final_conv
        mods = list(fc) if isinstance(fc, nn.Sequential) else [fc]
        if not mods:
            raise RuntimeError("unetsulc_b200.UNet3D: empty final_conv")
        for m in mods:
            if not isinstance(m, nn.Conv3d) or tuple(m.kernel_size) != (1, 1, 1):
                raise RuntimeError("unetsulc_b200.UNet3D: final_conv must be a 1x1x1 nn.Conv3d or an nn.Sequential "
                                   "of them (got %r)" % (m,))
        return mods

    def head_parameters(self):
        """[w0, b0, w1, b1, ...] of the head chain (bias-free convs are not supported by the head kernels)."""
        ps = []
        for m in self._head():
            if m.bias is None:
                raise RuntimeError("unetsulc_b200.UNet3D: final_conv without bias is unsupported")
            ps += [m.weight, m.bias]
        return ps

    def _head_effective(self):
        """The head as ONE affine map (W [Cout, Cin, 1, 1, 1], b [Cout]).  A chain of 1x1x1 convs without
        activations composes exactly: W = Wn ... W1, b = Wn(...(W2 b1 + b2)...) + bn.  Built with differentiable torch
        ops on the (<= 64 x 64) matrices: autograd carries dW / db of the fused head kernels back to every link."""
        mods = self._head()
        if len(mods) == 1:
            return mods[0].weight, mods[0].bias
        W = mods[0].weight.reshape(mods[0].out_channels, mods[0].in_channels)
        b = mods[0].bias
        for m in mods[1:]:
            Wk = m.weight.reshape(m.out_channels, m.in_channels)
            W = Wk @ W
            b = Wk @ b + m.bias
        return W.reshape(W.shape[0], W.shape[1], 1, 1, 1), b

    def trunk_parameters(self):
        """Parameters in the order the autograd functions take them (14 x (w, gamma, beta))."""
        ps = []
        for l in self._layers():
            ps += [l.conv.weight, l.norm.weight, l.norm.bias]
        return ps

    def _check_input(self, x):
        if not x.is_cuda:
            raise RuntimeError("unetsulc_b200.UNet3D runs on a B200 (sm_100a) only: input is on %s and there is no "
                               "CPU fallback" % x.device)
        if x.dim() != 5 or x.shape[1] != 1:
            raise RuntimeError("unetsulc_b200.UNet3D: expected input [B,1,D,H,W], got %s" % (tuple(x.shape),))
        p = self.final_conv.weight if isinstance(self.final_conv, nn.Conv3d) else None
        if not self.encoders[0].double_conv.conv1.weight.is_cuda:
            raise RuntimeError("unetsulc_b200.UNet3D: parameters are on CPU; call model.to('cuda') (no CPU fallback)")
        x = x.detach()
        if x.dtype != torch.float32:
            x = x.float()
        return x.contiguous()

    # ------------------------------------------------------------------------------------------ trunk forward
    def _trunk_forward(self, x, save, defer_last_apply=False):
        """x fp32 [B,1,D,H,W] -> feature ActView [B,D,H,W,f]; fills `save` (a _Saved) when not None.
        defer_last_apply (batch 1): the GroupNorm apply of the LAST layer is not run over the volume; returns
        (r, scale_shift) = its relu(conv) and fp32 [1,f,2] coefficients for the head kernels, which apply it to the
        rows they gather (labelled / skeleton voxels, 2-4 % of the volume)."""
        L = self._layers()
        force = self.__dict__.get("force_repack", False)
        stale = [l for l in L if l.stale() or (force and l.cin != 1 and l.conv.weight.requires_grad)]
        if stale:   # one launch re-packs every layer whose fp32 master changed (optimiser step, load_state_dict, .to())
            for l, (wf, wd) in zip(stale, ops.pack_conv_weights_multi([l.conv.weight for l in stale])):
                l.wf, l.wd, l._key = wf, wd, l.key()
        B, _, D0, H0, W0 = x.shape
        dev = x.device
        G = self.num_groups
        dims = [(D0, H0, W0)]
        for _ in range(3):
            d, h, w = dims[-1]
            dims.append((d // 2, h // 2, w // 2))
        if min(dims[3]) < 1:
            raise RuntimeError("unetsulc_b200.UNet3D: volume %s too small for 3 poolings" % ((D0, H0, W0),))
        f = self.init_channel_number
        skip_c = [f, 2 * f, 4 * f]                 # channels of encoder 0..2 outputs (skips)
        up_c = [2 * f, 4 * f, 8 * f]               # channels upsampled into cat at level 0..2
        cats = [ActView.alloc(B, *dims[l], skip_c[l] + up_c[l], dev) for l in range(3)]
        rec = []                                   # per conv layer: dict(x=ActView|tensor, r=ActView, mr=tensor)
        pool = None
        if B == 1:                                 # statistics accumulators of this step, zeroed with one fill
            pool = self.__dict__.get("_stat_pool")
            if pool is None or pool.buf.device != dev:
                pool = self.__dict__["_stat_pool"] = ops.StatPool(dev)
            pool.reset()

        deferred = []

        def conv_gn(layer, xin, out_view, pooled=None, first=False, defer=False):
            cin, cout = layer.cin, layer.cout
            d, h, w = (out_view.D, out_view.H, out_view.W)
            r = ActView.alloc(B, d, h, w, cout, dev)
            gamma, beta = layer.norm.weight.detach(), layer.norm.bias.detach()
            if first and B == 1:
                mr, ss = ops.conv3d_first_fwd_gn_stats(xin, layer.conv.weight.detach(), r, G, layer.norm.eps, gamma,
                                                       beta, pool)
            elif first:
                ops.conv3d_first_fwd(xin, layer.conv.weight.detach(), r, relu=True)
                mr, ss = ops.relu_gn_stats(r, G, layer.norm.eps, gamma, beta)
            elif B == 1 and cout <= 256 and B * d * h * w > ops.SPLITK_MAX_VOXELS:
                wf, _ = layer.packs()   # GroupNorm statistics come out of the conv epilogue (fixed-point accumulators)
                mr, ss = ops.conv3d_igemm_gn_stats(xin, wf, r, cin, cout, G, layer.norm.eps, gamma, beta, pool)
            else:
                wf, _ = layer.packs()
                ops.conv3d_igemm_auto(xin, wf, r, cin, cout, relu=True)   # split-K when the volume is tiny
                mr, ss = ops.relu_gn_stats(r, G, layer.norm.eps, gamma, beta)
            if defer:
                deferred.append((r, ss))
            else:
                ops.relu_gn_apply(r, ss, out_view, pooled)
            rec.append(dict(x=xin, r=r, mr=mr))

        cur = x
        li = 0
        # encoders
        for lvl in range(4):
            d, h, w = dims[lvl]
            y1 = ActView.alloc(B, d, h, w, L[li].cout, dev)
            conv_gn(L[li], cur, y1, first=(lvl == 0))
            li += 1
            if lvl < 3:
                out = cats[lvl].window(0, skip_c[lvl])
                pooled = ActView.alloc(B, *dims[lvl + 1], skip_c[lvl], dev)
                conv_gn(L[li], y1, out, pooled=pooled)
                cur = pooled
            else:
                out = ActView.alloc(B, d, h, w, L[li].cout, dev)
                conv_gn(L[li], y1, out)
                cur = out
            li += 1
        # decoders
        for k, lvl in enumerate((2, 1, 0)):
            d, h, w = dims[lvl]
            ops.upcat_fwd(cur, cats[lvl].window(skip_c[lvl], up_c[lvl]))
            y1 = ActView.alloc(B, d, h, w, L[li].cout, dev)
            conv_gn(L[li], cats[lvl], y1)
            li += 1
            last = defer_last_apply and B == 1 and lvl == 0
            y2 = None if last else ActView.alloc(B, d, h, w, L[li].cout, dev)
            conv_gn(L[li], y1, y2 if y2 is not None else y1, defer=last)
            li += 1
            cur = y2
        if save is not None:
            save.rec, save.cats, save.dims, save.x = rec, cats, dims, x
            save.skip_c, save.up_c, save.pool = skip_c, up_c, pool
        if deferred:
            return deferred[0]
        return cur

    # ------------------------------------------------------------------------------------------ trunk backward
    def _trunk_backward(self, save, dfeat, needs, outs=None, dfeat_stats=None, dfeat_row_labels=None):
        """dfeat: ActView gradient w.r.t. the trunk output.  needs: list of 42 bools (w, gamma, beta per layer).
        outs: optional list of 42 pre-allocated fp32 tensors the gradients are written into (views of the
        data-parallel buckets).  Returns list of 42 grads (None where not needed)."""
        L = self._layers()
        G = self.num_groups
        rec, cats, dims = save.rec, save.cats, save.dims
        skip_c, up_c = save.skip_c, save.up_c
        grads = [None] * 42
        first_needed = None
        for i in range(14):
            if needs[3 * i] or needs[3 * i + 1] or needs[3 * i + 2]:
                first_needed = i
                break
        if first_needed is None:
            return grads
        hook = self.grad_ready_hook
        if outs is None:
            outs = [None] * 42

        B = save.x.shape[0]
        # Weight gradients: the split reductions of the layers are deferred and run as ONE launch (b2_wgrad_reduce_multi)
        # at the end of backward — or, data parallel, whenever a gradient bucket closes (grad_flush_at, set by the
        # reducer), right before the layers' grad-ready hooks fire.
        pending, waiting = [], []
        flush_at = self.__dict__.get("grad_flush_at")

        def flush():
            ops.wgrad_reduce_multi(pending)
            del pending[:]
            if hook is not None:
                for j in waiting:
                    hook(j, [g for g in grads[3 * j:3 * j + 3] if g is not None])
            del waiting[:]

        def layer_bwd(i, dy, dy_stats=None):
            """dy: gradient w.r.t. the GN output of layer i (dy_stats: GroupNorm-backward statistics of dy when the
            dgrad that produced it fused them).  Returns gradient w.r.t. the layer input (or None); for the second
            conv of a block the return value is (dx, stats) so that the first conv's GroupNorm skips its pass."""
            layer, rc = L[i], rec[i]
            want_gb = needs[3 * i + 1] or needs[3 * i + 2]
            go, bo = (outs[3 * i + 1] if want_gb else None), (outs[3 * i + 2] if want_gb else None)
            if dy_stats is not None:
                dr, dg, db = ops.relu_gn_bwd_from_stats(dy_stats, dy, rc["r"], G, layer.norm.weight.detach(),
                                                        rc["mr"], want_gb, go, bo,
                                                        dy_row_labels=dfeat_row_labels if i == 13 else None)
            else:
                dr, dg, db = ops.relu_gn_bwd(dy, rc["r"], G, layer.norm.weight.detach(), rc["mr"], want_gb, go, bo)
            if needs[3 * i + 1]:
                grads[3 * i + 1] = dg
            if needs[3 * i + 2]:
                grads[3 * i + 2] = db
            if needs[3 * i]:
                if layer.cin == 1:
                    grads[3 * i] = ops.conv3d_first_wgrad(rc["x"], dr, layer.cout, outs[3 * i])
                elif _WGRAD_REDUCE == "inline":
                    grads[3 * i] = ops.conv3d_wgrad(rc["x"], dr, layer.cin, layer.cout, outs[3 * i])
                else:   # "defer"
                    desc = ops.conv3d_wgrad_partial(rc["x"], dr, layer.cin, layer.cout, i, outs[3 * i])
                    grads[3 * i] = desc["dw"]
                    pending.append(desc)
            waiting.append(i)
            if hook is not None and (flush_at is None or i in flush_at):
                flush()
            if i <= first_needed or layer.cin == 1:
                return None
            xin = rc["x"]
            dx = ActView.alloc(xin.N, xin.D, xin.H, xin.W, layer.cin, dr.buf.device)
            _, wd = layer.packs()
            if i % 2 == 1 and B == 1 and layer.cin <= 256 and xin.N * xin.V > ops.SPLITK_MAX_VOXELS:
                # conv2 of a block: dx IS the gradient at conv1's GroupNorm output -> fuse its backward statistics
                stats = ops.conv3d_dgrad_gn_bstats(dr, wd, dx, layer.cout, layer.cin, rec[i - 1]["r"], save.pool)
                return dx, stats
            ops.conv3d_igemm_auto(dr, wd, dx, layer.cout, layer.cin, relu=False)
            return dx

        dy = dfeat
        dcat = [None, None, None]
        # decoders: layers 13,12 (lvl 0), 11,10 (lvl 1), 9,8 (lvl 2)
        li = 13
        def split(res):
            return res if isinstance(res, tuple) else (res, None)

        # The kernel that PRODUCES the gradient at a GroupNorm output also accumulates that layer's GroupNorm-backward
        # statistics (batch 1): the upsample adjoint for layers 11, 9, 7, the pooling adjoint for layers 5, 3, 1.
        fuse = (B == 1)
        st_next = dfeat_stats    # layer 13: accumulated by the head kernel when it produced dfeat

        def done():
            flush()
            return grads

        for lvl in (0, 1, 2):
            dy, st = split(layer_bwd(li, dy, st_next))
            li -= 1
            if dy is None:
                return done()
            dc = layer_bwd(li, dy, st)
            li -= 1
            if dc is None:
                return done()
            dcat[lvl] = dc
            if fuse and 2048 % up_c[lvl] == 0:
                dy, st_next = ops.upcat_bwd(dc.window(skip_c[lvl], up_c[lvl]), *dims[lvl + 1], stat_r=rec[li]["r"],
                                            pool=save.pool)
            else:
                dy, st_next = ops.upcat_bwd(dc.window(skip_c[lvl], up_c[lvl]), *dims[lvl + 1]), None
        # encoders: layers 7,6 (lvl 3) ... 1,0 (lvl 0)
        for lvl in (3, 2, 1, 0):
            if lvl < 3:
                ywin = cats[lvl].window(0, skip_c[lvl])
                if fuse and 256 % (skip_c[lvl] // 8) == 0:
                    dy, st_next = ops.maxpool3d_bwd_add(ywin, dcat[lvl].window(0, skip_c[lvl]), dy,
                                                        stat_r=rec[li]["r"], pool=save.pool)
                else:
                    dy, st_next = ops.maxpool3d_bwd_add(ywin, dcat[lvl].window(0, skip_c[lvl]), dy), None
            dy, st = split(layer_bwd(li, dy, st_next))
            li -= 1
            if dy is None:
                return done()
            dy = layer_bwd(li, dy, st)
            li -= 1
            if dy is None:
                return done()
        return done()

    # ------------------------------------------------------------------------------------------ public API
    def forward(self, x):
        """Dense nn.Module surface: logits [B,C,D,H,W] fp32 in train(), Softmax(dim=1) in eval()."""
        x = self._check_input(x)
        hw, hb = self._head_effective()     # differentiable w.r.t. every link of a num_conv > 1 chain
        params = self.trunk_parameters() + [hw, hb]
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            return _DenseFunction.apply(self, x, not self.training, *params)
        feat = self._trunk_forward(x, None)
        return ops.head_dense_fwd(feat, hw.detach(), hb.detach(), softmax=not self.training)

    def loss_and_preds(self, x, labels):
        """Fused head: CrossEntropyLoss(ignore_index=-1)(model(x), labels) and torch.max(model(x), 1)[1] at the
        labelled voxels, without materialising the dense [B,C,D,H,W] tensor.  In eval() the loss is the reference's
        val-phase loss (CE applied to the Softmax outputs, training.py:189,205-208).
        Returns (loss: 0-dim fp32 tensor wired into autograd, preds: int32 [B,D,H,W], -1 where unlabelled)."""
        x = self._check_input(x)
        hw, hb = self._head_effective()
        params = self.trunk_parameters() + [hw, hb]
        if torch.is_grad_enabled() and self.training and any(p.requires_grad for p in params):
            return _FusedLossFunction.apply(self, x, labels, *params)
        feat, xss = self._split_feat(self._trunk_forward(x, None, defer_last_apply=True))
        out = ops.head_ce(feat, labels, hw.detach(), hb.detach(), compute_grad=False,
                          eval_softmax=not self.training, x_scale_shift=xss)
        return out["loss"][0], out["preds"]

    @staticmethod
    def _split_feat(res):
        """_trunk_forward result -> (feature ActView, deferred GroupNorm scale_shift or None)"""
        return res if isinstance(res, tuple) else (res, None)

    def forward_backward(self, x, labels, outs=None, loss_scale=1.0):
        """One fused training step without autograd: forward, CrossEntropyLoss(ignore_index=-1), backward.
        Gradients are returned (and written into `outs`, 44 tensors in ``parameters()`` order, when given) for the
        parameters with ``requires_grad``; nothing is accumulated into ``.grad``.
        Returns (loss_and_count: fp32 [2] = (mean, sum) device tensor, count int32 [1], preds int32 [B,D,H,W],
        grads: list of 44 tensors or None)."""
        x = self._check_input(x)
        hp = self.head_parameters()
        chain = len(hp) > 2
        params = list(self.trunk_parameters()) + hp
        needs = [bool(p.requires_grad) for p in params]
        if outs is None:
            outs = [None] * len(params)
        if chain:   # num_conv > 1: the kernels see the composed map; autograd on the small matrices splits dW / db
            with torch.enable_grad():
                hw, hb = self._head_effective()
        else:
            hw, hb = hp
        save = _Saved()
        with torch.no_grad():
            feat, xss = self._split_feat(self._trunk_forward(x, save, defer_last_apply=True))
            fuse13 = x.shape[0] == 1 and any(needs[:42])
            out = ops.head_ce(feat, labels, hw.detach(), hb.detach(), compute_grad=True,
                              eval_softmax=False, grad_scale=float(loss_scale), want_preds=True,
                              want_dx=any(needs[:42]), dW_out=None if chain else outs[42],
                              db_out=None if chain else outs[43],
                              stat_r=save.rec[13]["r"] if fuse13 else None, pool=save.pool, x_scale_shift=xss,
                              sparse_dx=fuse13)
            if self.post_head_hook is not None:    # CUDA-graph capture: segment boundary once the loss is final
                self.post_head_hook()
        if chain:
            head_grads = [None] * len(hp)
            live = [i for i, p in enumerate(hp) if p.requires_grad]
            if live:
                gs = torch.autograd.grad([hw, hb], [hp[i] for i in live], [out["dW"].view_as(hw), out["db"]],
                                         allow_unused=True)
                for i, g in zip(live, gs):
                    g = torch.zeros_like(hp[i]) if g is None else g
                    if outs[42 + i] is not None:
                        outs[42 + i].copy_(g)
                        g = outs[42 + i]
                    head_grads[i] = g
        else:
            head_grads = [out["dW"] if needs[42] else None, out["db"] if needs[43] else None]
        with torch.no_grad():
            if self.grad_ready_hook is not None:
                self.grad_ready_hook(14, [g for g in head_grads if g is not None])
            grads = (self._trunk_backward(save, out["dx"], needs[:42], outs[:42], out["dx_stats"],
                                          out["dx_row_labels"])
                     if any(needs[:42]) else [None] * 42)
        return out["loss"], out["count"], out["preds"], list(grads) + head_grads

    def ordered_parameters(self):
        """The parameters in the order forward_backward() reports gradients (42 trunk + 2 per head conv)."""
        return list(self.trunk_parameters()) + self.head_parameters()

    def scores_at(self, x, index, exact=False):
        """Eval forward + Softmax scores gathered at linear voxel indices (labeling(), pattern_class.py:266-277).
        Returns (scores fp32 [n, C], preds int32 [n]).  exact: the split-precision forward (see _exact_forward)."""
        x = self._check_input(x)
        if exact:
            return self._exact_scores_at(x, index)
        with torch.no_grad():
            hw, hb = self._head_effective()
            feat, xss = self._split_feat(self._trunk_forward(x, None, defer_last_apply=True))
            return ops.head_gather(feat, index, hw, hb, softmax=True, x_scale_shift=xss)


def _exact_methods():
    """exact-label inference: split-precision forward (see csrc/exact.cu)"""

    def _exact_packs(self):
        L = self._layers()
        key = tuple((l.conv.weight._version, l.conv.weight.data_ptr()) for l in L)
        cache = self.__dict__.get("_exact_pack_cache")
        if cache is not None and cache[0] == key:
            return cache[1]
        packs = []
        with torch.no_grad():
            for l in L:
                w = l.conv.weight.detach().float()
                hi = w.to(torch.bfloat16).float()
                lo = (w - hi).to(torch.bfloat16).float()
                if l.cin == 1:
                    w3 = torch.zeros((l.cout, 32, 3, 3, 3), dtype=torch.float32, device=w.device)
                    w3[:, 0] = hi[:, 0]
                    w3[:, 1] = lo[:, 0]
                else:
                    w3 = torch.cat([hi, hi, lo], dim=1).contiguous()
                packs.append(ops.pack_conv_weights(w3, want_dgrad=False)[0])
        self.__dict__["_exact_pack_cache"] = (key, packs)
        return packs

    def _exact_trunk(self, x):
        """x fp32 [1,1,D,H,W] -> fp32 features [V, f] (NDHWC) of the last decoder block"""
        if x.shape[0] != 1:
            raise RuntimeError("unetsulc_b200.UNet3D: exact inference handles one volume per call")
        L = self._layers()
        packs = self._exact_packs()
        G = self.num_groups
        f = self.init_channel_number
        _, _, D0, H0, W0 = x.shape
        dims = [(D0, H0, W0)]
        for _ in range(3):
            d, h, w = dims[-1]
            dims.append((d // 2, h // 2, w // 2))
        if min(dims[3]) < 1:
            raise RuntimeError("unetsulc_b200.UNet3D: volume %s too small for 3 poolings" % ((D0, H0, W0),))
        dev = x.device
        skip_c = [f, 2 * f, 4 * f]
        up_c = [2 * f, 4 * f, 8 * f]
        vol = [d * h * w for d, h, w in dims]
        cats = [torch.empty((vol[l], skip_c[l] + up_c[l]), dtype=torch.float32, device=dev) for l in range(3)]

        def conv_gn(i, xs, cin3, out, ld, off):
            layer = L[i]
            r = ops.exact_conv(xs, packs[i], cin3, layer.cout, relu=True)
            ops.exact_gn(r, G, layer.norm.eps, layer.norm.weight.detach().float(), layer.norm.bias.detach().float(),
                         out, ld, off)

        def block(i, src, ld, off, cin, lvl, out, out_ld, out_off):
            """two (conv, relu, gn) layers i, i+1 at level lvl; src = fp32 [V, ld] window or None for the network input"""
            d, h, w = dims[lvl]
            if src is None:
                xs, cin3 = ops.exact_split_first(x, d, h, w), 32
            else:
                xs, cin3 = ops.exact_split3(src, ld, off, cin, d, h, w), 3 * cin
            c1 = L[i].cout
            y1 = torch.empty((vol[lvl], c1), dtype=torch.float32, device=dev)
            conv_gn(i, xs, cin3, y1, c1, 0)
            xs2 = ops.exact_split3(y1, c1, 0, c1, d, h, w)
            conv_gn(i + 1, xs2, 3 * c1, out, out_ld, out_off)

        cur, cur_c = None, 1
        for lvl in range(4):
            if lvl < 3:
                block(2 * lvl, cur, cur_c, 0, cur_c, lvl, cats[lvl], skip_c[lvl] + up_c[lvl], 0)
                cur = ops.exact_maxpool(cats[lvl], skip_c[lvl] + up_c[lvl], 0, skip_c[lvl], *dims[lvl])
                cur_c = skip_c[lvl]
            else:
                out = torch.empty((vol[3], 8 * f), dtype=torch.float32, device=dev)
                block(6, cur, cur_c, 0, cur_c, 3, out, 8 * f, 0)
                cur, cur_c = out, 8 * f
        li = 8
        for lvl in (2, 1, 0):
            ld = skip_c[lvl] + up_c[lvl]
            ops.exact_upsample(cur, cur_c, dims[lvl + 1], cats[lvl], ld, skip_c[lvl], dims[lvl])
            cout = L[li + 1].cout
            out = torch.empty((vol[lvl], cout), dtype=torch.float32, device=dev)
            block(li, cats[lvl], ld, 0, ld, lvl, out, cout, 0)
            cur, cur_c = out, cout
            li += 2
        return cur

    def _exact_scores_at(self, x, index):
        with torch.no_grad():
            hw, hb = self._head_effective()
            feat = self._exact_trunk(x)
            return ops.exact_head_gather(feat, index, hw.detach(), hb.detach(), softmax=True)

    return _exact_packs, _exact_trunk, _exact_scores_at


UNet3D._exact_packs, UNet3D._exact_trunk, UNet3D._exact_scores_at = _exact_methods()


def _needs(ctx_needs, offset):
    return list(ctx_needs[offset:offset + 42])


class _DenseFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, x, softmax, *params):
        save = _Saved()
        feat = model._trunk_forward(x, save)
        hw, hb = params[42].detach(), params[43].detach()
        out = ops.head_dense_fwd(feat, hw, hb, softmax=softmax)
        ctx.model, ctx.save_, ctx.feat, ctx.softmax, ctx.hw = model, save, feat, softmax, hw
        if softmax:
            ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, g):
        model, save, feat = ctx.model, ctx.save_, ctx.feat
        g = g.contiguous().float()
        if ctx.softmax:  # d softmax: g_logit = p * (g - sum_c g*p)
            (p,) = ctx.saved_tensors
            g = p * (g - (g * p).sum(dim=1, keepdim=True))
        dfeat, dW, db = ops.head_dense_bwd(g, feat, ctx.hw)
        needs = list(ctx.needs_input_grad[3:3 + 42])
        grads = model._trunk_backward(save, dfeat, needs)
        nh = ctx.needs_input_grad[45:47]
        if model.grad_ready_hook is not None:
            model.grad_ready_hook(14, [t for t, n in zip((dW, db), nh) if n])
        return (None, None, None) + tuple(grads) + (dW if nh[0] else None, db if nh[1] else None)


class _FusedLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, x, labels, *params):
        save = _Saved()
        feat = model._trunk_forward(x, save)
        hw, hb = params[42].detach(), params[43].detach()
        out = ops.head_ce(feat, labels, hw, hb, compute_grad=False, eval_softmax=False)
        ctx.model, ctx.save_, ctx.feat, ctx.labels, ctx.hw, ctx.hb = model, save, feat, labels, hw, hb
        ctx.mark_non_differentiable(out["preds"])
        return out["loss"][0].clone(), out["preds"]

    @staticmethod
    def backward(ctx, gloss, _gpreds):
        model, save, feat = ctx.model, ctx.save_, ctx.feat
        gl = gloss.detach().float().reshape(1).contiguous()
        needs = list(ctx.needs_input_grad[3:3 + 42])
        nh = ctx.needs_input_grad[45:47]
        out = ops.head_ce(feat, ctx.labels, ctx.hw, ctx.hb, compute_grad=True,
                          eval_softmax=False, grad_scale=1.0, grad_scale_dev=gl, want_preds=False,
                          want_dx=any(needs))
        if model.grad_ready_hook is not None:
            model.grad_ready_hook(14, [t for t, n in zip((out["dW"], out["db"]), nh) if n])
        grads = model._trunk_backward(save, out["dx"], needs) if any(needs) else [None] * 42
        return (None, None, None) + tuple(grads) + (out["dW"] if nh[0] else None, out["db"] if nh[1] else None)
