"""GPU: U-Nets whose 14 trunk convolutions carry a bias (58-key checkpoints).

  * every kernel call of biased training steps against an fp64 reference of that call (the per-call oracle of
    tests/test_gpu_step_oracle.py plus bias-aware spies for the new entry points): fprop K = 27 Cin + 2, first conv
    K = 27 + 3, the split-K reduction adding the bias once, dbias against the fixed-point bound of gn_bwd_apply's launch
    plan.  The biases are large enough to flip a visible share of the ReLU masks, and that share is asserted.
  * the biased kernel variants at odd shapes against fp64, with the kernel each launch takes read from torch.profiler
  * end to end against the fp32 oracle (DESIGN.md §5 bounds, 58 gradients), exact mode, run-to-run determinism
  * the API classes with biased checkpoints
"""
import contextlib
import io
import os
import random
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import tests.test_gpu_step_oracle as so
from tests import harness
from tests.test_gpu_model import rel_l2, cosine

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIAS_STD = 0.2


def _quiet():
    return contextlib.redirect_stdout(io.StringIO())


def _perturb(m, seed):
    """non-trivial GroupNorm affine parameters and conv biases of both signs"""
    torch.manual_seed(seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "norm" in name and name.endswith("weight"):
                p.add_(0.2 * torch.randn_like(p))
            if "norm" in name and name.endswith("bias"):
                p.add_(0.1 * torch.randn_like(p))
            if "double_conv.conv" in name and name.endswith("bias"):
                p.copy_(BIAS_STD * torch.randn_like(p))


def _model(f=64, seed=42, n_classes=56):
    import unetsulc_b200
    torch.manual_seed(seed)
    m = unetsulc_b200.UNet3D(1, n_classes, init_channel_number=f, conv_bias=True)
    _perturb(m, seed + 1)
    return m.cuda().train()


@pytest.fixture
def biased_oracle(monkeypatch):
    from oracle import unet3d_ref
    monkeypatch.setattr(unet3d_ref, "CONV_BIAS_WHEN_NORM", True)

    def pair(f=64, seed=42, n_classes=56):
        """fp32 oracle and our model (built bias-free: load_state_dict switches it) with the same weights"""
        import unetsulc_b200
        torch.manual_seed(seed)
        ref = unet3d_ref.UNet3DRef(1, n_classes, init_channel_number=f)
        _perturb(ref, seed + 1)
        ours = unetsulc_b200.UNet3D(1, n_classes, init_channel_number=f)
        ours.load_state_dict(ref.state_dict())
        assert ours.conv_bias
        return ref.cuda(), ours.cuda()
    return pair


# ------------------------------------------------------------------------------------------------ bias-aware spies
def dbias_plan(sms, V, C, N):
    """(K, nb) of the dbias sums fused into gn_bwd_apply_kernel<.., true> (norm.cu): apply_blocks(V * C/8) blocks per
    sample of 256 threads, vpb = 256 / (C/8) voxel rows per sweep; a thread sums ceil(V / (blocks * vpb)) stored
    values, the block adds its vpb rows in order and commits once per channel"""
    C8 = C // 8
    items = V * C8
    wave = sms * 4
    nb8, nb2 = so._ceil(items, 2048), so._ceil(items, 512)
    nb = nb8 if nb8 >= wave else (nb2 if nb2 < wave else wave)
    nb = max(min(nb, sms * 16), 1)
    vpb = 256 // C8
    return so._ceil(V, nb * vpb) + vpb + 2, nb * N


def _flips(orc, pre, b):
    """share of ReLU masks the bias flips: (conv > 0) != (conv + b > 0)"""
    post = pre + b.view(1, -1, 1, 1, 1)
    orc.flips[0] += int(((pre > 0) != (post > 0)).sum())
    orc.flips[1] += pre.numel()


def _bias_conv_check(orc, op, x64, w64, b, got, relu, K, bf16=True):
    b64 = b.double().view(1, -1, 1, 1, 1)
    pre = so.conv3d_taps(x64, w64)
    ref = pre + b64
    A = so.conv3d_taps(x64.abs(), w64.abs()) + b64.abs()
    if relu:
        ref = ref.clamp_min(0)
    orc.dense(op, got, ref, A, K, bf16=bf16)
    _flips(orc, pre, b.double())


def spy_conv3d_igemm_bias(real, orc, x, wpack, bias, y, cin, cout, relu=True, y_fp32=False, stat_acc=None,
                          splitk=False):
    x64 = so.nc(x).clone()
    real(x, wpack, bias, y, cin, cout, relu, y_fp32, stat_acc, splitk)
    torch.cuda.synchronize()
    split = splitk and stat_acc is None and not y_fp32 and x.N * x.V <= so.SPLITK_MAX_VOXELS
    orc.seen.add("bias_fprop" + ("_stats" if stat_acc is not None else "") + ("_splitk" if split else "")
                 + ("_fp32" if y_fp32 else ""))
    _bias_conv_check(orc, "conv_fprop_bias", x64, so.unpack_wf(wpack, cout, cin), bias, so.nc(y), relu,
                     27 * cin + 2, bf16=not y_fp32)
    if stat_acc is not None:
        r = so.rows(y)
        K, nb = so.conv_epilogue_plan(orc.sms, y.D, y.H, y.W)
        orc.sums("stats_acc:conv_epilogue_bias", stat_acc, cout, r, r * r, K, nb, store=False)
        orc.fwd_meta[stat_acc.data_ptr()] = (r, K, nb)


def spy_conv3d_first_fwd_bias(real, orc, x, w, bias, y, relu=True, stat_acc=None):
    real(x, w, bias, y, relu, stat_acc)
    torch.cuda.synchronize()
    orc.seen.add("bias_first" + ("_stats" if stat_acc is not None else ""))
    _bias_conv_check(orc, "conv_first_bias", x.double(), w.double(), bias, so.nc(y), relu, 27 + 3)
    if stat_acc is not None:
        r = so.rows(y)
        K, nb = so.first_conv_plan(y.V)
        orc.sums("stats_acc:conv_first_bias", stat_acc, y.C, r, r * r, K, nb, store=False)
        orc.fwd_meta[stat_acc.data_ptr()] = (r, K, nb)


def spy_gn_finalize_acc(real, orc, acc, V, C, groups, eps, gamma, beta):
    mr, ss = real(acc, V, C, groups, eps, gamma, beta)
    meta = orc.fwd_meta.pop(acc.data_ptr(), None)
    if meta is not None:
        torch.cuda.synchronize()
        r, K, nb = meta
        orc.fwd_stats("gn_stats", r.view(1, V, C), C, groups, eps, gamma, beta, mr, ss, K, nb)
    return mr, ss


def _dbias_check(orc, dr, dbias):
    d = so.rows(dr)
    K, nb = dbias_plan(orc.sms, dr.V, dr.C, dr.N)
    orc.ratio("dbias", dbias, d.sum(0), K * so.U * d.abs().sum(0) + nb * so.FIX + so.FLOOR)


def spy_relu_gn_bwd_from_stats_dbias(real, orc, acc, dy, r, groups, gamma, mean_rstd, want_param_grads=True,
                                     dgamma_out=None, dbeta_out=None, dy_row_labels=None, dbias_out=None, pool=None):
    got = {}

    def real3(*a):
        dr, dg, db, dbias = real(*a, dbias_out=dbias_out, pool=pool)
        got["dbias"] = dbias
        return dr, dg, db
    dr, dg, db = so.spy_relu_gn_bwd_from_stats(real3, orc, acc, dy, r, groups, gamma, mean_rstd, want_param_grads,
                                               dgamma_out, dbeta_out, dy_row_labels)
    orc.seen.add("dbias_acc" + ("_rows" if dy_row_labels is not None else ""))
    _dbias_check(orc, dr, got["dbias"])
    return dr, dg, db, got["dbias"]


def spy_relu_gn_bwd_dbias(real, orc, dy, r, groups, gamma, mean_rstd, want_param_grads=True, dgamma_out=None,
                          dbeta_out=None, dbias_out=None):
    got = {}

    def real3(*a):
        dr, dg, db, dbias = real(*a, dbias_out=dbias_out)
        got["dbias"] = dbias
        return dr, dg, db
    dr, dg, db = so.spy_relu_gn_bwd(real3, orc, dy, r, groups, gamma, mean_rstd, want_param_grads, dgamma_out,
                                    dbeta_out)
    orc.seen.add("dbias_pass")
    _dbias_check(orc, dr, got["dbias"])
    return dr, dg, db, got["dbias"]


BIAS_SPIES = {
    "conv3d_igemm_bias": spy_conv3d_igemm_bias,
    "conv3d_first_fwd_bias": spy_conv3d_first_fwd_bias,
    "gn_finalize_acc": spy_gn_finalize_acc,
    "relu_gn_bwd_from_stats_dbias": spy_relu_gn_bwd_from_stats_dbias,
    "relu_gn_bwd_dbias": spy_relu_gn_bwd_dbias,
}


def install_spies(monkeypatch, orc):
    import functools
    from unetsulc_b200 import ops
    orc.flips = [0, 0]
    orc.fwd_meta = {}
    so.install_spies(monkeypatch, orc)
    for name, spy in BIAS_SPIES.items():
        monkeypatch.setattr(ops, name, functools.partial(spy, getattr(ops, name), orc))


def _report(orc, name):
    print("\n[bias %s] %d checks, ReLU masks flipped by the bias: %.3f; worst error / bound:"
          % (name, len(orc.worst), orc.flips[0] / max(orc.flips[1], 1)))
    for op in sorted(orc.worst):
        print("    %-34s %.3e" % (op, orc.worst[op]))
    bad = {op: w for op, w in orc.worst.items() if not w <= 1.0}
    assert not bad, "ops outside their fp64 bound: %s" % bad


# ------------------------------------------------------------------------------------------------ per-call oracle
BIAS_B1 = so.COMMON | {"bias_first_stats", "bias_fprop_stats", "conv_dgrad_bstats", "maxpool_bwd_stats",
                       "gn_bwd_acc", "gn_bwd_acc_rows", "dbias_acc", "dbias_acc_rows", "head_train_fused_sparse_xss"}
BIAS_B2 = so.COMMON | {"bias_first", "bias_fprop", "bias_fprop_splitk", "gn_stats_pass", "gn_bwd_pass", "dbias_pass",
                       "maxpool_bwd", "upcat_bwd_non2x", "head_train", "conv_dgrad"}
CONFIGS = {
    # name: (width, batch, shape, wgrad reduce mode, autograd surface, coverage set)
    "f64_b1_24x32x40": (64, 1, (24, 32, 40), "inline", False,
                        BIAS_B1 | {"upcat_bwd_stats_2x", "bias_fprop_splitk", "conv_dgrad_splitk", "gn_stats_pass"}),
    "f64_b1_24x32x40_defer": (64, 1, (24, 32, 40), "defer", False,
                              (BIAS_B1 - {"wgrad"}) | {"wgrad_defer", "upcat_bwd_stats_2x"}),
    "f64_b1_17x26x21": (64, 1, (17, 26, 21), "inline", False, BIAS_B1 | {"upcat_bwd_stats_non2x",
                                                                         "bias_fprop_splitk"}),
    "f64_b1_23x30x19": (64, 1, (23, 30, 19), "inline", False, BIAS_B1 | {"upcat_bwd_stats_non2x"}),
    "f64_b1_40x48x56": (64, 1, (40, 48, 56), "inline", False, BIAS_B1 | {"upcat_bwd_stats_2x"}),
    "f64_b1_48x56x64": (64, 1, (48, 56, 64), "inline", False, BIAS_B1 | {"upcat_bwd_stats_2x"}),
    "f64_b2_17x26x21": (64, 2, (17, 26, 21), "inline", False, BIAS_B2),
    "f64_b1_24x32x40_autograd": (64, 1, (24, 32, 40), "inline", True,
                                 so.COMMON | {"head_fwd", "head_train", "head_grad_scale_dev", "gn_bwd_pass",
                                              "dbias_pass", "gn_bwd_acc", "dbias_acc", "maxpool_bwd_stats",
                                              "upcat_bwd_stats_2x"}),
    "f32_b1_24x32x40": (32, 1, (24, 32, 40), "inline", False, BIAS_B1 | {"upcat_bwd_stats_2x", "bias_fprop_splitk"}),
    "f32_b2_17x26x21": (32, 2, (17, 26, 21), "inline", False, BIAS_B2),
}


def run_config(monkeypatch, name, cfg):
    from unetsulc_b200 import models
    f, B, shape, mode, autograd, expect = cfg
    model = _model(f)
    assert len(model.ordered_parameters()) == 58
    x, labels = so._data(B, shape)
    monkeypatch.setattr(models, "_WGRAD_REDUCE", mode)
    g_fb = None
    if autograd:
        _, _, _, g_fb = model.forward_backward(x, labels)
        g_fb = [g.clone() for g in g_fb]
        model.force_repack = True
    orc = so.Oracle()
    install_spies(monkeypatch, orc)
    if autograd:
        model.zero_grad(set_to_none=True)
        loss, _ = model.loss_and_preds(x, labels)
        (2.5 * loss).backward()
        grads = [p.grad for p in model.ordered_parameters()]
    else:
        _, _, _, grads = model.forward_backward(x, labels)
    torch.cuda.synchronize()
    _report(orc, name)
    assert orc.flips[0] >= 0.02 * orc.flips[1], orc.flips
    assert not expect - orc.seen, "entry points not reached: %s" % sorted(expect - orc.seen)
    assert len(grads) == 58 and all(g is not None and bool(torch.isfinite(g).all()) for g in grads)
    if autograd:
        names = [n for n, _ in model.named_parameters()]
        for i, (n, a, b) in enumerate(zip(names, grads, g_fb)):
            a, b = a.double().flatten(), (2.5 * b.double()).flatten()
            e = float((a - b).norm() / (b.norm() + 1e-30))
            assert e < (1e-5 if i >= 56 else 2e-2), (n, e)


@pytest.mark.parametrize("name", list(CONFIGS))
def test_biased_step_matches_fp64_per_call(monkeypatch, name):
    run_config(monkeypatch, name, CONFIGS[name])


def test_biased_step_matches_fp64_per_call_baseline_shape(monkeypatch):
    run_config(monkeypatch, "f64_b1_96x112x96", (64, 1, (96, 112, 96), "inline", False,
                                                 BIAS_B1 | {"upcat_bwd_stats_2x", "bias_fprop_splitk"}))


# ------------------------------------------------------------------------------------------------ kernel edge cases
def _kernels(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _act(N, C, D, H, W, seed, scale=1.0):
    from unetsulc_b200.ops import ActView
    g = torch.Generator(device="cuda").manual_seed(seed)
    t = (scale * torch.randn((N, D, H, W, C), generator=g, device="cuda")).to(torch.bfloat16)
    return ActView(t, N, D, H, W, C)


def _weights(cout, cin, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn((cout, cin, 3, 3, 3), generator=g, device="cuda") * (2.0 / (27 * cin)) ** 0.5


def _bias(c, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return 0.5 * torch.randn(c, generator=g, device="cuda")


@pytest.mark.parametrize("cin,cout,dims,splitk,kernel", [
    (16, 16, (13, 25, 27), False, "conv3d_igemm_kernel<16, false>"),   # KC = 16, N = 16 tile
    (32, 16, (9, 30, 31), False, "conv3d_igemm_kernel<32, false>"),    # KC = 32, N = 16 tile
    (48, 16, (7, 35, 34), False, "conv3d_igemm_kernel<16, false>"),    # three 16-channel chunks
    (16, 32, (22, 30, 46), False, "conv3d_slab_kernel<16, 16, true>"),  # slab, 16-channel chunk, 16 x 8 tile
    (96, 32, (22, 30, 46), False, "conv3d_slab_kernel<32, 16, true>"),  # slab, three 32-channel chunks
    (64, 64, (20, 33, 64), False, "conv3d_slab_kernel<64, 32, true>"),  # slab, 32 x 4 tile
    (128, 128, (20, 24, 28), False, "conv3d_igemm_kernel<64, true>"),  # h-halo implicit GEMM
    (256, 512, (10, 12, 14), False, "conv3d_igemm_kernel<64, true>"),  # two N tiles (n0 = 256)
    (256, 512, (10, 12, 14), True, "conv_splitk_reduce_kernel"),       # split-K: bias added once by the reduction
    (64, 128, (11, 13, 9), True, "conv_splitk_reduce_kernel"),
])
def test_biased_fprop_variants_against_fp64(monkeypatch, cin, cout, dims, splitk, kernel):
    from unetsulc_b200 import ops
    orc = so.Oracle()
    install_spies(monkeypatch, orc)
    x = _act(1, cin, *dims, seed=cin + cout)
    wf, _ = ops.pack_conv_weights(_weights(cout, cin, 7))
    b = _bias(cout, 3)
    y = ops.ActView.alloc(1, *dims, cout, "cuda")
    names = _kernels(lambda: ops.conv3d_igemm_bias(x, wf, b, y, cin, cout, splitk=splitk))
    assert any(kernel in n for n in names), names
    if splitk:   # the partials carry no bias: without split-K the same layer gives the same values within rounding
        assert any("conv3d_igemm_kernel<64, false>" in n for n in names), names
    if cout <= 256 and not splitk:   # fused statistics on the same launch
        acc = torch.zeros(4 * cout, dtype=torch.int64, device="cuda")
        y2 = ops.ActView.alloc(1, *dims, cout, "cuda")
        ops.conv3d_igemm_bias(x, wf, b, y2, cin, cout, stat_acc=acc)
        assert torch.equal(y.buf, y2.buf)
    _report(orc, "fprop %d->%d %s" % (cin, cout, dims))
    assert orc.flips[0] >= 0.02 * orc.flips[1]


def test_biased_exact_fp32_epilogue_two_n_tiles(monkeypatch):
    """fp32 output (exact mode) with Cout = 512: two N tiles, the bias index follows n0 + c"""
    from unetsulc_b200 import ops
    orc = so.Oracle()
    install_spies(monkeypatch, orc)
    x = _act(1, 192, 6, 7, 8, seed=1)
    wf, _ = ops.pack_conv_weights(_weights(512, 192, 2), want_dgrad=False)
    b = _bias(512, 4)
    y = ops.ActView(torch.empty((6 * 7 * 8, 512), dtype=torch.float32, device="cuda"), 1, 6, 7, 8, 512)
    ops.conv3d_igemm_bias(x, wf, b, y, 192, 512, y_fp32=True)
    _report(orc, "fp32 192->512")
    assert "bias_fprop_fp32" in orc.seen


@pytest.mark.parametrize("cout,dims,occ", [(16, (7, 9, 11), 0.05), (32, (33, 17, 40), 0.01), (64, (20, 24, 28), 0.002)])
def test_biased_first_layer_against_fp64(monkeypatch, cout, dims, occ):
    """mostly empty volumes: a voxel with no non-zero neighbour stores relu(b) and enters the statistics with it"""
    from unetsulc_b200 import ops
    from oracle.synth import synth_volume
    orc = so.Oracle()
    install_spies(monkeypatch, orc)
    x, _ = synth_volume(dims, 5, 77, occupancy=occ)
    x = x.reshape(1, 1, *dims).cuda().contiguous()
    w, b = _weights(cout, 1, 9), _bias(cout, 5)
    y = ops.ActView.alloc(1, *dims, cout, "cuda")
    ops.conv3d_first_fwd_bias(x, w, b, y)
    acc = torch.zeros(4 * cout, dtype=torch.int64, device="cuda")
    y2 = ops.ActView.alloc(1, *dims, cout, "cuda")
    ops.conv3d_first_fwd_bias(x, w, b, y2, stat_acc=acc)
    assert torch.equal(y.buf, y2.buf)
    empty = F.max_pool3d(x.abs(), 3, 1, 1)[0, 0] == 0
    assert bool(empty.any())
    want = b.relu().to(torch.bfloat16)
    assert bool((y.buf[0][empty] == want).all())
    _report(orc, "first %d" % cout)
    assert {"bias_first", "bias_first_stats"} <= orc.seen


@pytest.mark.parametrize("C,dims,N,labels", [(64, (24, 32, 40), 1, False), (64, (24, 32, 40), 1, True),
                                             (512, (3, 4, 5), 1, False), (32, (17, 26, 21), 2, False),
                                             (16, (9, 10, 11), 3, False)])
def test_dbias_against_fp64(monkeypatch, C, dims, N, labels):
    """dbias of both GroupNorm-backward forms (batch 1 accumulators, with and without label rows; the pass form over
    several samples) against fp64 sums of the stored dr, and bit-identical on a second run"""
    from unetsulc_b200 import ops
    orc = so.Oracle()
    install_spies(monkeypatch, orc)
    G = min(C // 2, 32)
    r = _act(N, C, *dims, seed=1)
    r.buf.relu_()
    dy = _act(N, C, *dims, seed=2, scale=1e-2)
    gamma = 1.0 + 0.2 * torch.randn(C, device="cuda")
    beta = 0.1 * torch.randn(C, device="cuda")
    mr, _ = ops.relu_gn_stats(r, G, 1e-5, gamma, beta)
    lab = None
    if labels:   # the same labelled rows (5 %) on both runs
        g = torch.Generator(device="cuda").manual_seed(3)
        lab = torch.where(torch.rand(r.V, generator=g, device="cuda") < 0.05, 1, -1).to(torch.int64)
    outs = []
    for _ in range(2):
        if N == 1:
            acc = torch.zeros(4 * C, dtype=torch.int64, device="cuda")
            dyr = so.rows(dy) * (1 if lab is None else (lab.view(-1, 1) >= 0))
            rr = so.rows(r)
            a4 = acc.view(C, 4)
            for k, v in ((0, dyr.sum(0)), (2, (dyr * rr).sum(0))):   # the fp64 sums as one fixed-point contribution
                hi = v.round()
                a4[:, k] = hi.to(torch.int64)
                a4[:, k + 1] = ((v - hi) * 2.0 ** 32).round().to(torch.int64)
            orc.acc_meta[acc.data_ptr()] = (1, 1)
            outs.append(ops.relu_gn_bwd_from_stats_dbias(acc, dy, r, G, gamma, mr, dy_row_labels=lab))
        else:
            outs.append(ops.relu_gn_bwd_dbias(dy, r, G, gamma, mr))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][3], outs[1][3]) and torch.equal(outs[0][0].buf, outs[1][0].buf)
    _report(orc, "dbias C=%d" % C)
    assert "dbias" in orc.worst and bool(outs[0][3].abs().sum() > 0)   # checked (exact sums give a ratio of 0)


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("shape", [(24, 32, 40), (96, 112, 96)])
def test_biased_end_to_end_against_fp32_oracle(biased_oracle, shape):
    """DESIGN.md §5 bounds: logits rel-L2 < 3e-2, argmax >= 97 %, all 58 gradients (the 14 biases included) cosine >
    0.9 and norm ratio in (0.8, 1.25)"""
    from oracle.synth import synth_volume
    ref, ours = biased_oracle()
    x, labels = synth_volume(shape, 56, 1234, occupancy=0.03 if shape[0] == 96 else 0.05)
    x, labels = x.unsqueeze(0).cuda(), labels.unsqueeze(0).cuda()
    ref.train(); ours.train()
    logits_r = ref(x)
    loss_r = F.cross_entropy(logits_r, labels, ignore_index=-1)
    loss_r.backward()
    with torch.no_grad():
        logits_o = ours(x)
    e = rel_l2(logits_o, logits_r.detach())
    del logits_o
    loss, count, preds, grads = ours.forward_backward(x, labels)
    m = labels >= 0
    agree = float((preds[m].long() == logits_r.detach().argmax(1)[m]).float().mean())
    print("bias %s: logits rel-L2 %.3e, loss ours %.6f oracle %.6f, argmax agreement %.4f"
          % (shape, e, float(loss[0]), float(loss_r), agree))
    assert e < 3e-2
    assert agree >= 0.97
    assert len(grads) == 58
    order = {id(p): k for k, p in enumerate(ours.ordered_parameters())}
    named = dict(ours.named_parameters())
    cmin, rmin, rmax, cbias = 1.0, 10.0, 0.0, 1.0
    for n, pr in ref.named_parameters():
        g = grads[order[id(named[n])]]
        c, ratio = cosine(g, pr.grad), float(g.norm() / pr.grad.norm())
        cmin, rmin, rmax = min(cmin, c), min(rmin, ratio), max(rmax, ratio)
        if "double_conv.conv" in n and n.endswith("bias"):
            cbias = min(cbias, c)
        assert c > 0.9 and 0.8 < ratio < 1.25, (n, c, ratio)
    print("bias %s: gradient cosine >= %.4f (conv biases >= %.4f), norm ratio %.3f..%.3f"
          % (shape, cmin, cbias, rmin, rmax))


@pytest.mark.parametrize("shape", [(24, 32, 40), (17, 26, 21)])
def test_biased_exact_mode(biased_oracle, shape):
    from oracle.synth import synth_volume
    ref, ours = biased_oracle()
    x, labels = synth_volume(shape, 56, 1234, occupancy=0.05)
    x, labels = x.unsqueeze(0).cuda(), labels.unsqueeze(0).cuda()
    ref.eval(); ours.eval()
    idx = torch.nonzero(labels.reshape(-1) >= 0).reshape(-1)
    with torch.no_grad():
        pr = ref(x)[0].reshape(56, -1)[:, idx].t().contiguous()
        po, preds = ours.scores_at(x, idx, exact=True)
    err = float((po - pr).abs().max())
    top2 = pr.topk(2, dim=1).values
    margin = top2[:, 0] - top2[:, 1]
    same = preds.long() == pr.argmax(1)
    print("bias exact %s: %d voxels, max |score err| %.3e, label agreement %.6f"
          % (shape, len(idx), err, float(same.float().mean())))
    assert err <= 1e-4
    assert bool(same[margin > 2e-4].all())


@pytest.mark.parametrize("f", [64, 32])
def test_biased_steps_are_deterministic(f):
    x, labels = so._data(1, (24, 32, 40))
    outs = []
    for _ in range(2):
        m = _model(f)
        loss, _, _, grads = m.forward_backward(x, labels)
        outs.append((loss.clone(), [g.clone() for g in grads]))
    assert len(outs[0][1]) == 58
    assert torch.equal(outs[0][0], outs[1][0])
    assert all(torch.equal(a, b) for a, b in zip(outs[0][1], outs[1][1]))


# ------------------------------------------------------------------------------------------------ API classes
def test_biased_learning_graph_replay_equals_eager(tmp_path):
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=5, shape=(14, 16, 12), n_classes=6, seed=2)
    files = sorted(bck2)
    out = []
    for use_graph in (False, True):
        random.seed(7); np.random.seed(7); torch.manual_seed(7)
        with _quiet():
            m = UnetTrainingSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path),
                                           dict_model={'name': 'cb', 'conv_bias': True, 'img_size': [24, 24, 24]},
                                           dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
            m.use_cuda_graph = use_graph
            m.learning(1e-2, 0.9, 2, files[:4], files[4:], batch_size=1)
        assert m.model.conv_bias
        r = m.results
        out.append((r['epoch_loss_train'], r['epoch_loss_val'], r['epoch_acc_train'], r['epoch_acc_val']))
        assert all(np.isfinite(np.asarray(r['epoch_loss_train'], float)).ravel())
    assert out[0] == out[1]


def _biased_checkpoint(tmp_path, sslist, name='cbase', num_conv=1):
    """a trained-looking biased .mdsm written through the API (state_dict of 58 + 2 (num_conv - 1) keys)"""
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    torch.manual_seed(11)
    with _quiet():
        base = UnetTrainingSulciLabelling([], 'L', cuda=0, working_path=str(tmp_path),
                                          dict_model={'name': name, 'conv_bias': True, 'num_conv': num_conv},
                                          dict_names={}, dict_bck2={}, sulci_side_list=sslist)
        base.load_network()
        _perturb(base.model, 12)
        base.save_model()
        base.save_params()
    path = tmp_path / 'models' / (name + '_model.mdsm')
    sd = torch.load(str(path), map_location='cpu')
    assert len(sd) == 58 + 2 * (num_conv - 1)
    params = __import__('json').load(open(str(tmp_path / 'models' / (name + '_params.json'))))
    assert params['dict_model']['conv_bias'] is True
    return path, sd


def test_biased_load_saved_model_labeling_and_thresholds(tmp_path):
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    from oracle.synth import synth_folds
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=2, shape=(24, 24, 24))
    files = sorted(bck2)
    for num_conv in (1, 2):
        path, sd = _biased_checkpoint(tmp_path, sslist, 'cb%d' % num_conv, num_conv)
        with _quiet():
            m = UnetTrainingSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path),
                                           dict_model={'name': 'lab%d' % num_conv},
                                           dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
            # built bias-free (no 'conv_bias' key), the checkpoint makes it biased
            m.load_saved_model({'model_file': str(path), 'out_channels': len(sslist), 'num_conv': num_conv})
        assert m.model.conv_bias
        for k, v in sd.items():
            assert torch.equal(m.model.state_dict()[k].cpu(), v), k
        with _quiet():
            ytrue, ypred, yscores = m.labeling(files[0])
        n = len(bck2[files[0]])
        assert len(ypred) == n and yscores.shape == (n, len(sslist))
        assert np.allclose(yscores.sum(1), 1.0, atol=1e-5) and ypred == np.argmax(yscores, axis=1).tolist()
        from oracle.synth import synth_volume
        x, l = synth_volume((24, 24, 24), len(sslist), 5, occupancy=0.08)
        m.model.train()
        loss, _, _, grads = m.model.forward_backward(x.unsqueeze(0).cuda(), l.unsqueeze(0).cuda())
        assert len(grads) == 56 + 2 * num_conv and all(bool(torch.isfinite(g).all()) for g in grads)
    rng = np.random.RandomState(0)
    for g in files:
        pts = np.asarray(bck2[g])
        nb = pts * 2 + 1
        perm = rng.permutation(len(pts))
        m.dict_graph_data[g] = {'nbck': nb.tolist(), 'bck2': pts.tolist(), 'names': names[g],
                                'vert': list(range(len(pts)))}
        m.dict_graph_data[g + '.notcut'] = {'nbck': nb[perm].tolist(), 'bck2': pts[perm].tolist(),
                                            'names': [names[g][i] for i in perm],
                                            'vert': synth_folds(pts[perm], (8, 8, 8)).tolist()}
    m.results = {'threshold_scores': {}}
    with _quiet():
        m.test_thresholds(files, [g + '.notcut' for g in files], [5, 50, 100])
    assert sorted(m.results['threshold_scores']) == [5, 50, 100]


def test_biased_transfer_learning_two_phases(tmp_path):
    """phase 1 trains final_conv only; from epoch int(0.8 * num_epochs) + 1 on the decoders (and their conv biases)
    train too.  The model ends on the best-validation weights, so the biases are watched during the steps."""
    from unetsulc_b200.transfer_learning import UnetTransferSulciLabelling
    bck2, names, sslist = harness.synthetic_cohort()
    files = sorted(bck2)
    path, sd = _biased_checkpoint(tmp_path, sslist)
    dec, enc = "decoders.2.double_conv.conv2.bias", "encoders.3.double_conv.conv2.bias"
    with _quiet():
        tl = UnetTransferSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path), dict_model={'name': 'tlb'},
                                        dict_trained_model={'out_channels': len(sslist), 'model_file': str(path)},
                                        dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
        seen = []   # (decoder bias trainable, decoder bias, encoder bias) before every step
        mask = tl._apply_freeze_mask

        def watch():
            mask()
            p = dict(tl.model.named_parameters())
            seen.append((p[dec].requires_grad, p[dec].detach().cpu().clone(), p[enc].detach().cpu().clone(),
                         p[enc].requires_grad))
        tl._apply_freeze_mask = watch
        tl.learning(1e-2, 0.9, 10, files[:2], files[2:], patience={'fine_tunning': 100})
    assert tl.model.conv_bias
    assert tl.results['fine_tunning_epoch'] == [8]
    phase1 = [s for s in seen if not s[0]]
    phase2 = [s for s in seen if s[0]]
    assert len(phase1) >= 2 and len(phase2) >= 2
    assert all(torch.equal(s[1], sd[dec]) for s in phase1)            # frozen in phase 1
    assert not torch.equal(phase2[-1][1], phase2[0][1])               # trained in phase 2
    assert all(torch.equal(s[2], sd[enc]) and not s[3] for s in seen)  # encoders frozen throughout
    assert tl.results['epoch_loss_train'][0][-1] < tl.results['epoch_loss_train'][0][0]


def _dp_worker(rank, world, port, tmp, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import unetsulc_b200
        from unetsulc_b200 import parallel
        from unetsulc_b200.training import UnetTrainingSulciLabelling
        from oracle.synth import synth_volume
        res = {}
        torch.manual_seed(100 + rank)
        model = unetsulc_b200.UNet3D(1, 56, conv_bias=True).to(dev).train()
        red = parallel.BucketedGradReducer(model)
        x, l = synth_volume((32, 40, 32), 56, 1000 + rank, occupancy=0.05)
        x, l = x.unsqueeze(0).to(dev), l.unsqueeze(0).to(dev)
        model.grad_ready_hook = None
        _, _, _, g_local = model.forward_backward(x, l)
        g_avg = []
        for g in g_local:
            t = g.clone()
            dist.all_reduce(t)
            g_avg.append(t / world)
        model.grad_ready_hook = red._on_layer_ready
        red.begin()
        model.forward_backward(x, l, outs=red.outs())
        views = red.finish()
        torch.cuda.synchronize()
        res["n"] = len(views)
        res["grad_worst"] = max(float((a - b).abs().max() / (b.abs().max() + 1e-30)) for a, b in zip(views, g_avg))
        model.grad_ready_hook = None
        del model, red
        bck2, names, sslist = harness.synthetic_cohort(n_subjects=7, shape=(14, 16, 12), n_classes=6, seed=2)
        files = sorted(bck2)
        random.seed(7); np.random.seed(7); torch.manual_seed(7 + rank)
        with contextlib.redirect_stdout(io.StringIO()):
            m = UnetTrainingSulciLabelling(files, 'L', cuda=rank, working_path=tmp,
                                           dict_model={'name': 'dpb', 'conv_bias': True, 'img_size': [24, 24, 24]},
                                           dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
            m.learning(1e-2, 0.9, 2, files[:5], files[5:], batch_size=1)
        res["learn"] = (m.results['epoch_loss_train'], m.results['epoch_loss_val'])
        res["sync"] = parallel.parameters_in_sync(m.model)
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_biased_data_parallel_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 300
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, str(tmp_path), q)) for r in range(world)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    for r in range(world):
        assert out[r]["n"] == 58 and out[r]["grad_worst"] < 1e-5 and out[r]["sync"]
    assert out[0]["learn"] == out[1]["learn"]
