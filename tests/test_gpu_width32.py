"""GPU: the 32-filter network (init_channel_number=32, 16 GroupNorm groups) on the tcgen05 path.

  * every kernel call of f = 32 training steps against an fp64 reference of that call (the per-call oracle of
    tests/test_gpu_step_oracle.py), with coverage sets that require the kernel variants only this width reaches:
    the first conv at Cout = 16, 16-channel K chunks (Cin = 16), the N = 16 dgrad with fused statistics, Cin = 96 and
    the Cout = 32 weight gradient
  * those variants at odd shapes against fp64, with the kernel each launch takes read from torch.profiler
  * end to end against the fp32 oracle (DESIGN.md §5 bounds), exact-label mode, run-to-run determinism
  * the API classes: learning() eager and graph-replayed, labeling / test_thresholds, the .mdsm round trip,
    transfer learning, the num_conv = 2 head, two-GPU data parallelism (skips on one GPU)
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


def _quiet():
    return contextlib.redirect_stdout(io.StringIO())


def _perturb_gn(m, seed):
    torch.manual_seed(seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "norm" in name and name.endswith("weight"):
                p.add_(0.2 * torch.randn_like(p))
            if "norm" in name and name.endswith("bias"):
                p.add_(0.1 * torch.randn_like(p))


def _model32(seed=42, n_classes=56):
    import unetsulc_b200
    torch.manual_seed(seed)
    m = unetsulc_b200.UNet3D(1, n_classes, init_channel_number=32)
    _perturb_gn(m, seed + 1)
    return m.cuda().train()


def _pair32(seed=42, n_classes=56):
    """fp32 oracle and our model with the same (GroupNorm-perturbed) weights"""
    import unetsulc_b200
    from oracle.unet3d_ref import UNet3DRef
    torch.manual_seed(seed)
    ref = UNet3DRef(1, n_classes, init_channel_number=32)
    _perturb_gn(ref, seed + 1)
    ours = unetsulc_b200.UNet3D(1, n_classes, init_channel_number=32)
    ours.load_state_dict(ref.state_dict())
    return ref.cuda(), ours.cuda()


# ------------------------------------------------------------------------------------------------ per-call oracle
def _record_shapes(monkeypatch, seen):
    """wraps the (spied) conv entry points of ops: records (kind, Cin, Cout) of every call"""
    from unetsulc_b200 import ops

    def wrap(name, key):
        f = getattr(ops, name)

        def g(*a, **k):
            seen.add(key(*a, **k))
            return f(*a, **k)
        monkeypatch.setattr(ops, name, g)

    wrap("conv3d_first_fwd", lambda x, w, y, *a, **k: ("first_fwd", w.shape[0]))
    wrap("conv3d_first_fwd_gn_stats", lambda x, w, y, *a, **k: ("first_fwd", w.shape[0]))
    wrap("conv3d_first_wgrad", lambda x, dy, cout, *a, **k: ("first_wgrad", cout))
    wrap("conv3d_igemm_gn_stats", lambda x, wp, y, cin, cout, *a, **k: ("fprop", cin, cout))
    wrap("conv3d_igemm_auto", lambda x, wp, y, cin, cout, relu: ("fprop" if relu else "dgrad", cin, cout))
    wrap("conv3d_dgrad_gn_bstats", lambda dy, wd, dx, cin, cout, *a, **k: ("dgrad_bstats", cin, cout))
    wrap("conv3d_wgrad", lambda x, dy, cin, cout, *a, **k: ("wgrad", cin, cout))
    wrap("conv3d_wgrad_partial", lambda x, dy, cin, cout, *a, **k: ("wgrad", cin, cout))


# the calls only a 32-filter network makes (dgrad calls name the dY channels first)
NEW_B1 = {("first_fwd", 16), ("first_wgrad", 16), ("fprop", 16, 32), ("dgrad_bstats", 32, 16), ("fprop", 96, 32),
          ("wgrad", 16, 32), ("wgrad", 32, 32), ("wgrad", 96, 32)}
NEW_B2 = {("first_fwd", 16), ("first_wgrad", 16), ("fprop", 16, 32), ("dgrad", 32, 16), ("fprop", 96, 32),
          ("wgrad", 16, 32), ("wgrad", 32, 32), ("wgrad", 96, 32)}
CONFIGS32 = {
    # name: (batch, shape, wgrad reduce mode, autograd surface, op coverage, call coverage)
    "b1_24x32x40": (1, (24, 32, 40), "inline", False,
                    so.FUSED_B1 | {"upcat_bwd_stats_2x", "conv_fprop_splitk", "conv_dgrad_splitk"}, NEW_B1),
    "b1_24x32x40_defer": (1, (24, 32, 40), "defer", False,
                          (so.FUSED_B1 - {"wgrad"}) | {"wgrad_defer", "upcat_bwd_stats_2x"}, NEW_B1),
    "b1_17x26x21": (1, (17, 26, 21), "inline", False, so.FUSED_B1 | {"upcat_bwd_stats_non2x"}, NEW_B1),
    "b1_40x48x56": (1, (40, 48, 56), "inline", False, so.FUSED_B1 | {"upcat_bwd_stats_2x"}, NEW_B1),
    "b2_17x26x21": (2, (17, 26, 21), "inline", False,
                    so.COMMON | {"conv_first", "gn_stats_pass", "gn_bwd_pass", "maxpool_bwd", "upcat_bwd_non2x",
                                 "head_train", "conv_fprop", "conv_dgrad"}, NEW_B2),
    "b1_24x32x40_autograd": (1, (24, 32, 40), "inline", True,
                             so.COMMON | {"head_fwd", "head_train", "head_grad_scale_dev", "gn_bwd_pass",
                                          "gn_bwd_acc", "maxpool_bwd_stats", "upcat_bwd_stats_2x"}, NEW_B1),
}


def _run_config32(monkeypatch, name, cfg):
    from unetsulc_b200 import models
    B, shape, mode, autograd, expect, expect_calls = cfg
    model = _model32()
    x, labels = so._data(B, shape)
    monkeypatch.setattr(models, "_WGRAD_REDUCE", mode)
    g_fb = None
    if autograd:
        _, _, _, g_fb = model.forward_backward(x, labels)
        g_fb = [g.clone() for g in g_fb]
        model.force_repack = True
    orc = so.Oracle()
    so.install_spies(monkeypatch, orc)
    calls = set()
    _record_shapes(monkeypatch, calls)
    if autograd:
        model.zero_grad(set_to_none=True)
        loss, _ = model.loss_and_preds(x, labels)
        (2.5 * loss).backward()
        grads = [p.grad for p in model.ordered_parameters()]
    else:
        _, _, _, grads = model.forward_backward(x, labels)
    torch.cuda.synchronize()
    print("\n[f32 %s] %d checks; worst error / bound:" % (name, len(orc.worst)))
    for op in sorted(orc.worst):
        print("    %-34s %.3e" % (op, orc.worst[op]))
    bad = {op: w for op, w in orc.worst.items() if not w <= 1.0}
    assert not bad, "ops outside their fp64 bound: %s" % bad
    assert not expect - orc.seen, "entry points not reached: %s" % sorted(expect - orc.seen)
    assert not expect_calls - calls, "f = 32 calls not reached: %s" % sorted(expect_calls - calls)
    assert all(g is not None and bool(torch.isfinite(g).all()) for g in grads)
    if autograd:
        so._compare_scaled(model, grads, g_fb, 2.5)


@pytest.mark.parametrize("name", list(CONFIGS32))
def test_width32_step_matches_fp64_per_call(monkeypatch, name):
    _run_config32(monkeypatch, name, CONFIGS32[name])


def test_width32_step_matches_fp64_per_call_baseline_shape(monkeypatch):
    _run_config32(monkeypatch, "b1_96x112x96",
                  (1, (96, 112, 96), "inline", False, so.FUSED_B1 | {"upcat_bwd_stats_2x"}, NEW_B1))


# ------------------------------------------------------------------------------------------------ kernel edge cases
def _kernels(fn):
    """names of the CUDA kernels fn launches (torch.profiler)"""
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


@pytest.mark.parametrize("cin,cout,dims,kernel", [
    # volumes above ops.SPLITK_MAX_VOXELS: the plain and the statistics launches take the same kernel
    (16, 16, (13, 25, 27), "conv3d_igemm_kernel<16"),     # KC = 16 chunk, N = 16 tile
    (16, 32, (5, 40, 41), "conv3d_igemm_kernel<16"),      # encoders.0.conv2 fprop where the slab would pad > 1.5x
    (32, 16, (9, 30, 31), "conv3d_igemm_kernel<32"),      # N = 16 tile; its dgrad is Cin = 16 on the slab kernel
    (48, 16, (7, 35, 34), "conv3d_igemm_kernel<16"),      # three 16-channel chunks (exact path, first two layers)
    (16, 32, (22, 30, 46), "conv3d_slab_kernel<16"),      # slab kernel, one 16-channel chunk, every side padded
    (96, 32, (22, 30, 46), "conv3d_slab_kernel<32"),      # decoders.2.conv1: three 32-channel chunks, padded box
])
def test_width32_conv_fprop_dgrad_against_fp64(monkeypatch, cin, cout, dims, kernel):
    from unetsulc_b200 import ops
    orc = so.Oracle()
    so.install_spies(monkeypatch, orc)
    x = _act(1, cin, *dims, seed=cin + cout)
    wf, wd = ops.pack_conv_weights(_weights(cout, cin, 7))
    y = ops.ActView.alloc(1, *dims, cout, "cuda")
    names = _kernels(lambda: ops.conv3d_igemm_auto(x, wf, y, cin, cout, relu=True))
    assert any(kernel in n for n in names), names
    # fused statistics on the same launch (batch 1)
    gamma, beta = torch.ones(cout, device="cuda"), torch.zeros(cout, device="cuda")
    y2 = ops.ActView.alloc(1, *dims, cout, "cuda")
    ops.conv3d_igemm_gn_stats(x, wf, y2, cin, cout, min(cout, 16), 1e-5, gamma, beta)
    assert torch.equal(y.buf, y2.buf)
    # dgrad of the same layer (dY has cout channels, dX cin), plain and with the GroupNorm-backward statistics
    dy = _act(1, cout, *dims, seed=3, scale=1e-3)
    dx = ops.ActView.alloc(1, *dims, cin, "cuda")
    ops.conv3d_igemm_auto(dy, wd, dx, cout, cin, relu=False)
    r = _act(1, cin, *dims, seed=5)
    r.buf.relu_()
    dx2 = ops.ActView.alloc(1, *dims, cin, "cuda")
    ops.conv3d_dgrad_gn_bstats(dy, wd, dx2, cout, cin, r)
    assert torch.equal(dx.buf, dx2.buf)
    print("worst error / bound:", orc.worst)
    assert {"conv_fprop", "conv_fprop_stats", "conv_dgrad", "conv_dgrad_bstats"} <= orc.seen
    assert all(w <= 1.0 for w in orc.worst.values()), orc.worst


@pytest.mark.parametrize("cin,cout,dims,defer", [
    (16, 32, (9, 13, 11), False), (16, 32, (16, 24, 32), True),   # Cin = 16 slots (odd box, then the halo box)
    (32, 32, (7, 10, 13), False), (32, 32, (48, 56, 48), True),   # Cout = 32 dY tiles, halo mode N = 96
    (96, 32, (11, 9, 14), False), (96, 32, (48, 56, 48), True),
])
def test_width32_wgrad_against_fp64(monkeypatch, cin, cout, dims, defer):
    from unetsulc_b200 import ops
    orc = so.Oracle()
    so.install_spies(monkeypatch, orc)
    x = _act(1, cin, *dims, seed=11)
    dy = _act(1, cout, *dims, seed=12, scale=1e-2)
    if defer:
        desc = ops.conv3d_wgrad_partial(x, dy, cin, cout, "w32")
        ops.wgrad_reduce_multi([desc])
        dw = desc["dw"]
    else:
        dw = ops.conv3d_wgrad(x, dy, cin, cout)
    again = ops.conv3d_wgrad(x, dy, cin, cout)
    assert torch.equal(dw, again)      # deterministic, and both reductions give the same bits
    print("worst error / bound:", orc.worst)
    assert all(w <= 1.0 for w in orc.worst.values()), orc.worst
    assert orc.worst["wgrad"] > 0.0


@pytest.mark.parametrize("dims", [(7, 9, 11), (33, 17, 40)])
def test_width32_first_layer_against_fp64(monkeypatch, dims):
    from unetsulc_b200 import ops
    from oracle.synth import synth_volume
    orc = so.Oracle()
    so.install_spies(monkeypatch, orc)
    x, _ = synth_volume(dims, 5, 77, occupancy=0.2)
    x = x.reshape(1, 1, *dims).cuda().contiguous()
    w = _weights(16, 1, 9)
    y = ops.ActView.alloc(1, *dims, 16, "cuda")
    ops.conv3d_first_fwd(x, w, y)
    y2 = ops.ActView.alloc(1, *dims, 16, "cuda")
    ops.conv3d_first_fwd_gn_stats(x, w, y2, 16, 1e-5, torch.ones(16, device="cuda"), torch.zeros(16, device="cuda"))
    assert torch.equal(y.buf, y2.buf)
    dy = _act(1, 16, *dims, seed=4, scale=1e-2)
    ops.conv3d_first_wgrad(x, dy, 16)
    print("worst error / bound:", orc.worst)
    assert {"conv_first", "conv_first_stats", "wgrad_first"} <= orc.seen
    assert all(w <= 1.0 for w in orc.worst.values()), orc.worst


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("shape", [(24, 32, 40), (96, 112, 96)])
def test_width32_end_to_end_against_fp32_oracle(shape):
    """DESIGN.md §5 bounds: logits rel-L2 <= 3e-2, loss <= 1e-2 rel, argmax >= 97 %, 44 gradients cos > 0.9 and norm
    ratio in (0.8, 1.25); with the oracle's ReLU masks aligned to ours 2.5e-2 above the first pooling boundary, 0.2
    below it, head 2e-2"""
    from oracle.synth import synth_volume
    from tests._aligned_oracle import run_aligned
    from unetsulc_b200 import models, ops
    assert not torch.backends.cudnn.allow_tf32 and not torch.backends.cuda.matmul.allow_tf32
    ref, ours = _pair32()
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
    print("f32 %s: logits rel-L2 %.3e, loss ours %.6f oracle %.6f, argmax agreement %.4f"
          % (shape, e, float(loss[0]), float(loss_r), agree))
    assert e < 3e-2
    assert abs(float(loss[0]) - float(loss_r)) < 1e-2 * abs(float(loss_r))
    assert agree >= 0.97
    order = {id(p): k for k, p in enumerate(ours.ordered_parameters())}
    named = dict(ours.named_parameters())
    cmin, rmin, rmax = 1.0, 10.0, 0.0
    for n, pr in ref.named_parameters():
        g = grads[order[id(named[n])]]
        c, ratio = cosine(g, pr.grad), float(g.norm() / pr.grad.norm())
        cmin, rmin, rmax = min(cmin, c), min(rmin, ratio), max(rmax, ratio)
        assert c > 0.9 and 0.8 < ratio < 1.25, (n, c, ratio)
    print("f32 %s: gradient cosine >= %.4f, norm ratio %.3f..%.3f" % (shape, cmin, rmin, rmax))
    # aligned ReLU masks
    ref.zero_grad(set_to_none=True)
    save = models._Saved()
    feat = ours._trunk_forward(x, save)
    head = ours.final_conv
    out = ops.head_ce(feat, labels, head.weight.detach(), head.bias.detach(), compute_grad=True)
    tg = ours._trunk_backward(save, out["dx"], [True] * 42)
    loss_a = run_aligned(ref, x, labels, [rc["r"].dense().float().permute(0, 4, 1, 2, 3) for rc in save.rec])
    assert abs(float(out["loss"][0]) - float(loss_a)) < 2e-3 * abs(float(loss_a))
    worst_above, worst_below = 0.0, 0.0
    names = [n for n, _ in ref.named_parameters() if not n.startswith("final_conv")]
    for n, g, (_, p) in zip(names, tg, [(n, p) for n, p in ref.named_parameters() if not n.startswith("final_conv")]):
        er = rel_l2(g, p.grad)
        below = n.startswith("encoders.0") or n.startswith("encoders.1") or n.startswith("encoders.2")
        if below:
            worst_below = max(worst_below, er)
        else:
            worst_above = max(worst_above, er)
        assert er < (0.2 if below else 2.5e-2), (n, er)
    print("f32 %s: aligned-mask gradients rel-L2 <= %.3e above / %.3e below the first pooling boundary"
          % (shape, worst_above, worst_below))
    assert rel_l2(out["dW"], ref.final_conv.weight.grad) < 2e-2
    assert rel_l2(out["db"], ref.final_conv.bias.grad) < 1e-2


@pytest.mark.parametrize("shape", [(24, 32, 40), (17, 26, 21)])
def test_width32_exact_mode(shape):
    from oracle.synth import synth_volume
    ref, ours = _pair32()
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
    print("f32 exact %s: %d voxels, max |score err| %.3e, label agreement %.6f" % (shape, len(idx), err,
                                                                                  float(same.float().mean())))
    assert err <= 1e-4
    assert bool(same[margin > 2e-4].all())


def test_width32_steps_are_deterministic():
    x, labels = so._data(1, (24, 32, 40))
    outs = []
    for _ in range(2):
        m = _model32()
        loss, _, _, grads = m.forward_backward(x, labels)
        outs.append((loss.clone(), [g.clone() for g in grads]))
    assert torch.equal(outs[0][0], outs[1][0])
    assert all(torch.equal(a, b) for a, b in zip(outs[0][1], outs[1][1]))


# ------------------------------------------------------------------------------------------------ API classes
def test_width32_learning_graph_replay_equals_eager_and_mdsm_round_trip(tmp_path):
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    from oracle.unet3d_ref import UNet3DRef
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=5, shape=(14, 16, 12), n_classes=6, seed=2)
    files = sorted(bck2)
    out = []
    for use_graph in (False, True):
        random.seed(7); np.random.seed(7); torch.manual_seed(7)
        with _quiet():
            m = UnetTrainingSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path),
                                           dict_model={'name': 'w32', 'num_filter': 32, 'img_size': [24, 24, 24]},
                                           dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
            m.use_cuda_graph = use_graph
            m.learning(1e-2, 0.9, 2, files[:4], files[4:], batch_size=1)
        assert m.model.init_channel_number == 32
        r = m.results
        out.append((r['epoch_loss_train'], r['epoch_loss_val'], r['epoch_acc_train'], r['epoch_acc_val']))
        assert all(np.isfinite(np.asarray(r['epoch_loss_train'], float)).ravel())
    assert out[0] == out[1]
    with _quiet():
        m.save_model(name='w32')
    path = tmp_path / 'models' / 'w32' / 'w32_model.mdsm'
    sd = torch.load(str(path), map_location='cpu')
    ref = UNet3DRef(1, len(sslist), init_channel_number=32)
    ref.load_state_dict(sd)
    for k, v in m.model.state_dict().items():
        assert torch.equal(v.cpu(), sd[k]), k
    with _quiet():
        m2 = UnetTrainingSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path),
                                        dict_model={'name': 'w32b', 'num_filter': 32},
                                        dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
        m2.load_network()
    m2.model.load_state_dict(ref.state_dict())
    for k, v in ref.state_dict().items():
        assert torch.equal(m2.model.state_dict()[k].cpu(), v), k


def test_width32_labeling_and_test_thresholds_and_two_conv_head(tmp_path):
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    from oracle.synth import synth_folds
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=2, shape=(24, 24, 24))
    files = sorted(bck2)
    for num_conv in (1, 2):
        torch.manual_seed(3)
        with _quiet():
            m = UnetTrainingSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path),
                                           dict_model={'name': 'lab32_%d' % num_conv, 'num_filter': 32,
                                                       'num_conv': num_conv},
                                           dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
            m.load_network()
        if num_conv == 2:
            assert [(c.in_channels, c.out_channels) for c in m.model.final_conv] == [(32, 19), (19, 6)]
        with _quiet():
            ytrue, ypred, yscores = m.labeling(files[0])
        n = len(bck2[files[0]])
        assert len(ypred) == n and yscores.shape == (n, len(sslist))
        assert np.allclose(yscores.sum(1), 1.0, atol=1e-5) and ypred == np.argmax(yscores, axis=1).tolist()
        # one training step through the chained head: gradients reach both links
        from oracle.synth import synth_volume
        x, l = synth_volume((24, 24, 24), len(sslist), 5, occupancy=0.08)
        m.model.train()
        loss, _, _, grads = m.model.forward_backward(x.unsqueeze(0).cuda(), l.unsqueeze(0).cuda())
        assert len(grads) == 42 + 2 * num_conv and all(bool(torch.isfinite(g).all()) for g in grads)
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


def test_width32_transfer_learning_two_phases(tmp_path):
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    from unetsulc_b200.transfer_learning import UnetTransferSulciLabelling
    bck2, names, sslist = harness.synthetic_cohort()
    files = sorted(bck2)
    torch.manual_seed(5)
    with _quiet():
        base = UnetTrainingSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path),
                                          dict_model={'name': 'base32', 'num_filter': 32},
                                          dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
        base.load_network()
        base.save_model()
    enc_before = base.model.encoders[0].double_conv.conv1.weight.detach().clone()
    with _quiet():
        tl = UnetTransferSulciLabelling(files, 'L', cuda=0, working_path=str(tmp_path), dict_model={'name': 'tl32'},
                                        dict_trained_model={'out_channels': len(sslist), 'init_channel_number': 32,
                                                            'model_file': str(tmp_path / 'models' /
                                                                              'base32_model.mdsm')},
                                        dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
        tl.learning(1e-2, 0.9, 5, files[:2], files[2:], patience={'fine_tunning': 100})
    assert tl.model.init_channel_number == 32
    assert tl.results['fine_tunning_epoch'] == [4]
    assert torch.equal(tl.model.encoders[0].double_conv.conv1.weight.detach().cpu(), enc_before)
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
        model = unetsulc_b200.UNet3D(1, 56, init_channel_number=32).to(dev).train()
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
        res["grad_worst"] = max(float((a - b).abs().max() / (b.abs().max() + 1e-30)) for a, b in zip(views, g_avg))
        model.grad_ready_hook = None
        del model, red
        bck2, names, sslist = harness.synthetic_cohort(n_subjects=7, shape=(14, 16, 12), n_classes=6, seed=2)
        files = sorted(bck2)
        random.seed(7); np.random.seed(7); torch.manual_seed(7 + rank)
        with contextlib.redirect_stdout(io.StringIO()):
            m = UnetTrainingSulciLabelling(files, 'L', cuda=rank, working_path=tmp,
                                           dict_model={'name': 'dp32', 'num_filter': 32, 'img_size': [24, 24, 24]},
                                           dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
            m.learning(1e-2, 0.9, 2, files[:5], files[5:], batch_size=1)
        res["learn"] = (m.results['epoch_loss_train'], m.results['epoch_loss_val'])
        res["sync"] = parallel.parameters_in_sync(m.model)
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_width32_data_parallel_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29900 + os.getpid() % 300
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, str(tmp_path), q)) for r in range(world)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    for r in range(world):
        assert out[r]["grad_worst"] < 1e-5 and out[r]["sync"]
    assert out[0]["learn"] == out[1]["learn"]
