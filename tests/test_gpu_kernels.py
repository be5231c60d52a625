"""GPU parity tests, kernel by kernel, through the C-ABI (ctypes) of libunetsulc_b200.so.

Checker = plain PyTorch fp32 ops on the same (bf16-rounded) inputs.  Tolerances (SURVEY.md §8(d)):
  * bf16-output conv kernels ............ rel-L2 <= 2e-3 (one bf16 rounding of an fp32-accumulated result)
  * fp32-output conv / wgrad kernels .... rel-L2 <= 1e-4 (summation order only)
  * GroupNorm / resample (bf16 out) ..... rel-L2 <= 4e-3
  * integer pass (fold vote, counters) .. bit-exact
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ops():
    import unetsulc_b200  # noqa: F401
    from unetsulc_b200 import ops
    return ops


def rel_l2(a, b):
    a = a.double().flatten()
    b = b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def bf16_round(t):
    return t.to(torch.bfloat16).float()


def to_ndhwc(t):   # [N,C,D,H,W] fp32 -> contiguous [N,D,H,W,C] bf16
    return t.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)


def from_view(v):  # ActView -> [N,C,D,H,W] fp32
    return v.dense().float().permute(0, 4, 1, 2, 3).contiguous()


CONV_SHAPES = [
    # N, Cin, Cout, D, H, W
    (1, 64, 64, 8, 16, 32),
    (1, 32, 64, 6, 10, 36),      # 64-byte swizzle path (Cin = 32)
    (1, 192, 64, 8, 8, 32),
    (1, 128, 256, 6, 7, 6),
    (1, 256, 512, 3, 4, 5),      # two N tiles
    (2, 64, 128, 5, 7, 9),       # odd sizes, batch 2
    (1, 64, 32, 4, 8, 16),       # dgrad shape of encoders.0.conv2
    (1, 128, 384, 4, 6, 8),      # N tile 192 (dgrad of decoders.1.conv1)
]


@pytest.mark.parametrize("shape", CONV_SHAPES)
@pytest.mark.parametrize("fp32_out", [True, False])
def test_conv_fprop(shape, fp32_out):
    ops = _ops()
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(1)
    x = bf16_round(torch.randn(N, Cin, D, H, W, device="cuda", generator=g))
    w = bf16_round(torch.randn(Cout, Cin, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * Cin) ** 0.5))
    ref = F.conv3d(x, w, padding=1)
    wf, _ = ops.pack_conv_weights(w)
    assert torch.equal(wf.float(), w.permute(2, 3, 4, 0, 1).reshape(27, Cout, Cin))
    xv = ops.ActView(to_ndhwc(x), N, D, H, W, Cin)
    if fp32_out:
        ybuf = torch.zeros(N, D, H, W, Cout, device="cuda", dtype=torch.float32)
        yv = ops.ActView(ybuf, N, D, H, W, Cout)
        ops.conv3d_igemm(xv, wf, yv, Cin, Cout, relu=False, y_fp32=True)
        torch.cuda.synchronize()
        got = ybuf.permute(0, 4, 1, 2, 3)
        err = rel_l2(got, ref)
        assert err < 1e-4, "fp32-out conv rel-L2 %.3e" % err
    else:
        yv = ops.ActView.alloc(N, D, H, W, Cout, "cuda", zero=True)
        ops.conv3d_igemm(xv, wf, yv, Cin, Cout, relu=True)
        torch.cuda.synchronize()
        err = rel_l2(from_view(yv), F.relu(ref))
        assert err < 2e-3, "bf16-out conv rel-L2 %.3e" % err


SLAB_SHAPES = [
    # shapes the shared-memory tap-reuse kernel (conv_slab.cu) takes: Cout in {32, 64}, tile-aligned volumes
    (1, 64, 64, 8, 12, 64),
    (1, 32, 64, 8, 12, 64),      # KC = 32 planes
    (1, 192, 64, 8, 8, 32),      # 3 channel chunks
    (1, 64, 32, 8, 12, 64),      # N = 32 (dgrad of encoders.0.conv2)
    (2, 64, 64, 8, 12, 60),      # ragged W edge (60 -> 64), batch 2
    (1, 64, 64, 4, 4, 32),       # a single tile: every plane touches the volume border
    (1, 64, 64, 10, 13, 72),     # 16 x 8 x 4 tile shape (W = 72 pads to 80, not 96); ragged H and D edges
    (1, 32, 64, 8, 16, 48),      # 16-wide tiles with 64-byte rows (KC = 32)
    (1, 192, 64, 6, 9, 40),      # 16-wide tiles, 3 channel chunks, ragged everywhere
    (1, 64, 32, 9, 11, 24),      # 16-wide tiles, N = 32
]


@pytest.mark.parametrize("shape", SLAB_SHAPES)
def test_conv_slab_kernel(shape):
    ops = _ops()
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(31)
    x = bf16_round(torch.randn(N, Cin, D, H, W, device="cuda", generator=g))
    w = bf16_round(torch.randn(Cout, Cin, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * Cin) ** 0.5))
    wf, wd = ops.pack_conv_weights(w)
    wide = torch.full((N, D, H, W, Cout + 16), 3.0, device="cuda", dtype=torch.bfloat16)
    yv = ops.ActView(wide, N, D, H, W, Cout, ld=Cout + 16, coff=8)
    ops.conv3d_igemm(ops.ActView(to_ndhwc(x), N, D, H, W, Cin), wf, yv, Cin, Cout, relu=True)
    torch.cuda.synchronize()
    ref = F.relu(F.conv3d(x, w, padding=1))
    err = rel_l2(from_view(yv), ref)
    assert err < 2e-3, "slab fprop rel-L2 %.3e" % err
    assert bool((wide[..., :8] == 3.0).all()) and bool((wide[..., Cout + 8:] == 3.0).all())
    # dgrad through the same kernel (roles of Cin / Cout swapped) when the output width allows it
    if Cin in (32, 64):
        dy = bf16_round(torch.randn(N, Cout, D, H, W, device="cuda", generator=g))
        xq = torch.zeros(N, Cin, D, H, W, device="cuda", requires_grad=True)
        F.conv3d(xq, w, padding=1).backward(dy)
        dx = ops.ActView.alloc(N, D, H, W, Cin, "cuda", zero=True)
        ops.conv3d_igemm(ops.ActView(to_ndhwc(dy), N, D, H, W, Cout), wd, dx, Cout, Cin, relu=False)
        torch.cuda.synchronize()
        err = rel_l2(from_view(dx), xq.grad)
        assert err < 2e-3, "slab dgrad rel-L2 %.3e" % err


@pytest.mark.parametrize("shape", [(1, 64, 64, 8, 12, 64), (1, 128, 256, 6, 7, 6), (1, 64, 128, 5, 7, 9),
                                   (1, 32, 64, 8, 12, 64), (1, 192, 64, 8, 8, 32)])
def test_conv_epilogue_groupnorm_statistics(shape):
    """GroupNorm statistics fused into the conv epilogue == statistics of a separate pass over the stored tensor."""
    ops = _ops()
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(41)
    x = bf16_round(torch.randn(N, Cin, D, H, W, device="cuda", generator=g))
    w = bf16_round(torch.randn(Cout, Cin, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * Cin) ** 0.5))
    gamma = torch.randn(Cout, device="cuda", generator=g) * 0.5 + 1.0
    beta = torch.randn(Cout, device="cuda", generator=g) * 0.1
    wf, _ = ops.pack_conv_weights(w)
    xv = ops.ActView(to_ndhwc(x), N, D, H, W, Cin)
    r1 = ops.ActView.alloc(N, D, H, W, Cout, "cuda", zero=True)
    mr1, ss1 = ops.conv3d_igemm_gn_stats(xv, wf, r1, Cin, Cout, 32, 1e-5, gamma, beta)   # exact accumulators
    r2 = ops.ActView.alloc(N, D, H, W, Cout, "cuda", zero=True)
    ops.conv3d_igemm(xv, wf, r2, Cin, Cout, relu=True)
    mr2, ss2 = ops.relu_gn_stats(r2, 32, 1e-5, gamma, beta)
    torch.cuda.synchronize()
    assert torch.equal(r1.buf, r2.buf)
    assert torch.allclose(mr1, mr2, rtol=1e-5, atol=1e-6)
    assert torch.allclose(ss1, ss2, rtol=1e-5, atol=1e-6)
    ref = F.group_norm(from_view(r2), 32, gamma, beta, 1e-5)
    y = ops.ActView.alloc(N, D, H, W, Cout, "cuda")
    ops.relu_gn_apply(r1, ss1, y)
    assert rel_l2(from_view(y), ref) < 4e-3
    # the accumulators hold the exact sums of the stored tensor: compare with an fp64 reduction
    lib = ops._lib.load()
    acc = torch.zeros(4 * Cout, dtype=torch.int64, device="cuda")
    r3 = ops.ActView.alloc(N, D, H, W, Cout, "cuda", zero=True)
    ops._lib.check(lib.b2_conv3d_igemm_stats(ops._p(xv.buf), xv.ld, xv.coff, ops._p(wf), ops._p(r3.buf), r3.ld, r3.coff,
                                             N, D, H, W, Cin, Cout, 1, ops._p(acc), ops._s()), "b2_conv3d_igemm_stats")
    torch.cuda.synchronize()
    a4 = acc.view(Cout, 4).double()
    rr = r2.buf.double().reshape(-1, Cout)
    assert torch.allclose(a4[:, 0] + a4[:, 1] / 2.0 ** 32, rr.sum(0), rtol=1e-6, atol=1e-3)
    assert torch.allclose(a4[:, 2] + a4[:, 3] / 2.0 ** 32, (rr * rr).sum(0), rtol=1e-6, atol=1e-3)


@pytest.mark.parametrize("shape", [(1, 256, 512, 12, 14, 12), (1, 256, 256, 6, 7, 6), (1, 64, 128, 5, 7, 9),
                                   (1, 128, 64, 3, 4, 5)])
def test_conv_splitk_small_volumes(shape):
    """fewer output tiles than half the SMs: split-K over the 27 taps + fp32 reduce (+ReLU) kernel."""
    ops = _ops()
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(61)
    x = bf16_round(torch.randn(N, Cin, D, H, W, device="cuda", generator=g))
    w = bf16_round(torch.randn(Cout, Cin, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * Cin) ** 0.5))
    wf, wd = ops.pack_conv_weights(w)
    wide = torch.full((N, D, H, W, Cout + 16), 5.0, device="cuda", dtype=torch.bfloat16)
    yv = ops.ActView(wide, N, D, H, W, Cout, ld=Cout + 16, coff=8)
    ops.conv3d_igemm_auto(ops.ActView(to_ndhwc(x), N, D, H, W, Cin), wf, yv, Cin, Cout, relu=True)
    torch.cuda.synchronize()
    ref = F.relu(F.conv3d(x, w, padding=1))
    assert rel_l2(from_view(yv), ref) < 2e-3
    assert bool((wide[..., :8] == 5.0).all()) and bool((wide[..., Cout + 8:] == 5.0).all())
    dy = bf16_round(torch.randn(N, Cout, D, H, W, device="cuda", generator=g))
    xq = torch.zeros(N, Cin, D, H, W, device="cuda", requires_grad=True)
    F.conv3d(xq, w, padding=1).backward(dy)
    dx = ops.ActView.alloc(N, D, H, W, Cin, "cuda", zero=True)
    ops.conv3d_igemm_auto(ops.ActView(to_ndhwc(dy), N, D, H, W, Cout), wd, dx, Cout, Cin, relu=False)
    torch.cuda.synchronize()
    assert rel_l2(from_view(dx), xq.grad) < 2e-3


def test_conv_fprop_channel_windows():
    """input read from / output written into channel windows of wider buffers (concat buffers)."""
    ops = _ops()
    N, Cin, Cout, D, H, W = 1, 64, 64, 4, 8, 16
    g = torch.Generator(device="cuda").manual_seed(2)
    x = bf16_round(torch.randn(N, Cin, D, H, W, device="cuda", generator=g))
    w = bf16_round(torch.randn(Cout, Cin, 3, 3, 3, device="cuda", generator=g) * 0.03)
    wide_in = torch.randn(N, D, H, W, 192, device="cuda", generator=g).to(torch.bfloat16)
    wide_in[..., 128:192] = to_ndhwc(x)
    wide_out = torch.full((N, D, H, W, 160), 7.0, device="cuda", dtype=torch.bfloat16)
    wf, _ = ops.pack_conv_weights(w)
    xv = ops.ActView(wide_in, N, D, H, W, Cin, ld=192, coff=128)
    yv = ops.ActView(wide_out, N, D, H, W, Cout, ld=160, coff=32)
    ops.conv3d_igemm(xv, wf, yv, Cin, Cout, relu=True)
    torch.cuda.synchronize()
    ref = F.relu(F.conv3d(x, w, padding=1))
    assert rel_l2(from_view(yv), ref) < 2e-3
    assert bool((wide_out[..., :32] == 7.0).all()) and bool((wide_out[..., 96:] == 7.0).all())


@pytest.mark.parametrize("shape", CONV_SHAPES[:6])
def test_conv_dgrad(shape):
    ops = _ops()
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(3)
    dy = bf16_round(torch.randn(N, Cout, D, H, W, device="cuda", generator=g))
    w = bf16_round(torch.randn(Cout, Cin, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * Cout) ** 0.5))
    x = torch.zeros(N, Cin, D, H, W, device="cuda", requires_grad=True)
    F.conv3d(x, w, padding=1).backward(dy)
    ref = x.grad
    _, wd = ops.pack_conv_weights(w)
    dyv = ops.ActView(to_ndhwc(dy), N, D, H, W, Cout)
    dxbuf = torch.zeros(N, D, H, W, Cin, device="cuda", dtype=torch.float32)
    ops.conv3d_igemm(dyv, wd, ops.ActView(dxbuf, N, D, H, W, Cin), Cout, Cin, relu=False, y_fp32=True)
    torch.cuda.synchronize()
    err = rel_l2(dxbuf.permute(0, 4, 1, 2, 3), ref)
    assert err < 1e-4, "dgrad rel-L2 %.3e" % err


WGRAD_SHAPES = [
    (1, 64, 64, 8, 16, 32),
    (1, 32, 64, 6, 10, 36),      # 64-byte swizzle slots (Cin = 32)
    (1, 192, 64, 8, 8, 32),
    (1, 128, 256, 6, 7, 6),
    (1, 256, 512, 3, 4, 5),
    (2, 64, 128, 5, 7, 9),
    (1, 384, 128, 4, 6, 8),
    # 64-wide fixed operand with one-plane tile boxes: the "dY-halo" mode (three h taps per MMA)
    (1, 32, 64, 5, 12, 32),
    (2, 64, 64, 3, 9, 16),       # ragged h tiles: the halo lines of the last tile are out of range
    (1, 96, 64, 3, 8, 16),       # three 32-channel chunks
    (1, 64, 64, 2, 3, 128),      # one-line tiles (bh = 1): the halo is two thirds of the box
    (1, 768, 256, 4, 8, 32),     # 81 (group chunk) columns > SMs / 2: stream-K runs, two segments per CTA
    (1, 704, 256, 5, 9, 24),     # ... ragged tiles, last chunk with one group
]


@pytest.mark.parametrize("shape", WGRAD_SHAPES)
def test_conv_wgrad(shape):
    ops = _ops()
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(4)
    x = bf16_round(torch.randn(N, Cin, D, H, W, device="cuda", generator=g))
    dy = bf16_round(torch.randn(N, Cout, D, H, W, device="cuda", generator=g))
    w = torch.zeros(Cout, Cin, 3, 3, 3, device="cuda", requires_grad=True)
    F.conv3d(x, w, padding=1).backward(dy)
    ref = w.grad
    got = ops.conv3d_wgrad(ops.ActView(to_ndhwc(x), N, D, H, W, Cin), ops.ActView(to_ndhwc(dy), N, D, H, W, Cout),
                           Cin, Cout)
    torch.cuda.synchronize()
    err = rel_l2(got, ref)
    assert err < 1e-4, "wgrad rel-L2 %.3e" % err


@pytest.mark.parametrize("cin,cout,dims", [(64, 128, (48, 56, 48)), (192, 64, (40, 56, 96)), (768, 256, (24, 28, 24))])
def test_conv_full_size_layers_deterministic_and_exact(cin, cout, dims):
    """BASELINE-sized layers: many tiles per persistent CTA (exercises the smem ring and the TMEM double buffer);
    results must be bit-identical run to run and match the fp32 checker."""
    ops = _ops()
    D, H, W = dims
    g = torch.Generator(device="cuda").manual_seed(21)
    x = bf16_round(torch.randn(1, cin, D, H, W, device="cuda", generator=g))
    dy = bf16_round(torch.randn(1, cout, D, H, W, device="cuda", generator=g))
    w = bf16_round(torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * cin) ** 0.5))
    wf, wd = ops.pack_conv_weights(w)
    xv = ops.ActView(to_ndhwc(x), 1, D, H, W, cin)
    dyv = ops.ActView(to_ndhwc(dy), 1, D, H, W, cout)
    outs = []
    for _ in range(2):
        y = ops.ActView.alloc(1, D, H, W, cout, "cuda", zero=True)
        ops.conv3d_igemm(xv, wf, y, cin, cout, relu=True)
        dx = ops.ActView.alloc(1, D, H, W, cin, "cuda", zero=True)
        ops.conv3d_igemm(dyv, wd, dx, cout, cin, relu=False)
        dw = ops.conv3d_wgrad(xv, dyv, cin, cout)
        torch.cuda.synchronize()
        outs.append((y.buf.clone(), dx.buf.clone(), dw.clone()))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)
    xq = x.clone().requires_grad_(True)
    wq = w.clone().requires_grad_(True)
    ref = F.conv3d(xq, wq, padding=1)
    ref.backward(dy)
    assert rel_l2(outs[0][0].float().permute(0, 4, 1, 2, 3), F.relu(ref)) < 2e-3
    assert rel_l2(outs[0][1].float().permute(0, 4, 1, 2, 3), xq.grad) < 2e-3
    e = rel_l2(outs[0][2], wq.grad)
    print("full-size wgrad rel-L2 %.3e" % e)
    assert e < 2e-4


@pytest.mark.parametrize("cin,cout,dims", [(64, 64, (32, 56, 96)), (192, 64, (16, 28, 96)), (32, 64, (32, 56, 96)),
                                           (128, 128, (48, 56, 48)), (256, 512, (12, 14, 12))])
def test_conv_pipelines_stress_bitwise(cin, cout, dims):
    """30 back-to-back launches of fprop (+ fused GroupNorm statistics), dgrad and wgrad must be bit-identical:
    a barrier-protocol race in the TMA / tcgen05 / TMEM pipelines would show up as run-to-run differences."""
    ops = _ops()
    D, H, W = dims
    g = torch.Generator(device="cuda").manual_seed(51)
    x = ops.ActView(torch.randn(1, D, H, W, cin, device="cuda", generator=g).to(torch.bfloat16), 1, D, H, W, cin)
    dy = ops.ActView(torch.randn(1, D, H, W, cout, device="cuda", generator=g).to(torch.bfloat16), 1, D, H, W, cout)
    w = torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) * 0.02
    gamma = torch.ones(cout, device="cuda"); beta = torch.zeros(cout, device="cuda")
    wf, wd = ops.pack_conv_weights(w)
    first = None
    for it in range(30):
        y = ops.ActView.alloc(1, D, H, W, cout, "cuda")
        if cout <= 256:
            mr, _ = ops.conv3d_igemm_gn_stats(x, wf, y, cin, cout, 32, 1e-5, gamma, beta)
        else:
            ops.conv3d_igemm(x, wf, y, cin, cout, relu=True)
            mr, _ = ops.relu_gn_stats(y, 32, 1e-5, gamma, beta)
        dx = ops.ActView.alloc(1, D, H, W, cin, "cuda")
        ops.conv3d_igemm(dy, wd, dx, cout, cin, relu=False)
        dw = ops.conv3d_wgrad(x, dy, cin, cout)
        cur = (y.buf, mr, dx.buf, dw)
        if first is None:
            first = tuple(t.clone() for t in cur)
        else:
            for name, a, b in zip(("fprop", "stats", "dgrad", "wgrad"), first, cur):
                assert torch.equal(a, b), "%s differs at iteration %d" % (name, it)
    torch.cuda.synchronize()


def test_conv_first_layer():
    ops = _ops()
    N, Cout, D, H, W = 2, 32, 9, 12, 17
    g = torch.Generator(device="cuda").manual_seed(5)
    x = (torch.rand(N, 1, D, H, W, device="cuda", generator=g) < 0.05).float()
    w = torch.randn(Cout, 1, 3, 3, 3, device="cuda", generator=g) * 0.2
    yv = ops.ActView.alloc(N, D, H, W, Cout, "cuda")
    ops.conv3d_first_fwd(x, w, yv, relu=True)
    ref = F.relu(F.conv3d(x, w, padding=1))
    assert rel_l2(from_view(yv), ref) < 2e-3
    dy = bf16_round(torch.randn(N, Cout, D, H, W, device="cuda", generator=g))
    wp = w.clone().requires_grad_(True)
    F.conv3d(x, wp, padding=1).backward(dy)
    got = ops.conv3d_first_wgrad(x, ops.ActView(to_ndhwc(dy), N, D, H, W, Cout), Cout)
    torch.cuda.synchronize()
    assert rel_l2(got, wp.grad) < 1e-5


_PAIR_SNIPPET = r"""
import sys, torch, torch.nn.functional as F
sys.path.insert(0, %r)
import unetsulc_b200
from unetsulc_b200 import ops
g = torch.Generator(device="cuda").manual_seed(3)
worst = 0.0
for (cin, cout, D, H, W) in [(64, 128, 16, 24, 40), (128, 256, 9, 20, 24), (192, 192, 8, 16, 24)]:
    x = torch.randn(1, cin, D, H, W, device="cuda", generator=g).to(torch.bfloat16).float()
    w = (torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) / (27 * cin) ** 0.5).to(torch.bfloat16).float()
    wf, _ = ops.pack_conv_weights(w)
    xv = ops.ActView(x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16), 1, D, H, W, cin)
    y = ops.ActView.alloc(1, D, H, W, cout, "cuda")
    ops.conv3d_igemm(xv, wf, y, cin, cout, relu=True)
    ref = F.relu(F.conv3d(x, w, padding=1))
    got = y.buf.float().permute(0, 4, 1, 2, 3)
    worst = max(worst, float((got - ref).norm() / ref.norm()))
torch.cuda.synchronize()
print("PAIR_REL_L2 %%.3e" %% worst)
"""


def test_conv_cta_pair_kernel_opt_in():
    """the cta_group::2 variant (B2_2CTA=1, read once per process) against fp32 torch on bf16-rounded inputs, with an
    odd number of 128-voxel tiles in one case"""
    import subprocess
    import sys
    env = dict(os.environ, B2_2CTA="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _PAIR_SNIPPET % root], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    rel = float(r.stdout.split("PAIR_REL_L2")[1].split()[0])
    assert rel < 3e-3, rel


@pytest.mark.parametrize("shape", [(64, 64, 8, 12, 64), (128, 64, 6, 8, 32), (256, 128, 6, 7, 6)])
def test_dgrad_fused_groupnorm_backward_statistics(shape):
    """dgrad with (sum dX, sum dX*r) accumulated in its epilogue + the one-launch GroupNorm backward that finalises
    them in its prologue == plain dgrad followed by the two-pass GroupNorm backward."""
    ops = _ops()
    Cdy, Cdx, D, H, W = shape
    G = 32
    g = torch.Generator(device="cuda").manual_seed(61)
    dy = ops.ActView(torch.randn(1, D, H, W, Cdy, device="cuda", generator=g).to(torch.bfloat16), 1, D, H, W, Cdy)
    w = torch.randn(Cdy, Cdx, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * Cdy) ** 0.5)
    _, wd = ops.pack_conv_weights(w)
    r = ops.ActView(torch.randn(1, D, H, W, Cdx, device="cuda", generator=g).relu().to(torch.bfloat16), 1, D, H, W, Cdx)
    gamma = torch.randn(Cdx, device="cuda", generator=g) * 0.5 + 1.0
    beta = torch.zeros(Cdx, device="cuda")
    mr, _ = ops.relu_gn_stats(r, G, 1e-5, gamma, beta)
    dx1 = ops.ActView.alloc(1, D, H, W, Cdx, "cuda")
    acc = ops.conv3d_dgrad_gn_bstats(dy, wd, dx1, Cdy, Cdx, r)
    dr1, dg1, db1 = ops.relu_gn_bwd_from_stats(acc, dx1, r, G, gamma, mr)
    dx2 = ops.ActView.alloc(1, D, H, W, Cdx, "cuda")
    ops.conv3d_igemm(dy, wd, dx2, Cdy, Cdx, relu=False)
    dr2, dg2, db2 = ops.relu_gn_bwd(dx2, r, G, gamma, mr)
    torch.cuda.synchronize()
    assert torch.equal(dx1.buf, dx2.buf)
    assert rel_l2(dr1.buf.float(), dr2.buf.float()) < 2e-3
    assert torch.allclose(dg1, dg2, rtol=1e-4, atol=1e-3)
    assert torch.allclose(db1, db2, rtol=1e-4, atol=1e-3)


def test_conv_first_layer_fused_gn_stats():
    """first conv with the GroupNorm statistics fused in == first conv followed by the statistics kernel"""
    ops = _ops()
    Cout, D, H, W, G = 32, 19, 21, 37, 32
    g = torch.Generator(device="cuda").manual_seed(15)
    x = (torch.rand(1, 1, D, H, W, device="cuda", generator=g) < 0.05).float()
    w = torch.randn(Cout, 1, 3, 3, 3, device="cuda", generator=g) * 0.2
    gamma = torch.randn(Cout, device="cuda", generator=g) * 0.5 + 1.0
    beta = torch.randn(Cout, device="cuda", generator=g) * 0.1
    y0 = ops.ActView.alloc(1, D, H, W, Cout, "cuda")
    ops.conv3d_first_fwd(x, w, y0, relu=True)
    mr0, ss0 = ops.relu_gn_stats(y0, G, 1e-5, gamma, beta)
    y1 = ops.ActView.alloc(1, D, H, W, Cout, "cuda")
    mr1, ss1 = ops.conv3d_first_fwd_gn_stats(x, w, y1, G, 1e-5, gamma, beta)
    torch.cuda.synchronize()
    assert torch.equal(y0.buf, y1.buf)
    assert torch.allclose(mr0, mr1, rtol=1e-5, atol=1e-6)
    assert torch.allclose(ss0, ss1, rtol=1e-5, atol=1e-6)
    ref = F.relu(F.conv3d(x, w, padding=1))
    assert rel_l2(from_view(y1), ref) < 2e-3


@pytest.mark.parametrize("C,D,H,W,N", [(32, 8, 10, 12, 1), (64, 9, 11, 13, 2), (256, 4, 6, 6, 1), (512, 3, 4, 5, 1)])
def test_relu_groupnorm_fwd_bwd(C, D, H, W, N):
    ops = _ops()
    G = 32
    g = torch.Generator(device="cuda").manual_seed(6)
    conv_out = torch.randn(N, C, D, H, W, device="cuda", generator=g)
    r = bf16_round(F.relu(conv_out))                     # what the conv epilogue stores
    gamma = torch.randn(C, device="cuda", generator=g) * 0.5 + 1.0
    beta = torch.randn(C, device="cuda", generator=g) * 0.1
    rv = ops.ActView(to_ndhwc(r), N, D, H, W, C)
    mr, ss = ops.relu_gn_stats(rv, G, 1e-5, gamma, beta)
    # plain apply into a channel window
    wide = torch.zeros(N, D, H, W, C + 16, device="cuda", dtype=torch.bfloat16)
    yv = ops.ActView(wide, N, D, H, W, C, ld=C + 16, coff=8)
    ops.relu_gn_apply(rv, ss, yv)
    rq = r.clone().requires_grad_(True)
    gq, bq = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    ref = F.group_norm(rq, G, gq, bq, 1e-5)
    torch.cuda.synchronize()
    assert rel_l2(from_view(yv), ref) < 4e-3
    # apply + pool
    y2 = ops.ActView.alloc(N, D, H, W, C, "cuda")
    pooled = ops.ActView.alloc(N, D // 2, H // 2, W // 2, C, "cuda")
    ops.relu_gn_apply(rv, ss, y2, pooled)
    torch.cuda.synchronize()
    assert torch.equal(y2.dense(), yv.dense())
    assert torch.equal(from_view(pooled), F.max_pool3d(from_view(y2), 2))
    # backward
    dy = bf16_round(torch.randn(N, C, D, H, W, device="cuda", generator=g))
    ref.backward(dy)
    dr, dg, db = ops.relu_gn_bwd(ops.ActView(to_ndhwc(dy), N, D, H, W, C), rv, G, gamma, mr)
    torch.cuda.synchronize()
    ref_dr = rq.grad * (r > 0).float()
    assert rel_l2(from_view(dr), ref_dr) < 4e-3
    assert rel_l2(dg, gq.grad) < 1e-3
    assert rel_l2(db, bq.grad) < 1e-3


@pytest.mark.parametrize("D,H,W", [(8, 10, 12), (7, 9, 11)])
def test_maxpool_bwd_add(D, H, W):
    ops = _ops()
    N, C = 1, 64
    g = torch.Generator(device="cuda").manual_seed(7)
    y = bf16_round(torch.randn(N, C, D, H, W, device="cuda", generator=g)).requires_grad_(True)
    dskip = bf16_round(torch.randn(N, C, D, H, W, device="cuda", generator=g))
    dpool = bf16_round(torch.randn(N, C, D // 2, H // 2, W // 2, device="cuda", generator=g))
    F.max_pool3d(y, 2).backward(dpool)
    ref = y.grad + dskip
    wide = torch.zeros(N, D, H, W, 192, device="cuda", dtype=torch.bfloat16)
    wide[..., :C] = to_ndhwc(y.detach())
    dwide = torch.zeros(N, D, H, W, 192, device="cuda", dtype=torch.bfloat16)
    dwide[..., :C] = to_ndhwc(dskip)
    out = ops.maxpool3d_bwd_add(ops.ActView(wide, N, D, H, W, C, ld=192), ops.ActView(dwide, N, D, H, W, C, ld=192),
                                ops.ActView(to_ndhwc(dpool), N, D // 2, H // 2, W // 2, C))
    torch.cuda.synchronize()
    assert rel_l2(from_view(out), ref) < 4e-3


@pytest.mark.parametrize("C,D,H,W", [(64, 8, 10, 12), (128, 7, 9, 11), (256, 6, 6, 8), (40, 6, 8, 10)])
def test_maxpool_bwd_add_with_groupnorm_backward_statistics(C, D, H, W):
    """pooling adjoint that also accumulates (sum out, sum out*r) of the tensor it produces: same output as the plain
    entry point, accumulators == fp64 sums of the stored tensor (C = 40: plain entry point only)"""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(17)
    y = bf16_round(torch.randn(1, C, D, H, W, device="cuda", generator=g)).requires_grad_(True)
    dskip = bf16_round(torch.randn(1, C, D, H, W, device="cuda", generator=g))
    dpool = bf16_round(torch.randn(1, C, D // 2, H // 2, W // 2, device="cuda", generator=g))
    r = bf16_round(torch.randn(1, C, D, H, W, device="cuda", generator=g).relu())
    F.max_pool3d(y, 2).backward(dpool)
    ref = y.grad + dskip
    yv = ops.ActView(to_ndhwc(y.detach()), 1, D, H, W, C)
    dv = ops.ActView(to_ndhwc(dskip), 1, D, H, W, C)
    pv = ops.ActView(to_ndhwc(dpool), 1, D // 2, H // 2, W // 2, C)
    out0 = ops.maxpool3d_bwd_add(yv, dv, pv)
    torch.cuda.synchronize()
    assert rel_l2(from_view(out0), ref) < 4e-3
    if 256 % (C // 8) != 0:
        return          # the fused statistics need C/8 to divide the block size
    out1, acc = ops.maxpool3d_bwd_add(yv, dv, pv, stat_r=ops.ActView(to_ndhwc(r), 1, D, H, W, C))
    torch.cuda.synchronize()
    assert torch.equal(out0.buf, out1.buf)
    a4 = acc.view(C, 4).double()
    o = out1.buf.double().reshape(-1, C)
    rr = to_ndhwc(r).double().reshape(-1, C)
    assert torch.allclose(a4[:, 0] + a4[:, 1] / 2.0 ** 32, o.sum(0), rtol=1e-5, atol=1e-3)
    assert torch.allclose(a4[:, 2] + a4[:, 3] / 2.0 ** 32, (o * rr).sum(0), rtol=1e-5, atol=1e-3)


@pytest.mark.parametrize("din,dout", [((4, 5, 6), (8, 10, 12)), ((3, 4, 5), (7, 9, 11)), ((6, 7, 6), (12, 14, 12))])
def test_upsample_concat_fwd_bwd(din, dout):
    ops = _ops()
    N, C, Cs = 1, 128, 64
    g = torch.Generator(device="cuda").manual_seed(8)
    x = bf16_round(torch.randn(N, C, *din, device="cuda", generator=g)).requires_grad_(True)
    ref = F.interpolate(x, size=dout, mode="trilinear", align_corners=False)
    cat = torch.zeros(N, *dout, Cs + C, device="cuda", dtype=torch.bfloat16)
    ops.upcat_fwd(ops.ActView(to_ndhwc(x.detach()), N, *din, C), ops.ActView(cat, N, *dout, C, ld=Cs + C, coff=Cs))
    torch.cuda.synchronize()
    got = cat[..., Cs:].float().permute(0, 4, 1, 2, 3)
    assert rel_l2(got, ref) < 4e-3
    assert bool((cat[..., :Cs] == 0).all())
    dcat = bf16_round(torch.randn(N, Cs + C, *dout, device="cuda", generator=g))
    ref.backward(dcat[:, Cs:])
    for separable in (False, True):
        dx = ops.upcat_bwd(ops.ActView(to_ndhwc(dcat), N, *dout, C, ld=Cs + C, coff=Cs), *din, separable=separable)
        torch.cuda.synchronize()
        assert rel_l2(from_view(dx), x.grad) < 4e-3, separable
    # with the fused GroupNorm-backward statistics (two-pass kernels on the non-2x ratios): same dx, accumulators ==
    # fp64 sums of the stored tensor within the fixed-point bound (tests/test_gpu_step_oracle.py)
    from tests.test_gpu_step_oracle import Oracle, spy_upcat_bwd
    orc = Oracle()
    r = ops.ActView(to_ndhwc(bf16_round(torch.randn(N, C, *din, device="cuda", generator=g).relu())), N, *din, C)
    dx2, _ = spy_upcat_bwd(ops.upcat_bwd, orc, ops.ActView(to_ndhwc(dcat), N, *dout, C, ld=Cs + C, coff=Cs), *din,
                           stat_r=r)
    assert torch.equal(dx2.buf, dx.buf)
    assert all(v <= 1.0 for v in orc.worst.values()), orc.worst


@pytest.mark.parametrize("N,C,din", [(1, 64, (5, 6, 9)), (1, 128, (24, 28, 24)), (2, 256, (3, 5, 4)), (1, 512, (6, 7, 6))])
def test_upsample2x_adjoint_single_pass(N, C, din):
    """exact-2x levels: the single-pass TMA-staged stencil kernel (upsample2x_bwd_kernel) == PyTorch's adjoint, ==
    the two-pass separable kernels (B2_NO_UP1PASS), with and without the fused GroupNorm-backward statistics;
    partial tiles (5x6x9), several D segments and work items per CTA (24x28x24), batch 2."""
    ops = _ops()
    Cs = 64
    dout = tuple(2 * d for d in din)
    g = torch.Generator(device="cuda").manual_seed(21)
    x = bf16_round(torch.randn(N, C, *din, device="cuda", generator=g)).requires_grad_(True)
    ref = F.interpolate(x, size=dout, mode="trilinear", align_corners=False)
    dcat = bf16_round(torch.randn(N, Cs + C, *dout, device="cuda", generator=g))
    ref.backward(dcat[:, Cs:])
    win = ops.ActView(to_ndhwc(dcat), N, *dout, C, ld=Cs + C, coff=Cs)
    dx = ops.upcat_bwd(win, *din)
    torch.cuda.synchronize()
    e = rel_l2(from_view(dx), x.grad)
    assert e < 4e-3, e
    if N == 1:
        r = bf16_round(torch.randn(1, C, *din, device="cuda", generator=g).relu())
        dx2, acc = ops.upcat_bwd(win, *din, stat_r=ops.ActView(to_ndhwc(r), 1, *din, C))
        torch.cuda.synchronize()
        assert torch.equal(dx.buf, dx2.buf)
        a4 = acc.view(C, 4).double()
        o = dx2.buf.double().reshape(-1, C)
        rr = to_ndhwc(r).double().reshape(-1, C)
        assert torch.allclose(a4[:, 0] + a4[:, 1] / 2.0 ** 32, o.sum(0), rtol=1e-5, atol=1e-3)
        assert torch.allclose(a4[:, 2] + a4[:, 3] / 2.0 ** 32, (o * rr).sum(0), rtol=1e-5, atol=1e-3)
        dx3, _ = ops.upcat_bwd(win, *din, stat_r=ops.ActView(to_ndhwc(r), 1, *din, C))   # bit-identical run to run
        torch.cuda.synchronize()
        assert torch.equal(dx2.buf, dx3.buf)


def _head_inputs(seed, N=1, D=6, H=7, W=8, Cin=64, Cout=56, frac=0.2):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = bf16_round(torch.randn(N, Cin, D, H, W, device="cuda", generator=g))
    Wt = torch.randn(Cout, Cin, 1, 1, 1, device="cuda", generator=g) * 0.2
    b = torch.randn(Cout, device="cuda", generator=g) * 0.1
    labels = torch.randint(0, Cout, (N, D, H, W), device="cuda", generator=g)
    mask = torch.rand(N, D, H, W, device="cuda", generator=g) < frac
    labels = torch.where(mask, labels, torch.full_like(labels, -1))
    return x, Wt, b, labels


@pytest.mark.parametrize("Cout", [56, 64, 3])
def test_head_ce_fused(Cout):
    ops = _ops()
    x, Wt, b, labels = _head_inputs(9, Cout=Cout)
    N, Cin, D, H, W = x.shape
    xq = x.clone().requires_grad_(True)
    Wq, bq = Wt.clone().requires_grad_(True), b.clone().requires_grad_(True)
    logits = F.conv3d(xq, Wq, bq)
    loss = F.cross_entropy(logits, labels, ignore_index=-1)
    loss.backward()
    xv = ops.ActView(to_ndhwc(x), N, D, H, W, Cin)
    out = ops.head_ce(xv, labels, Wt, b, compute_grad=True)
    torch.cuda.synchronize()
    assert abs(float(out["loss"][0]) - float(loss)) < 1e-4 * max(1.0, abs(float(loss)))
    assert int(out["count"]) == int((labels >= 0).sum())
    m = labels >= 0
    assert torch.equal(out["preds"][m].long(), logits.argmax(1)[m])
    assert bool((out["preds"][~m] == -1).all())
    assert rel_l2(out["dW"], Wq.grad) < 1e-4
    assert rel_l2(out["db"], bq.grad) < 1e-4
    assert rel_l2(from_view(out["dx"]), xq.grad) < 4e-3
    # reference val-phase loss: CrossEntropyLoss applied to Softmax outputs (training.py:189,205-208)
    out2 = ops.head_ce(xv, labels, Wt, b, compute_grad=False, eval_softmax=True)
    ref2 = F.cross_entropy(torch.softmax(logits.detach(), 1), labels, ignore_index=-1)
    assert abs(float(out2["loss"][0]) - float(ref2)) < 1e-4 * max(1.0, abs(float(ref2)))


def test_head_deferred_groupnorm_apply_is_bit_identical():
    """head kernels fed relu(conv) + GroupNorm scale/shift (apply deferred to the gathered rows) == head kernels fed
    the tensor the dense apply pass would have written"""
    ops = _ops()
    x, Wt, b, labels = _head_inputs(12, N=1, D=9, H=11, W=13)
    N, Cin, D, H, W = x.shape
    g = torch.Generator(device="cuda").manual_seed(13)
    r = ops.ActView(to_ndhwc(x.relu()), N, D, H, W, Cin)
    gamma = torch.randn(Cin, device="cuda", generator=g) * 0.5 + 1.0
    beta = torch.randn(Cin, device="cuda", generator=g) * 0.2
    mr, ss = ops.relu_gn_stats(r, 32, 1e-5, gamma, beta)
    y = ops.ActView.alloc(N, D, H, W, Cin, "cuda")
    ops.relu_gn_apply(r, ss, y)
    a = ops.head_ce(y, labels, Wt, b, compute_grad=True)
    d = ops.head_ce(r, labels, Wt, b, compute_grad=True, x_scale_shift=ss)
    idx = torch.nonzero(labels.reshape(-1) >= 0).reshape(-1)
    sa, pa = ops.head_gather(y, idx, Wt, b, softmax=True)
    sd, pd = ops.head_gather(r, idx, Wt, b, softmax=True, x_scale_shift=ss)
    torch.cuda.synchronize()
    for k in ("loss", "preds", "dW", "db"):
        assert torch.equal(a[k], d[k]), k
    assert torch.equal(a["dx"].buf, d["dx"].buf)
    assert torch.equal(sa, sd) and torch.equal(pa, pd)


def test_head_ce_no_labelled_voxel_is_nan():
    ops = _ops()
    x, Wt, b, labels = _head_inputs(10)
    labels = torch.full_like(labels, -1)
    N, Cin, D, H, W = x.shape
    out = ops.head_ce(ops.ActView(to_ndhwc(x), N, D, H, W, Cin), labels, Wt, b, compute_grad=True)
    assert bool(torch.isnan(out["loss"][0]))          # same as PyTorch's mean over an empty set
    assert int(out["count"]) == 0
    assert float(out["dW"].abs().sum()) == 0.0


def test_head_gather_and_dense():
    ops = _ops()
    x, Wt, b, labels = _head_inputs(11, N=2)
    N, Cin, D, H, W = x.shape
    xv = ops.ActView(to_ndhwc(x), N, D, H, W, Cin)
    logits = F.conv3d(x, Wt, b)
    probs = torch.softmax(logits, 1)
    dense_l = ops.head_dense_fwd(xv, Wt, b, softmax=False)
    dense_p = ops.head_dense_fwd(xv, Wt, b, softmax=True)
    torch.cuda.synchronize()
    assert dense_l.shape == logits.shape
    assert rel_l2(dense_l, logits) < 1e-5
    assert rel_l2(dense_p, probs) < 1e-5
    idx = torch.nonzero(labels.flatten() >= 0).flatten()
    sc, pr = ops.head_gather(xv, idx, Wt, b, softmax=True)
    torch.cuda.synchronize()
    pflat = probs.permute(0, 2, 3, 4, 1).reshape(-1, probs.shape[1])
    assert rel_l2(sc, pflat[idx]) < 1e-5
    assert torch.equal(pr.long(), logits.permute(0, 2, 3, 4, 1).reshape(-1, logits.shape[1])[idx].argmax(1))
    # dense backward (grad of an arbitrary loss on the dense logits, mostly-zero rows)
    gq = torch.zeros_like(logits)
    m = (labels >= 0).unsqueeze(1).expand_as(gq)
    gq[m] = torch.randn(int(m.sum()), device="cuda")
    xq = x.clone().requires_grad_(True)
    Wq, bq = Wt.clone().requires_grad_(True), b.clone().requires_grad_(True)
    F.conv3d(xq, Wq, bq).backward(gq)
    dx, dW, db = ops.head_dense_bwd(gq, xv, Wt)
    torch.cuda.synchronize()
    assert rel_l2(dW, Wq.grad) < 1e-4
    assert rel_l2(db, bq.grad) < 1e-4
    assert rel_l2(from_view(dx), xq.grad) < 4e-3


def test_sgd_matches_torch():
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(12)
    shapes = [(64, 32, 3, 3, 3), (64,), (56, 64, 1, 1, 1), (5000,)]
    ps = [torch.randn(s, device="cuda", generator=g) for s in shapes]
    ref_ps = [p.clone().requires_grad_(True) for p in ps]
    opt = torch.optim.SGD(ref_ps, lr=1e-2, momentum=0.9, weight_decay=0)
    moms = [torch.zeros_like(p) for p in ps]
    for step in range(3):
        grads = [torch.randn(s, device="cuda", generator=g) for s in shapes]
        for rp, gr in zip(ref_ps, grads):
            rp.grad = gr.clone()
        opt.step()
        ops.sgd_step(ps, grads, moms, 1e-2, 0.9)
    torch.cuda.synchronize()
    for p, rp in zip(ps, ref_ps):
        assert torch.allclose(p, rp.detach(), rtol=1e-6, atol=1e-7)


def test_sgd_multi_launch_odd_views_and_grad_scale():
    """> 64 tensors (two launches of sgd_multi_kernel), numels that are not multiples of 4, parameters that are views
    at odd float offsets of one flat buffer (as the data-parallel buckets are: the scalar path), grad_scale != 1.
    Against the fp64 recurrence v <- mu v + s g, p <- p - lr v with lr, mu, s rounded to fp32 as the kernel receives
    them.  Bound per element after k steps: 5 k u P, P = |p0| + sum_j lr Av_j, Av_j = mu Av_(j-1) + |s g_j|: step j
    adds at most 3 u Av_j to the error of v (mu v, s g, their sum), the error of v carries through mu, so
    e_v(j) <= 3 j u Av_j, and p takes lr e_v(j) plus 2 u (|p| + lr |v|) per step: e_p(k) <= 3 k u P + 2 k u P."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(13)
    numels = [(i * 37) % 301 + 1 for i in range(70)] + [4099, 8192 + 3, 4096]
    flat = torch.randn(sum(numels) + len(numels), device="cuda", generator=g)
    ps, off = [], 1
    for n in numels:                       # every view starts one float after the end of the previous one
        ps.append(flat[off:off + n])
        off += n + 1
    moms = [torch.zeros_like(p) for p in ps]
    lr, mu, s, steps = 1e-2, 0.9, 0.37, 3
    lr32, mu32, s32 = (float(torch.tensor(c, dtype=torch.float32)) for c in (lr, mu, s))
    p64 = [p.double().clone() for p in ps]
    v64 = [torch.zeros_like(q) for q in p64]
    P = [q.abs() for q in p64]
    Vabs = [torch.zeros_like(q) for q in p64]
    for _ in range(steps):
        grads = [torch.randn(n, device="cuda", generator=g) for n in numels]
        ops.sgd_step(ps, grads, moms, lr, mu, grad_scale=s)
        for i, gr in enumerate(grads):
            v64[i] = mu32 * v64[i] + s32 * gr.double()
            p64[i] = p64[i] - lr32 * v64[i]
            Vabs[i] = mu32 * Vabs[i] + abs(s32) * gr.double().abs()
            P[i] = P[i] + lr32 * Vabs[i]
    torch.cuda.synchronize()
    u = 2.0 ** -24
    for i, (p, ref, mag) in enumerate(zip(ps, p64, P)):
        err = (p.double() - ref).abs()
        assert bool((err <= 5 * steps * u * mag + 1e-30).all()), (i, numels[i], float(err.max()))


def test_pack_conv_weights_multi_many_layers():
    """> 16 layers (several launches, kMaxPackLayers): every trunk (cout, cin) and Cin in {384, 768}; bit-equal to
    pack_conv_weights and to the bf16 permutation of the fp32 master (Wf[tap][co][ci], Wd[26 - tap][ci][co])."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(14)
    trunk = [(64, 32), (64, 64), (128, 64), (128, 128), (256, 128), (256, 256), (512, 256), (256, 768), (256, 256),
             (128, 384), (128, 128), (64, 192), (64, 64)]
    shapes = trunk + trunk[::-1] + [(64, 384), (128, 768), (512, 512)]
    ws = [torch.randn(co, ci, 3, 3, 3, device="cuda", generator=g) * 0.05 for co, ci in shapes]
    outs = ops.pack_conv_weights_multi(ws)
    torch.cuda.synchronize()
    assert len(outs) == len(ws)
    for (co, ci), w, (wf, wd) in zip(shapes, ws, outs):
        wb = w.to(torch.bfloat16)
        assert torch.equal(wf, wb.permute(2, 3, 4, 0, 1).reshape(27, co, ci)), (co, ci)
        assert torch.equal(wd, wb.flip(2, 3, 4).permute(2, 3, 4, 1, 0).reshape(27, ci, co)), (co, ci)
        wf1, wd1 = ops.pack_conv_weights(w)
        assert torch.equal(wf, wf1) and torch.equal(wd, wd1), (co, ci)


BSTATS_CASES = [
    ("dgrad", (64, 64, 8, 12, 64)), ("dgrad", (128, 64, 6, 8, 32)), ("dgrad", (256, 128, 6, 7, 6)),
    ("pool", (64, 8, 10, 12)), ("pool", (128, 7, 9, 11)), ("pool", (256, 6, 6, 8)),
    ("up", (64, (5, 6, 9), (10, 12, 18))), ("up", (128, (24, 28, 24), (48, 56, 48))), ("up", (512, (6, 7, 6), (12, 14, 12))),
    ("up", (128, (8, 13, 10), (17, 26, 21))), ("up", (256, (4, 6, 5), (8, 13, 10))), ("up", (512, (2, 3, 2), (4, 6, 5))),
]


@pytest.mark.parametrize("scale", [1.0, 1e-4, 1e-6])
@pytest.mark.parametrize("case", BSTATS_CASES, ids=lambda c: "%s-%s" % (c[0], "x".join(str(v) for v in c[1][:2])))
def test_bstats_producers_at_gradient_scale(case, scale):
    """The kernels that produce a gradient at a GroupNorm output and accumulate its backward statistics (dgrad
    epilogue, pooling adjoint, upsample adjoint: single-pass 2x and two-pass non-2x), with the gradient scaled to the
    magnitudes of a real step (mean cross-entropy over ~2e4 voxels: 1e-5 .. 1e-6 per voxel).  Each output against fp64,
    the accumulators against fp64 sums of the stored tensor with the fixed-point bound, and dr / dgamma / dbeta of the
    accumulator route against the closed-form fp64 GroupNorm backward, relative to the sum of |terms| per channel
    (bounds: tests/test_gpu_step_oracle.py)."""
    ops = _ops()
    from tests.test_gpu_step_oracle import (Oracle, spy_conv3d_dgrad_gn_bstats, spy_maxpool3d_bwd_add,
                                            spy_relu_gn_bwd_from_stats, spy_upcat_bwd)
    kind, shp = case
    G = 32
    orc = Oracle()
    g = torch.Generator(device="cuda").manual_seed(71)

    def act(C, dims, s=1.0, relu=False):
        t = torch.randn(1, *dims, C, device="cuda", generator=g) * s
        return ops.ActView((t.relu() if relu else t).to(torch.bfloat16), 1, *dims, C)

    if kind == "dgrad":
        Cdy, Cdx, D, H, W = shp
        dims, C = (D, H, W), Cdx
        w = torch.randn(Cdy, Cdx, 3, 3, 3, device="cuda", generator=g) * (1.0 / (27 * Cdy) ** 0.5)
        _, wd = ops.pack_conv_weights(w)
        r = act(C, dims, relu=True)
        dx = ops.ActView.alloc(1, D, H, W, C, "cuda")
        acc = spy_conv3d_dgrad_gn_bstats(ops.conv3d_dgrad_gn_bstats, orc, act(Cdy, dims, scale), wd, dx, Cdy, Cdx, r)
    elif kind == "pool":
        C, D, H, W = shp
        dims = (D, H, W)
        r = act(C, dims, relu=True)
        dx, acc = spy_maxpool3d_bwd_add(ops.maxpool3d_bwd_add, orc, act(C, dims), act(C, dims, scale),
                                        act(C, (D // 2, H // 2, W // 2), scale), stat_r=r)
    else:
        C, din, dout = shp
        dims = din
        r = act(C, din, relu=True)
        dx, acc = spy_upcat_bwd(ops.upcat_bwd, orc, act(C, dout, scale), *din, stat_r=r)
    gamma = torch.randn(C, device="cuda", generator=g) * 0.5 + 1.0
    beta = torch.randn(C, device="cuda", generator=g) * 0.1
    mr, _ = ops.relu_gn_stats(r, G, 1e-5, gamma, beta)
    spy_relu_gn_bwd_from_stats(ops.relu_gn_bwd_from_stats, orc, acc, dx, r, G, gamma, mr)
    print("%s scale %g: %s" % (case, scale, " ".join("%s=%.2e" % kv for kv in sorted(orc.worst.items()))))
    assert all(v <= 1.0 for v in orc.worst.values()), orc.worst


def _head_ce_bstats_call(ops, xv, labels, Wt, b, r, dx, xss):
    """b2_head_ce_bstats with skip_dx_memset = 1 into the caller's dX buffer (ops.head_ce allocates its own)"""
    lib = ops._lib.load()
    N, Cin = xv.N, xv.C
    Cout = Wt.shape[0]
    dev = xv.buf.device
    loss = torch.empty(2, dtype=torch.float32, device=dev)
    count = torch.empty(1, dtype=torch.int32, device=dev)
    preds = torch.full((N, xv.D, xv.H, xv.W), -1, dtype=torch.int32, device=dev)
    dW = torch.empty(Cout, Cin, dtype=torch.float32, device=dev)
    db = torch.empty(Cout, dtype=torch.float32, device=dev)
    acc = torch.zeros(4 * Cin, dtype=torch.int64, device=dev)
    ws = ops.Workspace.get(lib.b2_head_workspace_bytes(Cin), dev, "head")
    Wc = Wt.reshape(Cout, Cin).contiguous()
    ops._lib.check(lib.b2_head_ce_bstats(ops._p(xv.buf), ops._p(labels), N * xv.V, ops._p(Wc), ops._p(b), Cin, Cout,
                                         1.0, ops._p(None), ops._p(preds), ops._p(dx.buf), ops._p(dW), ops._p(db),
                                         ops._p(loss), ops._p(count), ops._p(ws), ws.numel(), ops._p(r.buf),
                                         ops._p(acc), ops._p(xss), 1, ops._s()), "b2_head_ce_bstats")
    return dict(loss=loss, count=count, preds=preds, dx=dx, dW=dW, db=db, dx_stats=acc)


@pytest.mark.parametrize("Cout", [3, 56, 64])
@pytest.mark.parametrize("deferred_apply", [False, True])
@pytest.mark.parametrize("frac", [0.2, 0.0])
def test_head_sparse_dx_rows_never_read(Cout, deferred_apply, frac):
    """b2_head_ce_bstats with skip_dx_memset = 1 writes only the labelled rows of dX (the buffer is pre-filled with bf16
    NaN here); relu_gn_bwd_from_stats(dy_row_labels=labels) must read the other rows as zero: dr, dgamma, dbeta finite
    and equal to the fp64 reference with those rows zero.  frac = 0: no labelled voxel -> NaN loss, zero accumulators,
    zero dr."""
    ops = _ops()
    from tests.test_gpu_step_oracle import Oracle, _block_count_max, _gn_bwd_check, head_check
    x, Wt, b, labels = _head_inputs(19, D=9, H=11, W=13, Cout=Cout, frac=frac)
    if frac == 0.0:
        labels = torch.full_like(labels, -1)
    N, Cin, D, H, W = x.shape
    g = torch.Generator(device="cuda").manual_seed(20)
    r = ops.ActView(to_ndhwc(x.relu()), N, D, H, W, Cin)
    gamma = torch.randn(Cin, device="cuda", generator=g) * 0.5 + 1.0
    beta = torch.randn(Cin, device="cuda", generator=g) * 0.2
    mr, ss = ops.relu_gn_stats(r, 32, 1e-5, gamma, beta)
    if deferred_apply:
        xv, xss = r, ss
    else:
        xv = ops.ActView.alloc(N, D, H, W, Cin, "cuda")
        ops.relu_gn_apply(r, ss, xv)
        xss = None
    dx = ops.ActView(torch.full((N, D, H, W, Cin), float("nan"), device="cuda", dtype=torch.bfloat16), N, D, H, W, Cin)
    out = _head_ce_bstats_call(ops, xv, labels, Wt, b, r, dx, xss)
    dr, dg, db = ops.relu_gn_bwd_from_stats(out["dx_stats"], dx, r, 32, gamma, mr, dy_row_labels=labels)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(dr.buf.float()).all()) and bool(torch.isfinite(dg).all() and torch.isfinite(db).all())
    orc = Oracle()
    head_check(orc, xv, labels, Wt, b, out, True, 1.0, r, xss, True)
    _gn_bwd_check(orc, "gn_bwd", dx, r, 32, gamma, mr, dr, dg, db, _block_count_max(labels, N * D * H * W) + 6, 296,
                  labels)
    assert all(v <= 1.0 for v in orc.worst.values()), orc.worst
    if frac == 0.0:
        assert bool(torch.isnan(out["loss"][0])) and int(out["count"]) == 0
        assert int(out["dx_stats"].abs().sum()) == 0
        assert float(dr.buf.float().abs().sum()) == 0.0 and float(dg.abs().sum()) == 0.0


def test_fold_vote_bit_exact_vs_oracle():
    ops = _ops()
    from oracle.cutting_ref import cutting_ref
    from oracle.synth import synth_scores
    rng = np.random.RandomState(0)
    n, C = 20000, 56
    scores = synth_scores(n, C, seed=7)
    fold_raw = rng.randint(0, 64, size=n) * 17 + 3          # arbitrary (non-dense) vertex ids
    uniq, inv = np.unique(fold_raw, return_inverse=True)
    ths = [50, 100, 150]
    got = ops.fold_vote(scores.cuda(), torch.from_numpy(inv.astype(np.int32)).cuda(), len(uniq), ths).cpu().numpy()
    for t, th in enumerate(ths):
        ref = np.asarray(cutting_ref(scores.numpy(), fold_raw, np.zeros((n, 3), int), th))
        assert np.array_equal(got[t], ref), "threshold %d mismatch" % th
    # empty input
    e = ops.fold_vote(torch.zeros(0, C, device="cuda"), torch.zeros(0, dtype=torch.int32, device="cuda"), 1, ths)
    assert e.shape == (3, 0)


def test_esi_counts_exact():
    ops = _ops()
    from oracle.stats_ref import esi_counts_ref
    rng = np.random.RandomState(1)
    yt = rng.randint(0, 56, size=50000).astype(np.int32)
    yp = np.where(rng.rand(50000) < 0.7, yt, rng.randint(0, 56, size=50000)).astype(np.int32)
    c = ops.esi_counts(torch.from_numpy(yt).cuda(), torch.from_numpy(yp).cuda(), 56).cpu().numpy()
    tp, fp, fn = esi_counts_ref(yt, yp, list(range(56)))
    assert np.array_equal(c[0], tp) and np.array_equal(c[1], fp) and np.array_equal(c[2], fn)
