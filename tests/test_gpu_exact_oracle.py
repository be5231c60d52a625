"""fp64 oracle of every kernel call of exact-label inference (UNet3D.scores_at(exact=True)).

The eight ``ops.exact_*`` entry points are replaced by spies that clone what the call reads, run the real call,
synchronise, and compare what the call wrote with the same operation computed in float64 (tests/test_gpu_step_oracle.py
does the same for a training step).  Nothing compounds from one call to the next.  Notation as there: u = 2^-24,
``ref`` the fp64 result, ``A`` the operation on absolute values, ``K`` the longest fp32 chain.  Bounds (a ratio
error / bound <= 1 passes):
  * exact_split3 ......... bit-exact: [hi | lo | hi] with hi = bf16_rn(x), lo = bf16_rn(x - hi) (the subtraction is
                           exact in fp32), read from the (ld, off) window; and |x - hi - lo| <= 2^-16 |x| (+ FLOOR)
  * exact_split_first .... bit-exact: [hi, hi, lo, 0 ...] (32 channels)
  * exact_conv(_bias) .... (a) against the fp64 conv of the stored bf16 split operands and the packed weights:
                           K u A, K = 27 cin3 + 1 (+ 1 with a bias; products of bf16 values are exact in fp32).
                           (b) against the fp64 conv of the fp32 activation the split was made from and the layer's
                           fp32 weight: (a) + 3.02 2^-16 A, A = conv(|x|, |w|).  The three kept products lose at most
                           x_lo w_lo + e_x w + x_hi e_w, each <= 2^-18 |x| |w| (e_x = x - hi - lo).  ReLU on both.
  * exact_gn ............. the written window against fp64 GroupNorm of r: u (|ref| + |r sc| + |shift|) (the fp32
                           roundings of scale and shift and the one fma), plus the error of the fp64 statistics pushed
                           through mean, var = Q/m - mean^2 and rstd as Oracle.fwd_stats does, with 2^-53 and
                           K = V + 1024 (per-thread chains, the in-block rows, <= 296 block partials, the group).
                           Columns outside [off, off + C) are untouched (bit patterns).
  * exact_maxpool ........ exact: the max of each 2x2x2 cell (odd sizes floored), NaN propagated as torch does
  * exact_upsample ....... fp32, K = 8 + 4 max(D, H, W), A over the touched samples (upcat_fwd without the bf16 term);
                           columns outside the window untouched
  * exact_head_gather .... logits (softmax=False): (Cin + 1) u A_l.  Softmax scores: p (4 e + (Cout + 6) u
                           + u |z - z_max|), e = the row's largest logit bound (head_ce's softmax bound plus the
                           rounding of the exp argument).  Preds == the fp64 argmax wherever the top-2 margin exceeds
                           2 e, and always == the argmax of the kernel's own scores, ties to the lowest index.
End to end, per configuration: scores within 1e-4 of UNet3DRef(...).double() with the same weights, labels identical
wherever the fp64 top-2 margin exceeds 2e-4.  The fp32 oracle's own distance from fp64 is printed beside ours.
Every configuration also runs a non-binary input (binary skeleton x U(0.5, 1)), which the split first layer must carry
without rounding it to bf16.
"""
import copy
import functools
import time

import pytest
import torch
import torch.nn.functional as F

import tests.test_gpu_step_oracle as so

U, FLOOR = so.U, so.FLOOR
U53 = 2.0 ** -53
SPLIT_LOST = 3.02 * 2.0 ** -16
SCORE_TOL = 1e-4
MARGIN_EPS = 2e-4


# ------------------------------------------------------------------------------------------------ fp64 references
def split3_ref(x):
    """fp32 [V, C] -> bf16 [V, 3C] = [hi | lo | hi] (round to nearest even, as the kernel)"""
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.cat([hi, lo, hi], 1)


def gn_ref(r, G, eps, gamma, beta):
    """fp64 GroupNorm of r [V, C] over (V, C/G) per group (biased variance, two-pass).  Returns (y, mean_c, rstd_c)."""
    V, C = r.shape
    cpg = C // G
    g = r.view(V, G, cpg)
    mean = g.mean((0, 2))
    var = ((g - mean.view(1, G, 1)) ** 2).mean((0, 2))
    rstd = 1.0 / torch.sqrt(var + eps)
    mean_c, rstd_c = mean.repeat_interleave(cpg), rstd.repeat_interleave(cpg)
    return (r - mean_c) * rstd_c * gamma + beta, mean_c, rstd_c


def gn_bound(r, G, eps, gamma, beta):
    """(ref, bound) of exact_gn on r [V, C] float64 (module docstring)"""
    V, C = r.shape
    cpg = C // G
    m = V * cpg
    ref, mean_c, rstd_c = gn_ref(r, G, eps, gamma, beta)
    K = V + 1024
    eS = (K * U53 * r.abs().sum(0)).view(G, cpg).sum(1)
    eQ = (K * U53 * (r * r).sum(0)).view(G, cpg).sum(1)
    Qm = (r * r).sum(0).view(G, cpg).sum(1) / m
    mean = r.sum(0).view(G, cpg).sum(1) / m
    var = (Qm - mean * mean).clamp_min(0)
    dmean = eS / m + U53 * mean.abs()
    dvar = eQ / m + 2 * mean.abs() * dmean + dmean * dmean + 4 * U53 * (Qm + mean * mean)
    drstd = 1.0 / torch.sqrt(var + eps) * (0.5 * dvar / (var + eps) + 4 * U53)
    dmean_c, drstd_c = dmean.repeat_interleave(cpg), drstd.repeat_interleave(cpg)
    sc = rstd_c * gamma
    sh = beta - mean_c * sc
    stat = gamma.abs() * (rstd_c * dmean_c + (r - mean_c).abs() * drstd_c)
    bound = U * (ref.abs() + (r * sc).abs() + sh.abs()) * (1 + 1e-6) + (1 + 1e-6) * stat + FLOOR
    return ref, bound


def maxpool_ref(x):
    """MaxPool3d(2) of x [N, C, D, H, W] (floor mode), NaN in a cell -> NaN"""
    N, C, D, H, W = x.shape
    Dp, Hp, Wp = D // 2, H // 2, W // 2
    cells = x[:, :, :2 * Dp, :2 * Hp, :2 * Wp].reshape(N, C, Dp, 2, Hp, 2, Wp, 2)
    cells = cells.permute(0, 1, 2, 4, 6, 3, 5, 7).reshape(N, C, Dp, Hp, Wp, 8)
    m = cells.max(-1).values
    return torch.where(torch.isnan(cells).any(-1), torch.full_like(m, float("nan")), m)


def same_values(a, b):
    """equal values with NaN where the other has NaN"""
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


def head_ref(xg, W64, b64, softmax):
    """fp64 head on gathered rows: (logits, scores, e [n, Cout] logit bound, e_row [n] its row max)"""
    Cin = xg.shape[1]
    logits = xg @ W64.t() + b64
    e = (Cin + 1) * U * (xg.abs() @ W64.abs().t() + b64.abs())
    e_row = e.max(1).values if e.shape[0] and e.shape[1] else torch.zeros(e.shape[0], dtype=e.dtype, device=e.device)
    scores = torch.softmax(logits, 1) if softmax else logits
    return logits, scores, e, e_row


def first_argmax(s):
    """index of the first maximum of each row (CPU: ties -> lowest index)"""
    s = s.cpu()
    return (s == s.max(1, keepdim=True).values).to(torch.int8).argmax(1)


# ------------------------------------------------------------------------------------------------ spies
class ExactOracle(so.Oracle):
    def __init__(self):
        super(ExactOracle, self).__init__()
        self.src = {}       # split buffer data_ptr -> fp32 source (float64 [1, C, D, H, W])
        self.wmap = {}      # weight pack data_ptr -> (layer name, fp32 weight as float64, bias as float64 or None)

    def exact(self, op, ok):
        self.worst[op] = max(self.worst.get(op, 0.0), 0.0 if ok else float("inf"))


def _untouched(orc, op, before, after, off, C):
    """bit patterns of the columns outside [off, off + C) of a [.., ld] fp32 buffer are unchanged"""
    ld = before.shape[-1]
    outside = torch.ones(ld, dtype=torch.bool, device=before.device)
    outside[off:off + C] = False
    bits_before, bits_after = before.view(torch.int32)[..., outside], after.view(torch.int32)[..., outside]
    orc.exact(op + ":outside", torch.equal(bits_before, bits_after))


def _ncdhw(rows, D, H, W):
    """[V, C] -> [1, C, D, H, W]"""
    return rows.reshape(1, D, H, W, -1).permute(0, 4, 1, 2, 3)


def spy_exact_split3(real, orc, x, ld, off, C, D, H, W):
    V = D * H * W
    xw = x.reshape(-1, ld)[:V, off:off + C].clone()
    out = real(x, ld, off, C, D, H, W)
    torch.cuda.synchronize()
    orc.seen.add("split3")
    got = out.buf.reshape(V, 3 * C)
    orc.exact("split3", torch.equal(got.view(torch.int16), split3_ref(xw).view(torch.int16)))
    x64 = xw.double()
    hi, lo = got[:, :C].double(), got[:, C:2 * C].double()
    orc.ratio("split3:residual", hi + lo, x64, 2.0 ** -16 * x64.abs() + FLOOR)
    orc.src[out.buf.data_ptr()] = _ncdhw(x64, D, H, W)
    return out


def spy_exact_split_first(real, orc, x, D, H, W):
    V = D * H * W
    xv = x.reshape(V).clone()
    out = real(x, D, H, W)
    torch.cuda.synchronize()
    orc.seen.add("split_first")
    want = torch.zeros((V, 32), dtype=torch.bfloat16, device=x.device)
    s = split3_ref(xv.view(V, 1))
    want[:, 0], want[:, 1], want[:, 2] = s[:, 0], s[:, 0], s[:, 1]
    orc.exact("split_first", torch.equal(out.buf.reshape(V, 32).view(torch.int16), want.view(torch.int16)))
    orc.src[out.buf.data_ptr()] = xv.double().view(1, 1, D, H, W)
    return out


def _exact_conv_check(orc, xsplit, x64, wpack, bias, cin3, cout, relu, r):
    D, H, W = xsplit.D, xsplit.H, xsplit.W
    got = _ncdhw(r, D, H, W).double()
    name, w32, b64 = orc.wmap[wpack.data_ptr()]
    tag = "conv_first" if cin3 == 32 else "conv"
    orc.seen.add(tag)
    orc.seen.add("conv_cin3_%d" % cin3)
    if cin3 % 32:
        orc.seen.add("conv_kc16")
    if cin3 == 32 and cout == 16:
        orc.seen.add("conv_first_n16")
    bb = 0.0 if bias is None else bias.double().view(1, -1, 1, 1, 1)
    if bias is not None:
        orc.seen.add("conv_bias")
        assert torch.equal(bias.double(), b64)
    K = 27 * cin3 + 1 + (0 if bias is None else 1)
    # (a) the stored split operands and the packed weights
    wa = so.unpack_wf(wpack, cout, cin3)
    ref_a = so.conv3d_taps(x64, wa) + bb
    A_a = so.conv3d_taps(x64.abs(), wa.abs()) + (0.0 if bias is None else bb.abs())
    if relu:
        ref_a = ref_a.clamp_min(0)
    e_a = K * U * A_a + K * FLOOR
    orc.ratio("conv(a)", got, ref_a, e_a)
    del ref_a
    # (b) the fp32 activation the split was made from and the layer's fp32 weight
    xs = orc.src[xsplit.buf.data_ptr()]
    ref_b = so.conv3d_taps(xs, w32) + bb
    A_b = so.conv3d_taps(xs.abs(), w32.abs()) + (0.0 if bias is None else bb.abs())
    if relu:
        ref_b = ref_b.clamp_min(0)
    orc.ratio("conv(b):" + name, got, ref_b, e_a + SPLIT_LOST * A_b)


def spy_exact_conv(real, orc, xsplit, wpack, cin3, cout, relu=True):
    x64 = so.nc(xsplit).clone()
    r = real(xsplit, wpack, cin3, cout, relu)
    torch.cuda.synchronize()
    _exact_conv_check(orc, xsplit, x64, wpack, None, cin3, cout, relu, r)
    return r


def spy_exact_conv_bias(real, orc, xsplit, wpack, bias, cin3, cout, relu=True):
    x64 = so.nc(xsplit).clone()
    r = real(xsplit, wpack, bias, cin3, cout, relu)
    torch.cuda.synchronize()
    _exact_conv_check(orc, xsplit, x64, wpack, bias, cin3, cout, relu, r)
    return r


def spy_exact_gn(real, orc, r, groups, eps, gamma, beta, out, ld, off):
    C = r.shape[1]
    r64 = r.double().clone()
    before = out.clone()
    real(r, groups, eps, gamma, beta, out, ld, off)
    torch.cuda.synchronize()
    orc.seen.add("gn")
    ref, bound = gn_bound(r64, groups, eps, gamma.double(), beta.double())
    orc.ratio("gn", out.reshape(-1, ld)[:, off:off + C], ref, bound)
    _untouched(orc, "gn", before, out, off, C)


def spy_exact_maxpool(real, orc, x, ld, off, C, D, H, W):
    xw = x.reshape(-1, ld)[:D * H * W, off:off + C].clone()
    y = real(x, ld, off, C, D, H, W)
    torch.cuda.synchronize()
    orc.seen.add("maxpool")
    if D % 2 or H % 2 or W % 2:
        orc.seen.add("maxpool_odd")
    want = maxpool_ref(_ncdhw(xw, D, H, W))
    orc.exact("maxpool", same_values(_ncdhw(y, D // 2, H // 2, W // 2), want))
    return y


def spy_exact_upsample(real, orc, x, C, din, out, ld, off, dout):
    x64 = _ncdhw(x.reshape(-1, C)[:din[0] * din[1] * din[2]].double(), *din).clone()
    before = out.clone()
    real(x, C, din, out, ld, off, dout)
    torch.cuda.synchronize()
    two = all(o == 2 * i for i, o in zip(din, dout))
    orc.seen.add("upsample_2x" if two else "upsample_non2x")
    size = tuple(dout)
    got = _ncdhw(out.reshape(-1, ld)[:, off:off + C], *size)
    K = 8 + 4 * max(size)
    orc.dense("upsample", got, so.upsample_ref(x64, size), so.upsample_ref(x64.abs(), size, touch=True), K, bf16=False)
    _untouched(orc, "upsample", before, out, off, C)


def head_check(orc, op, xg, W, b, scores, preds, softmax):
    """fp64 reference of one gathered head call on the rows xg [n, Cin] float64 it read"""
    Cout, Cin = W.shape[0], xg.shape[1]
    W64, b64 = W.reshape(Cout, Cin).double(), b.double()
    logits, ref, e, e_row = head_ref(xg, W64, b64, softmax)
    n = xg.shape[0]
    assert scores.shape == (n, Cout) and preds.shape == (n,)
    if softmax:
        zmax = logits.max(1, keepdim=True).values if n else logits
        bound = ref * (4 * e_row.view(-1, 1) + (Cout + 6) * U + U * (logits - zmax).abs()) + FLOOR
        orc.ratio(op + ":scores", scores, ref, bound)
    else:
        orc.ratio(op + ":logits", scores, ref, e + FLOOR)
    if not n:
        return
    pl = preds.long().cpu()
    if Cout > 1:
        top2 = logits.topk(2, 1).values
        sure = ((top2[:, 0] - top2[:, 1]) > 2 * e_row).cpu()
    else:
        sure = torch.ones(n, dtype=torch.bool)
    orc.exact(op + ":preds", torch.equal(pl[sure], logits.argmax(1).cpu()[sure]))
    s = scores.cpu()
    own = first_argmax(s)
    tied = (s == s.max(1, keepdim=True).values).sum(1) > 1
    if softmax:   # distinct logits may round to equal probabilities: the pred is one of the tied maxima
        at_max = s.gather(1, pl.view(-1, 1)).view(-1) == s.max(1).values
        ok = torch.equal(pl[~tied], own[~tied]) and bool(at_max.all())
    else:
        ok = torch.equal(pl, own)
    orc.exact(op + ":own_argmax", ok)


def spy_exact_head_gather(real, orc, feat, index, W, b, softmax=True):
    xg = feat[index].double().clone() if index.numel() else feat[:0].double()
    scores, preds = real(feat, index, W, b, softmax)
    torch.cuda.synchronize()
    orc.seen.add("head_exact")
    head_check(orc, "head_exact", xg, W, b, scores, preds, softmax)
    return scores, preds


def spy_head_gather(real, orc, x, index, W, b, softmax=True, x_scale_shift=None):
    """bf16 inference head (scores_at(exact=False)): bf16 features, optional deferred GroupNorm apply of the last layer
    rounded to bf16 before the head (as head_ce)"""
    xr = x.dense().reshape(-1, x.C)[index].double().clone()
    ss = None if x_scale_shift is None else x_scale_shift.double().reshape(x.C, 2).clone()
    scores, preds = real(x, index, W, b, softmax, x_scale_shift)
    torch.cuda.synchronize()
    orc.seen.add("head_gather")
    xg = xr if ss is None else (xr * ss[:, 0] + ss[:, 1]).float().to(torch.bfloat16).double()
    head_check(orc, "head_gather", xg, W, b, scores, preds, softmax)
    return scores, preds


EXACT_SPIES = {
    "exact_split3": spy_exact_split3,
    "exact_split_first": spy_exact_split_first,
    "exact_conv": spy_exact_conv,
    "exact_conv_bias": spy_exact_conv_bias,
    "exact_gn": spy_exact_gn,
    "exact_maxpool": spy_exact_maxpool,
    "exact_upsample": spy_exact_upsample,
    "exact_head_gather": spy_exact_head_gather,
}


def install_exact_spies(monkeypatch, orc, model):
    from unetsulc_b200 import ops
    packs = model._exact_packs()
    layers = model._layers()
    for i, (p, l) in enumerate(zip(packs, layers)):
        name = "%s.%d.conv%d" % ("encoders" if i < 8 else "decoders", (i % 8) // 2, i % 2 + 1)
        b = None if l.conv.bias is None else l.conv.bias.detach().double()
        orc.wmap[p.data_ptr()] = (name, l.conv.weight.detach().double(), b)
    for name, spy in EXACT_SPIES.items():
        monkeypatch.setattr(ops, name, functools.partial(spy, getattr(ops, name), orc))


def _report(orc, name, wall=None):
    print("\n[exact %s] %d checks%s; worst error / bound:" % (name, len(orc.worst),
                                                            "" if wall is None else " in %.1f s" % wall))
    for op in sorted(orc.worst):
        print("    %-34s %.3e" % (op, orc.worst[op]))
    bad = {op: w for op, w in orc.worst.items() if not w <= 1.0}
    assert not bad, "ops outside their fp64 bound: %s" % bad


# ------------------------------------------------------------------------------------------------ direct edge cases
def _orc():
    return ExactOracle()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [16, 48, 64, 192])
def test_exact_split3_bit_patterns(C):
    """round-half-to-even, subnormals, signed zeros and large magnitudes in a window of a wider row"""
    from unetsulc_b200 import ops
    g = torch.Generator().manual_seed(C)
    D, H, W = 3, 5, 7
    V, ld, off = D * H * W, C + 40, 24
    x = torch.randn((V, ld), generator=g) * torch.exp2(torch.randint(-30, 30, (V, ld), generator=g).float())
    special = torch.tensor([
        1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8), 1.0 + 2.0 ** -8 + 2.0 ** -23,   # ties of hi
        1.0 + 2.0 ** -10 + 2.0 ** -18, 1.0 + 2.0 ** -10 + 3 * 2.0 ** -18,                          # ties of lo
        2.0 ** -149, -2.0 ** -149, 3 * 2.0 ** -149, 1e-40, -1.17e-38, 2.0 ** -126 * (1 + 2.0 ** -8),  # subnormals
        0.0, -0.0, 1e38, -3.0e38, 3.3e38, 1e30, -65504.0, 0.1, 1.0 / 3.0], dtype=torch.float32)
    flat = x[:, off:off + C].reshape(-1)
    flat[:special.numel()] = special
    x[:, off:off + C] = flat.view(V, C)
    xg = x.cuda()
    orc = _orc()
    out = spy_exact_split3(ops.exact_split3, orc, xg, ld, off, C, D, H, W)
    # the reference itself on the hand-made cases: hi ties to even, lo exact
    s = split3_ref(special.view(-1, 1))
    assert float(s[0, 0]) == 1.0 and float(s[1, 0]) == 1.0 + 2.0 ** -6 and float(s[3, 0]) == 1.0 + 2.0 ** -7
    assert torch.equal(s[12:14, 0].view(torch.int16), torch.tensor([0, -32768], dtype=torch.int16))
    got = out.buf.reshape(V, 3 * C).cpu()
    assert torch.equal(got.view(torch.int16), split3_ref(x[:, off:off + C]).view(torch.int16))
    _report(orc, "split3 C=%d" % C)


@pytest.mark.gpu
def test_exact_split_first_layout():
    from unetsulc_b200 import ops
    D, H, W = 5, 6, 7
    g = torch.Generator().manual_seed(7)
    x = torch.randn((1, 1, D, H, W), generator=g)
    x.view(-1)[:4] = torch.tensor([0.0, -0.0, 1.0 + 2.0 ** -8, 2.0 ** -149])
    orc = _orc()
    out = spy_exact_split_first(ops.exact_split_first, orc, x.cuda(), D, H, W)
    b = out.buf.reshape(-1, 32).cpu()
    assert bool((b[:, 3:] == 0).all()) and bool((b[:, 2] != 0).any())
    _report(orc, "split_first")


def _gn_case(C, V, seed, G=8):
    g = torch.Generator().manual_seed(seed)
    r = torch.randn((V, C), generator=g).relu() * 3
    cpg = C // G
    r[:, :cpg] = 0                                         # a group of zeros: var = 0
    if G > 2:
        r[:, cpg:2 * cpg] = 1000.0 + torch.randn((V, cpg), generator=g)   # |mean| / std ~ 1e3
    gamma = 1 + 0.3 * torch.randn(C, generator=g)
    beta = 0.2 * torch.randn(C, generator=g)
    return r.cuda(), gamma.cuda(), beta.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [16, 32, 64, 128, 256, 512])
def test_exact_gn_edges(C):
    """V = 1, V below one block's rows, V above 296 blocks of rows (grid-stride over the capped grid); a zero group, a
    group with |mean| / std ~ 1e3; a window inside a wider row with NaN sentinels; bit-identical run to run"""
    from unetsulc_b200 import ops
    rows = 256 // min(C, 256)
    orc = _orc()
    for V in sorted({1, max(rows // 2, 1) + (1 if rows > 2 else 0), 296 * rows + 37, 1500}):
        r, gamma, beta = _gn_case(C, V, seed=C + V)
        ld, off = C + 24, 8
        outs = []
        for _ in range(2):
            out = torch.full((V, ld), float("nan"), device="cuda")
            spy_exact_gn(ops.exact_gn, orc, r, 8, 1e-5, gamma, beta, out, ld, off)
            outs.append(out)
        orc.exact("gn:run_to_run", torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32)))
        assert bool(torch.isfinite(outs[0][:, off:off + C]).all())
    _report(orc, "gn C=%d" % C)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [48, 768])
def test_exact_gn_refuses_unsupported_widths(C):
    from unetsulc_b200 import ops
    r = torch.rand((64, C), device="cuda")
    out = torch.full((64, C), float("nan"), device="cuda")
    ones = torch.ones(C, device="cuda")
    with pytest.raises(RuntimeError, match="b2_exact_gn_stats"):
        ops.exact_gn(r, 8, 1e-5, ones, ones, out, C, 0)
    torch.cuda.synchronize()
    assert bool(torch.isnan(out).all())


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(5, 7, 9), (4, 6, 8), (2, 3, 2), (9, 4, 5)])
def test_exact_maxpool_edges(dims):
    """odd sizes, a channel window at xoff > 0 of a wider row, +-inf, one NaN in a cell, a cell that is all NaN:
    exactly F.max_pool3d"""
    from unetsulc_b200 import ops
    D, H, W = dims
    C, ld, off = 32, 80, 16
    V = D * H * W
    g = torch.Generator().manual_seed(V)
    x = torch.randn((V, ld), generator=g)
    x[:, off:off + C] = x[:, off:off + C].round()          # ties inside cells
    vol = x[:, off:off + C].contiguous().view(D, H, W, C)
    vol[0, 0, 0, 0] = float("inf")
    vol[1, 1, 1, 1] = float("-inf")
    vol[0, 1, 1, 2] = float("nan")                         # one NaN in cell (0, 0, 0), channel 2
    vol[0:2, 0:2, 0:2, 3] = float("nan")                   # a cell of NaN, channel 3
    vol[:2, :2, :2, 4] = float("-inf")                     # a cell of -inf, channel 4
    vol[D - 1, H - 1, W - 1, 5] = float("nan")             # in the floored tail when a size is odd
    x[:, off:off + C] = vol.reshape(V, C)
    orc = _orc()
    y = spy_exact_maxpool(ops.exact_maxpool, orc, x.cuda(), ld, off, C, D, H, W)
    want = F.max_pool3d(_ncdhw(x[:, off:off + C], D, H, W), 2)
    got = _ncdhw(y.cpu(), D // 2, H // 2, W // 2)
    assert same_values(got, want), "differs from torch.max_pool3d at %d places" % int(
        ((got != want) & ~(torch.isnan(got) & torch.isnan(want))).sum())
    assert bool(torch.isnan(got[0, 2, 0, 0, 0])) and bool(torch.isnan(got[0, 3, 0, 0, 0]))
    _report(orc, "maxpool %s" % (dims,))


@pytest.mark.gpu
@pytest.mark.parametrize("din,dout", [
    ((4, 6, 5), (8, 12, 10)),
    ((4, 6, 5), (9, 12, 10)), ((4, 6, 5), (8, 13, 10)), ((4, 6, 5), (8, 12, 11)),   # one axis non-2x
    ((1, 6, 5), (2, 12, 10)), ((4, 1, 5), (8, 3, 10)), ((3, 4, 1), (6, 8, 1)),        # an input extent of 1
    ((2, 3, 2), (4, 6, 5))])
def test_exact_upsample_edges(din, dout):
    from unetsulc_b200 import ops
    orc = _orc()
    for C in (32, 64):
        Vi, Vo = din[0] * din[1] * din[2], dout[0] * dout[1] * dout[2]
        g = torch.Generator().manual_seed(Vi + C)
        x = torch.randn((Vi, C), generator=g).cuda()
        ld, off = C + 40, 24
        out = torch.full((Vo, ld), float("nan"), device="cuda")
        out[:, :off] = torch.randn((Vo, off), generator=g).cuda()
        spy_exact_upsample(ops.exact_upsample, orc, x, C, din, out, ld, off, dout)
        assert bool(torch.isfinite(out[:, off:off + C]).all())
    _report(orc, "upsample %s -> %s" % (din, dout))


@pytest.mark.gpu
@pytest.mark.parametrize("cout", [1, 2, 31, 32, 33, 56, 64])
def test_exact_head_gather_edges(cout):
    """Cin 16 / 32 / 64, n = 0, 1, 7, 8 and a few thousand with duplicated unsorted indices, softmax on and off, exact
    ties (a duplicated W row and bias, in the same and in different lane halves) -> the lower index"""
    from unetsulc_b200 import ops
    orc = _orc()
    for cin in (16, 32, 64):
        g = torch.Generator().manual_seed(cout * 100 + cin)
        V = 5000
        feat = torch.randn((V, cin), generator=g).cuda()
        W = (torch.randn((cout, cin), generator=g) / cin ** 0.5).cuda()
        b = (0.1 * torch.randn(cout, generator=g)).cuda()
        tie_pairs = [(a, c) for a, c in ((3, 17), (5, 40), (0, cout - 1)) if c < cout and a < c]
        Wt, bt = W.clone(), b.clone()
        for a, c in tie_pairs:
            Wt[c], bt[c] = Wt[a], bt[a]
        for n in (0, 1, 7, 8, 3001):
            idx = torch.randint(0, V, (n,), generator=g)
            if n > 2:
                idx[n // 2:] = idx[:n - n // 2].flip(0)    # duplicates, unsorted
            idx = idx.cuda()
            for softmax in (True, False):
                spy_exact_head_gather(ops.exact_head_gather, orc, feat, idx, W, b, softmax)
                if tie_pairs and n:
                    s, p = spy_exact_head_gather(ops.exact_head_gather, orc, feat, idx, Wt, bt, softmax)
                    pl = p.long().cpu()
                    for a, c in tie_pairs:
                        assert not bool((pl == c).any()), "a tie went to the higher index %d (not %d)" % (c, a)
        # a row whose tied pair is its maximum: boost both
        if tie_pairs:
            a, c = tie_pairs[0]
            bt2 = bt.clone()
            bt2[a] = bt2[c] = 50.0
            idx = torch.randint(0, V, (257,), generator=g).cuda()
            for softmax in (True, False):
                _, p = spy_exact_head_gather(ops.exact_head_gather, orc, feat, idx, Wt, bt2, softmax)
                assert bool((p.long() == a).all()), "ties must go to the lowest index"
    _report(orc, "head_gather Cout=%d" % cout)


@pytest.mark.gpu
@pytest.mark.parametrize("cout,cin", [(64, 384), (65, 32)])
def test_exact_head_gather_refuses_oversized_heads(cout, cin):
    from unetsulc_b200 import ops
    feat = torch.randn((100, cin), device="cuda")
    with pytest.raises(RuntimeError, match="b2_exact_head_gather"):
        ops.exact_head_gather(feat, torch.arange(10, device="cuda"), torch.randn((cout, cin), device="cuda"),
                              torch.zeros(cout, device="cuda"))


# ------------------------------------------------------------------------------------------------ the exact forward
BASE = {"split_first", "split3", "conv_first", "conv", "gn", "maxpool", "head_exact"}
F32 = {"conv_kc16", "conv_first_n16", "conv_cin3_48"}
CONFIGS = {
    # name: (width, conv bias, shape, seed of the non-binary input, coverage set)
    "f64_24x32x40": (64, False, (24, 32, 40), 2001, BASE | {"upsample_2x"}),
    "f64_17x26x21": (64, False, (17, 26, 21), 2002, BASE | {"upsample_non2x", "maxpool_odd"}),
    "f64_23x30x19": (64, False, (23, 30, 19), 2003, BASE | {"upsample_non2x", "maxpool_odd"}),
    "f64_40x48x56": (64, False, (40, 48, 56), 2004, BASE | {"upsample_2x"}),
    "f32_24x32x40": (32, False, (24, 32, 40), 2005, BASE | F32 | {"upsample_2x"}),
    "f32_17x26x21": (32, False, (17, 26, 21), 2006, BASE | F32 | {"upsample_non2x", "maxpool_odd"}),
    "bias_f64_24x32x40": (64, True, (24, 32, 40), 2007, BASE | {"upsample_2x", "conv_bias"}),
}
CASES = [(n, "graded") for n in CONFIGS] + [(n, "binary") for n, c in CONFIGS.items() if c[2] == (24, 32, 40)]


def _pair(monkeypatch, f, bias, seed=42, n_classes=56):
    """fp32 oracle and our model with the same weights (non-trivial GroupNorm affine parameters; biases N(0, 0.2^2))"""
    import unetsulc_b200
    from oracle import unet3d_ref
    from tests.test_gpu_conv_bias import _perturb
    monkeypatch.setattr(unet3d_ref, "CONV_BIAS_WHEN_NORM", bias)
    torch.manual_seed(seed)
    ref = unet3d_ref.UNet3DRef(1, n_classes, init_channel_number=f)
    _perturb(ref, seed + 1)
    ours = unetsulc_b200.UNet3D(1, n_classes, init_channel_number=f)
    ours.load_state_dict(ref.state_dict())
    assert ours.conv_bias == bias
    return ref.cuda().eval(), ours.cuda().eval()


def _input(shape, kind, seed, n_classes=56):
    """binary skeleton (the labelling pipeline's input), or the skeleton times U(0.5, 1) with its own seed"""
    from oracle.synth import synth_volume
    occ = 0.03 if shape[0] >= 96 else 0.05
    x, labels = synth_volume(shape, n_classes, 1234 if kind == "binary" else seed, occupancy=occ)
    if kind == "graded":
        g = torch.Generator().manual_seed(seed + 1)
        x = x * (0.5 + 0.5 * torch.rand(x.shape, generator=g))
        assert bool((x.to(torch.bfloat16).float() != x).any())
    return x.unsqueeze(0).cuda(), labels


def run_exact(monkeypatch, name, cfg, kind, bf16_head=False):
    f, bias, shape, seed, expect = cfg
    ref, ours = _pair(monkeypatch, f, bias)
    x, labels = _input(shape, kind, seed)
    idx = torch.nonzero(labels.reshape(-1) >= 0).reshape(-1).cuda()
    with torch.no_grad():
        p32 = ref(x)[0].reshape(ref.final_conv.out_channels, -1)[:, idx].t().double()
        ref64 = copy.deepcopy(ref).double()
        p64 = ref64(x.double())[0].reshape(ref.final_conv.out_channels, -1)[:, idx].t()
        del ref64
    orc = ExactOracle()
    install_exact_spies(monkeypatch, orc, ours)
    t0 = time.time()
    po, preds = ours.scores_at(x, idx, exact=True)
    torch.cuda.synchronize()
    wall = time.time() - t0
    if bf16_head:   # the bf16 inference path under the step oracle's spies: its one call the step does not make
        from unetsulc_b200 import ops
        so.install_spies(monkeypatch, orc)
        monkeypatch.setattr(ops, "head_gather", functools.partial(spy_head_gather, ops.head_gather, orc))
        ours.scores_at(x, idx, exact=False)
        torch.cuda.synchronize()
    err = float((po.double() - p64).abs().max())
    err32 = float((p32 - p64).abs().max())
    top2 = p64.topk(2, 1).values
    margin = top2[:, 0] - top2[:, 1]
    sure = margin > MARGIN_EPS
    same = preds.long() == p64.argmax(1)
    print("\n[exact %s %s] %d voxels: max |score - fp64| ours %.3e, fp32 oracle %.3e; labels == fp64 argmax on %d / %d "
          "(margin > %.0e: %d / %d)" % (name, kind, idx.numel(), err, err32, int(same.sum()), idx.numel(), MARGIN_EPS,
                                       int(same[sure].sum()), int(sure.sum())))
    _report(orc, "%s %s" % (name, kind), wall)
    missing = expect - orc.seen
    assert not missing, "entry points the forward did not reach (or that lost their spy): %s" % sorted(missing)
    assert err <= SCORE_TOL, err
    assert bool(same[sure].all())
    return orc


@pytest.mark.gpu
@pytest.mark.parametrize("name,kind", CASES, ids=["%s-%s" % c for c in CASES])
def test_exact_forward_matches_fp64_per_call(monkeypatch, name, kind):
    orc = run_exact(monkeypatch, name, CONFIGS[name], kind, bf16_head=(name == "f64_24x32x40" and kind == "binary"))
    if name == "f64_24x32x40" and kind == "binary":
        assert "head_gather" in orc.seen


@pytest.mark.gpu
def test_exact_forward_matches_fp64_per_call_baseline_shape(monkeypatch):
    """the BASELINE box 96 x 112 x 96 (its own function: deselect with -k 'not baseline_shape')"""
    run_exact(monkeypatch, "f64_96x112x96", (64, False, (96, 112, 96), 2008, BASE | {"upsample_2x"}), "graded")


# ------------------------------------------------------------------------------------------------ CPU
def test_exact_fp64_references_match_torch_functional():
    """this file's own references (CPU, float64) == torch.nn.functional: GroupNorm written into a window, max-pool with
    +-inf and NaN, softmax and the argmax with ties to the lowest index; the split layout on hand-made cases"""
    g = torch.Generator().manual_seed(0)
    V, C, G = 60, 16, 4
    r = torch.randn((V, C), generator=g, dtype=torch.float64).relu()
    r[:, 4:8] = 0
    gam, bet = torch.randn(C, generator=g, dtype=torch.float64), torch.randn(C, generator=g, dtype=torch.float64)
    y, _, _ = gn_ref(r, G, 1e-5, gam, bet)
    want = F.group_norm(r.t().unsqueeze(0), G, gam, bet, 1e-5)[0].t()
    buf = torch.full((V, C + 8), float("nan"), dtype=torch.float64)
    buf[:, 3:3 + C] = y
    assert torch.allclose(buf[:, 3:3 + C], want, rtol=1e-12, atol=1e-12)
    assert bool(torch.isnan(buf[:, :3]).all()) and bool(torch.isnan(buf[:, 3 + C:]).all())
    ref, bound = gn_bound(r, G, 1e-5, gam, bet)
    assert torch.equal(ref, y) and bool((bound > 0).all()) and bool((bound < 1e-5 * (y.abs() + 1)).all())

    x = torch.randn((1, 3, 5, 7, 4), generator=g, dtype=torch.float64).round()
    x[0, 0, 0, 0, 0] = float("nan")
    x[0, 1, :2, :2, :2] = float("nan")
    x[0, 2, 0, 0, 1] = float("inf")
    x[0, 2, 2, 3, 0] = float("-inf")
    x[0, 0, 4, 6, 3] = float("nan")      # floored tail
    assert same_values(maxpool_ref(x), F.max_pool3d(x, 2))
    assert bool(torch.isnan(maxpool_ref(x)[0, 0, 0, 0, 0]))

    xg = torch.randn((9, 8), generator=g, dtype=torch.float64)
    W = torch.randn((5, 8), generator=g, dtype=torch.float64)
    b = torch.randn(5, generator=g, dtype=torch.float64)
    W[3], b[3] = W[1], b[1]
    logits, p, e, e_row = head_ref(xg, W, b, True)
    assert torch.allclose(p, F.softmax(F.linear(xg, W, b), 1), rtol=1e-14, atol=0)
    assert torch.equal(e_row, e.max(1).values) and bool((e > 0).all())
    s = torch.tensor([[0.1, 0.7, 0.2, 0.7], [0.5, 0.5, 0.5, 0.5], [0.0, 0.0, 1.0, 0.0]])
    assert first_argmax(s).tolist() == [1, 0, 2]

    sp = torch.tensor([[1.0 + 2.0 ** -8], [1.0 + 3 * 2.0 ** -8], [2.0 ** -149], [-0.0], [1.0 / 3.0]])
    s3 = split3_ref(sp)
    assert s3.shape == (5, 3) and torch.equal(s3[:, 0].view(torch.int16), s3[:, 2].view(torch.int16))
    assert s3[:, 0].float().tolist()[:2] == [1.0, 1.0 + 2.0 ** -6]              # ties to even
    assert float(s3[0, 1]) == 2.0 ** -8 and float(s3[1, 1]) == -(2.0 ** -8)   # lo carries the rest exactly
    assert float(s3[2, 0]) == 0.0 and float(s3[2, 1]) == 0.0     # below half the least bf16 subnormal (2^-133)
    assert int(s3[3, 0].view(torch.int16)) == -32768
    third = sp[4, 0].double()
    assert abs(float(s3[4, 0]) + float(s3[4, 1]) - float(third)) <= 2.0 ** -16 * float(third)
