"""Teacher-forced fp64 oracle inside a real training step.

Every kernel entry point ``models.py`` reaches through ``unetsulc_b200.ops`` is replaced by a spy that clones what the
call reads, runs the real call, synchronises, and compares what the call wrote with the same operation computed in
float64 from the exact (bf16 / fp32) tensors it read.  Nothing compounds from one call to the next, so every bound
below is derived from the arithmetic of one call, element by element, at the magnitudes a real step produces.

Notation: u = 2^-24 (fp32 unit roundoff), ``ref`` the fp64 result, ``A`` the same operation applied to absolute values
(e.g. conv3d(|x|, |w|)), ``K`` the number of terms of the longest fp32 chain.  Bounds (a ratio error / bound <= 1 passes):
  * bf16-stored result .............. |got - ref| <= 2^-8 |ref| + (1 + 2^-8) K u A  (one bf16 rounding: 8 significant
                                      bits, round to nearest, at most 2^-8 of the value it rounds; recursive fp32
                                      summation of K terms is within K u A in any order, tensor-core and split-K orders
                                      included)
  * fp32 result ..................... the same without the bf16 term
  * conv fprop / dgrad / split-K .... K = 27 Cin + 1 (the products of bf16 operands are exact in fp32)
  * first conv (fp32 weights) ....... K = 27 + 2 (one fp32 rounding per product as well)
  * wgrad, first-layer wgrad ........ fp32, K = N V + 2 (reduction over every voxel; split partials + the reduce are part
                                      of the same sum)
  * fixed-point statistics ......... |got - ref| <= K u sum|terms| + nb 2^-33: per-block fp32 partial sums (chain K),
                                      then one committed contribution per block and channel whose fraction limb is rounded
                                      to 2^-32 (common.h).  nb and K per producer, from its launch code:
        head_ce_kernel .............. nb = 296 (kCeBlocks); K = labelled voxels of the busiest block's range (one running
                                      fp32 sum per thread over the staged rows)
        pool_bwd_add_kernel ......... nb = min(ceil(cells*C/8 / 256), 8*148); K = 8 * (cells per thread) + 256/(C/8)
        upsample_bwd_hd_kernel ...... nb = N Di Hi (one block per coarse row); K = ceil(Wi C / 2048) + 256/(C/8)
        conv epilogues .............. conv3d_igemm_kernel (plain and h-halo) and conv3d_slab_kernel launch
                                      grid = min(T, 148) persistent CTAs, each commits once: nb = min(T, 148);
                                      K = 4 ceil(T / nb) + 8: a thread's running sum visits at most 4 planes (slab kTD)
                                      of each of its tiles, plus the 32-row warp_column_sums tree (5) and the combine of
                                      <= 8 warps (3).  T = the largest tile count of the boxes the launch code can pick
                                      (choose_box, the three h-halo boxes, the two slab boxes), see conv_epilogue_plan
        conv_first_fwd_kernel ....... blocks = min(ceil(V / 128), 592); K = ceil(V / (128 blocks)) + 7 (one 32-row
                                      column sum per warp pass, 4 warps combined); nb = blocks
        upsample2x_bwd_kernel ....... grid = min(items, 2*148 rounded to the channel slices); K = ceil(items / grid) * ds
                                      + 32 (ds coarse planes per item, then the 32 rows of the tile); nb = grid
        relu_gn_stats / relu_gn_bwd . nblk = stat_blocks(V, C) blocks, fp32 partials reduced in fp64 (nb = 0);
                                      K = ceil(V / (nblk vpi)) + 2 + vpi, vpi = 256 / (C / 8) rows per block
  * GroupNorm statistics (mean, rstd, scale, shift) from those sums: the sum errors above pushed through
    mean = S/m, var = Q/m - mean^2, rstd = 1/sqrt(var + eps) (first order), plus 4 u relative for the fp32 conversions and
    rsqrt + Newton step, plus 2 u (|beta| + |mean scale|) for the shift
  * GroupNorm apply ................. bf16: 2^-8 |ref| + 2 u (|r scale| + |shift|) (one fma); the pooled tensor must equal
                                      the max of the stored 2x2x2 cell exactly
  * GroupNorm backward (closed form, saved mean/rstd, ReLU mask of the stored r):
                                      dr: 2^-8 |ref| + rstd (dS1 + |xhat| dS2)/m + 6 u (|a dy| + |kb r| + |kb mu| + |kc|),
                                      the 6 covering the coefficient folding (a, kb, kc) and the two fmas;
                                      dS1, dS2 = the statistics bound of the sums the call consumed (the producer's, when
                                      they come from an accumulator), weighted by |gamma|;
                                      dgamma/dbeta: the statistics bound + u |ref|
  * maxpool3d_bwd_add ............... one correctly rounded bf16 add: 2^-8 |ref|
  * upcat_fwd / upcat_bwd ........... K = (taps: 8 fwd, 64 adjoint) + 4 max(D, H, W) (source coordinates are computed in
                                      fp32: each weight carries an absolute error <= (4 size) u), with A over all touched
                                      samples; the two-pass adjoint stores a bf16 intermediate: + 2^-8 A
  * head_ce (training) .............. logits: (Cin + 1) u A_l; per-voxel loss: 2 e_l + (Cout + 4) u + 2 u (|lse| + |l_y|);
                                      d(logits): |gs| (p (4 e_l + (Cout + 6) u) + 2 u |p - y|) + 3 u |d|; dW, db: sum of
                                      those over voxels + K u sum|terms| (K as for the statistics); dX rows: bf16 with
                                      K = Cout; preds must match wherever the fp64 top-2 margin exceeds 2 e_l
Each configuration prints the worst error / bound per op, so that the slack is visible in the log.
"""
import functools
import time

import pytest
import torch
import torch.nn.functional as F

U = 2.0 ** -24
FIX = 2.0 ** -33          # rounding of one committed fixed-point contribution (fraction limb in units of 2^-32)
FLOOR = 2.0 ** -126       # gradual-underflow floor

SPLITK_MAX_VOXELS = 8192  # ops.SPLITK_MAX_VOXELS (not imported: the module must import without the library)


# ------------------------------------------------------------------------------------------------ fp64 references
def conv3d_taps(x, w):
    """3x3x3 conv, padding 1, as 27 shifted matrix products in the dtype of the inputs (float64 here).
    x [N, Cin, D, H, W], w [Cout, Cin, 3, 3, 3] -> [N, Cout, D, H, W].  Same operation as F.conv3d(x, w, padding=1)."""
    N, Ci, D, H, W = x.shape
    xp = F.pad(x, (1, 1, 1, 1, 1, 1))
    out = torch.zeros((N, w.shape[0], D * H * W), dtype=x.dtype, device=x.device)
    for t in range(27):
        kd, kh, kw = t // 9, (t // 3) % 3, t % 3
        xs = xp[:, :, kd:kd + D, kh:kh + H, kw:kw + W].reshape(N, Ci, -1)
        out += torch.matmul(w[:, :, kd, kh, kw], xs)
    return out.view(N, -1, D, H, W)


def wgrad_taps(x, dy):
    """dW of conv3d_taps: [Cout, Cin, 3, 3, 3] = sum over voxels of dy * shifted x."""
    N, Ci, D, H, W = x.shape
    Co = dy.shape[1]
    xp = F.pad(x, (1, 1, 1, 1, 1, 1))
    dw = torch.zeros((Co, Ci, 27), dtype=x.dtype, device=x.device)
    g = dy.reshape(N, Co, -1)
    for t in range(27):
        kd, kh, kw = t // 9, (t // 3) % 3, t % 3
        xs = xp[:, :, kd:kd + D, kh:kh + H, kw:kw + W].reshape(N, Ci, -1)
        dw[:, :, t] = torch.einsum("nov,ncv->oc", g, xs)
    return dw.view(Co, Ci, 3, 3, 3)


def interp_matrix(n_in, n_out, touch=False, dtype=torch.float64, device="cpu"):
    """[n_out, n_in] linear-interpolation weights of PyTorch's align_corners=False rule (in float64); touch=True puts a 1
    on every source sample an output reads (both neighbours), the absolute-value operand of the bounds."""
    M = torch.zeros((n_out, n_in), dtype=dtype)
    scale = n_in / n_out
    for o in range(n_out):
        src = max(scale * (o + 0.5) - 0.5, 0.0)
        i0 = min(int(src), n_in - 1)
        i1 = i0 + (1 if i0 < n_in - 1 else 0)
        l1 = src - i0
        if touch:   # a source coordinate at an integer may round to either side in fp32: mark both neighbours too
            near = abs(src - round(src)) < 1e-5
            lo, hi = (max(i0 - 1, 0), min(i1 + 1, n_in - 1)) if near else (i0, i1)
            M[o, lo:hi + 1] = 1.0
        else:
            M[o, i0] += 1.0 - l1
            M[o, i1] += l1
    return M.to(device)


def separable(x, Md, Mh, Mw):
    """x [N, C, D, H, W] -> sum over (d, h, w) of Md[D', d] Mh[H', h] Mw[W', w] x"""
    x = torch.einsum("ncdhw,Ed->ncEhw", x, Md)
    x = torch.einsum("ncdhw,Eh->ncdEw", x, Mh)
    return torch.einsum("ncdhw,Ew->ncdhE", x, Mw)


def upsample_ref(x, size, touch=False):
    dev = x.device
    Ms = [interp_matrix(i, o, touch, device=dev) for i, o in zip(x.shape[2:], size)]
    return separable(x, *Ms)


def upsample_adjoint_ref(g, size_in, touch=False):
    dev = g.device
    Ms = [interp_matrix(i, o, touch, device=dev).t() for i, o in zip(size_in, g.shape[2:])]
    return separable(g, *Ms)


def groupnorm_bwd_ref(dy, r, mu, rstd, gamma, G):
    """Closed-form backward of y = GroupNorm(relu(c)) w.r.t. c, with the saved per-channel mean / rstd and the mask of
    the stored r.  dy, r [V, C] float64; mu, rstd, gamma [C].  Returns (dr, dgamma, dbeta, S1 [C], S2 [C])."""
    V, C = r.shape
    cpg = C // G
    xhat = (r - mu) * rstd
    sdy = dy.sum(0)
    sdyx = (dy * xhat).sum(0)
    S1 = (gamma * sdy).view(G, cpg).sum(1).repeat_interleave(cpg)
    S2 = (gamma * sdyx).view(G, cpg).sum(1).repeat_interleave(cpg)
    m = V * cpg
    dr = rstd * (gamma * dy - S1 / m - xhat * S2 / m)
    dr = torch.where(r > 0, dr, torch.zeros_like(dr))
    return dr, sdyx, sdy, S1, S2


def pool_adjoint_ref(y, g):
    """adjoint of MaxPool3d(2) (floor mode): g [N, C, D/2, H/2, W/2] routed to the FIRST maximum of each 2x2x2 cell of y
    in (d, h, w) scan order (PyTorch's max_pool3d_with_indices); voxels of the odd tails receive nothing."""
    N, C, D, H, W = y.shape
    Dp, Hp, Wp = D // 2, H // 2, W // 2
    cells = y[:, :, :2 * Dp, :2 * Hp, :2 * Wp].reshape(N, C, Dp, 2, Hp, 2, Wp, 2)
    cells = cells.permute(0, 1, 2, 4, 6, 3, 5, 7).reshape(N, C, Dp, Hp, Wp, 8)
    first = (cells == cells.max(-1, keepdim=True).values).to(torch.int8).argmax(-1, keepdim=True)
    routed = torch.zeros_like(cells).scatter_(-1, first, g.unsqueeze(-1))
    routed = routed.view(N, C, Dp, Hp, Wp, 2, 2, 2).permute(0, 1, 2, 5, 3, 6, 4, 7).reshape(N, C, 2 * Dp, 2 * Hp, 2 * Wp)
    out = torch.zeros_like(y)
    out[:, :, :2 * Dp, :2 * Hp, :2 * Wp] = routed
    return out


# ------------------------------------------------------------------------------------------------ bookkeeping
def nc(v):
    """ActView -> float64 [N, C, D, H, W]"""
    return v.dense().double().permute(0, 4, 1, 2, 3)


def rows(v):
    """ActView -> float64 [N*V, C]"""
    return v.dense().double().reshape(-1, v.C)


def unpack_wf(wf, cout, cin):
    """bf16 [27, cout, cin] pack -> float64 [cout, cin, 3, 3, 3]"""
    return wf.double().permute(1, 2, 0).reshape(cout, cin, 3, 3, 3)


def acc_sums(acc, C):
    a = acc.view(C, 4).double()
    return a[:, 0] + a[:, 1] / 2.0 ** 32, a[:, 2] + a[:, 3] / 2.0 ** 32


class Oracle(object):
    def __init__(self):
        self.worst = {}
        self.seen = set()
        self.acc_meta = {}     # accumulator data_ptr -> (K, nb) of the producer that filled it
        self.pending = {}      # deferred wgrad: dw data_ptr -> (ref, A, K)
        self.sms = torch.cuda.get_device_properties(0).multi_processor_count

    def ratio(self, op, got, ref, bound):
        got, ref = got.double(), ref.double()
        diff = (got - ref).abs()
        r = torch.where(diff == 0, torch.zeros_like(diff), diff / bound)
        # a non-finite result, reference or bound is a failure (max() would drop a NaN ratio)
        bad = ~torch.isfinite(got) | ~torch.isfinite(ref) | ~torch.isfinite(r)
        worst = float("inf") if bool(bad.any()) else (float(r.max()) if r.numel() else 0.0)
        self.worst[op] = max(self.worst.get(op, 0.0), worst)
        return worst

    def dense(self, op, got, ref, A, K, bf16=True, extra=0.0):
        b16 = 2.0 ** -8 if bf16 else 0.0
        bound = b16 * ref.abs() + (1.0 + b16) * K * U * A + extra + K * FLOOR
        return self.ratio(op, got, ref, bound)

    def sums(self, op, acc, C, terms_s, terms_q, K, nb, store=True):
        """fixed-point accumulators vs fp64 sums over the stored terms [n, C]"""
        s, q = acc_sums(acc, C)
        self.ratio(op, s, terms_s.sum(0), K * U * terms_s.abs().sum(0) + nb * FIX + FLOOR)
        self.ratio(op, q, terms_q.sum(0), K * U * terms_q.abs().sum(0) + nb * FIX + FLOOR)
        if store:
            self.acc_meta[acc.data_ptr()] = (K, nb)

    def fwd_stats(self, op, r, C, G, eps, gamma, beta, mr, ss, K, nb):
        """mean_rstd / scale_shift [N, C, 2] against fp64 statistics of the stored r [N, V, C]"""
        N, V = r.shape[0], r.shape[1]
        cpg = C // G
        m = V * cpg
        for n in range(N):
            x = r[n]
            S, Q = x.sum(0), (x * x).sum(0)
            eS = K * U * x.abs().sum(0) + nb * FIX
            eQ = K * U * (x * x).sum(0) + nb * FIX
            Sg, Qg = S.view(G, cpg).sum(1), Q.view(G, cpg).sum(1)
            eSg, eQg = eS.view(G, cpg).sum(1), eQ.view(G, cpg).sum(1)
            mean = Sg / m
            var = (Qg / m - mean * mean).clamp_min(0)
            rstd = 1.0 / torch.sqrt(var + eps)
            dmean = eSg / m
            dvar = eQg / m + 2 * mean.abs() * dmean + dmean * dmean
            drstd = rstd * (0.5 * dvar / (var + eps) + 4 * U)
            mean_c, rstd_c = mean.repeat_interleave(cpg), rstd.repeat_interleave(cpg)
            dmean_c, drstd_c = (dmean + U * mean.abs()).repeat_interleave(cpg), drstd.repeat_interleave(cpg)
            g64, b64 = gamma.double(), beta.double()
            self.ratio(op + ":mean", mr[n, :, 0], mean_c, dmean_c + FLOOR)
            self.ratio(op + ":rstd", mr[n, :, 1], rstd_c, drstd_c + FLOOR)
            sc = rstd_c * g64
            dsc = g64.abs() * drstd_c + U * sc.abs()
            self.ratio(op + ":scale", ss[n, :, 0], sc, dsc + FLOOR)
            sh = b64 - mean_c * sc
            dsh = mean_c.abs() * dsc + sc.abs() * dmean_c + 2 * U * (b64.abs() + (mean_c * sc).abs())
            self.ratio(op + ":shift", ss[n, :, 1], sh, dsh + FLOOR)


def _ceil(a, b):
    return -(-a // b)


def conv_epilogue_plan(sms, D, H, W):
    """(K, nb) of the statistics fused into conv3d_igemm_kernel / conv3d_slab_kernel (batch 1): both launch
    min(T, sms) persistent CTAs over T tiles of 128 voxel rows, and every CTA commits once.  T is bounded by the largest
    tile count among the boxes the launch code chooses from: choose_box (conv_igemm.cu), the h-halo boxes 8x16, 16x8,
    32x4 (one plane) and the slab boxes 16x8 / 32x4 (kTD = 4 planes)."""
    best = None
    for lw in range(8):      # choose_box: least padded volume, then longer W runs, then H
        for lh in range(8 - lw):
            cw, ch, cd = 1 << lw, 1 << lh, 1 << (7 - lw - lh)
            cost = _ceil(W, cw) * cw * _ceil(H, ch) * ch * _ceil(D, cd) * cd
            score = cost * 1024 - cw * 8 - ch
            if best is None or score < best[0]:
                best = (score, cw, ch, cd)
    boxes = [best[1:], (8, 16, 1), (16, 8, 1), (32, 4, 1), (16, 8, 4), (32, 4, 4)]
    T = max(_ceil(W, bw) * _ceil(H, bh) * _ceil(D, bd) for bw, bh, bd in boxes)
    nb = min(T, sms)
    return 4 * _ceil(T, nb) + 8, nb


def first_conv_plan(V):
    """(K, nb) of conv_first_fwd_kernel's statistics: min(ceil(V / 128), 148 * 4) blocks of 4 warps; a warp adds one
    32-row column sum per pass over 32 voxels, the block combines its 4 warps and commits once"""
    blocks = min(_ceil(V, 128), 148 * 4)
    return _ceil(V, 128 * blocks) + 5 + 2, blocks


def upsample2x_plan(sms, N, Di, Hi, Wi, C):
    """(K, nb) of upsample2x_bwd_kernel's statistics: the launch code's D segment length ds and grid
    (resample.cu, upcat_bwd_separable_impl); a thread accumulates one value per coarse plane of each of its items,
    then the 4 x 8 rows of the tile are combined in order"""
    tiles_h, tiles_w, n_slices = _ceil(Hi, 4), _ceil(Wi, 8), C // 64
    slots = 2 * sms // n_slices * n_slices
    best_ds, best = Di, -1.0
    for ds in range(1, Di + 1):
        items = N * _ceil(Di, ds) * tiles_h * tiles_w * n_slices
        waves = items / slots
        eff = (waves / float(_ceil(items, slots))) * (2.0 * ds / (2.0 * ds + 2.0))
        if eff > best + 1e-9:
            best, best_ds = eff, ds
    items = N * _ceil(Di, best_ds) * tiles_h * tiles_w * n_slices
    grid = min(items, slots)
    return _ceil(items, grid) * best_ds + 32, grid


def gn_pass_plan(V, C):
    """(K, nb) of the fp32 partial sums of gn_stats_kernel / gn_bwd_stats_kernel (norm.cu): stat_blocks(V, C) blocks
    of 256 threads, vpi = 256 / (C / 8) voxel rows per pass, per-thread sums in groups of <= 4, the vpi rows combined in
    order; the block partials are reduced in fp64 (no fixed point: nb = 0)"""
    nblk = max(min((V * C * 2) // 16384, 16384 // C, 296), 1)
    vpi = 256 // (C // 8)
    return _ceil(V, nblk * vpi) + 2 + vpi, 0


def _block_count_max(labels, NV):
    """labelled voxels of the busiest head_ce_kernel block (head.cu: per_block = ceil(NV / 296) rounded up to 256)"""
    pb = (NV + 295) // 296
    pb = (pb + 255) // 256 * 256
    lab = (labels.reshape(-1) >= 0).to(torch.int64)
    pad = torch.zeros(pb * 296 - NV, dtype=torch.int64, device=lab.device) if pb * 296 > NV else lab[:0]
    return int(torch.cat([lab, pad])[:pb * 296].view(296, pb).sum(1).max())


# ------------------------------------------------------------------------------------------------ spies
def _conv_check(orc, op, x64, w64, got, relu, K):
    ref = conv3d_taps(x64, w64)
    A = conv3d_taps(x64.abs(), w64.abs())
    if relu:
        ref = ref.clamp_min(0)
    orc.dense(op, got, ref, A, K)


def spy_pack_conv_weights_multi(real, orc, ws):
    outs = real(ws)
    torch.cuda.synchronize()
    orc.seen.add("pack_multi")
    for w, (wf, wd) in zip(ws, outs):
        _pack_check(orc, w, wf, wd)
    return outs


def _pack_check(orc, w, wf, wd):
    cout, cin = w.shape[0], w.shape[1]
    wb = w.detach().to(torch.bfloat16)
    ok = torch.equal(wf, wb.permute(2, 3, 4, 0, 1).reshape(27, cout, cin))
    if wd is not None:
        ok = ok and torch.equal(wd, wb.flip(2, 3, 4).permute(2, 3, 4, 1, 0).reshape(27, cin, cout))
    orc.worst["pack"] = max(orc.worst.get("pack", 0.0), 0.0 if ok else float("inf"))


def spy_pack_conv_weights(real, orc, w, want_dgrad=True):
    wf, wd = real(w, want_dgrad)
    torch.cuda.synchronize()
    _pack_check(orc, w, wf, wd)
    return wf, wd


def spy_conv3d_first_fwd(real, orc, x, w, y, relu=True):
    real(x, w, y, relu)
    torch.cuda.synchronize()
    orc.seen.add("conv_first")
    _conv_check(orc, "conv_first", x.double(), w.double(), nc(y), relu, 27 + 2)


def spy_conv3d_first_fwd_gn_stats(real, orc, x, w, y, groups, eps, gamma, beta, pool=None):
    mr, ss = real(x, w, y, groups, eps, gamma, beta, pool)
    torch.cuda.synchronize()
    orc.seen.add("conv_first_stats")
    _conv_check(orc, "conv_first", x.double(), w.double(), nc(y), True, 27 + 2)
    r = rows(y)
    K, nb = first_conv_plan(y.V)
    orc.sums("stats_acc:conv_first", orc.last_acc, y.C, r, r * r, K, nb, store=False)
    orc.fwd_stats("gn_stats", r.view(1, y.V, y.C), y.C, groups, eps, gamma, beta, mr, ss, K, nb)
    return mr, ss


def spy_conv3d_igemm_gn_stats(real, orc, x, wpack, y, cin, cout, groups, eps, gamma, beta, pool=None):
    x64 = nc(x).clone()
    mr, ss = real(x, wpack, y, cin, cout, groups, eps, gamma, beta, pool)
    torch.cuda.synchronize()
    orc.seen.add("conv_fprop_stats")
    _conv_check(orc, "conv_fprop", x64, unpack_wf(wpack, cout, cin), nc(y), True, 27 * cin + 1)
    r = rows(y)
    K, nb = conv_epilogue_plan(orc.sms, y.D, y.H, y.W)
    orc.sums("stats_acc:conv_epilogue", orc.last_acc, cout, r, r * r, K, nb, store=False)
    orc.fwd_stats("gn_stats", r.view(1, y.V, cout), cout, groups, eps, gamma, beta, mr, ss, K, nb)
    return mr, ss


def spy_conv3d_igemm_auto(real, orc, x, wpack, y, cin, cout, relu):
    x64 = nc(x).clone()
    real(x, wpack, y, cin, cout, relu)
    torch.cuda.synchronize()
    kind = "conv_fprop" if relu else "conv_dgrad"
    orc.seen.add(kind + ("_splitk" if x.N * x.V <= SPLITK_MAX_VOXELS else ""))
    _conv_check(orc, kind, x64, unpack_wf(wpack, cout, cin), nc(y), relu, 27 * cin + 1)


def spy_conv3d_dgrad_gn_bstats(real, orc, dy, wd, dx, cin, cout, r, pool=None):
    dy64 = nc(dy).clone()
    acc = real(dy, wd, dx, cin, cout, r, pool)
    torch.cuda.synchronize()
    orc.seen.add("conv_dgrad_bstats")
    _conv_check(orc, "conv_dgrad", dy64, unpack_wf(wd, cout, cin), nc(dx), False, 27 * cin + 1)
    o = rows(dx)
    K, nb = conv_epilogue_plan(orc.sms, dx.D, dx.H, dx.W)
    orc.sums("bstats_acc:conv_dgrad", acc, cout, o, o * rows(r), K, nb)
    return acc


def spy_relu_gn_stats(real, orc, r, groups, eps, gamma, beta):
    mr, ss = real(r, groups, eps, gamma, beta)
    torch.cuda.synchronize()
    orc.seen.add("gn_stats_pass")
    orc.fwd_stats("gn_stats", r.dense().double().reshape(r.N, r.V, r.C), r.C, groups, eps, gamma, beta, mr, ss,
                  *gn_pass_plan(r.V, r.C))
    return mr, ss


def spy_relu_gn_apply(real, orc, r, scale_shift, y, pooled=None):
    real(r, scale_shift, y, pooled)
    torch.cuda.synchronize()
    orc.seen.add("gn_apply_pool" if pooled is not None else "gn_apply")
    ss = scale_shift.double()
    sc = ss[:, :, 0].view(r.N, -1, 1, 1, 1)
    sh = ss[:, :, 1].view(r.N, -1, 1, 1, 1)
    x = nc(r)
    orc.dense("gn_apply", nc(y), x * sc + sh, 2 * ((x * sc).abs() + sh.abs()), 1)
    if pooled is not None:
        want = F.max_pool3d(nc(y), 2)
        ok = torch.equal(nc(pooled), want)
        orc.worst["gn_apply"] = max(orc.worst["gn_apply"], 0.0 if ok else float("inf"))


def spy_upcat_fwd(real, orc, x, cat_window):
    before = cat_window.buf.clone()
    real(x, cat_window)
    torch.cuda.synchronize()
    orc.seen.add("upcat_fwd")
    c = cat_window
    size = (c.D, c.H, c.W)
    x64 = nc(x)
    K = 8 + 4 * max(size)
    orc.dense("upcat_fwd", nc(c), upsample_ref(x64, size), upsample_ref(x64.abs(), size, touch=True), K)
    outside = torch.ones(c.ld, dtype=torch.bool, device=before.device)
    outside[c.coff:c.coff + c.C] = False
    ok = torch.equal(before[..., outside], c.buf[..., outside])
    orc.worst["upcat_fwd"] = max(orc.worst["upcat_fwd"], 0.0 if ok else float("inf"))


def spy_upcat_bwd(real, orc, dcat_window, Di, Hi, Wi, separable=True, stat_r=None, pool=None):
    g64 = nc(dcat_window).clone()
    res = real(dcat_window, Di, Hi, Wi, separable, stat_r, pool)
    torch.cuda.synchronize()
    dx, acc = res if stat_r is not None else (res, None)
    c = dcat_window
    exact2x = (c.D == 2 * Di and c.H == 2 * Hi and c.W == 2 * Wi and c.C % 64 == 0)
    two_pass = separable and not exact2x
    tag = "upcat_bwd" + ("_stats" if acc is not None else "") + ("_2x" if exact2x else "_non2x")
    orc.seen.add(tag)
    size_in = (Di, Hi, Wi)
    A = upsample_adjoint_ref(g64.abs(), size_in, touch=True)
    K = 64 + (0 if exact2x else 4 * max(c.D, c.H, c.W))
    orc.dense("upcat_bwd_2x" if exact2x else "upcat_bwd_non2x", nc(dx), upsample_adjoint_ref(g64, size_in), A, K,
              extra=(2.0 ** -8) * A if two_pass else 0.0)
    if acc is not None:
        C = c.C
        o = rows(dx)
        if exact2x:
            Ks, nb = upsample2x_plan(orc.sms, c.N, Di, Hi, Wi, C)
        else:   # upsample_bwd_hd_kernel: one block per coarse (n, d, h) row
            Ks, nb = -(-Wi * C // 2048) + 256 // (C // 8), c.N * Di * Hi
        orc.sums("bstats_acc:upcat_bwd", acc, C, o, o * rows(stat_r), Ks, nb)
    return res


def spy_maxpool3d_bwd_add(real, orc, y, dskip, dpool, stat_r=None, pool=None):
    y64, ds64, dp64 = nc(y).clone(), nc(dskip).clone(), nc(dpool).clone()
    res = real(y, dskip, dpool, stat_r, pool)
    torch.cuda.synchronize()
    out, acc = res if stat_r is not None else (res, None)
    orc.seen.add("maxpool_bwd" + ("_stats" if acc is not None else ""))
    ref = ds64 + pool_adjoint_ref(y64, dp64)
    orc.ratio("maxpool_bwd", nc(out), ref, (2.0 ** -8) * ref.abs() + FLOOR)
    if acc is not None:
        N, C, D, H, W = y64.shape
        cells = N * ((D + 1) // 2) * ((H + 1) // 2) * ((W + 1) // 2)
        total = cells * (C // 8)
        nb = min(min(-(-total // 256), orc.sms * 16), orc.sms * 8)
        Ks = 8 * -(-total // (nb * 256)) + 256 // (C // 8)
        o = rows(out)
        orc.sums("bstats_acc:maxpool_bwd", acc, C, o, o * rows(stat_r), Ks, nb)
    return res


def _gn_bwd_check(orc, op, dy, r, G, gamma, mean_rstd, dr, dg, db, K, nb, row_labels=None):
    C = r.C
    dy64 = rows(dy)
    if row_labels is not None:
        dy64 = torch.where((row_labels.reshape(-1, 1) >= 0), dy64, torch.zeros_like(dy64))
    r64 = rows(r)
    mu, rstd = mean_rstd[0, :, 0].double(), mean_rstd[0, :, 1].double()
    g64 = gamma.double()
    ref, dgam, dbet, S1, S2 = groupnorm_bwd_ref(dy64, r64, mu, rstd, g64, G)
    xhat = (r64 - mu) * rstd
    # statistics of the consumed sums (producer chain K, nb commits) and their group sums
    e_sdy = K * U * dy64.abs().sum(0) + nb * FIX
    T = (dy64.abs() * (r64.abs() + mu.abs())).sum(0)
    e_sdyx = rstd * (K * U * T + 3 * U * T + nb * FIX * (1 + mu.abs()))
    cpg = C // G
    m = r.V * cpg
    dS1 = (g64.abs() * e_sdy).view(G, cpg).sum(1).repeat_interleave(cpg) + U * S1.abs()
    dS2 = (g64.abs() * e_sdyx).view(G, cpg).sum(1).repeat_interleave(cpg) + U * S2.abs()
    kb = rstd * rstd * S2.abs() / m
    mag = rstd * g64.abs() * dy64.abs() + kb * r64.abs() + kb * mu.abs() + rstd * S1.abs() / m
    e = (rstd * (dS1 + xhat.abs() * dS2) / m) * (r64 > 0) + 6 * U * mag
    bound = (2.0 ** -8) * ref.abs() + (1.0 + 2.0 ** -8) * e + FLOOR
    orc.ratio(op, rows(dr), ref, bound)
    if dg is not None:
        orc.ratio(op + ":dgamma", dg, dgam, e_sdyx + U * dgam.abs() + FLOOR)
        orc.ratio(op + ":dbeta", db, dbet, e_sdy + U * dbet.abs() + FLOOR)


def spy_relu_gn_bwd_from_stats(real, orc, acc, dy, r, groups, gamma, mean_rstd, want_param_grads=True, dgamma_out=None,
                               dbeta_out=None, dy_row_labels=None):
    dy_rows = rows(dy).clone()
    out = real(acc, dy, r, groups, gamma, mean_rstd, want_param_grads, dgamma_out, dbeta_out, dy_row_labels)
    torch.cuda.synchronize()
    orc.seen.add("gn_bwd_acc" + ("_rows" if dy_row_labels is not None else ""))
    K, nb = orc.acc_meta[acc.data_ptr()]
    dr, dg, db = out
    dyv = _RowsView(dy_rows, r)
    _gn_bwd_check(orc, "gn_bwd", dyv, r, groups, gamma, mean_rstd, dr, dg, db, K, nb, dy_row_labels)
    return out


def spy_relu_gn_bwd(real, orc, dy, r, groups, gamma, mean_rstd, want_param_grads=True, dgamma_out=None, dbeta_out=None):
    dy_rows = rows(dy).clone()
    out = real(dy, r, groups, gamma, mean_rstd, want_param_grads, dgamma_out, dbeta_out)
    torch.cuda.synchronize()
    orc.seen.add("gn_bwd_pass")
    dr, dg, db = out
    V = r.V
    for n in range(r.N):   # per sample: its own statistics; dgamma / dbeta are summed over the samples
        sl = slice(n * V, (n + 1) * V)
        _gn_bwd_check(orc, "gn_bwd", _RowsView(dy_rows[sl], r), _RowsView(rows(r)[sl], r), groups, gamma,
                      mean_rstd[n:n + 1], _RowsView(rows(dr)[sl], r), None, None, *gn_pass_plan(V, r.C))
    if dg is not None:
        dy64 = dy_rows.view(r.N, V, r.C)
        r64 = rows(r).view(r.N, V, r.C)
        mu, rstd = mean_rstd[:, :, 0].double().unsqueeze(1), mean_rstd[:, :, 1].double().unsqueeze(1)
        T = dy64.abs() * (r64.abs() + mu.abs()) * rstd
        Kp = gn_pass_plan(V, r.C)[0]   # per-sample fp32 partials, then the samples summed in fp32
        orc.ratio("gn_bwd:dgamma", dg, (dy64 * (r64 - mu) * rstd).sum((0, 1)), (Kp + 3 + r.N) * U * T.sum((0, 1)) + FLOOR)
        orc.ratio("gn_bwd:dbeta", db, dy64.sum((0, 1)), (Kp + r.N) * U * dy64.abs().sum((0, 1)) + FLOOR)
    return out


class _RowsView(object):
    """float64 rows [V, C] posing as an ActView for _gn_bwd_check"""

    def __init__(self, t, like):
        self.t, self.C, self.V = t, like.C, t.shape[0]

    def dense(self):
        return self.t


def spy_conv3d_wgrad(real, orc, x, dy, cin, cout, out=None):
    x64, dy64 = nc(x).clone(), nc(dy).clone()
    dw = real(x, dy, cin, cout, out)
    torch.cuda.synchronize()
    orc.seen.add("wgrad")
    orc.dense("wgrad", dw, wgrad_taps(x64, dy64), wgrad_taps(x64.abs(), dy64.abs()), x.N * x.V + 2, bf16=False)
    return dw


def spy_conv3d_wgrad_partial(real, orc, x, dy, cin, cout, slot, out=None):
    x64, dy64 = nc(x), nc(dy)
    orc.pending_ref = (wgrad_taps(x64, dy64), wgrad_taps(x64.abs(), dy64.abs()), x.N * x.V + 2)
    desc = real(x, dy, cin, cout, slot, out)
    orc.pending[desc["dw"].data_ptr()] = orc.pending_ref
    return desc


def spy_wgrad_reduce_multi(real, orc, descs):
    real(descs)
    torch.cuda.synchronize()
    if descs:
        orc.seen.add("wgrad_defer")
    for d in descs:
        ref, A, K = orc.pending.pop(d["dw"].data_ptr())
        orc.dense("wgrad", d["dw"], ref, A, K, bf16=False)


def spy_conv3d_first_wgrad(real, orc, x, dy, cout, out=None):
    x64, dy64 = x.double(), nc(dy).clone()
    dw = real(x, dy, cout, out)
    torch.cuda.synchronize()
    orc.seen.add("wgrad_first")
    orc.dense("wgrad_first", dw, wgrad_taps(x64, dy64), wgrad_taps(x64.abs(), dy64.abs()), dy.N * dy.V + 2,
              bf16=False)
    return dw


def spy_head_ce(real, orc, x, labels, W, b, compute_grad, eval_softmax=False, grad_scale=1.0, grad_scale_dev=None,
                want_preds=True, want_dx=True, dW_out=None, db_out=None, stat_r=None, pool=None, x_scale_shift=None,
                sparse_dx=False):
    gdev = None if grad_scale_dev is None else float(grad_scale_dev.reshape(-1)[0])
    out = real(x, labels, W, b, compute_grad, eval_softmax, grad_scale, grad_scale_dev, want_preds, want_dx, dW_out,
               db_out, stat_r, pool, x_scale_shift, sparse_dx)
    torch.cuda.synchronize()
    fused = out["dx_stats"] is not None
    if not compute_grad:
        orc.seen.add("head_fwd")
    elif fused:
        orc.seen.add("head_train_fused" + ("_sparse" if sparse_dx else "") + ("_xss" if x_scale_shift is not None else ""))
    else:
        orc.seen.add("head_train")
    if grad_scale_dev is not None:
        orc.seen.add("head_grad_scale_dev")
    head_check(orc, x, labels, W, b, out, compute_grad, grad_scale * (1.0 if gdev is None else gdev), stat_r,
               x_scale_shift, sparse_dx, eval_softmax)
    return out


def head_check(orc, x, labels, W, b, out, compute_grad, gsc, stat_r, x_scale_shift, sparse_dx, eval_softmax=False):
    """fp64 reference of one head_ce call (training form: loss, count, preds, dW, db, dX rows, dX statistics)"""
    NV, Cin = x.N * x.V, x.C
    Cout = W.shape[0]
    lab = labels.reshape(-1).to(torch.int64)
    idx = torch.nonzero(lab >= 0).reshape(-1)
    n = idx.numel()
    assert int(out["count"][0]) == n
    if eval_softmax:
        return
    xr = x.dense().reshape(NV, Cin)[idx]
    if x_scale_shift is not None:
        ss = x_scale_shift.double().reshape(Cin, 2)
        xg = (xr.double() * ss[:, 0] + ss[:, 1]).float().to(torch.bfloat16).double()
    else:
        xg = xr.double()
    W64, b64 = W.reshape(Cout, Cin).double(), b.double()
    y = lab[idx]
    logits = xg @ W64.t() + b64
    A_l = xg.abs() @ W64.abs().t() + b64.abs()
    e_l = ((Cin + 1) * U * A_l).max(1).values if n else A_l.sum(1)
    lse = torch.logsumexp(logits, 1)
    ly = logits.gather(1, y.view(-1, 1)).view(-1)
    lv = lse - ly
    e_lv = 2 * e_l + (Cout + 4) * U + 2 * U * (lse.abs() + ly.abs())
    kblk = _block_count_max(labels, NV) + 6
    loss_sum = lv.sum()
    e_sum = e_lv.sum() + kblk * U * lv.abs().sum()
    if n:
        orc.ratio("head:loss_sum", out["loss"][1:2], loss_sum.view(1), e_sum.view(1) + FLOOR)
        orc.ratio("head:loss_mean", out["loss"][0:1], (loss_sum / n).view(1),
                  (e_sum / n + U * (loss_sum / n).abs()).view(1) + FLOOR)
    else:
        ok = bool(torch.isnan(out["loss"][0])) and float(out["loss"][1]) == 0.0
        orc.worst["head:loss_mean"] = max(orc.worst.get("head:loss_mean", 0.0), 0.0 if ok else float("inf"))
    preds = out["preds"]
    if preds is not None:
        pf = preds.reshape(-1)
        top2 = logits.topk(min(2, Cout), 1).values if n else logits
        margin = (top2[:, 0] - top2[:, 1]) if (n and Cout > 1) else torch.full((n,), float("inf"), dtype=torch.float64,
                                                                                 device=logits.device)
        sure = margin > 2 * e_l
        ok = torch.equal(pf[idx][sure].long(), logits.argmax(1)[sure]) and bool((pf[lab < 0] == -1).all())
        orc.worst["head:preds"] = max(orc.worst.get("head:preds", 0.0), 0.0 if ok else float("inf"))
    if not compute_grad:
        return
    p = torch.softmax(logits, 1)
    onehot = F.one_hot(y, Cout).double()
    gs = gsc / n if n else 0.0
    d = (p - onehot) * gs
    e_d = abs(gs) * (p * (4 * e_l.view(-1, 1) + (Cout + 6) * U) + 2 * U * (p - onehot).abs()) + 3 * U * d.abs()
    dW_ref = d.t() @ xg
    e_dW = e_d.t() @ xg.abs() + kblk * U * (d.abs().t() @ xg.abs())
    orc.ratio("head:dW", out["dW"].reshape(Cout, Cin), dW_ref, e_dW + FLOOR)
    orc.ratio("head:db", out["db"], d.sum(0), e_d.sum(0) + kblk * U * d.abs().sum(0) + FLOOR)
    if out["dx"] is None:
        return
    dxr = out["dx"].dense().reshape(NV, Cin)
    dx_ref = d @ W64
    e_dx = e_d @ W64.abs() + Cout * U * (d.abs() @ W64.abs())
    orc.ratio("head:dx", dxr[idx], dx_ref, (2.0 ** -8) * dx_ref.abs() + (1.0 + 2.0 ** -8) * e_dx + FLOOR)
    if not sparse_dx:
        unl = lab < 0
        ok = bool((dxr[unl] == 0).all())
        orc.worst["head:dx"] = max(orc.worst["head:dx"], 0.0 if ok else float("inf"))
    if out["dx_stats"] is not None:
        g = dxr[idx].double()
        rr = stat_r.dense().reshape(NV, Cin)[idx].double()
        orc.sums("bstats_acc:head", out["dx_stats"], Cin, g, g * rr, kblk, 296)


SPIES = {
    "pack_conv_weights_multi": spy_pack_conv_weights_multi,
    "pack_conv_weights": spy_pack_conv_weights,
    "conv3d_first_fwd": spy_conv3d_first_fwd,
    "conv3d_first_fwd_gn_stats": spy_conv3d_first_fwd_gn_stats,
    "conv3d_igemm_gn_stats": spy_conv3d_igemm_gn_stats,
    "conv3d_igemm_auto": spy_conv3d_igemm_auto,
    "conv3d_dgrad_gn_bstats": spy_conv3d_dgrad_gn_bstats,
    "relu_gn_stats": spy_relu_gn_stats,
    "relu_gn_apply": spy_relu_gn_apply,
    "upcat_fwd": spy_upcat_fwd,
    "upcat_bwd": spy_upcat_bwd,
    "maxpool3d_bwd_add": spy_maxpool3d_bwd_add,
    "relu_gn_bwd_from_stats": spy_relu_gn_bwd_from_stats,
    "relu_gn_bwd": spy_relu_gn_bwd,
    "conv3d_wgrad": spy_conv3d_wgrad,
    "conv3d_wgrad_partial": spy_conv3d_wgrad_partial,
    "wgrad_reduce_multi": spy_wgrad_reduce_multi,
    "conv3d_first_wgrad": spy_conv3d_first_wgrad,
    "head_ce": spy_head_ce,
}


def install_spies(monkeypatch, orc):
    from unetsulc_b200 import ops
    real_acc = ops._acc

    def acc_spy(pool, C, device):   # remembers the accumulator a fused producer takes from the StatPool
        t = real_acc(pool, C, device)
        orc.last_acc = t
        return t

    monkeypatch.setattr(ops, "_acc", acc_spy)
    for name, spy in SPIES.items():
        monkeypatch.setattr(ops, name, functools.partial(spy, getattr(ops, name), orc))


# ------------------------------------------------------------------------------------------------ the step
COMMON = {"pack_multi", "upcat_fwd", "gn_apply", "gn_apply_pool", "wgrad", "wgrad_first"}
FUSED_B1 = COMMON | {"conv_first_stats", "conv_fprop_stats", "conv_dgrad_bstats", "maxpool_bwd_stats",
                     "gn_bwd_acc", "gn_bwd_acc_rows", "head_train_fused_sparse_xss"}
CONFIGS = {
    # name: (batch, shape, wgrad reduce mode, autograd surface, coverage set)
    "b1_24x32x40": (1, (24, 32, 40), "inline", False,
                    FUSED_B1 | {"upcat_bwd_stats_2x", "conv_fprop_splitk", "conv_dgrad_splitk", "gn_stats_pass"}),
    "b1_24x32x40_defer": (1, (24, 32, 40), "defer", False,
                          (FUSED_B1 - {"wgrad"}) | {"wgrad_defer", "upcat_bwd_stats_2x"}),
    "b1_17x26x21": (1, (17, 26, 21), "inline", False, FUSED_B1 | {"upcat_bwd_stats_non2x", "conv_fprop_splitk"}),
    "b1_23x30x19": (1, (23, 30, 19), "inline", False, FUSED_B1 | {"upcat_bwd_stats_non2x"}),
    "b1_40x48x56": (1, (40, 48, 56), "inline", False, FUSED_B1 | {"upcat_bwd_stats_2x"}),
    # level 1 (24x28x32): the Cout = 128 layers run conv3d_igemm_kernel over 168 tiles, more than the SMs, so its
    # persistent loop carries the fused statistics across tiles (at 40x48x56 only the slab kernel of level 0 does)
    "b1_48x56x64": (1, (48, 56, 64), "inline", False, FUSED_B1 | {"upcat_bwd_stats_2x"}),
    "b2_17x26x21": (2, (17, 26, 21), "inline", False,
                    COMMON | {"conv_first", "gn_stats_pass", "gn_bwd_pass", "maxpool_bwd", "upcat_bwd_non2x",
                              "head_train", "conv_fprop", "conv_dgrad"}),
    "b1_24x32x40_autograd": (1, (24, 32, 40), "inline", True,
                             COMMON | {"head_fwd", "head_train", "head_grad_scale_dev", "gn_bwd_pass", "gn_bwd_acc",
                                       "maxpool_bwd_stats", "upcat_bwd_stats_2x"}),
}


def _pair(seed=42, n_classes=56):
    """model with non-trivial GroupNorm affine parameters (as tests/test_gpu_model.py builds it)"""
    import unetsulc_b200
    torch.manual_seed(seed)
    m = unetsulc_b200.UNet3D(1, n_classes)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "norm" in name and name.endswith("weight"):
                p.add_(0.2 * torch.randn_like(p))
            if "norm" in name and name.endswith("bias"):
                p.add_(0.1 * torch.randn_like(p))
    return m.cuda().train()


def _data(B, shape, n_classes=56):
    from oracle.synth import synth_volume
    xs, ls = [], []
    for s in range(B):
        x, l = synth_volume(shape, n_classes, 1234 + s, occupancy=0.05)
        xs.append(x)
        ls.append(l)
    return torch.stack(xs).cuda(), torch.stack(ls).cuda()


def run_config(monkeypatch, name, cfg):
    from unetsulc_b200 import models
    B, shape, mode, autograd, expect = cfg
    model = _pair()
    x, labels = _data(B, shape)
    monkeypatch.setattr(models, "_WGRAD_REDUCE", mode)
    g_fb = None
    if autograd:   # gradients of the fused step, without spies
        _, _, _, g_fb = model.forward_backward(x, labels)
        g_fb = [g.clone() for g in g_fb]
        model.force_repack = True   # the spied step re-packs its weights as well
    orc = Oracle()
    install_spies(monkeypatch, orc)
    t0 = time.time()
    if autograd:
        model.zero_grad(set_to_none=True)
        loss, _ = model.loss_and_preds(x, labels)
        (2.5 * loss).backward()
        grads = [p.grad for p in model.ordered_parameters()]
    else:
        _, _, _, grads = model.forward_backward(x, labels)
    torch.cuda.synchronize()
    wall = time.time() - t0
    print("\n[%s] %d checks in %.1f s; worst error / bound:" % (name, len(orc.worst), wall))
    for op in sorted(orc.worst):
        print("    %-34s %.3e" % (op, orc.worst[op]))
    bad = {op: w for op, w in orc.worst.items() if not w <= 1.0}
    assert not bad, "ops outside their fp64 bound: %s" % bad
    missing = expect - orc.seen
    assert not missing, "entry points the step did not reach (or that lost their spy): %s" % sorted(missing)
    assert all(g is not None and bool(torch.isfinite(g).all()) for g in grads)
    if autograd:
        _compare_scaled(model, grads, g_fb, 2.5)


def _compare_scaled(model, grads, g_fb, s):
    """autograd surface with an upstream gradient s == s x the fused step.  The head gradients come from the same
    logits and differ only by the fp32 roundings of the scale (gs = s/n against 1/n, then one product per term):
    rel-L2 <= 1e-5.  The trunk gradients pass through a different (unfused) GroupNorm backward at the last layer and
    re-round every bf16 activation gradient after the scale, so they agree within the bf16 storage of the 14 layers:
    rel-L2 <= 2e-2 (the tolerance of the fused / dense autograd comparison in test_gpu_model.py)."""
    names = [n for n, _ in model.named_parameters()]
    for i, (n, a, b) in enumerate(zip(names, grads, g_fb)):
        a, b = a.double().flatten(), (s * b.double()).flatten()
        e = float((a - b).norm() / (b.norm() + 1e-30))
        assert e < (1e-5 if i >= 42 else 2e-2), (n, e)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_step_matches_fp64_per_call(monkeypatch, name):
    run_config(monkeypatch, name, CONFIGS[name])


@pytest.mark.gpu
def test_step_matches_fp64_per_call_baseline_shape(monkeypatch):
    """one batch-1 step at the BASELINE box 96 x 112 x 96 (its own function: deselect with -k 'not baseline_shape')"""
    run_config(monkeypatch, "b1_96x112x96", (1, (96, 112, 96), "inline", False, FUSED_B1 | {"upcat_bwd_stats_2x"}))


def test_fp64_references_match_torch_functional():
    """the oracle's own references (CPU, float64) == torch.nn.functional on small odd shapes"""
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 5, 4, 7, 6, generator=g, dtype=torch.float64)
    w = torch.randn(3, 5, 3, 3, 3, generator=g, dtype=torch.float64)
    assert torch.allclose(conv3d_taps(x, w), F.conv3d(x, w, padding=1), rtol=1e-12, atol=1e-12)
    wq = w.clone().requires_grad_(True)
    dy = torch.randn(2, 3, 4, 7, 6, generator=g, dtype=torch.float64)
    F.conv3d(x, wq, padding=1).backward(dy)
    assert torch.allclose(wgrad_taps(x, dy), wq.grad, rtol=1e-12, atol=1e-12)
    for din, dout in (((2, 3, 2), (4, 6, 5)), ((9, 13, 10), (19, 26, 21)), ((3, 4, 5), (6, 8, 10))):
        xi = torch.randn(1, 4, *din, generator=g, dtype=torch.float64, requires_grad=True)
        ref = F.interpolate(xi, size=dout, mode="trilinear", align_corners=False)
        assert torch.allclose(upsample_ref(xi.detach(), dout), ref, rtol=1e-12, atol=1e-12)
        gy = torch.randn(ref.shape, generator=g, dtype=torch.float64)
        ref.backward(gy)
        assert torch.allclose(upsample_adjoint_ref(gy, din), xi.grad, rtol=1e-12, atol=1e-12)
    y = torch.randn(1, 3, 5, 7, 4, generator=g, dtype=torch.float64).round()   # many ties
    yq = y.clone().requires_grad_(True)
    gp = torch.randn(1, 3, 2, 3, 2, generator=g, dtype=torch.float64)
    F.max_pool3d(yq, 2).backward(gp)
    assert torch.equal(pool_adjoint_ref(y, gp), yq.grad)
    r = torch.randn(50, 8, generator=g, dtype=torch.float64).relu()
    c = torch.randn(50, 8, generator=g, dtype=torch.float64)
    gam, bet = torch.randn(8, generator=g, dtype=torch.float64), torch.randn(8, generator=g, dtype=torch.float64)
    cq, gq, bq = c.clone().requires_grad_(True), gam.clone().requires_grad_(True), bet.clone().requires_grad_(True)
    rr = cq.relu()
    out = F.group_norm(rr.t().unsqueeze(0), 4, gq, bq, 1e-5)
    dyn = torch.randn(50, 8, generator=g, dtype=torch.float64)
    out.backward(dyn.t().unsqueeze(0))
    rd = c.relu()
    grp = rd.view(50, 4, 2)
    mu = grp.mean((0, 2)).repeat_interleave(2)
    rstd = 1.0 / torch.sqrt(grp.var((0, 2), unbiased=False) + 1e-5).repeat_interleave(2)
    dr, dgam, dbet, _, _ = groupnorm_bwd_ref(dyn, rd, mu, rstd, gam, 4)
    assert torch.allclose(dr, cq.grad, rtol=1e-10, atol=1e-12)
    assert torch.allclose(dgam, gq.grad, rtol=1e-10, atol=1e-12)
    assert torch.allclose(dbet, bq.grad, rtol=1e-10, atol=1e-12)
