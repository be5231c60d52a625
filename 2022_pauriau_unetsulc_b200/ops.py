"""Thin torch-tensor wrappers over the C-ABI (include/unetsulc_b200.h).

PyTorch here is plumbing only: device memory, the current stream, autograd bookkeeping.  Every function below
enqueues hand-written sm_100a kernels from libunetsulc_b200.so on ``torch.cuda.current_stream()``.
"""
import ctypes as C

import torch

from . import _lib

BF16 = torch.bfloat16

# Number of kernels of libunetsulc_b200.so enqueued so far (bench.py reports the delta over its timed region).
LAUNCHES = [0]
# Optional per-op CUDA-event profile: name -> list of (start_event, end_event, work) ; enabled by bench.py only.
PROFILE = None


def _count(n):
    LAUNCHES[0] += n


class _Prof(object):
    """with _Prof("igemm", flops): ...  records CUDA events on the launching stream when PROFILE is a dict."""

    def __init__(self, name, work=0.0):
        self.name, self.work = name, work

    def __enter__(self):
        if PROFILE is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            self.b.record()
            PROFILE.setdefault(self.name, []).append((self.a, self.b, self.work))
        return False


def _s():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("unetsulc_b200: tensor on %s — the B200 path has no CPU fallback" % t.device)


class Workspace(object):
    """Grow-only scratch buffer per device (the C-ABI never allocates).

    A captured CUDA graph bakes the buffer's address into its kernel nodes, so a buffer that has to be replaced by a
    larger one is RETIRED (kept alive), never freed: graphs captured earlier keep reading / writing valid, private
    scratch memory instead of memory the caching allocator may have handed to somebody else."""
    _bufs = {}
    _retired = []

    @classmethod
    def get(cls, nbytes, device, tag="ws"):
        key = (str(device), tag)
        buf = cls._bufs.get(key)
        nbytes = int(nbytes)
        if buf is None or buf.numel() < nbytes:
            if buf is not None:
                cls._retired.append(buf)
            buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
            cls._bufs[key] = buf
        return buf


_COUNTERS = {}


def _counters(device):
    """zero-initialised int32 tickets for the "last block done" reductions (the kernels leave them zero)"""
    key = str(device)
    t = _COUNTERS.get(key)
    if t is None:
        t = torch.zeros(2048, dtype=torch.int32, device=device)
        _COUNTERS[key] = t
    return t


class ActView(object):
    """A channel window [coff, coff+C) of an NDHWC bf16 buffer [N, D, H, W, ld]."""
    __slots__ = ("buf", "N", "D", "H", "W", "C", "ld", "coff")

    def __init__(self, buf, N, D, H, W, C, ld=None, coff=0):
        self.buf, self.N, self.D, self.H, self.W, self.C = buf, N, D, H, W, C
        self.ld = C if ld is None else ld
        self.coff = coff

    @property
    def V(self):
        return self.D * self.H * self.W

    @staticmethod
    def alloc(N, D, H, W, C, device, zero=False):
        f = torch.zeros if zero else torch.empty
        return ActView(f((N, D, H, W, C), dtype=BF16, device=device), N, D, H, W, C)

    def window(self, coff, C):
        return ActView(self.buf, self.N, self.D, self.H, self.W, C, self.ld, self.coff + coff)

    def dense(self):
        """[N, D, H, W, C] torch view (strided if this is a window)."""
        return self.buf.view(self.N, self.D, self.H, self.W, self.ld)[..., self.coff:self.coff + self.C]


def conv3d_igemm(x, wpack, y, cin, cout, relu, y_fp32=False):
    """x, y: ActView; wpack bf16 [27, cout, cin]."""
    lib = _lib.load()
    _need_cuda(x.buf, wpack, y.buf)
    with _Prof("conv3d_igemm", 2.0 * x.N * x.V * 27 * cin * cout):
        _lib.check(lib.b2_conv3d_igemm(_p(x.buf), x.ld, x.coff, _p(wpack), _p(y.buf), y.ld, y.coff, int(y_fp32),
                                       x.N, x.D, x.H, x.W, cin, cout, int(relu), _s()), "b2_conv3d_igemm")
    _count(1)


SPLITK_MAX_VOXELS = 8192   # below this the layer cannot fill 148 SMs with 128-voxel tiles


def conv3d_igemm_auto(x, wpack, y, cin, cout, relu):
    """conv3d_igemm that switches to the split-K path for very small volumes (the 12x14x12 level)."""
    if x.N * x.V > SPLITK_MAX_VOXELS:
        return conv3d_igemm(x, wpack, y, cin, cout, relu)
    lib = _lib.load()
    _need_cuda(x.buf, wpack, y.buf)
    ws = Workspace.get(lib.b2_conv3d_splitk_workspace_bytes(x.N, x.D, x.H, x.W, cout), x.buf.device, "splitk")
    with _Prof("conv3d_igemm", 2.0 * x.N * x.V * 27 * cin * cout):
        _lib.check(lib.b2_conv3d_igemm_splitk(_p(x.buf), x.ld, x.coff, _p(wpack), _p(y.buf), y.ld, y.coff, x.N, x.D,
                                              x.H, x.W, cin, cout, int(relu), _p(ws), ws.numel(), _s()),
                   "b2_conv3d_igemm_splitk")
    _count(2)


class StatPool(object):
    """Fixed-point GroupNorm statistics accumulators (int64 [C][4] per layer, see include/unetsulc_b200.h) carved out of
    one buffer that is zeroed with a single fill at the start of a step.  `take(C)` hands out the next slot."""
    SLOT = 512 * 4

    def __init__(self, device, slots=32):
        self.buf = torch.zeros(slots * self.SLOT, dtype=torch.int64, device=device)
        self.next = 0

    def reset(self):
        self.buf.zero_()
        self.next = 0
        _count(1)

    def take(self, C):
        if C > 512:
            raise RuntimeError("unetsulc_b200: statistics accumulators support <= 512 channels, got %d" % C)
        if (self.next + 1) * self.SLOT > self.buf.numel():
            raise RuntimeError("unetsulc_b200: StatPool exhausted (reset() it once per step)")
        t = self.buf[self.next * self.SLOT:self.next * self.SLOT + 4 * C]
        self.next += 1
        return t


def _acc(pool, C, device):
    return pool.take(C) if pool is not None else torch.zeros(4 * C, dtype=torch.int64, device=device)


def conv3d_igemm_gn_stats(x, wpack, y, cin, cout, groups, eps, gamma, beta, pool=None):
    """fprop + ReLU with the GroupNorm statistics fused into the conv epilogue (batch 1, cout <= 256): exact
    accumulators + a one-block finalize.  Returns (mean_rstd [1,C,2], scale_shift [1,C,2]) like relu_gn_stats,
    without re-reading the output tensor."""
    lib = _lib.load()
    _need_cuda(x.buf, wpack, y.buf, gamma, beta)
    acc = _acc(pool, cout, x.buf.device)
    with _Prof("conv3d_igemm", 2.0 * x.N * x.V * 27 * cin * cout):
        _lib.check(lib.b2_conv3d_igemm_stats(_p(x.buf), x.ld, x.coff, _p(wpack), _p(y.buf), y.ld, y.coff, x.N, x.D,
                                             x.H, x.W, cin, cout, 1, _p(acc), _s()), "b2_conv3d_igemm_stats")
    _count(1)
    return gn_finalize_acc(acc, x.V, cout, groups, eps, gamma, beta)


def gn_finalize_acc(acc, V, C, groups, eps, gamma, beta):
    """fixed-point accumulators int64 [C][4] -> (mean_rstd [1,C,2], scale_shift [1,C,2])"""
    lib = _lib.load()
    mean_rstd = torch.empty((1, C, 2), dtype=torch.float32, device=acc.device)
    scale_shift = torch.empty((1, C, 2), dtype=torch.float32, device=acc.device)
    _lib.check(lib.b2_relu_gn_finalize_acc(_p(acc), V, C, groups, float(eps), _p(gamma), _p(beta), _p(mean_rstd),
                                           _p(scale_shift), _s()), "b2_relu_gn_finalize_acc")
    _count(1)
    return mean_rstd, scale_shift


def conv3d_dgrad_gn_bstats(dy, wd, dx, cin, cout, r, pool=None):
    """dgrad (dy: gradient w.r.t. the conv output with `cin` channels -> dx with `cout` channels, dense) with the
    GroupNorm-backward statistics of the layer that produced dx's forward tensor fused into the epilogue.
    r: that layer's stored relu(conv) (dense ActView, `cout` channels).  Returns the accumulator tensor."""
    lib = _lib.load()
    acc = _acc(pool, cout, dy.buf.device)
    with _Prof("conv3d_igemm", 2.0 * dy.N * dy.V * 27 * cin * cout):
        _lib.check(lib.b2_conv3d_igemm_bstats(_p(dy.buf), dy.ld, dy.coff, _p(wd), _p(dx.buf), dy.N, dy.D, dy.H, dy.W,
                                              cin, cout, _p(r.buf), _p(acc), _s()), "b2_conv3d_igemm_bstats")
    _count(1)
    return acc


def relu_gn_bwd_from_stats(acc, dy, r, groups, gamma, mean_rstd, want_param_grads=True, dgamma_out=None,
                           dbeta_out=None, dy_row_labels=None):
    """GroupNorm backward using (sum dy, sum dy*r) accumulated by the kernel that produced `dy` (batch 1): a
    one-block finalize + the apply pass, no statistics pass over (dy, r)."""
    lib = _lib.load()
    dev = r.buf.device
    dr = ActView.alloc(r.N, r.D, r.H, r.W, r.C, dev)
    dgamma = dgamma_out if dgamma_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    dbeta = dbeta_out if dbeta_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    ws = Workspace.get(r.C * 16, dev, "gncoef")
    _lib.check(lib.b2_relu_gn_bwd_acc(_p(acc), _p(dy.buf), dy.ld, dy.coff, _p(r.buf), r.V, r.C, groups, _p(gamma),
                                      _p(mean_rstd), _p(dr.buf), _p(dgamma), _p(dbeta), _p(ws), ws.numel(),
                                      _p(dy_row_labels), _s()),
               "b2_relu_gn_bwd_acc")
    _count(2)
    return dr, dgamma, dbeta


# ---- layers with a conv bias (58-key checkpoints); the bias-free layers never call these ----------------------------
def conv3d_igemm_bias(x, wpack, bias, y, cin, cout, relu=True, y_fp32=False, stat_acc=None, splitk=False):
    """fprop of a biased layer: bias fp32 [cout] is added to the accumulator before ReLU.  stat_acc: fixed-point
    statistics accumulators (batch 1, see conv3d_igemm_gn_stats); splitk: allow the split-K path on tiny volumes."""
    lib = _lib.load()
    _need_cuda(x.buf, wpack, y.buf, bias)
    if not bias.is_contiguous() or bias.data_ptr() % 8:
        bias = bias.contiguous().clone()
    ws = None
    if splitk and stat_acc is None and not y_fp32 and x.N * x.V <= SPLITK_MAX_VOXELS:
        ws = Workspace.get(lib.b2_conv3d_splitk_workspace_bytes(x.N, x.D, x.H, x.W, cout), x.buf.device, "splitk")
    with _Prof("conv3d_igemm", 2.0 * x.N * x.V * 27 * cin * cout):
        _lib.check(lib.b2_conv3d_igemm_bias(_p(x.buf), x.ld, x.coff, _p(wpack), _p(y.buf), y.ld, y.coff, int(y_fp32),
                                            x.N, x.D, x.H, x.W, cin, cout, int(relu), _p(bias), _p(stat_acc), _p(ws),
                                            ws.numel() if ws is not None else 0, _s()), "b2_conv3d_igemm_bias")
    _count(2 if ws is not None else 1)


def conv3d_first_fwd_bias(x, w, bias, y, relu=True, stat_acc=None):
    """first conv (Cin = 1) + bias + ReLU; stat_acc: fused GroupNorm statistics (batch 1)"""
    lib = _lib.load()
    _need_cuda(x, w, bias, y.buf)
    _lib.check(lib.b2_conv3d_first_fwd_bias(_p(x), _p(w), _p(bias), _p(y.buf), y.ld, y.coff, y.N, y.D, y.H, y.W,
                                            w.shape[0], int(relu), _p(stat_acc), _s()), "b2_conv3d_first_fwd_bias")
    _count(1)


def _dbias_acc(pool, C, device):
    """int64 [C][2] zeroed dbias accumulators (half of a StatPool slot)"""
    return (pool.take(C) if pool is not None else torch.zeros(4 * C, dtype=torch.int64, device=device))[:2 * C]


def relu_gn_bwd_from_stats_dbias(acc, dy, r, groups, gamma, mean_rstd, want_param_grads=True, dgamma_out=None,
                                 dbeta_out=None, dy_row_labels=None, dbias_out=None, pool=None):
    """relu_gn_bwd_from_stats that also returns the conv-bias gradient sum_v dr (fp32 [C], into dbias_out if given).
    Returns (dr, dgamma, dbeta, dbias)."""
    lib = _lib.load()
    dev = r.buf.device
    dr = ActView.alloc(r.N, r.D, r.H, r.W, r.C, dev)
    dgamma = dgamma_out if dgamma_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    dbeta = dbeta_out if dbeta_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    dbias = dbias_out if dbias_out is not None else torch.empty(r.C, dtype=torch.float32, device=dev)
    dacc = _dbias_acc(pool, r.C, dev)
    ws = Workspace.get(r.C * 16, dev, "gncoef")
    _lib.check(lib.b2_relu_gn_bwd_acc_dbias(_p(acc), _p(dy.buf), dy.ld, dy.coff, _p(r.buf), r.V, r.C, groups,
                                            _p(gamma), _p(mean_rstd), _p(dr.buf), _p(dgamma), _p(dbeta), _p(ws),
                                            ws.numel(), _p(dy_row_labels), _p(dacc), _p(dbias), _s()),
               "b2_relu_gn_bwd_acc_dbias")
    _count(3)
    return dr, dgamma, dbeta, dbias


def relu_gn_bwd_dbias(dy, r, groups, gamma, mean_rstd, want_param_grads=True, dgamma_out=None, dbeta_out=None,
                      dbias_out=None):
    """relu_gn_bwd that also returns the conv-bias gradient (summed over the samples).  Returns (dr, dgamma, dbeta,
    dbias)."""
    lib = _lib.load()
    dev = r.buf.device
    dr = ActView.alloc(r.N, r.D, r.H, r.W, r.C, dev)
    dgamma = dgamma_out if dgamma_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    dbeta = dbeta_out if dbeta_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    dbias = dbias_out if dbias_out is not None else torch.empty(r.C, dtype=torch.float32, device=dev)
    dacc = _dbias_acc(None, r.C, dev)
    ws = Workspace.get(lib.b2_relu_gn_bwd_workspace_bytes(r.N, r.C), dev, "gn")
    _lib.check(lib.b2_relu_gn_bwd_dbias(_p(dy.buf), dy.ld, dy.coff, _p(r.buf), r.N, r.V, r.C, groups, _p(gamma),
                                        _p(mean_rstd), _p(dr.buf), _p(dgamma), _p(dbeta), _p(ws), ws.numel(),
                                        _p(_counters(dev)), _p(dacc), _p(dbias), _s()), "b2_relu_gn_bwd_dbias")
    _count(4)   # zero fill of the accumulators, statistics, apply, dbias finalize
    return dr, dgamma, dbeta, dbias


def conv3d_wgrad(x, dy, cin, cout, out=None):
    """returns dW fp32 [cout, cin, 3, 3, 3] (written into `out` when given)"""
    lib = _lib.load()
    _need_cuda(x.buf, dy.buf)
    need = lib.b2_conv3d_wgrad_workspace_bytes(x.N, x.D, x.H, x.W, cin, cout)
    if need < 0:
        raise RuntimeError("b2_conv3d_wgrad: unsupported shape Cin=%d Cout=%d" % (cin, cout))
    ws = Workspace.get(need, x.buf.device, "wgrad")
    dw = out if out is not None else torch.empty((cout, cin, 3, 3, 3), dtype=torch.float32, device=x.buf.device)
    with _Prof("conv3d_wgrad", 2.0 * x.N * x.V * 27 * cin * cout):
        _lib.check(lib.b2_conv3d_wgrad(_p(x.buf), x.ld, x.coff, _p(dy.buf), dy.ld, dy.coff, _p(dw), _p(ws),
                                       ws.numel(), x.N, x.D, x.H, x.W, cin, cout, _s()), "b2_conv3d_wgrad")
    _count(2)
    return dw


def conv3d_wgrad_partial(x, dy, cin, cout, slot, out=None):
    """The tensor-core half of conv3d_wgrad: split partials stay in the workspace of `slot` (one per layer) until
    wgrad_reduce_multi() runs.  Returns the descriptor to hand to it; desc["dw"] is the (not yet valid) gradient."""
    lib = _lib.load()
    _need_cuda(x.buf, dy.buf)
    need = lib.b2_conv3d_wgrad_workspace_bytes(x.N, x.D, x.H, x.W, cin, cout)
    if need < 0:
        raise RuntimeError("b2_conv3d_wgrad: unsupported shape Cin=%d Cout=%d" % (cin, cout))
    ws = Workspace.get(need, x.buf.device, "wgrad_p%s" % slot)
    dw = out if out is not None else torch.empty((cout, cin, 3, 3, 3), dtype=torch.float32, device=x.buf.device)
    splits, swapped = C.c_int(0), C.c_int(0)
    with _Prof("conv3d_wgrad", 2.0 * x.N * x.V * 27 * cin * cout):
        _lib.check(lib.b2_conv3d_wgrad_partial(_p(x.buf), x.ld, x.coff, _p(dy.buf), dy.ld, dy.coff, _p(ws), ws.numel(),
                                               x.N, x.D, x.H, x.W, cin, cout, C.byref(splits), C.byref(swapped), _s()),
                   "b2_conv3d_wgrad_partial")
    _count(1)
    return dict(ws=ws, dw=dw, splits=splits.value, swapped=swapped.value, cin=cin, cout=cout)


def wgrad_reduce_multi(descs):
    """one launch: dW of every pending layer (descriptors of conv3d_wgrad_partial) from its split partials"""
    n = len(descs)
    if n == 0:
        return
    lib = _lib.load()
    vp, ia = C.c_void_p * n, C.c_int * n
    _lib.check(lib.b2_wgrad_reduce_multi(vp(*[d["ws"].data_ptr() for d in descs]), vp(*[d["dw"].data_ptr() for d in descs]),
                                         ia(*[d["splits"] for d in descs]), ia(*[d["cin"] for d in descs]),
                                         ia(*[d["cout"] for d in descs]), ia(*[d["swapped"] for d in descs]), n, _s()),
               "b2_wgrad_reduce_multi")
    _count((n + 15) // 16)


def conv3d_first_fwd(x, w, y, relu=True):
    """x fp32 [N, 1, D, H, W] contiguous; w fp32 [cout, 1, 3, 3, 3]; y ActView"""
    lib = _lib.load()
    _need_cuda(x, w, y.buf)
    _lib.check(lib.b2_conv3d_first_fwd(_p(x), _p(w), _p(y.buf), y.ld, y.coff, y.N, y.D, y.H, y.W, w.shape[0],
                                       int(relu), _s()), "b2_conv3d_first_fwd")
    _count(1)


def conv3d_first_fwd_gn_stats(x, w, y, groups, eps, gamma, beta, pool=None):
    """first conv + ReLU with the GroupNorm statistics fused in (batch 1).  Returns (mean_rstd, scale_shift)."""
    lib = _lib.load()
    _need_cuda(x, w, y.buf, gamma, beta)
    cout = w.shape[0]
    acc = _acc(pool, cout, x.device)
    _lib.check(lib.b2_conv3d_first_fwd_stats(_p(x), _p(w), _p(y.buf), y.ld, y.coff, y.N, y.D, y.H, y.W, cout, 1,
                                             _p(acc), _s()), "b2_conv3d_first_fwd_stats")
    _count(1)
    return gn_finalize_acc(acc, y.V, cout, groups, eps, gamma, beta)


def conv3d_first_wgrad(x, dy, cout, out=None):
    lib = _lib.load()
    _need_cuda(x, dy.buf)
    need = lib.b2_conv3d_first_wgrad_workspace_bytes(cout)
    ws = Workspace.get(need, x.device, "wgrad")
    dw = out if out is not None else torch.empty((cout, 1, 3, 3, 3), dtype=torch.float32, device=x.device)
    _lib.check(lib.b2_conv3d_first_wgrad(_p(x), _p(dy.buf), dy.ld, dy.coff, _p(dw), _p(ws), ws.numel(), dy.N, dy.D,
                                         dy.H, dy.W, cout, _s()), "b2_conv3d_first_wgrad")
    _count(2)
    return dw


def relu_gn_stats(r, groups, eps, gamma, beta):
    """r: dense ActView (post-ReLU conv output).  Returns (mean_rstd [N,C,2], scale_shift [N,C,2]) fp32."""
    lib = _lib.load()
    _need_cuda(r.buf, gamma, beta)
    dev = r.buf.device
    mean_rstd = torch.empty((r.N, r.C, 2), dtype=torch.float32, device=dev)
    scale_shift = torch.empty((r.N, r.C, 2), dtype=torch.float32, device=dev)
    ws = Workspace.get(lib.b2_gn_workspace_bytes(r.N, r.C), dev, "gn")
    _lib.check(lib.b2_relu_gn_stats(_p(r.buf), r.N, r.V, r.C, groups, float(eps), _p(gamma), _p(beta), _p(mean_rstd),
                                    _p(scale_shift), _p(ws), ws.numel(), _p(_counters(dev)), _s()),
               "b2_relu_gn_stats")
    _count(1)
    return mean_rstd, scale_shift


def relu_gn_apply(r, scale_shift, y, pooled=None):
    lib = _lib.load()
    _lib.check(lib.b2_relu_gn_apply(_p(r.buf), r.N, r.D, r.H, r.W, r.C, _p(scale_shift), _p(y.buf), y.ld, y.coff,
                                    _p(pooled.buf) if pooled is not None else C.c_void_p(0), _s()),
               "b2_relu_gn_apply")
    _count(1)


def relu_gn_bwd(dy, r, groups, gamma, mean_rstd, want_param_grads=True, dgamma_out=None, dbeta_out=None):
    """dy: ActView (any window); r dense.  Returns (dr ActView dense, dgamma, dbeta)."""
    lib = _lib.load()
    dev = r.buf.device
    dr = ActView.alloc(r.N, r.D, r.H, r.W, r.C, dev)
    dgamma = dgamma_out if dgamma_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    dbeta = dbeta_out if dbeta_out is not None else (
        torch.empty(r.C, dtype=torch.float32, device=dev) if want_param_grads else None)
    ws = Workspace.get(lib.b2_relu_gn_bwd_workspace_bytes(r.N, r.C), dev, "gn")
    _lib.check(lib.b2_relu_gn_bwd(_p(dy.buf), dy.ld, dy.coff, _p(r.buf), r.N, r.V, r.C, groups, _p(gamma),
                                  _p(mean_rstd), _p(dr.buf), _p(dgamma), _p(dbeta), _p(ws), ws.numel(),
                                  _p(_counters(dev)), _s()),
               "b2_relu_gn_bwd")
    _count(2)
    return dr, dgamma, dbeta


def maxpool3d_bwd_add(y, dskip, dpool, stat_r=None, pool=None):
    """y: forward tensor window (pre-pool); dskip: ActView or None; dpool: dense ActView at half res.
    stat_r (batch 1): the saved relu(conv) of the layer whose output gradient this is — the kernel then also
    accumulates that layer's GroupNorm-backward statistics; returns (out, acc) instead of out."""
    lib = _lib.load()
    out = ActView.alloc(y.N, y.D, y.H, y.W, y.C, y.buf.device)
    args = (_p(y.buf), y.ld, y.coff, _p(dskip.buf) if dskip is not None else C.c_void_p(0),
            dskip.ld if dskip is not None else 8, dskip.coff if dskip is not None else 0,
            _p(dpool.buf), _p(out.buf), y.N, y.D, y.H, y.W, y.C)
    if stat_r is not None:
        acc = _acc(pool, y.C, y.buf.device)
        _lib.check(lib.b2_maxpool3d_bwd_add_bstats(*(args + (_p(stat_r.buf), _p(acc), _s()))),
                   "b2_maxpool3d_bwd_add_bstats")
        _count(1)
        return out, acc
    _lib.check(lib.b2_maxpool3d_bwd_add(*(args + (_s(),))), "b2_maxpool3d_bwd_add")
    _count(1)
    return out


def upcat_fwd(x, cat_window):
    lib = _lib.load()
    c = cat_window
    _lib.check(lib.b2_upcat_fwd(_p(x.buf), x.N, x.D, x.H, x.W, x.C, _p(c.buf), c.ld, c.coff, c.D, c.H, c.W, _s()),
               "b2_upcat_fwd")
    _count(1)


def upcat_bwd(dcat_window, Di, Hi, Wi, separable=True, stat_r=None, pool=None):
    """adjoint of the trilinear upsample.  stat_r (batch 1, separable): see maxpool3d_bwd_add; returns (dx, acc)."""
    lib = _lib.load()
    c = dcat_window
    dx = ActView.alloc(c.N, Di, Hi, Wi, c.C, c.buf.device)
    if separable:
        ws = Workspace.get(lib.b2_upcat_bwd_workspace_bytes(c.N, c.D, c.H, Wi, c.C), c.buf.device, "upbwd")
        # exact 2x levels run the single-pass stencil kernel (one launch), other ratios the two separable passes
        n_launch = 1 if (c.D == 2 * Di and c.H == 2 * Hi and c.W == 2 * Wi and c.C % 64 == 0) else 2
        if stat_r is not None:
            acc = _acc(pool, c.C, c.buf.device)
            _lib.check(lib.b2_upcat_bwd_separable_bstats(_p(c.buf), c.ld, c.coff, c.N, c.D, c.H, c.W, _p(dx.buf), Di,
                                                         Hi, Wi, c.C, _p(ws), ws.numel(), _p(stat_r.buf), _p(acc),
                                                         _s()), "b2_upcat_bwd_separable_bstats")
            _count(n_launch)
            return dx, acc
        _lib.check(lib.b2_upcat_bwd_separable(_p(c.buf), c.ld, c.coff, c.N, c.D, c.H, c.W, _p(dx.buf), Di, Hi, Wi,
                                              c.C, _p(ws), ws.numel(), _s()), "b2_upcat_bwd_separable")
        _count(n_launch)
    else:
        _lib.check(lib.b2_upcat_bwd(_p(c.buf), c.ld, c.coff, c.N, c.D, c.H, c.W, _p(dx.buf), Di, Hi, Wi, c.C, _s()),
                   "b2_upcat_bwd")
        _count(1)
    return dx


def head_ce(x, labels, W, b, compute_grad, eval_softmax=False, grad_scale=1.0, grad_scale_dev=None,
            want_preds=True, want_dx=True, dW_out=None, db_out=None, stat_r=None, pool=None, x_scale_shift=None,
            sparse_dx=False):
    """x: dense ActView [N,D,H,W,Cin]; labels int64 [N,D,H,W] (-1 = ignore).
    x_scale_shift (batch 1): x is the last layer's relu(conv) and its GroupNorm apply is deferred to this kernel
    (performed on the labelled rows only).
    sparse_dx (with stat_r): dx is not cleared, only the rows of labelled voxels are written; hand `labels` to
    relu_gn_bwd_from_stats(dy_row_labels=...) so that the other rows read as zero.
    Returns dict(loss [2] fp32 (mean, sum), count int32 [1], preds int32 [N,D,H,W] or None, dx ActView, dW, db)."""
    lib = _lib.load()
    _need_cuda(x.buf, labels, W, b)
    dev = x.buf.device
    cout, cin = W.shape[0], W.shape[1]
    if labels.dtype != torch.int64 or not labels.is_contiguous():
        labels = labels.to(torch.int64).contiguous()
    NV = x.N * x.V
    loss = torch.empty(2, dtype=torch.float32, device=dev)
    count = torch.empty(1, dtype=torch.int32, device=dev)
    preds = torch.full((x.N, x.D, x.H, x.W), -1, dtype=torch.int32, device=dev) if want_preds else None
    dx = ActView.alloc(x.N, x.D, x.H, x.W, cin, dev) if (compute_grad and want_dx) else None
    dW = (dW_out if dW_out is not None else torch.empty_like(W, dtype=torch.float32)) if compute_grad else None
    db = (db_out if db_out is not None else torch.empty(cout, dtype=torch.float32, device=dev)) if compute_grad else None
    ws = Workspace.get(lib.b2_head_workspace_bytes(cin), dev, "head")
    Wc = W.reshape(cout, cin)
    if not Wc.is_contiguous():
        Wc = Wc.contiguous()
    dx_stats = None
    if stat_r is not None and dx is not None and not eval_softmax:
        # dx is the gradient at the last GroupNorm output: its backward statistics come out of this kernel too
        dx_stats = _acc(pool, cin, dev)
        _lib.check(lib.b2_head_ce_bstats(_p(x.buf), _p(labels), NV, _p(Wc), _p(b), cin, cout, float(grad_scale),
                                         _p(grad_scale_dev), _p(preds), _p(dx.buf), _p(dW), _p(db), _p(loss),
                                         _p(count), _p(ws), ws.numel(), _p(stat_r.buf), _p(dx_stats),
                                         _p(x_scale_shift), int(bool(sparse_dx)), _s()),
                   "b2_head_ce_bstats")
    else:
        _lib.check(lib.b2_head_ce(_p(x.buf), _p(labels), NV, _p(Wc), _p(b), cin, cout, float(grad_scale),
                                  _p(grad_scale_dev), int(compute_grad), int(eval_softmax), _p(preds),
                                  _p(dx.buf) if dx is not None else C.c_void_p(0), _p(dW), _p(db), _p(loss), _p(count),
                                  _p(ws), ws.numel(), _p(x_scale_shift), _s()), "b2_head_ce")
    _count(3)
    return dict(loss=loss, count=count, preds=preds, dx=dx, dW=dW, db=db, dx_stats=dx_stats,
                dx_row_labels=labels if (sparse_dx and dx_stats is not None) else None)


def head_gather(x, index, W, b, softmax=True, x_scale_shift=None):
    """index: int64 linear voxel indices into [N*D*H*W].  Returns (scores fp32 [n, cout], preds int32 [n]).
    x_scale_shift: see head_ce."""
    lib = _lib.load()
    dev = x.buf.device
    cout, cin = W.shape[0], W.shape[1]
    n = index.numel()
    scores = torch.empty((n, cout), dtype=torch.float32, device=dev)
    preds = torch.empty(n, dtype=torch.int32, device=dev)
    Wc = W.reshape(cout, cin).contiguous()
    _lib.check(lib.b2_head_gather(_p(x.buf), _p(index), n, _p(Wc), _p(b), cin, cout, int(softmax), _p(scores),
                                  _p(preds), _p(x_scale_shift), _s()), "b2_head_gather")
    _count(1)
    return scores, preds


def head_dense_fwd(x, W, b, softmax):
    lib = _lib.load()
    dev = x.buf.device
    cout, cin = W.shape[0], W.shape[1]
    out = torch.empty((x.N, cout, x.D, x.H, x.W), dtype=torch.float32, device=dev)
    Wc = W.reshape(cout, cin).contiguous()
    _lib.check(lib.b2_head_dense_fwd(_p(x.buf), x.N, x.V, _p(Wc), _p(b), cin, cout, int(softmax), _p(out), _s()),
               "b2_head_dense_fwd")
    _count(1)
    return out


def head_dense_bwd(g, x, W):
    """g fp32 [N, cout, D, H, W] contiguous.  Returns (dx ActView, dW, db)."""
    lib = _lib.load()
    dev = x.buf.device
    cout, cin = W.shape[0], W.shape[1]
    g = g.contiguous().float()
    dx = ActView.alloc(x.N, x.D, x.H, x.W, cin, dev)
    dW = torch.empty_like(W, dtype=torch.float32)
    db = torch.empty(cout, dtype=torch.float32, device=dev)
    ws = Workspace.get(lib.b2_head_workspace_bytes(cin), dev, "head")
    Wc = W.reshape(cout, cin).contiguous()
    _lib.check(lib.b2_head_dense_bwd(_p(g), _p(x.buf), x.N, x.V, _p(Wc), cin, cout, _p(dx.buf), _p(dW), _p(db),
                                     _p(ws), ws.numel(), _s()), "b2_head_dense_bwd")
    _count(2)
    return dx, dW, db


def sgd_step(params, grads, moms, lr, momentum, grad_scale=1.0):
    lib = _lib.load()
    n = len(params)
    if n == 0:
        return
    arr = C.c_void_p * n
    ll = C.c_longlong * n
    P = arr(*[p.data_ptr() for p in params])
    G = arr(*[g.data_ptr() for g in grads])
    M = arr(*[m.data_ptr() for m in moms])
    Nn = ll(*[p.numel() for p in params])
    _lib.check(lib.b2_sgd_step(P, G, M, Nn, n, float(lr), float(momentum), float(grad_scale), _s()), "b2_sgd_step")
    _count((n + 63) // 64)


def pack_conv_weights(w, want_dgrad=True):
    """w fp32 [cout, cin, 3, 3, 3] -> (wf bf16 [27, cout, cin], wd bf16 [27, cin, cout])"""
    lib = _lib.load()
    _need_cuda(w)
    cout, cin = w.shape[0], w.shape[1]
    wf = torch.empty((27, cout, cin), dtype=BF16, device=w.device)
    wd = torch.empty((27, cin, cout), dtype=BF16, device=w.device) if want_dgrad else None
    wc = w.detach()
    if not wc.is_contiguous():
        wc = wc.contiguous()
    _lib.check(lib.b2_pack_conv_weights(_p(wc), _p(wf), _p(wd), cout, cin, _s()), "b2_pack_conv_weights")
    _count(1)
    return wf, wd


def pack_conv_weights_multi(ws):
    """ws: list of fp32 [cout, cin, 3, 3, 3] CUDA tensors -> list of (wf, wd), one kernel launch for all of them."""
    lib = _lib.load()
    n = len(ws)
    if n == 0:
        return []
    outs, W, WF, WD, CO, CI = [], [], [], [], [], []
    keep = []
    for w in ws:
        _need_cuda(w)
        cout, cin = w.shape[0], w.shape[1]
        wc = w.detach()
        if not wc.is_contiguous():
            wc = wc.contiguous()
        keep.append(wc)
        wf = torch.empty((27, cout, cin), dtype=BF16, device=w.device)
        wd = torch.empty((27, cin, cout), dtype=BF16, device=w.device)
        outs.append((wf, wd))
        W.append(wc.data_ptr()); WF.append(wf.data_ptr()); WD.append(wd.data_ptr()); CO.append(cout); CI.append(cin)
    vp, ia = C.c_void_p * n, C.c_int * n
    _lib.check(lib.b2_pack_conv_weights_multi(vp(*W), vp(*WF), vp(*WD), ia(*CO), ia(*CI), n, _s()),
               "b2_pack_conv_weights_multi")
    _count((n + 15) // 16)
    return outs


def scatter_volume(points, point_labels, size, device, background=-1):
    """points: int array-like [n, 3] (host), point_labels: int [n] (host), size: (D, H, W).
    Returns (x fp32 [1, D, H, W], labels int64 [D, H, W]) on `device`, identical to the reference's CPU index_put
    (last duplicate wins); 16 bytes per point are copied to the device instead of 12 bytes per voxel."""
    import numpy as np
    lib = _lib.load()
    D, H, W = int(size[0]), int(size[1]), int(size[2])
    pts = np.ascontiguousarray(np.asarray(points, dtype=np.int32).reshape(-1, 3))
    lab = np.ascontiguousarray(np.asarray(point_labels, dtype=np.int32).reshape(-1))
    n = pts.shape[0]
    if n and (pts.min() < 0 or (pts.max(axis=0) >= np.array([D, H, W])).any()):
        raise IndexError("scatter_volume: point outside the %dx%dx%d volume" % (D, H, W))
    x = torch.empty((1, D, H, W), dtype=torch.float32, device=device)
    labels = torch.empty((D, H, W), dtype=torch.int64, device=device)
    ws = Workspace.get(lib.b2_scatter_volume_workspace_bytes(D, H, W), x.device, "scatter")
    packed = torch.from_numpy(np.concatenate([pts.reshape(-1), lab])).to(device, non_blocking=True) if n else None
    _lib.check(lib.b2_scatter_volume(_p(packed), C.c_void_p(packed.data_ptr() + 12 * n) if n else C.c_void_p(0), n,
                                     D, H, W, _p(x), _p(labels), int(background), _p(ws), ws.numel(), _s()),
               "b2_scatter_volume")
    _count(3 if n else 1)
    return x, labels


class ResidentPoints(object):
    """A subject's point list: base points (minus their minimum) int32 [n,3] + label ids int32 [n], held in pinned
    host memory and — after the first `on(device)` with keep=True — on the device."""
    __slots__ = ("h_pts", "h_lab", "n", "pts", "lab")

    def __init__(self, pts_host, lab_host):
        import numpy as np
        pts = np.ascontiguousarray(np.asarray(pts_host, dtype=np.int32).reshape(-1, 3))
        lab = np.ascontiguousarray(np.asarray(lab_host, dtype=np.int32).reshape(-1))
        self.n = pts.shape[0]
        self.h_pts, self.h_lab = torch.from_numpy(pts), torch.from_numpy(lab)
        if torch.cuda.is_available():
            self.h_pts, self.h_lab = self.h_pts.pin_memory(), self.h_lab.pin_memory()
        self.pts = self.lab = None

    def on(self, device, keep=True):
        """(pts, lab) on `device`; keep=False uploads them again on every call (16 bytes per point, asynchronous)"""
        if self.pts is not None and self.pts.device == torch.device(device):
            return self.pts, self.lab
        pts = self.h_pts.to(device, non_blocking=True)
        lab = self.h_lab.to(device, non_blocking=True)
        if keep:
            self.pts, self.lab = pts, lab
        return pts, lab


_OOB = {}


def oob_counter(device):
    """device int32 [1]: points that fell outside their volume since the last check (see scatter_volume_rot)"""
    key = str(torch.device(device))
    t = _OOB.get(key)
    if t is None:
        t = _OOB[key] = torch.zeros(1, dtype=torch.int32, device=device)
    return t


def check_oob(device):
    """One D2H read: raises IndexError (what the reference's index_put raises per sample) if any point of the samples
    built since the last check fell outside its volume."""
    t = _OOB.get(str(torch.device(device)))
    if t is None:
        return
    n = int(t.item())
    if n:
        t.zero_()
        raise IndexError("scatter_volume: %d point(s) outside the volume (img_size too small for the rotated "
                         "skeleton)" % n)


def scatter_volume_rot(res, xform, size, device, background=-1, keep=True):
    """res: ResidentPoints; xform: 12 floats (R row-major, t) or None for the identity; size: (D, H, W).
    Returns (x fp32 [1, D, H, W], labels int64 [D, H, W]): the dense volumes of the rotated, truncated, min-shifted
    point list (reference dataset.py:33-43, 66-88), built entirely on the device.  keep: see ResidentPoints.on."""
    lib = _lib.load()
    D, H, W = int(size[0]), int(size[1]), int(size[2])
    dev = torch.device(device)
    pts, lab = res.on(dev, keep)
    x = torch.empty((1, D, H, W), dtype=torch.float32, device=dev)
    labels = torch.empty((D, H, W), dtype=torch.int64, device=dev)
    ws = Workspace.get(lib.b2_scatter_volume_rot_workspace_bytes(res.n, D, H, W), dev, "scatter")
    if xform is None:
        xform = (1., 0., 0., 0., 1., 0., 0., 0., 1., 0., 0., 0.)
    xf = (C.c_double * 12)(*[float(v) for v in xform])
    _lib.check(lib.b2_scatter_volume_rot(_p(pts), _p(lab), res.n, xf, D, H, W, _p(x), _p(labels),
                                         int(background), _p(oob_counter(dev)), _p(ws), ws.numel(), _s()),
               "b2_scatter_volume_rot")
    _count(5 if res.n else 1)
    return x, labels


def step_metrics(labels, preds, n_classes, counts, loss=None, loss_weight=1.0, loss_acc=None):
    """labels int64 [...], preds int32 [...] (same numel); counts int64 [3, n_classes] += TP/FP/FN over the labelled
    voxels; loss_acc float64 [2] += (loss[0] * loss_weight, loss_weight).  No host synchronisation."""
    lib = _lib.load()
    _need_cuda(labels, preds, counts)
    if labels.dtype != torch.int64 or not labels.is_contiguous():
        labels = labels.to(torch.int64).contiguous()
    if preds.dtype != torch.int32 or not preds.is_contiguous():
        preds = preds.to(torch.int32).contiguous()
    _lib.check(lib.b2_step_metrics(_p(labels), _p(preds), labels.numel(), n_classes, _p(counts), _p(loss),
                                   float(loss_weight), _p(loss_acc), _s()), "b2_step_metrics")
    _count(1)


def fold_vote(scores, fold_dense, n_folds, thresholds):
    """scores fp32 [n, C] cuda; fold_dense int32 [n] in [0, n_folds); thresholds: list of ints.
    Returns int32 [T, n]."""
    lib = _lib.load()
    _need_cuda(scores, fold_dense)
    dev = scores.device
    n, Cc = scores.shape
    T = len(thresholds)
    out = torch.empty((T, n), dtype=torch.int32, device=dev)
    if n == 0:
        return out
    th = torch.tensor(list(thresholds), dtype=torch.int32, device=dev)
    ws = Workspace.get(lib.b2_fold_vote_workspace_bytes(n, Cc, n_folds, T), dev, "vote")
    _lib.check(lib.b2_fold_vote(_p(scores.contiguous()), _p(fold_dense.contiguous()), n, Cc, n_folds, _p(th), T,
                                _p(out), _p(ws), ws.numel(), _s()), "b2_fold_vote")
    _count(3)
    return out


def match_voxels(pts_a, pts_b, val_b):
    """pts_a, pts_b: int32 cuda [n, 3] (same voxel set, two orders); val_b int32 cuda [n].  Returns int32 [n]:
    val_b re-ordered to list a by pairing equal ranks of the stable (x, y, z) sorts (pattern_class.py:205-228)."""
    lib = _lib.load()
    _need_cuda(pts_a, pts_b, val_b)
    n = pts_a.shape[0]
    out = torch.empty(n, dtype=torch.int32, device=pts_a.device)
    if n == 0:
        return out
    ws = Workspace.get(lib.b2_match_voxels_workspace_bytes(n), pts_a.device, "match")
    _lib.check(lib.b2_match_voxels(_p(pts_a.contiguous()), _p(pts_b.contiguous()), _p(val_b.contiguous()), n, _p(out),
                                   _p(ws), ws.numel(), _s()), "b2_match_voxels")
    _count(5)
    return out


def esi_counts(y_true, y_pred, n_classes, counts=None):
    """int32 cuda vectors -> uint64-valued int64 tensor [3, n_classes] (TP, FP, FN), accumulated into `counts`."""
    lib = _lib.load()
    _need_cuda(y_true, y_pred)
    if counts is None:
        counts = torch.zeros((3, n_classes), dtype=torch.int64, device=y_true.device)
    _lib.check(lib.b2_esi_counts(_p(y_true.contiguous()), _p(y_pred.contiguous()), y_true.numel(), n_classes,
                                 _p(counts), _s()), "b2_esi_counts")
    _count(1)
    return counts


# ---------------------------------------------------------------------------------------------------- exact inference
F32 = torch.float32


def exact_split3(x, ld, off, C, D, H, W):
    """fp32 [V, ld] channel window [off, off + C) -> ActView bf16 [1, D, H, W, 3C] = [hi | lo | hi]"""
    lib = _lib.load()
    V = D * H * W
    out = ActView.alloc(1, D, H, W, 3 * C, x.device)
    _lib.check(lib.b2_exact_split3(_p(x), V, C, ld, off, _p(out.buf), _s()), "b2_exact_split3")
    _count(1)
    return out


def exact_split_first(x, D, H, W):
    """network input fp32 [1, 1, D, H, W] -> ActView bf16 [1, D, H, W, 32] = [hi, hi, lo, 0 ...]"""
    lib = _lib.load()
    out = ActView.alloc(1, D, H, W, 32, x.device)
    _lib.check(lib.b2_exact_split_first(_p(x), D * H * W, _p(out.buf), _s()), "b2_exact_split_first")
    _count(1)
    return out


def exact_conv(xsplit, wpack, cin3, cout, relu=True):
    """split-operand 3x3x3 conv on the tcgen05 implicit-GEMM kernel, fp32 output [V, cout] (+ ReLU)"""
    dev = xsplit.buf.device
    r = torch.empty((xsplit.V, cout), dtype=F32, device=dev)
    y = ActView(r, 1, xsplit.D, xsplit.H, xsplit.W, cout)
    conv3d_igemm(xsplit, wpack, y, cin3, cout, relu=relu, y_fp32=True)
    return r


def exact_conv_bias(xsplit, wpack, bias, cin3, cout, relu=True):
    """exact_conv of a biased layer: the fp32 bias joins the fp32 accumulator before ReLU"""
    dev = xsplit.buf.device
    r = torch.empty((xsplit.V, cout), dtype=F32, device=dev)
    y = ActView(r, 1, xsplit.D, xsplit.H, xsplit.W, cout)
    conv3d_igemm_bias(xsplit, wpack, bias, y, cin3, cout, relu=relu, y_fp32=True)
    return r


def exact_gn(r, groups, eps, gamma, beta, out, ld, off):
    """GroupNorm(groups, C) of the fp32 [V, C] tensor r (fp64 statistics) written to out[:, off:off+C] (fp32 [V, ld])"""
    lib = _lib.load()
    V, Cc = r.shape
    ss = torch.empty((Cc, 2), dtype=F32, device=r.device)
    ws = Workspace.get(lib.b2_exact_gn_workspace_bytes(Cc), r.device, "exgn")
    _lib.check(lib.b2_exact_gn_stats(_p(r), V, Cc, groups, float(eps), _p(gamma), _p(beta), _p(ss), _p(ws), ws.numel(),
                                     _s()), "b2_exact_gn_stats")
    _lib.check(lib.b2_exact_gn_apply(_p(r), V, Cc, _p(ss), _p(out), ld, off, _s()), "b2_exact_gn_apply")
    _count(3)


def exact_maxpool(x, ld, off, C, D, H, W):
    lib = _lib.load()
    y = torch.empty(((D // 2) * (H // 2) * (W // 2), C), dtype=F32, device=x.device)
    _lib.check(lib.b2_exact_maxpool(_p(x), 1, D, H, W, C, ld, off, _p(y), _s()), "b2_exact_maxpool")
    _count(1)
    return y


def exact_upsample(x, C, din, out, ld, off, dout):
    lib = _lib.load()
    _lib.check(lib.b2_exact_upsample(_p(x), 1, din[0], din[1], din[2], C, _p(out), ld, off, dout[0], dout[1], dout[2],
                                     _s()), "b2_exact_upsample")
    _count(1)


def exact_head_gather(feat, index, W, b, softmax=True):
    lib = _lib.load()
    cout, cin = W.shape[0], W.shape[1]
    n = index.numel()
    scores = torch.empty((n, cout), dtype=F32, device=feat.device)
    preds = torch.empty(n, dtype=torch.int32, device=feat.device)
    Wc = W.reshape(cout, cin).contiguous().float()
    _lib.check(lib.b2_exact_head_gather(_p(feat), _p(index.contiguous()), n, _p(Wc), _p(b.contiguous().float()), cin,
                                        cout, int(softmax), _p(scores), _p(preds), _s()), "b2_exact_head_gather")
    _count(1)
    return scores, preds
