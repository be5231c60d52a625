"""Fused multi-tensor SGD (one launch of sgd_multi_kernel for all 44 tensors, 58 with trunk conv biases).

Semantics of ``torch.optim.SGD(params, lr, momentum, weight_decay=0)`` as the reference builds it
(training.py:140, rebuilt at :252 on LR division => momentum buffers reset): v <- mu*v + g ; p <- p - lr*v.
Parameters whose ``.grad`` is None are skipped (frozen layers, transfer_learning.py:330-335).
"""
import torch

from . import ops


class SGD(object):
    def __init__(self, params, lr, momentum=0.0, weight_decay=0):
        if weight_decay != 0:
            raise ValueError("unetsulc_b200.SGD: weight_decay=%r unsupported (reference uses 0)" % weight_decay)
        self.params = [p for p in params]
        self.lr, self.momentum = float(lr), float(momentum)
        self.param_groups = [{"params": self.params, "lr": self.lr, "momentum": self.momentum, "weight_decay": 0}]
        self._mom = {}

    def zero_grad(self, set_to_none=True):
        for p in self.params:
            if p.grad is not None:
                if set_to_none:
                    p.grad = None
                else:
                    p.grad.zero_()

    def _buf(self, p):
        b = self._mom.get(id(p))
        if b is None or b.device != p.device:
            b = torch.zeros_like(p, memory_format=torch.contiguous_format)
            self._mom[id(p)] = b
        return b

    @torch.no_grad()
    def step(self, grads=None, grad_scale=1.0):
        """grads: optional list aligned with ``params`` (None = skip); defaults to ``p.grad``."""
        lr = float(self.param_groups[0]["lr"])
        ps, gs, ms = [], [], []
        for i, p in enumerate(self.params):
            g = p.grad if grads is None else grads[i]
            if g is None:
                continue
            if not g.is_contiguous():
                g = g.contiguous()
            ps.append(p.data)
            gs.append(g)
            ms.append(self._buf(p))
        ops.sgd_step(ps, gs, ms, lr, self.momentum, grad_scale)
        # the kernel wrote through raw pointers: bump the version counters (no kernel launch) so that the bf16
        # weight packs are refreshed on the next forward
        for i, p in enumerate(self.params):
            g = p.grad if grads is None else grads[i]
            if g is not None:
                torch.autograd.graph.increment_version(p)
