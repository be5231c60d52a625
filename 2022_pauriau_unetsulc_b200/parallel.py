"""Data parallelism over subjects: one process per GPU, gradients all-reduced with NCCL over NVLink/NVSwitch,
bucketed in reverse layer order and overlapped with the rest of the backward pass.

The reference has no distributed code (single process, single device, pattern_class.py:109-114); this is the
north-star's "training partitions across the 8 GPUs of one box data-parallel over subjects".

Semantics (SURVEY.md §8(e)): every rank computes the reference's batch-1 loss (mean over ITS labelled voxels) and
its gradient; the all-reduce AVERAGES the gradients over ranks = gradient of the mean of the per-sample means, i.e.
the reference run with gradient accumulation over W subjects divided by W.  GroupNorm statistics are per sample, so
normalisation is unchanged by the partitioning.

Buckets (fp32, 65.3 MB in total), in the order backward produces them:
  0: final_conv + decoders.2 + decoders.1      (2.2 M)      3: encoders.2 + encoders.1   (1.66 M)
  1: decoders.0                                (7.1 M)      4: encoders.0                (56 k)
  2: encoders.3                                (5.3 M)
The last bucket closes when backward ends, so its all-reduce is fully exposed in front of the optimiser step: it holds
only encoders.0 (225 KB, latency-bound).  Round 1 had encoders.2/1/0 (6.8 MB) there.
Gradients are written by the wgrad / GroupNorm-backward kernels directly into views of the flat bucket (no copy);
when the last layer of a bucket reports ready, an event is recorded on the compute stream and the all-reduce is
enqueued on a dedicated communication stream.  ``finish()`` makes the compute stream wait for all of them.
"""
import torch
import torch.distributed as dist

# layer index (0..13 trunk conv layers in forward order, 14 = head) -> bucket id
_BUCKET_OF_LAYER = {14: 0, 13: 0, 12: 0, 11: 0, 10: 0, 9: 1, 8: 1, 7: 2, 6: 2, 5: 3, 4: 3, 3: 3, 2: 3, 1: 4, 0: 4}
N_BUCKETS = 5
# the layer whose completion closes each bucket (backward runs 14, 13, ..., 0)
_LAST_LAYER_OF_BUCKET = {0: 10, 1: 8, 2: 6, 3: 2, 4: 0}


def layer_of_param(i, stride=3):
    """index in UNet3D.ordered_parameters() -> layer index; stride = UNet3D.trunk_stride() (3 trunk parameters per
    layer, 4 with conv biases)"""
    return 14 if i >= 14 * stride else i // stride


class BucketedGradReducer(object):
    def __init__(self, model, process_group=None, average=True, sync_params=True):
        self.model = model
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.average = average
        params = model.ordered_parameters()
        dev = params[0].device
        if self.world > 1 and sync_params:
            # every process built (and randomly initialised) its own network: replicas must start from rank 0's
            # weights or the averaged gradients are taken at different points and the replicas never agree
            broadcast_parameters(model, process_group)
        self.params = params
        self.stride = model.trunk_stride()
        sizes = [0] * N_BUCKETS
        self.slot = []
        for i, p in enumerate(params):
            b = _BUCKET_OF_LAYER[layer_of_param(i, self.stride)]
            n = (p.numel() + 3) // 4 * 4          # keep every view 16-byte aligned
            self.slot.append((b, sizes[b], p.numel()))
            sizes[b] += n
        self.flat = [torch.zeros(max(s, 4), dtype=torch.float32, device=dev) for s in sizes]
        self.views = [self.flat[b][off:off + n].view_as(p) for (b, off, n), p in zip(self.slot, params)]
        self.comm_stream = torch.cuda.Stream(device=dev) if dev.type == "cuda" else None
        self._pending = []
        self._needed_last = dict(_LAST_LAYER_OF_BUCKET)
        # CUDA-graph capture of a data-parallel step (pattern_class._graphed_step): NCCL is never captured; while
        # `segment_cb` is set, a bucket launch / the final wait only report where the step has to be cut into graph
        # segments, and the collectives are enqueued eagerly between the replays of those segments.
        self.segment_cb = None
        self.force_segments = False   # tests: cut the step at the bucket boundaries even on one rank
        model.grad_ready_hook = self._on_layer_ready

    def outs(self):
        """pre-allocated gradient tensors to hand to UNet3D.forward_backward(outs=...)"""
        return self.views

    def begin(self):
        """call before each backward: decides which layer closes each bucket given the requires_grad masks"""
        self._pending = []
        needs = [bool(p.requires_grad) for p in self.params]
        active_layers = sorted({layer_of_param(i, self.stride) for i, n in enumerate(needs) if n})
        self._close_at = {}
        for b in range(N_BUCKETS):
            layers = [l for l in active_layers if _BUCKET_OF_LAYER[l] == b]
            if layers:
                self._close_at[min(layers)] = b    # backward visits layers in decreasing order
        self.model.grad_flush_at = set(self._close_at)   # deferred weight-gradient reductions flush where buckets close
        # gradients of frozen parameters are not produced: keep their slots at zero
        for v, n in zip(self.views, needs):
            if not n:
                v.zero_()

    def _on_layer_ready(self, layer, grads):
        b = self._close_at.get(layer)
        if b is None or (self.world == 1 and not self.force_segments):
            return
        self._launch(b)

    def _launch(self, b):
        if self.segment_cb is not None:            # capturing: cut the graph here, the all-reduce runs at replay
            self.segment_cb(("reduce", b))
            return
        if self.world == 1:                        # force_segments on a single rank: nothing to exchange
            return
        if self.comm_stream is None:               # CPU tensors (gloo tests)
            dist.all_reduce(self.flat[b], group=self.group)
            if self.average:
                self.flat[b].div_(self.world)
            return
        ev = torch.cuda.Event()
        ev.record()                                # on the compute stream, after the bucket's last producer
        with torch.cuda.stream(self.comm_stream):
            self.comm_stream.wait_event(ev)
            if self.average:
                dist.all_reduce(self.flat[b], op=dist.ReduceOp.AVG, group=self.group)
            else:
                dist.all_reduce(self.flat[b], group=self.group)
            done = torch.cuda.Event()
            done.record()
        self._pending.append(done)

    def finish(self):
        """compute stream waits for every outstanding all-reduce; returns the reduced gradient views"""
        if self.segment_cb is not None:
            self.segment_cb(("finish", None))
            return self.views
        for ev in self._pending:
            torch.cuda.current_stream().wait_event(ev)
        self._pending = []
        return self.views


def broadcast_parameters(model, group=None, src=0):
    """rank `src`'s parameters and buffers -> every rank (in place; version counters bumped so that the bf16 weight
    packs are rebuilt)"""
    with torch.no_grad():
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, src=src, group=group)
            torch.autograd.graph.increment_version(t)


def parameters_in_sync(model, group=None):
    """True when every rank holds bit-identical parameters (compares per-tensor fp64 sums and abs-sums)"""
    chk = torch.stack([torch.stack((p.detach().double().sum(), p.detach().double().abs().sum()))
                       for p in model.parameters()])
    lo, hi = chk.clone(), chk.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
    return bool(torch.equal(lo, hi))


def shard_subjects(items, rank, world):
    """Rank r takes items[r::world]; the tail is padded by repeating the last item with weight 0 so that every
    rank runs the same number of steps (SURVEY.md §8(e)).  Returns list of (item, weight)."""
    items = list(items)
    if not items:
        return []
    steps = (len(items) + world - 1) // world
    mine = items[rank::world]
    out = [(it, 1.0) for it in mine]
    while len(out) < steps:
        out.append((items[-1], 0.0))
    return out


def allreduce_metrics(counts, loss_sum, n_samples, group=None):
    """Epoch metrics across ranks: int64 TP/FP/FN counters [3, C], fp64 loss sum, sample count."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return counts, loss_sum, n_samples
    dist.all_reduce(counts, group=group)
    t = torch.tensor([loss_sum, float(n_samples)], dtype=torch.float64, device=counts.device)
    dist.all_reduce(t, group=group)
    return counts, float(t[0]), int(round(float(t[1])))
