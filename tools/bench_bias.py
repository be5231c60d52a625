"""Training-step throughput of U-Nets with and without trunk conv biases at 96 x 112 x 96, measured in one run.

    python tools/bench_bias.py [--steps 30] [--repeats 5] [--out profiles/r04_conv_bias.json]

* card name and power limit (nvidia-smi) are read in the same run and stored with the numbers;
* graph-replayed training steps (UnetTrainingSulciLabelling.train_step_device, SGD included) of four arms, f = 64 and
  f = 32, each bias-free and biased, alternated `--repeats` times so that all see the same machine state;
* per-kernel device time of one eager step of each arm (torch.profiler, a separate step), summed by kernel name, so
  that the GroupNorm-backward apply pass and the conv epilogues can be compared biased vs bias-free.
Every arm is warmed up (and its graph captured) before it is timed.  Inputs: four resident synthetic volumes, ~3 %
occupancy (tools/bench_width.py).
"""
import argparse
import contextlib
import io
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_width import SHAPE, N_CLASSES, card, _data   # noqa: E402


class Arm(object):
    def __init__(self, f, bias, dev, xs, ls):
        import torch
        from unetsulc_b200.optim import SGD
        from unetsulc_b200.training import UnetTrainingSulciLabelling
        self.name = "f%d_%s" % (f, "bias" if bias else "nobias")
        with contextlib.redirect_stdout(io.StringIO()):
            dm = {"name": self.name, "num_filter": f}
            if bias:
                dm["conv_bias"] = True
            self.trainer = UnetTrainingSulciLabelling(
                [], "L", cuda=dev.index or 0, working_path="/tmp/unetsulc_bench_bias", dict_model=dm,
                dict_names={}, dict_bck2={}, sulci_side_list=["S%02d_left" % i for i in range(N_CLASSES)])
            torch.manual_seed(42)
            self.trainer.load_network()
        self.model = self.trainer.model.train()
        assert self.model.conv_bias == bias
        if bias:
            with torch.no_grad():
                for n, p in self.model.named_parameters():
                    if "double_conv.conv" in n and n.endswith("bias"):
                        p.copy_(0.2 * torch.randn_like(p))
        self.opt = SGD(self.model.ordered_parameters(), lr=1e-2, momentum=0.9, weight_decay=0)
        self.xs, self.ls, self.i = xs, ls, 0

    def step(self):
        i = self.i
        self.i += 1
        return self.trainer.train_step_device(self.xs[i % len(self.xs)], self.ls[i % len(self.ls)], self.opt, None)

    def timed(self, steps):
        import torch
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            self.step()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    def kernel_times(self):
        """device time per kernel name (us) of one eager step"""
        import torch
        from torch.profiler import profile, ProfilerActivity
        m = self.model
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.forward_backward(self.xs[0], self.ls[0])
            torch.cuda.synchronize()
        out = {}
        for e in prof.key_averages():
            if e.device_type == torch.autograd.DeviceType.CUDA:
                out[e.key] = {"us": e.device_time_total, "calls": e.count}
        return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_bias: no CUDA device (this benchmark measures the B200 path only)")
    import __graft_entry__ as ge
    ge.build()
    dev = torch.device("cuda", 0)
    xs, ls = _data(dev)
    arms = [Arm(f, b, dev, xs, ls) for f in (64, 32) for b in (False, True)]
    for a in arms:
        for _ in range(args.warmup):
            a.step()
    torch.cuda.synchronize()
    ms = {a.name: [] for a in arms}
    for _ in range(args.repeats):
        for a in arms:
            ms[a.name].append(a.timed(args.steps))
    res = {"card": card(), "shape": list(SHAPE), "steps_per_window": args.steps, "windows": args.repeats,
           "arms": {}}
    for a in arms:
        t = sorted(ms[a.name])
        res["arms"][a.name] = {"ms_per_step": ms[a.name], "median_ms": t[len(t) // 2],
                               "volumes_per_s_median": 1000.0 / t[len(t) // 2]}
    for f in (64, 32):
        b, n = res["arms"]["f%d_bias" % f]["median_ms"], res["arms"]["f%d_nobias" % f]["median_ms"]
        res["f%d_bias_overhead" % f] = b / n - 1.0
    kt = {a.name: a.kernel_times() for a in arms}
    res["kernels_us"] = kt
    for f in (64, 32):
        nb, bb = kt["f%d_nobias" % f], kt["f%d_bias" % f]
        sel = lambda d, key: sum(v["us"] for k, v in d.items() if key in k)   # noqa: E731
        res["f%d_kernel_compare_us" % f] = {
            key: {"nobias": sel(nb, key), "bias": sel(bb, key)}
            for key in ("gn_bwd_apply_kernel", "dbias_finalize_kernel", "conv3d_slab_kernel", "conv3d_igemm_kernel",
                        "conv_splitk_reduce_kernel", "conv_first_fwd_kernel")}
    print(json.dumps({k: v for k, v in res.items() if k != "kernels_us"}, indent=1))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
