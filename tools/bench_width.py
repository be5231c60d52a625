"""Training-step throughput of the 32- and 64-filter networks at 96 x 112 x 96, measured in one run.

    python tools/bench_width.py [--steps 30] [--repeats 5] [--out profiles/width32_vs_64.json]

* card name and power limit (nvidia-smi) are read in the same run and stored with the numbers;
* graph-replayed training steps (UnetTrainingSulciLabelling.train_step_device, SGD included) of f = 32 and f = 64,
  alternated `--repeats` times so that both see the same machine state; volumes/s per repeat, median and spread;
* CUDA-event times of every fprop / dgrad / wgrad launch of an eager step, per layer, with FLOP/s from the shapes
  (2 x voxels x 27 x Cin x Cout per pass), and the kernel each launch ran (torch.profiler, a separate eager step);
* stock PyTorch eager at f = 32 (oracle/unet3d_ref.py: torch.nn modules, cuDNN / ATen kernels), fp32 and bf16
  autocast + channels_last_3d, as the kernel to beat.
Every shape is warmed up before it is timed.  Inputs are four resident synthetic volumes, ~3 % occupancy.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPE = (96, 112, 96)
N_CLASSES = 56


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # report, do not guess
        return {"unavailable": str(e)[:200]}


def _data(dev, n=4):
    from oracle.synth import synth_volume
    xs, ls = [], []
    for i in range(n):
        x, l = synth_volume(SHAPE, N_CLASSES, 1234 + i, occupancy=0.03)
        xs.append(x.unsqueeze(0).to(dev))
        ls.append(l.unsqueeze(0).to(dev))
    return xs, ls


class Arm(object):
    """one network width: trainer, optimiser, graph-replayed step"""

    def __init__(self, f, dev, xs, ls):
        import torch
        from unetsulc_b200.optim import SGD
        from unetsulc_b200.training import UnetTrainingSulciLabelling
        with contextlib.redirect_stdout(io.StringIO()):
            self.trainer = UnetTrainingSulciLabelling(
                [], "L", cuda=dev.index or 0, working_path="/tmp/unetsulc_bench_width",
                dict_model={"name": "w%d" % f, "num_filter": f}, dict_names={}, dict_bck2={},
                sulci_side_list=["S%02d_left" % i for i in range(N_CLASSES)])
            torch.manual_seed(42)
            self.trainer.load_network()
        self.f = f
        self.model = self.trainer.model.train()
        self.opt = SGD(self.model.ordered_parameters(), lr=1e-2, momentum=0.9, weight_decay=0)
        self.xs, self.ls = xs, ls
        self.i = 0

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


CONV_OPS = {
    # ops function -> (kind, how to read (cin, cout, view with the voxel count) from its arguments)
    "conv3d_first_fwd_gn_stats": ("fprop", lambda x, w, y, *a, **k: (1, w.shape[0], y)),
    "conv3d_igemm_gn_stats": ("fprop", lambda x, wp, y, cin, cout, *a, **k: (cin, cout, y)),
    "conv3d_igemm_auto": (None, lambda x, wp, y, cin, cout, relu: (cin, cout, y)),
    "conv3d_dgrad_gn_bstats": ("dgrad", lambda dy, wd, dx, cin, cout, *a, **k: (cout, cin, dx)),
    "conv3d_wgrad": ("wgrad", lambda x, dy, cin, cout, *a, **k: (cin, cout, x)),
    "conv3d_first_wgrad": ("wgrad", lambda x, dy, cout, *a, **k: (1, cout, dy)),
}


@contextlib.contextmanager
def conv_recorder(records, with_events=True):
    """wraps the conv entry points of ops: appends dict(kind, cin, cout, voxels, events) per call, in call order.
    (cin, cout) are the layer's, for dgrad too."""
    import torch
    from unetsulc_b200 import ops
    saved = {}
    for name, (kind, shape) in CONV_OPS.items():
        real = saved[name] = getattr(ops, name)

        def spy(*a, _real=real, _kind=kind, _shape=shape, **k):
            cin, cout, v = _shape(*a, **k)
            knd = _kind or ("fprop" if (k.get("relu", a[5] if len(a) > 5 else None)) else "dgrad")
            if knd == "dgrad" and _kind is None:   # conv3d_igemm_auto(dy, wd, dx, layer.cout, layer.cin)
                cin, cout = cout, cin
            rec = dict(kind=knd, cin=cin, cout=cout, voxels=v.N * v.V, dims=[v.D, v.H, v.W])
            if with_events:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            out = _real(*a, **k)
            if with_events:
                e1.record()
                rec["events"] = (e0, e1)
            records.append(rec)
            return out
        setattr(ops, name, spy)
    try:
        yield records
    finally:
        for name, real in saved.items():
            setattr(ops, name, real)


def per_layer(arm, steps=5):
    """eager steps: CUDA-event time of every conv launch, averaged per (kind, layer)"""
    import torch
    graph_flag, arm.trainer.use_cuda_graph = arm.trainer.use_cuda_graph, False
    for _ in range(2):
        arm.step()
    torch.cuda.synchronize()
    rows = {}
    for _ in range(steps):
        recs = []
        with conv_recorder(recs):
            arm.step()
        torch.cuda.synchronize()
        for r in recs:
            key = (r["kind"], r["cin"], r["cout"], tuple(r["dims"]))
            ms = r["events"][0].elapsed_time(r["events"][1])
            rows.setdefault(key, []).append(ms)
    arm.trainer.use_cuda_graph = graph_flag
    out = []
    for (kind, cin, cout, dims), ms in rows.items():
        ms_med = sorted(ms)[len(ms) // 2]
        flops = 2.0 * dims[0] * dims[1] * dims[2] * 27 * cin * cout
        out.append({"kind": kind, "cin": cin, "cout": cout, "dims": list(dims), "ms_median": ms_med,
                    "ms_min": min(ms), "ms_max": max(ms), "calls": len(ms), "gflop": flops / 1e9,
                    "tflop_per_s": flops / (ms_med * 1e-3) / 1e12})
    return out


def kernels_taken(arm):
    """one eager step under torch.profiler: the conv kernel each fprop / dgrad / wgrad launch ran"""
    import torch
    from torch.profiler import profile, ProfilerActivity
    graph_flag, arm.trainer.use_cuda_graph = arm.trainer.use_cuda_graph, False
    arm.step()
    torch.cuda.synchronize()
    recs = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with conv_recorder(recs, with_events=False):
            arm.step()
        torch.cuda.synchronize()
    arm.trainer.use_cuda_graph = graph_flag
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    evs.sort(key=lambda e: e.time_range.start)
    conv = [e.name for e in evs if ("conv3d_" in e.name or "conv_first" in e.name) and "reduce" not in e.name]
    short = [n.split("(")[0].replace("void ", "").replace("b2::", "") for n in conv]
    if len(short) != len(recs):
        return {"error": "%d conv kernels for %d conv calls" % (len(short), len(recs)), "kernels": short}
    return [dict(kind=r["kind"], cin=r["cin"], cout=r["cout"], dims=r["dims"], kernel=k) for r, k in zip(recs, short)]


def torch_eager(f, dev, xs, ls, steps, warmup):
    """stock torch.nn network (the oracle module) at width f: fp32, and bf16 autocast + channels_last_3d"""
    import torch
    import torch.nn.functional as F
    from oracle.unet3d_ref import UNet3DRef
    out = {}
    for name in ("fp32", "bf16_autocast_channels_last_3d"):
        torch.manual_seed(42)
        net = UNet3DRef(1, N_CLASSES, init_channel_number=f).to(dev).train()
        x, l = xs[0], ls[0]
        if name != "fp32":
            net = net.to(memory_format=torch.channels_last_3d)
            x = x.contiguous(memory_format=torch.channels_last_3d)
        opt = torch.optim.SGD(net.parameters(), lr=1e-2, momentum=0.9)

        def step():
            opt.zero_grad()
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(name != "fp32")):
                o = net(x)
            F.cross_entropy(o.float(), l, ignore_index=-1).backward()
            opt.step()
        try:
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                step()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / steps
            out[name] = {"volumes_per_s": 1e3 / ms, "ms_per_step": ms, "steps": steps}
        except Exception as e:   # e.g. out of memory on a shared card: report, do not fail the run
            out[name] = {"unavailable": str(e)[:200]}
        del net, opt
        torch.cuda.empty_cache()
    out["cudnn_allow_tf32"] = bool(torch.backends.cudnn.allow_tf32)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30, help="graph-replayed steps per timed window")
    ap.add_argument("--repeats", type=int, default=5, help="alternated (f=32, f=64) windows")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--eager-steps", type=int, default=5, help="steps of the stock PyTorch arm")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "width32_vs_64.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_width.py: no CUDA device (the B200 path has no CPU fallback)")
    dev = torch.device("cuda", 0)
    res = {"card": card(), "shape": list(SHAPE), "classes": N_CLASSES, "steps": args.steps, "repeats": args.repeats}
    xs, ls = _data(dev)
    arms = {f: Arm(f, dev, xs, ls) for f in (32, 64)}
    for arm in arms.values():        # eager steps, graph capture, then replays of every shape
        arm.trainer.use_cuda_graph = True
        for _ in range(args.warmup + arm.trainer._graph_capture_after):
            arm.step()
    torch.cuda.synchronize()
    ms = {32: [], 64: []}
    for _ in range(args.repeats):
        for f in (32, 64):
            ms[f].append(arms[f].timed(args.steps))
    for f in (32, 64):
        v = sorted(1e3 / m for m in ms[f])
        res["f%d" % f] = {"volumes_per_s": v, "median": v[len(v) // 2], "spread": v[-1] - v[0],
                          "ms_per_step": sorted(ms[f])}
    res["f32_over_f64"] = res["f32"]["median"] / res["f64"]["median"]
    for f in (32, 64):
        res["f%d" % f]["layers"] = per_layer(arms[f])
        res["f%d" % f]["kernels"] = kernels_taken(arms[f])
    del arms
    torch.cuda.empty_cache()
    res["torch_eager_f32"] = torch_eager(32, dev, xs, ls, args.eager_steps, 2)
    res["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "f32_over_f64")}))
    for f in (32, 64):
        print("f=%d: %.2f volumes/s median (spread %.2f over %d windows of %d steps)"
              % (f, res["f%d" % f]["median"], res["f%d" % f]["spread"], args.repeats, args.steps))
    print("torch eager f=32:", json.dumps(res["torch_eager_f32"]))
    print("wrote", args.out)


if __name__ == "__main__":
    main()
