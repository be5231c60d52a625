#!/usr/bin/env python
"""bench.py — headline benchmark: UNet3D (in 1, out 56, 'crg', 64 filters) full-training steps per second on
synthetic 1x1x96x112x96 skeleton volumes (BASELINE.json configs[1]; configs[3] under torchrun with N ranks).

  python bench.py --gpus 1 --steps K --warmup W            our arm (hand-written sm_100a kernels)
      ... --dump-outputs DIR                               also writes the last timed step's loss and updated
                                                            parameters as DIR/*.npy (see dump_outputs)
  python bench.py --impl reference --steps K --warmup W     the reference's CPU path (oracle port, host cores), on the
                                                            SAME full 96x112x96 volume
  torchrun ... bench.py --gpus N ...                        data parallel over subjects, one rank per GPU
  python bench.py --inference [--steps S]                   BASELINE configs[4]: batched inference + cutting sweep,
                                                            (subject, hemisphere) pairs dealt over the ranks

A "step" = forward + CrossEntropyLoss(ignore_index=-1) + backward + SGD(lr 1e-2, momentum 0.9) on ONE volume per
rank (weak scaling: global batch = N).  One JSON line on stdout (rank 0):
  value ....... volumes/s of the whole job, inputs resident in HBM, the step replayed from a CUDA graph
  e2e ......... the same through the reference-facing API: UnetTrainingSulciLabelling.learning() over a synthetic
                cohort held as host point lists (the form main.py caches, dict_bck2 / dict_names); every step copies
                the subject's point list host -> device, builds the volumes there (rotation augmentation included),
                trains, and reads the loss back (step_callback); timed = the train phase of the second epoch
  roofline .... the fprop + dgrad tcgen05 kernels (conv3d_igemm_kernel + conv3d_slab_kernel): algorithmic FLOPs /
                CUDA-event time of their 26 launches per step, against the measured bf16 peak (burst when the SM clock
                sampled during the run is >= 1.8 GHz, else sustained; both fractions are printed)
  torch_gpu ... "the kernel to beat": stock PyTorch eager (cuDNN) on the same GPU, fp32 (the reference's real GPU path,
                training.py:199-212) and bf16 autocast + channels_last_3d
  cpu_baseline  the oracle port on the host cores, full volume (N = 1 only)
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPE = (96, 112, 96)
N_CLASSES = 56
FWD_BWD_GFLOP = 5612.086          # SURVEY.md §8(d): full training step, one volume
FWD_GFLOP = 1871.290
METRIC = "training volumes/sec"
WORKLOAD = ("UNet3D(in=1,out=56,'crg',f=64) full training step (SGD lr 1e-2 momentum 0.9), synthetic "
            "1x1x96x112x96 skeleton volumes, batch 1 per rank")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def load_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/): the
    newest profiles/r*_traffic.json.  Returns (bytes_per_launch or None, source)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    if not files:
        return None, None
    try:
        d = json.load(open(files[-1]))
        return float(d["dram_bytes_per_launch"]), os.path.relpath(files[-1], ROOT)
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------------------------------- synthetic data
def synth_volume(shape, n_classes, seed, occupancy=0.03):
    """SURVEY.md §8(d): x = (U < occupancy) with Generator(seed); labels = randint(0, n_classes) on the skeleton,
    -1 elsewhere (what reference dataset.py:78-88 produces)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(shape, generator=g) < occupancy)
    labels = torch.full(shape, -1, dtype=torch.long)
    lab = torch.randint(0, n_classes, shape, generator=g)
    labels[x] = lab[x]
    return x.to(torch.float32).unsqueeze(0), labels


def synth_dataset(n, rank, shape=SHAPE):
    xs, ls = [], []
    for i in range(n):
        x, l = synth_volume(shape, N_CLASSES, 1234 + 100 * rank + i, occupancy=0.03)
        xs.append(x.unsqueeze(0))
        ls.append(l.unsqueeze(0))
    return xs, ls


_ELLIPSOID = {}


def synth_cohort(n_subjects, seed0, shape=SHAPE, n_points=31000, only=None):
    """Synthetic subjects in the form main.py caches them (dict_bck2: integer point lists, dict_names: one sulcus name
    per point).  The points fill an ellipsoid inscribed in the volume with margin, so that the rotation augmentation
    (sigma = pi/16 about the centre, dataset.py:304-326) keeps every subject inside the fixed 96x112x96 img_size.
    only: predicate on the subject position — the other subjects get empty lists (ranks never touch the subjects of
    other ranks)."""
    import numpy as np
    names = ["S%02d_left" % i for i in range(N_CLASSES)]
    dict_bck2, dict_names = {}, {}
    cells = _ELLIPSOID.get(shape)
    if cells is None:
        radii = np.array([shape[0] / 2.0 - 10, shape[1] / 2.0 - 10, shape[2] / 2.0 - 10])
        grid = np.stack(np.meshgrid(*[np.arange(s) for s in shape], indexing="ij"), -1).reshape(-1, 3)
        inside = ((((grid + 0.5) - np.array(shape) / 2.0) / radii) ** 2).sum(1) <= 1.0
        cells = _ELLIPSOID[shape] = grid[inside]
    for s in range(n_subjects):
        g = "bench_subject%04d.arg" % (seed0 + s)
        if only is not None and not only(s):
            dict_bck2[g], dict_names[g] = [], []
            continue
        rng = np.random.RandomState(seed0 + s)
        pts = cells[rng.choice(len(cells), size=n_points, replace=False)]
        lab = rng.randint(0, N_CLASSES, size=n_points)
        dict_bck2[g] = pts.tolist()
        dict_names[g] = [names[l] for l in lab]
    return dict_bck2, dict_names, names


# ------------------------------------------------------------------------------------------------------------ CPU arm
def cpu_train_steps(steps, warmup, shape=SHAPE):
    """The reference's CPU path for this metric: the oracle port (fp32 PyTorch on the host cores; the reference runs
    torch.device('cpu') when cuda=-1, pattern_class.py:109-110) doing the same training step on the same volume."""
    import torch
    from oracle.unet3d_ref import UNet3DRef
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(42)
    model = UNet3DRef(1, N_CLASSES)
    opt = torch.optim.SGD(model.parameters(), lr=1e-2, momentum=0.9, weight_decay=0)
    crit = torch.nn.CrossEntropyLoss(ignore_index=-1)
    x, l = synth_volume(shape, N_CLASSES, 1234, occupancy=0.03)
    x, l = x.unsqueeze(0), l.unsqueeze(0)
    model.train()

    def step():
        opt.zero_grad()
        loss = crit(model(x), l)
        loss.backward()
        opt.step()
        return float(loss.detach())

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return 1.0 / dt, dt, cores


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    vps, dt, cores = cpu_train_steps(args.steps, args.warmup)
    desc = ("oracle port (fp32 PyTorch restatement of the reference's UNet3D CPU path), %d host threads; each step = "
            "one full SGD training step on one 96x112x96 volume (the headline workload, not a crop); %.2f s/step"
            % (cores, dt))
    line = {
        "impl": "reference", "metric": METRIC, "value": vps, "unit": "volumes/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "cpu_baseline": {"value": vps, "unit": "volumes/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": vps, "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------- stock PyTorch on the GPU
def torch_gpu_arm(dev, steps, warmup):
    """'The kernel to beat' (SURVEY.md §2.1 / §8(d)): the same network written with stock torch.nn modules, eager, on
    the same GPU — fp32 exactly as the reference runs it on a GPU (training.py:199-212: no autocast, default cuDNN
    settings) and bf16 autocast with channels_last_3d weights/inputs.  Library kernels only (cuDNN / ATen)."""
    import torch
    import torch.nn as nn
    import torch.nn.functional as F

    def dconv(ci, co, enc):
        c1 = (ci, max(co // 2, ci)) if enc else (ci, co)
        c2 = (c1[1], co)
        layers = []
        for a, b in (c1, c2):
            layers += [nn.Conv3d(a, b, 3, padding=1, bias=False), nn.ReLU(), nn.GroupNorm(32, b, eps=1e-5)]
        return nn.Sequential(*layers)

    class Net(nn.Module):
        def __init__(self, f=64, out=N_CLASSES):
            super().__init__()
            self.enc = nn.ModuleList([dconv(1, f, True), dconv(f, 2 * f, True), dconv(2 * f, 4 * f, True),
                                      dconv(4 * f, 8 * f, True)])
            self.dec = nn.ModuleList([dconv(12 * f, 4 * f, False), dconv(6 * f, 2 * f, False), dconv(3 * f, f, False)])
            self.head = nn.Conv3d(f, out, 1)

        def forward(self, x):
            feats = []
            for i, e in enumerate(self.enc):
                if i:
                    x = F.max_pool3d(x, 2)
                x = e(x)
                feats.insert(0, x)
            for d, skip in zip(self.dec, feats[1:]):
                x = F.interpolate(x, size=skip.shape[2:], mode="trilinear", align_corners=False)
                x = d(torch.cat((skip, x), 1))
            return self.head(x)

    x, l = synth_volume(SHAPE, N_CLASSES, 1234, occupancy=0.03)
    x, l = x.unsqueeze(0).to(dev), l.unsqueeze(0).to(dev)
    out = {}
    for name in ("fp32", "bf16_autocast_channels_last_3d"):
        torch.manual_seed(42)
        net = Net().to(dev).train()
        xin = x
        if name != "fp32":
            net = net.to(memory_format=torch.channels_last_3d)
            xin = x.contiguous(memory_format=torch.channels_last_3d)
        opt = torch.optim.SGD(net.parameters(), lr=1e-2, momentum=0.9, weight_decay=0)
        crit = nn.CrossEntropyLoss(ignore_index=-1)

        def step():
            opt.zero_grad()
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(name != "fp32")):
                o = net(xin)
            loss = crit(o.float(), l)
            loss.backward()
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
            out[name] = {"value": 1e3 / ms, "unit": "volumes/s", "ms_per_step": ms, "steps": steps, "warmup": warmup}
        except Exception as e:   # e.g. out of memory on a shared box: report, do not fail the bench
            out[name] = {"unavailable": str(e)[:200]}
        del net, opt
        torch.cuda.empty_cache()
    out["what"] = ("stock torch.nn UNet3D (cuDNN/ATen library kernels), eager, same GPU, same volume, resident inputs; "
                   "cudnn.allow_tf32=%s (PyTorch default, what the reference would run)"
                   % torch.backends.cudnn.allow_tf32)
    return out


# ------------------------------------------------------------------------------------------------------------ GPU arm
def _quiet():
    import contextlib
    import io
    return contextlib.redirect_stdout(io.StringIO())


DUMP_SAMPLE = 1 << 20     # elements kept of a larger tensor: the 44 fp32 parameters alone are 65 MB


def dump_outputs(out_dir, loss, model):
    """--dump-outputs: what the last timed step hands its caller, as out_dir/<name>.npy (float32): `loss` = the
    (mean, sum) the step returns, and `param.<name>` = every parameter as the step's SGD update left it.  A tensor of
    more than DUMP_SAMPLE elements is flattened and sampled at DUMP_SAMPLE positions drawn by a fixed-seed generator,
    the same positions on every run, so that the dumps of two builds compare element for element (about 31 MB)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = [("loss", loss)] + [("param." + n, p) for n, p in model.named_parameters()]
    for name, t in arrays:
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_SAMPLE:
            pick = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[pick]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import unetsulc_b200
    from unetsulc_b200 import ops, parallel
    from unetsulc_b200.optim import SGD
    from unetsulc_b200.training import UnetTrainingSulciLabelling

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks, peak_src = load_peaks()

    # the public training class; its model/optimiser are what `learning()` would build (training.py:60-74,140)
    sslist = ["S%02d_left" % i for i in range(N_CLASSES)]
    with _quiet():
        trainer = UnetTrainingSulciLabelling([], "L", cuda=local, working_path="/tmp/unetsulc_bench",
                                             dict_model={"name": "bench"}, dict_names={}, dict_bck2={},
                                             sulci_side_list=sslist)
        torch.manual_seed(42)
        trainer.load_network()
    model = trainer.model
    model.train()
    opt = SGD(model.ordered_parameters(), lr=1e-2, momentum=0.9, weight_decay=0)
    reducer = parallel.BucketedGradReducer(model) if world > 1 else None

    n_data = 4
    xs_h, ls_h = synth_dataset(n_data, rank)
    xs_d = [x.to(dev) for x in xs_h]
    ls_d = [l.to(dev) for l in ls_h]

    # the step is replayed from CUDA graphs: one graph on one rank; under data parallelism one graph segment per
    # gradient bucket with the NCCL all-reduces enqueued eagerly in between (NCCL itself is never captured)
    trainer.use_cuda_graph = not args.no_cuda_graph

    last_loss = [None]

    def step_resident(i):
        last_loss[0] = trainer.train_step_device(xs_d[i % n_data], ls_d[i % n_data], opt, reducer)
        return last_loss[0]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, collective=True):
        """collective=False: rank-local timing (no barrier / all-reduce) for work only one rank does"""
        sync = sync_all if collective else torch.cuda.synchronize
        sync()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for i in range(steps):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = a.elapsed_time(b)
        if world > 1 and collective:
            t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        sync()
        return ms / 1e3, wall

    # per-kernel CUDA-event profile of the dominant kernels: taken on eager steps (events cannot be recorded inside a
    # replayed graph), same kernels, same shapes, same stream
    graph_flag, trainer.use_cuda_graph = trainer.use_cuda_graph, False
    for i in range(2):
        step_resident(i)
    torch.cuda.synchronize()
    ops.PROFILE = {}
    l0 = ops.LAUNCHES[0]
    prof_steps = min(args.steps, 5)
    prof_secs, _ = timed(step_resident, prof_steps)
    launches_per_step = (ops.LAUNCHES[0] - l0) / prof_steps
    prof, ops.PROFILE = ops.PROFILE, None
    trainer.use_cuda_graph = graph_flag

    for i in range(max(args.warmup, 3) + trainer._graph_capture_after):
        step_resident(i)
    sampler = ClockSampler(local)
    sampler.start()
    secs, wall = timed(step_resident, args.steps)
    launches = int(round(launches_per_step * args.steps))
    clocks = sampler.stop()
    value = world * args.steps / secs
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_loss[0], model)

    # roofline of the dominant kernels: 26 launches / step, fprop + dgrad of the 13 Cin >= 32 convs (implicit GEMM on
    # tcgen05: conv3d_igemm_kernel, and conv3d_slab_kernel for the Cout <= 64 layers)
    ig = prof.get("conv3d_igemm", [])
    ig_ms = sum(a.elapsed_time(b) for a, b, _ in ig)
    ig_flop = sum(w for _, _, w in ig)
    achieved = ig_flop / (ig_ms * 1e-3) / 1e12 if ig_ms > 0 else 0.0
    burst = float(peaks.get("bf16_tflops", 0) or 0)
    sustained = float(peaks.get("bf16_tflops_sustained", burst) or burst)
    at_burst_clock = bool(clocks.get("sm_mhz")) and clocks["sm_mhz"] >= 1800
    peak = burst if at_burst_clock else sustained
    wg = prof.get("conv3d_wgrad", [])
    wg_ms = sum(a.elapsed_time(b) for a, b, _ in wg)
    wg_tf = (sum(w for _, _, w in wg) / (wg_ms * 1e-3) / 1e12) if wg_ms > 0 else None
    traffic, traffic_src = load_traffic()
    step_tf = value / world * FWD_BWD_GFLOP * 1e9 / 1e12
    roofline = {
        "bound": "tensor", "kernel": "conv3d_igemm_kernel + conv3d_slab_kernel (fprop + dgrad, 26 launches/step)",
        "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
        "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": "%s %s bf16 (SM clock sampled during the timed region: %s MHz)"
                       % (peak_src, "burst" if at_burst_clock else "sustained", clocks.get("sm_mhz")),
        "frac_vs_burst": achieved / burst if burst else None,
        "frac_vs_sustained": achieved / sustained if sustained else None,
        "launches_per_step": len(ig) / max(prof_steps, 1), "avg_launch_ms": ig_ms / max(len(ig), 1),
        # share of the TIMED (graph-replayed) step: kernel time per step from the eager event profile / replayed step time
        # (the profiled eager steps themselves are slower: two events per conv launch keep the host busy)
        "share_of_step": (ig_ms / max(prof_steps, 1)) / (secs / args.steps * 1e3) if secs > 0 else None,
        "wgrad_kernel_tflops": wg_tf, "wgrad_frac": (wg_tf / peak) if (wg_tf and peak) else None,
        "wgrad_share_of_step": (wg_ms / max(prof_steps, 1)) / (secs / args.steps * 1e3) if secs > 0 else None,
        "profiled": "%d eager steps (%.3f ms/step) with CUDA events around every conv launch; the timed region "
                    "replays the same step as a CUDA graph" % (prof_steps, prof_secs / prof_steps * 1e3),
        "step_tflops": step_tf, "step_frac_vs_burst": step_tf / burst if burst else None,
        "step_frac_vs_sustained": step_tf / sustained if sustained else None,
    }

    # ---- end to end through the reference-facing API: UnetTrainingSulciLabelling.learning() ----------------------
    e2e = None if args.no_e2e else run_e2e_learning(args, world, rank, local, dev)

    # secondary metric of BASELINE.json: inference ms per hemisphere = eval forward + Softmax scores gathered at the
    # skeleton voxels + the cutting / fold-vote pass for thresholds [50, 100, 150] (pattern_class.py:177-245), device
    # resident, CUDA events, rank 0 only
    inference = None
    if rank == 0:
        import numpy as _np
        model.eval()
        xi = xs_d[0]
        idx = torch.nonzero(xi.reshape(-1) > 0).reshape(-1)
        coords = torch.nonzero(xi[0, 0] > 0).cpu().numpy()
        vert = (coords[:, 2] // 12) * 64 + (coords[:, 1] // 14) * 8 + (coords[:, 0] // 12)
        _, inv = _np.unique(vert, return_inverse=True)
        fold = torch.from_numpy(inv.astype(_np.int32)).to(dev)
        nf = int(inv.max()) + 1

        def infer(_i):
            with torch.no_grad():
                scores, preds = model.scores_at(xi, idx)
                return ops.fold_vote(scores, fold, nf, [50, 100, 150])

        for i in range(3):
            infer(i)
        isecs, _ = timed(infer, 10, collective=False)   # rank 0 only: no barrier
        inference = {"ms_per_hemi": isecs / 10 * 1e3, "voxels": int(idx.numel()), "folds": nf,
                     "ceiling_ms": FWD_GFLOP / peak if peak else None,
                     "what": "eval forward + softmax gather at skeleton voxels + fold vote for 3 thresholds, "
                             "inputs resident in HBM"}
        model.train()

    torch_gpu = None
    if rank == 0 and world == 1 and not args.no_torch_gpu:
        del xs_d, ls_d
        trainer.__dict__.pop("_graphs", None)
        torch.cuda.empty_cache()
        torch_gpu = torch_gpu_arm(dev, steps=5, warmup=3)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        vps, dt, cores = cpu_train_steps(2, 1)
        cpu = {"value": vps, "unit": "volumes/s", "cores": cores, "kind": "port",
               "sample": "oracle port (fp32 PyTorch, %d host threads): 2 full SGD training steps on one 96x112x96 "
                         "volume after 1 warm-up; %.2f s/step" % (cores, dt)}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "volumes/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "parallelism": "dp%d over subjects" % world,
                       "cuda_graph": bool(trainer.use_cuda_graph),
                       "l2": "no explicit flush: a step streams ~2 GB of activations (>> 126 MB L2) and cycles "
                             "through %d distinct volumes" % n_data},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "torch_gpu": torch_gpu, "wall_s_timed_region": wall, "inference": inference,
        }
        print(json.dumps(line), flush=True)
    _shutdown(world, [trainer])
    return 0


def _shutdown(world, holders):
    """Tears the process group down without ever hanging the launcher: captured CUDA graphs that contain NCCL kernels
    are released first (destroying a communicator that live graphs still reference can block), and the destroy itself
    runs under a watchdog."""
    import gc
    import torch
    import torch.distributed as dist
    if world <= 1:
        return
    for h in holders:
        h.__dict__.pop("_graphs", None)
        h.__dict__.pop("_graph_seen", None)
    gc.collect()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    t = threading.Thread(target=dist.destroy_process_group, daemon=True)
    t.start()
    t.join(20)
    if t.is_alive():
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def run_e2e_learning(args, world, rank, local, dev):
    """e2e: UnetTrainingSulciLabelling.learning() (the reference's public call, training.py:77) for 2 epochs over a
    synthetic cohort of `steps` subjects per rank held as HOST point lists; img_size fixed to 96x112x96 (dict_model
    extension), batch 1.  Epoch 0 warms up (eager steps, graph capture); the timed region is the train phase of epoch
    1 as learning() itself clocks it (wall time between two device synchronisations): per step the subject's point
    list is copied host -> device (pinned, 16 B per point), the volumes are built there with the rotation
    augmentation, the captured step runs, and the loss is read back (step_callback)."""
    import torch
    import torch.distributed as dist
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    k = args.steps
    bck2, names, sslist = synth_cohort(k * world + 1, seed0=5000,
                                       only=lambda s: s >= k * world or s % world == rank)
    files = sorted(bck2)
    train_files, val_files = files[:k * world], files[k * world:]
    import random
    import numpy as np
    random.seed(42)
    np.random.seed(42)
    torch.manual_seed(42)
    losses = []
    with _quiet():
        tr = UnetTrainingSulciLabelling(files, "L", cuda=local, working_path="/tmp/unetsulc_bench",
                                        dict_model={"name": "bench_e2e", "img_size": list(SHAPE)},
                                        dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
        tr.use_cuda_graph = not args.no_cuda_graph
        tr.resident_points = False          # every step uploads its subject's point list: a real per-step H2D copy
        tr.step_callback = lambda phase, step, loss: losses.append(loss)
        tr.learning(1e-2, 0.9, 2, train_files, val_files, batch_size=1, patience={}, save_results=False)
    t = tr.timings["train"][-1]
    secs, steps = t["seconds"], t["steps"]
    if world > 1:
        tt = torch.tensor([secs], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        secs = float(tt[0])
    n_pts = sum(len(bck2[g]) for g in train_files) / max(len(train_files), 1)
    del tr
    torch.cuda.empty_cache()
    return {"value": world * steps / secs, "unit": "volumes/s", "h2d_bytes_per_step": int(16 * n_pts + 96),
            "d2h_bytes_per_step": 8, "ms_per_step": secs / steps * 1e3, "steps": steps,
            "api": "UnetTrainingSulciLabelling.learning(lr=1e-2, momentum=0.9, num_epochs=2, batch_size=1), "
                   "dict_model.img_size=[96,112,96]; timed: train phase of epoch 1 (epoch 0 = warm-up + graph capture)",
            "last_loss": losses[-1] if losses else None}


# ------------------------------------------------------------------------------------------- config 5: batched inference
def run_inference(args):
    """BASELINE configs[4]: batched inference with cutting thresholds [50, 100, 150] and the per-elementary-fold vote,
    both hemispheres, (subject, hemisphere) pairs dealt round-robin over the ranks; through the public
    test_thresholds() (pattern_class.py:177-245).  `--steps S` = subjects per hemisphere per rank."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks, _ = load_peaks()
    S = args.steps * world
    trainers = {}
    files = {}
    for hemi, seed0 in (("L", 7000), ("R", 8000)):
        bck2, names, sslist = synth_cohort(S, seed0=seed0)
        fl = sorted(bck2)
        with _quiet():
            t = UnetTrainingSulciLabelling(fl, hemi, cuda=local, working_path="/tmp/unetsulc_bench",
                                           dict_model={"name": "bench_inf_" + hemi}, dict_names=names, dict_bck2=bck2,
                                           sulci_side_list=sslist)
            torch.manual_seed(42)
            t.load_network()
        rng = np.random.RandomState(seed0)
        for g in fl:      # pre-extracted graph data (what soma.aims would give): cut graph + shuffled not-cut graph
            pts = np.asarray(bck2[g])
            nb = pts * 2 + 1
            perm = rng.permutation(len(pts))
            q = pts[perm]
            vert = (q[:, 2] // 12) * 64 + (q[:, 1] // 14) * 8 + (q[:, 0] // 12)
            t.dict_graph_data[g] = {"nbck": nb, "bck2": bck2[g], "names": names[g], "vert": np.arange(len(pts))}
            t.dict_graph_data[g + ".notcut"] = {"nbck": nb[perm], "bck2": q, "names": None, "vert": vert}
        trainers[hemi], files[hemi] = t, fl

    def sweep():
        for hemi in ("L", "R"):
            t = trainers[hemi]
            t.results = {"threshold_scores": {}}
            with _quiet():
                t.test_thresholds(files[hemi], [g + ".notcut" for g in files[hemi]], [50, 100, 150])

    sweep()                                            # warm-up (workspaces, weight packs)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = time.perf_counter()
    sweep()
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    clocks = sampler.stop()
    if world > 1:
        tt = torch.tensor([secs], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        secs = float(tt[0])
    hemis = 2 * S
    if rank == 0:
        sc = trainers["L"].results["threshold_scores"]
        print(json.dumps({
            "metric": "inference ms/hemi", "value": secs / hemis * 1e3 * world, "unit": "ms per hemisphere per GPU",
            "hemis_per_s": hemis / secs, "n_gpus": world, "steps": args.steps, "higher_is_better": False,
            "scaling": "weak", "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "test_thresholds(): eval forward 1x1x96x112x96 + softmax gather at ~31k skeleton "
                                   "points + voxel matching + fold vote for thresholds [50,100,150] + ESI, both "
                                   "hemispheres (two models), %d subjects per hemisphere, pairs round-robin over "
                                   "%d rank(s); wall clock incl. host point-list handling" % (S, world)},
            "clocks": clocks, "ceiling_ms": FWD_GFLOP / float(peaks.get("bf16_tflops", 1678.4)),
            "threshold_scores_L_first": {str(k): v[0][:2] for k, v in sc.items()}}), flush=True)
    _shutdown(world, list(trainers.values()))
    return 0


# ------------------------------------------------------------------------------------- variable bounding boxes (sweep)
def run_sweep(args):
    """VERDICT r1 item 9 / SURVEY §8(d): a cohort of 16 subjects whose bounding boxes are drawn around 80x104x72 +- 8
    (what real cohorts look like, dataset.py:68-75) through learning(), batch 1:
      (a) as the reference runs it — no fixed img_size, rotation augmentation on: every sample has its own box, the
          step runs eagerly (shapes never repeat, nothing to replay);
      (b) the same cohort with dict_model['img_size'] = the largest box + margin: one shape, CUDA-graph replay.
    Prints one JSON line with the train-phase volumes/s of the last epoch of both."""
    import random
    import numpy as np
    import torch
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    rng = np.random.RandomState(11)
    names = ["S%02d_left" % i for i in range(N_CLASSES)]
    bck2, nm, boxes = {}, {}, []
    for s in range(16):
        box = tuple(int(v) for v in (np.array([80, 104, 72]) + rng.randint(-8, 9, size=3)))
        boxes.append(box)
        n_pts = int(0.03 * box[0] * box[1] * box[2])
        lin = rng.choice(box[0] * box[1] * box[2], size=n_pts, replace=False)
        pts = np.stack(np.unravel_index(lin, box), 1)
        pts = np.concatenate([pts, [[0, 0, 0], [box[0] - 1, box[1] - 1, box[2] - 1]]])   # pin the bounding box
        g = "sweep_subject%02d.arg" % s
        bck2[g] = pts.tolist()
        nm[g] = [names[l] for l in rng.randint(0, N_CLASSES, size=len(pts))]
    files = sorted(bck2)
    out = {}
    # (b): the fixed size comes from the reference's own pre-scan for batch > 1 (training.py:119-134): largest box over
    # the augmented draws of all epochs, then the generators are re-seeded so that the same draws are made again
    from unetsulc_b200.dataset import SulciDataset
    random.seed(42); np.random.seed(42)
    scan = SulciDataset(files[:15], {n_: i for i, n_ in enumerate(names)}, train=True, dict_bck2=bck2, dict_names=nm)
    big = [0, 0, 0]
    for _ in range(4):
        for k in range(15):
            big = [max(a_, b_) for a_, b_ in zip(big, scan.item_size(k))]
    big = [max(a_, b_ ) for a_, b_ in zip(big, [max(b[k] for b in boxes) for k in range(3)])]
    for mode, dm in (("variable_boxes_eager", {"name": "sweep_a"}),
                     ("padded_to_%dx%dx%d_graph" % tuple(big), {"name": "sweep_b", "img_size": big})):
        random.seed(42); np.random.seed(42); torch.manual_seed(42)
        with _quiet():
            tr = UnetTrainingSulciLabelling(files, "L", cuda=0, working_path="/tmp/unetsulc_bench", dict_model=dm,
                                            dict_names=nm, dict_bck2=bck2, sulci_side_list=names)
            tr.learning(1e-2, 0.9, 4, files[:15], files[15:], batch_size=1, patience={}, save_results=False)
        t = tr.timings["train"]
        out[mode] = {"volumes_per_s": [round(x["steps"] / x["seconds"], 2) for x in t],
                     "ms_per_step_last_epoch": t[-1]["seconds"] / t[-1]["steps"] * 1e3}
        del tr
        torch.cuda.empty_cache()
    vox = float(np.mean([b[0] * b[1] * b[2] for b in boxes]))
    print(json.dumps({"metric": "training volumes/sec (variable bounding boxes)", "unit": "volumes/s", "n_gpus": 1,
                      "boxes": boxes, "mean_voxels": vox, "voxels_vs_96x112x96": vox / (96 * 112 * 96),
                      "epochs": 4, "subjects": 15, "results": out,
                      "note": "train-phase wall clock per epoch incl. host-side sample building; epoch 0 includes "
                              "first-use workspace allocation (a) / eager steps before the capture (b)"}))
    return 0


def main():
    if os.environ.get("B2_DEBUG_DP") == "1":   # debugging aid: dump every thread's Python stack if the run stalls
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ.get("B2_DEBUG_DP_AFTER", "75")), exit=False)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--inference", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="variable bounding boxes through learning() (1 GPU)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-gpu", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the learning() leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss and updated parameters to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.inference or args.sweep):
        ap.error("--dump-outputs applies to the training benchmark of our arm only")
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.inference:
        return run_inference(args)
    if args.sweep:
        return run_sweep(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
