"""``UnetPatternSulciLabelling`` — API-keeping base class (reference pattern_class.py:32-368).

Same constructor, attributes, methods, file layout and result keys as the reference; the arithmetic underneath is
the B200 path: ``labeling`` runs the eval forward and gathers Softmax scores at the skeleton voxels on the GPU
(``UNet3D.scores_at``), ``test_thresholds`` evaluates all cutting thresholds in one ``b2_fold_vote`` pass, and the
epoch loop shared by the training classes (``_fit``) uses the fused forward+loss+backward step, the fused SGD and
on-device ESI counters.  Data-parallel training over subjects is enabled when ``torch.distributed`` is initialised.
"""
import copy
import json
import os
import sys
import os.path as op
import time

import numpy as np
import torch
import torch.nn as nn

from . import ops, parallel
from .dataset import SulciDataset, extract_data
from .early_stopping import EarlyStopping
from .models import UNet3D
from .optim import SGD
from .stats import esi_from_counts

_BV_MODELS = '/casa/host/build/share/brainvisa-share-5.1/models/models_2019/cnn_models/'

_MODEL_DEFAULTS = (  # attribute, dict_model key, default, printed label
    ('num_filter', 'num_filter', 64, 'Number of filters : '),
    ('num_channel', 'num_channel', 1, 'Number of channels : '),
    ('interpolate', 'interpolate', True, 'Interpolate : '),
    ('final_sigmoid', 'final_sigmoid', False, 'Final Sigmoid : '),
    ('conv_layer_order', 'conv_layer_order', 'crg', 'Convolutional Layer Order : '),
    # B200 extension: trunk convolutions with a bias (58-key checkpoints); a loaded checkpoint overrides it
    ('conv_bias', 'conv_bias', False, 'Conv bias : '),
)


def _summary_writer(log_dir):
    try:
        from torch.utils.tensorboard import SummaryWriter
        return SummaryWriter(log_dir=log_dir)
    except Exception:  # tensorboard not installed: results dict / JSON still carry every number
        return None


def make_head(init_channels, out_channels, num_conv):
    """final_conv as the reference builds it (pattern_class.py:357-365): one 1x1x1 conv, or a chain of them."""
    if num_conv > 1:
        fac = (init_channels - out_channels) / num_conv
        seq = nn.Sequential()
        for n in range(num_conv):
            seq.add_module(str(n), nn.Conv3d(init_channels - round(n * fac), init_channels - round((n + 1) * fac), 1))
        return seq
    return nn.Conv3d(init_channels, out_channels, 1)


class UnetPatternSulciLabelling(object):

    def __init__(self, graphs, hemi, cuda=-1, working_path=None, dict_model={},
                 dict_names=None, dict_bck2=None, sulci_side_list=None):
        self.graphs = graphs
        self.hemi = hemi
        self.dict_bck2 = dict_bck2
        self.dict_names = dict_names
        self.background = -1
        self._set_sulci(sulci_side_list)
        self.working_path = os.getcwd() if working_path is None else working_path

        self.model = None
        self.dict_model = dict_model
        if 'name' in dict_model:
            self.model_name = dict_model['name']
            print('Model name: ', self.model_name)
        else:
            self.model_name = 'UnknownModel_hemi' + hemi
        for attr, key, default, label in _MODEL_DEFAULTS:
            if key in dict_model:
                setattr(self, attr, dict_model[key])
                print(label, dict_model[key])
            else:
                setattr(self, attr, default)
        self.num_conv = dict_model.get('num_conv', 1)
        # B200 extension (not in the reference's dict_model): a fixed volume size for batch_size 1 as well — the
        # reference only fixes it for batch_size > 1 (training.py:119-134) or through labeling(imgsize=...).  With a
        # fixed size the whole training step is replayed from a CUDA graph and the samples are built on the device.
        self.img_size = dict_model.get('img_size')
        # optional hook called as step_callback(phase, step, loss_float) after every training step (one D2H read
        # per step, taken right after the head so that it overlaps the backward pass); None = no per-step host sync
        self.step_callback = None
        # keep every subject's point list on the device after its first use (False: upload it again every sample)
        self.resident_points = True
        self.timings = {}

        self.results = {}
        self.dict_scores = {}
        self.trfile = None
        # optional pre-extracted graph data {gfile: {'nbck','bck2','names','vert'}} (avoids soma.aims in test_thresholds)
        self.dict_graph_data = {}

        if cuda == -1:
            self.device = torch.device('cpu')
        else:
            self.device = torch.device("cuda" if torch.cuda.is_available() else "cpu", index=cuda)
        print('Working on', self.device)

    # ------------------------------------------------------------------------------------------ label dictionaries
    def _set_sulci(self, sulci_side_list):
        self.sulci_side_list = sulci_side_list
        if sulci_side_list is None:
            self.dict_sulci = None
            self.sslist = None
            return
        self.dict_sulci = {s: i for i, s in enumerate(sulci_side_list)}
        self.dict_sulci.setdefault('background', -1)
        self.sslist = [s for s in sulci_side_list if not s.startswith('unknown') and not s.startswith('ventricle')]

    def _graph_data(self, gfile):
        if gfile in self.dict_graph_data:
            return self.dict_graph_data[gfile]
        from soma import aims
        graph = aims.read(gfile)
        if self.trfile is not None:
            self.flt.translate(graph)
        return extract_data(graph)

    def extract_data_from_graphs(self):
        print('Creating sulci side list...')
        found = set()
        dict_bck2, dict_names = {}, {}
        for gfile in self.graphs:
            data = self._graph_data(gfile)
            dict_bck2[gfile] = data['bck2']
            dict_names[gfile] = data['names']
            found.update(data['names'])
        self._set_sulci(sorted(found))
        print(len(self.sulci_side_list), ' sulci detected')
        self.dict_bck2 = dict_bck2
        self.dict_names = dict_names

    def fill_dict_model(self, dict_model):
        side = 'left' if self.hemi == 'L' else 'right'
        dict_model.setdefault('in_channels', 1)
        if 'out_channels' not in dict_model:
            dict_model['out_channels'] = _BV_MODELS + 'sulci_unet_model_params_%s.json' % side
        if isinstance(dict_model['out_channels'], str):
            with open(dict_model['out_channels'], 'r') as f:
                dict_model['out_channels'] = len(json.load(f)['sulci_side_list'])
        dict_model.setdefault('final_sigmoid', False)
        dict_model.setdefault('interpolate', True)
        dict_model.setdefault('conv_layer_order', 'crg')
        dict_model.setdefault('init_channel_number', 64)
        dict_model.setdefault('model_file', _BV_MODELS + 'sulci_unet_model_%s.mdsm' % side)
        dict_model.setdefault('num_conv', 1)
        return dict_model

    # ------------------------------------------------------------------------------------------ inference
    def _subject_arrays(self, gfile, bck2, names):
        """(points minus their minimum int64 [n,3], label ids int32 [n]) of a subject, converted from the Python lists
        of dict_bck2 / dict_names once (the reference converts them on every call, dataset.py:47-49, 82-86)."""
        cache = self.__dict__.setdefault("_subject_cache", {})
        c = cache.get(gfile)
        if c is None or c[0] is not bck2 or c[1] is not names:
            pts = np.asarray(bck2).reshape(-1, 3).astype(np.int64)
            ids = np.asarray([self.dict_sulci[n] for n in names], dtype=np.int32)
            c = cache[gfile] = (bck2, names, pts - np.min(pts, axis=0), ids)
        return c[2], c[3]

    def _name_ids(self, names):
        """int32 class ids of a list of sulcus names (-2 for names outside sulci_side_list); converted once per list
        object — 30 k dictionary look-ups per graph otherwise"""
        cache = self.__dict__.setdefault("_name_id_cache", {})
        c = cache.get(id(names))
        if c is None or c[0] is not names:
            if len(cache) > 256:
                cache.clear()
            c = cache[id(names)] = (names, np.asarray([self.dict_sulci.get(nm, -2) for nm in names], dtype=np.int32))
        return c[1]

    def _labeling_device(self, gfile, bck2=None, names=None, imgsize=None, exact=None):
        """The device half of labeling(): eval forward + Softmax scores gathered at the skeleton points.
        Returns (scores fp32 [n, C], preds int32 [n], ytrue int64 [n]) as DEVICE tensors."""
        self.model = self.model.to(self.device)
        self.model.eval()
        if bck2 is None:
            bck2 = self.dict_bck2[gfile]
        if names is None:
            names = self.dict_names[gfile]
        if self.device.type == "cuda":
            # same volumes as SulciDataset(train=False)[0] (dataset.py:45-88) from per-subject cached arrays
            pts, ids = self._subject_arrays(gfile, bck2, names)
            size = (np.max(pts, axis=0) + 1) if imgsize is None else imgsize
            inputs, labels = ops.scatter_volume(pts, ids, size, self.device, background=self.dict_sulci['background'])
        else:
            dataset = SulciDataset([gfile], self.dict_sulci, train=False, translation_file=self.trfile,
                                   dict_bck2={gfile: bck2}, dict_names={gfile: names}, img_size=imgsize,
                                   device=self.device if self.device.type == "cuda" else None)
            inputs, labels = dataset[0]
            pts = np.asarray(bck2) - np.min(bck2, axis=0)
        D, H, W = labels.shape
        lin = torch.as_tensor((pts[:, 0] * H + pts[:, 1]) * W + pts[:, 2], dtype=torch.long).to(self.device)
        exact = self.exact_inference if exact is None else exact
        with torch.no_grad():
            x = inputs.unsqueeze(0).to(self.device)
            scores, preds = self.model.scores_at(x, lin, exact=exact)
        return scores, preds, labels.to(self.device).reshape(-1)[lin]

    # exact_inference (B200 extension): labeling() runs the split-precision forward (bf16x3 tensor-core convolutions,
    # fp32 activations; models.UNet3D.scores_at(exact=True)) whose per-voxel arg-max equals the fp32 reference's
    # wherever the reference's top-2 margin exceeds the documented epsilon.  About 3x the inference time.
    exact_inference = False

    def labeling(self, gfile, bck2=None, names=None, imgsize=None):
        """Returns (ytrue, ypred, yscores): lists over the skeleton points and a float64 [Npoints, C] array."""
        print('Labeling', gfile)
        scores, preds, ytrue = self._labeling_device(gfile, bck2, names, imgsize)
        return ytrue.cpu().tolist(), preds.cpu().tolist(), scores.cpu().numpy().astype(np.float64)

    def test_thresholds(self, gfile_list_test, gfile_list_notcut_test, threshold_range, save_results=True):
        """Threshold sweep of the cutting pass (pattern_class.py:177-245).  Per graph everything between the forward
        pass and the per-threshold ESI stays on the device: scores -> voxel matching (b2_match_voxels) -> fold vote
        for all thresholds (b2_fold_vote) -> TP/FP/FN counters (b2_esi_counts); one small D2H read per graph.
        With torch.distributed initialised, graphs are dealt round-robin to the ranks (no collective on the data
        path) and the per-graph scores are gathered at the end, so every rank returns the reference's result."""
        print('test thresholds')
        since = time.time()
        threshold_range = list(threshold_range)
        for th in threshold_range:
            self.dict_scores[th] = []
        rank, world = self._dist()
        n_classes = len(self.sulci_side_list)
        keep = [self.dict_sulci[ss] for ss in self.sslist]
        mine = {}                                   # graph position -> [score per threshold] or None (ignored)
        pairs = list(zip(gfile_list_test, gfile_list_notcut_test))
        for k, (gfile, gfile_notcut) in enumerate(pairs):
            if k % world != rank:
                continue
            data = self._graph_data(gfile)
            data_nc = self._graph_data(gfile_notcut)
            nbck = np.asarray(data['nbck'], dtype=np.int32).reshape(-1, 3)
            nbck_nc = np.asarray(data_nc['nbck'], dtype=np.int32).reshape(-1, 3)
            vert_nc = np.asarray(data_nc['vert']).reshape(-1)

            print('Labeling', gfile)
            scores, _, _ = self._labeling_device(gfile)

            if len(nbck) != len(nbck_nc):
                print()
                print('ERROR no matches between %s and %s' % (gfile, gfile_notcut))
                print('--- Files ignored to fix the threshold')
                print()
                mine[k] = None
                continue
            # elementary-fold ids: the not-cut graph's vertex ids used directly when they are small non-negative
            # integers (they are vertex indices), else compacted on the host
            if len(vert_nc) and (vert_nc.min() < 0 or vert_nc.max() >= (1 << 20)):
                vert_nc = np.unique(vert_nc, return_inverse=True)[1]
            n_folds = int(vert_nc.max()) + 1 if len(vert_nc) else 1
            dev = self.device
            fold = ops.match_voxels(torch.from_numpy(nbck).to(dev), torch.from_numpy(nbck_nc).to(dev),
                                    torch.from_numpy(vert_nc.astype(np.int32)).to(dev))
            cut = ops.fold_vote(scores, fold, n_folds, [int(t) for t in threshold_range])     # int32 [T, n]
            true_ids = torch.from_numpy(self._name_ids(data['names'])).to(dev)
            counts = torch.zeros((len(threshold_range), 3, n_classes), dtype=torch.int64, device=dev)
            for t in range(len(threshold_range)):
                ops.esi_counts(true_ids, cut[t], n_classes, counts[t])
            counts = counts.cpu()
            mine[k] = [(1 - esi_from_counts(counts[t], keep)) * 100 for t in range(len(threshold_range))]
        if world > 1:
            import torch.distributed as dist
            parts = [None] * world
            dist.all_gather_object(parts, mine)
            mine = {k: v for part in parts for k, v in part.items()}
        for k in sorted(mine):
            if mine[k] is not None:
                for th, sc in zip(threshold_range, mine[k]):
                    self.dict_scores[th].append(sc)
        if save_results:
            store = self.results.setdefault('threshold_scores', {})
            for th, sc in self.dict_scores.items():
                store.setdefault(th, []).append(sc)
        elapsed = time.time() - since
        print('Cutting complete in {:.0f}m {:.0f}s'.format(elapsed // 60, elapsed % 60))

    # ------------------------------------------------------------------------------------------ persistence
    def _dump(self, sub, fname, payload):
        os.makedirs(op.join(self.working_path, sub), exist_ok=True)
        with open(op.join(self.working_path, sub, fname), 'w') as f:
            json.dump(payload, f)

    def save_data(self, name=None):
        fname = self.model_name + '.json' if name is None else name + '_data.json'
        self._dump('data', fname, {'dict_bck2': self.dict_bck2, 'dict_names': self.dict_names,
                                   'sulci_side_list': self.sulci_side_list})
        print('Data saved')

    def _model_path(self, name):
        if name is None:
            return op.join(self.working_path, 'models', self.model_name + '_model.mdsm')
        return op.join(self.working_path, 'models', self.model_name, name + '_model.mdsm')

    def save_model(self, name=None):
        path = self._model_path(name)
        os.makedirs(op.dirname(path), exist_ok=True)
        self.model.to(torch.device('cpu'))          # the reference leaves the model on the CPU (pattern_class.py:303)
        torch.save(self.model.state_dict(), path)
        print('Model saved')

    def save_results(self, name=None):
        self._dump('results', (self.model_name if name is None else name) + '_results.json', self.results)
        print('Results saved')

    def save_params(self, best_threshold=None, name=None):
        os.makedirs(op.join(self.working_path, 'models'), exist_ok=True)
        self.dict_model['model_file'] = self._model_path(name)
        self.dict_model['out_channels'] = len(self.sulci_side_list)
        if self.model is not None and self.model.conv_bias:   # bias-free runs write the reference's keys only
            self.dict_model['conv_bias'] = True
        else:
            self.dict_model.pop('conv_bias', None)
        params = {'dict_bck2': self.dict_bck2, 'dict_names': self.dict_names,
                  'sulci_side_list': self.sulci_side_list, 'dict_model': self.dict_model}
        if best_threshold is not None:
            params['cutting_threshold'] = best_threshold
        folder = op.join(self.working_path, 'models', self.model_name)
        if not op.exists(folder):
            folder = op.join(self.working_path, 'models')
        fname = (self.model_name if name is None else name) + '_params.json'
        with open(op.join(folder, fname), 'w') as f:
            json.dump(params, f)
        print('Parameters saved')

    def reset_results(self):
        self.results = {}

    def load_saved_model(self, dict_model):
        dict_model = self.fill_dict_model(dict_model)
        self.model = UNet3D(dict_model['in_channels'], dict_model['out_channels'],
                            final_sigmoid=dict_model['final_sigmoid'], interpolate=dict_model['interpolate'],
                            conv_layer_order=dict_model['conv_layer_order'],
                            init_channel_number=dict_model['init_channel_number'],
                            conv_bias=dict_model.get('conv_bias', False))
        self.model.final_conv = make_head(dict_model['init_channel_number'], dict_model['out_channels'],
                                          dict_model['num_conv'])
        self.model.load_state_dict(torch.load(dict_model['model_file'], map_location='cpu'))
        self.model.to(self.device)
        print("Model Loaded !")

    # ------------------------------------------------------------------------------------------ shared epoch loop
    def _loaders(self, gfile_list_train, gfile_list_test, batch_size, num_epochs):
        """Train / val DataLoaders as the reference builds them (training.py:84-136): batch 1 uses each subject's own
        bounding box; batch > 1 pads every volume to the largest box seen over `num_epochs` augmented passes."""
        import random

        def make(files, train, img_size=None):
            # volumes are built on the device from the point list (b2_scatter_volume, SURVEY §8 f-1)
            return SulciDataset(files, self.dict_sulci, train=train, translation_file=self.trfile,
                                dict_bck2=self.dict_bck2, dict_names=self.dict_names, img_size=img_size,
                                device=self.device if self.device.type == "cuda" else None,
                                resident=self.resident_points)

        def loader(ds):
            return torch.utils.data.DataLoader(ds, batch_size=batch_size, shuffle=False, num_workers=0)

        def max_size(ds, passes):
            size = [0, 0, 0]
            for _ in range(passes):
                for k in range(len(ds)):                 # same random draws as building the samples, no volumes
                    shp = ds.item_size(k)
                    size = [max(size[i], shp[i]) for i in range(3)]
            return size

        sizes = {}
        print('Extract validation dataloader...')
        if batch_size == 1:
            valloader = loader(make(gfile_list_test, False, self.img_size))
        else:
            sizes['val'] = max_size(make(gfile_list_test, False), 1)
            print('Val dataset image size:', sizes['val'], sep=' ')
            valloader = loader(make(gfile_list_test, False, sizes['val']))
        print('Extract train dataloader...')
        if batch_size == 1:
            trainloader = loader(make(gfile_list_train, True, self.img_size))
        else:
            random.seed(42)
            np.random.seed(42)
            sizes['train'] = max_size(make(gfile_list_train, True), num_epochs)
            print('Train dataset image size:', sizes['train'], sep=' ')
            trainloader = loader(make(gfile_list_train, True, sizes['train']))
            np.random.seed(42)
            random.seed(42)
        return trainloader, valloader, sizes

    def _dist(self):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist.get_rank(), dist.get_world_size()
        return 0, 1

    # -- CUDA-graph replay of the whole step ---------------------------------------------------------------------
    # A step is ~125 kernel launches; enqueueing them from Python costs ~5 ms against ~7 ms of GPU time.  When the
    # same volume shape keeps coming back (dict_model['img_size'], the batch > 1 padding of training.py:119-134,
    # benchmarks) the step — forward, loss, backward, SGD and the epoch-metric counters — is captured once into CUDA
    # graphs and replayed; shapes that do not repeat (every subject of a cohort trained with batch 1 and no img_size
    # has its own bounding box) keep running eagerly.  `use_cuda_graph = False` turns replay off.
    # Data parallel: NCCL is NOT captured.  The step is cut into graph segments at the points where a gradient bucket
    # closes; between the replays of two segments the bucket's all-reduce is enqueued eagerly on the communication
    # stream, so it still overlaps the rest of the backward pass; the last segment (fused SGD) is replayed after the
    # compute stream has waited for every all-reduce.
    use_cuda_graph = True
    # data parallel: capture the NCCL all-reduces INSIDE the step's graph (fork / join of the communication stream is
    # recorded by the capture) instead of cutting the step into segments around eager collectives: one replay per
    # step.  B2_DP_CAPTURE_NCCL=0 selects the segmented form.
    dp_capture_nccl = os.environ.get("B2_DP_CAPTURE_NCCL", "1") != "0"
    _graph_cache_limit = 24       # captured shapes kept (each holds its own ~2.5 GB activation pool at 96x112x96);
    _graph_min_free_frac = 0.30   # ... but never capture another one with less than this fraction of HBM free
    _graph_capture_after = 2      # eager sightings of a (shape, optimiser, mask) key before it is captured

    def _graph_key(self, shape, optimizer):
        mask = tuple(bool(p.requires_grad) for p in self.model.ordered_parameters())
        return (tuple(shape), id(optimizer), float(optimizer.param_groups[0]["lr"]), float(optimizer.momentum), mask)

    def _step_metrics(self):
        """Persistent device accumulators of the epoch metrics (training.py:215-225): TP/FP/FN int64 [3, C] and
        float64 [2] = (sum of batch-mean loss x batch size, samples).  Static addresses: the captured step adds to them."""
        m = self.__dict__.get("_metrics")
        n_classes = len(self.sulci_side_list)
        if m is None or m["counts"].shape[1] != n_classes or m["counts"].device != self.device:
            m = self.__dict__["_metrics"] = dict(
                counts=torch.zeros((3, n_classes), dtype=torch.int64, device=self.device),
                loss=torch.zeros(2, dtype=torch.float64, device=self.device), n_classes=n_classes)
        return m

    def _eager_step(self, x, y, optimizer, reducer, metrics=None, loss_scale=1.0):
        """forward + loss + backward (+ bucketed all-reduce) + SGD, enqueued kernel by kernel.  loss_scale 0 = the
        zero-weight padding step of an uneven data-parallel tail: same collectives, zero gradient contribution, no
        metrics."""
        if reducer is not None:
            reducer.begin()
        loss, _, preds, grads = self.model.forward_backward(x, y, outs=reducer.outs() if reducer is not None else None,
                                                            loss_scale=loss_scale)
        if reducer is not None:
            grads = [g if n is not None else None for g, n in zip(reducer.finish(), grads)]
        optimizer.step(grads=grads)
        if metrics is not None and loss_scale != 0:
            ops.step_metrics(y, preds, metrics["n_classes"], metrics["counts"], loss, float(x.shape[0]),
                             metrics["loss"])
        return loss

    def _capture_segments(self, sx, sy, optimizer, reducer, metrics):
        """Records one eager step into a list of (CUDAGraph, actions) segments; actions = list of ("reduce", bucket)
        / ("finish", None): what has to be enqueued eagerly after that segment's replay."""
        import gc
        segs, cur = [], []
        pool = torch.cuda.graph_pool_handle()
        side = torch.cuda.Stream(device=sx.device)

        dbg = os.environ.get("B2_DEBUG_DP") == "1"

        def begin():
            if dbg:
                print("[b2 dp-graph] capture segment %d" % len(segs), file=sys.stderr, flush=True)
            g = torch.cuda.CUDAGraph()
            # thread_local: the NCCL watchdog thread may query events while this thread captures
            g.capture_begin(pool=pool, capture_error_mode="thread_local")
            cur.append(g)

        mark = [ops.LAUNCHES[0]]

        def cut(action):
            if ops.LAUNCHES[0] == mark[0] and segs:     # nothing enqueued since the last cut: no empty graph
                segs[-1][1].append(action)
                return
            g = cur.pop()
            g.capture_end()
            segs.append((g, [action]))
            mark[0] = ops.LAUNCHES[0]
            begin()

        gc.collect()
        torch.cuda.synchronize()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            if reducer is not None and not (self.dp_capture_nccl and reducer.world > 1):
                reducer.segment_cb = cut
            # the loss is final once the head has run: a cut here lets train_step() read it back (and return, and
            # start the next step's H2D copies) while the backward pass of this step is still running
            self.model.post_head_hook = lambda: cut(("loss", None))
            # the captured step must contain the bf16 re-pack of every trainable layer even if the packs happen to be
            # fresh right now (an eval / labeling pass since the last SGD step): replays follow SGD steps
            self.model.force_repack = True
            begin()
            try:
                loss = self._eager_step(sx, sy, optimizer, reducer, metrics)
            finally:
                self.model.force_repack = False
                self.model.post_head_hook = None
                if reducer is not None:
                    reducer.segment_cb = None
                g = cur.pop()
                g.capture_end()
            segs.append((g, []))
        torch.cuda.current_stream().wait_stream(side)
        return segs, loss

    def _graphed_step(self, x, y, optimizer, reducer=None, metrics=None, read_loss=False):
        """x, y: device tensors, or HOST tensors (pinned).  Host inputs are software-pipelined: they are copied into
        staging buffers on a copy stream (this overlaps the PREVIOUS step's backward pass, because train_step()
        returns as soon as that step's loss is final), then device-to-device into the graph's static inputs.
        read_loss: the loss is copied to pinned host memory right after the head (see _take_loss).
        Returns the [2] loss tensor (mean, sum) of the step that was just enqueued."""
        cache = self.__dict__.setdefault("_graphs", {})
        seen = self.__dict__.setdefault("_graph_seen", {})
        key = self._graph_key(x.shape, optimizer) + (id(reducer), id(metrics) if metrics is not None else 0)
        ent = cache.get(key)
        if ent is None and not x.is_cuda:
            x = x.to(self.device, non_blocking=True)
            y = y.to(self.device, non_blocking=True)
        if ent is None:
            n_seen = seen.get(key, 0)
            if n_seen < self._graph_capture_after:   # real eager steps first (workspaces, momentum buffers; and the
                if len(seen) > 4096:                  # shape has to prove that it comes back)
                    seen.clear()
                seen[key] = n_seen + 1
                return self._eager_step(x, y, optimizer, reducer, metrics)
            free, total = torch.cuda.mem_get_info(self.device)
            while cache and (len(cache) >= self._graph_cache_limit or free < self._graph_min_free_frac * total):
                cache.pop(next(iter(cache)))          # oldest first; its private pool goes back to the allocator
                torch.cuda.empty_cache()
                free, total = torch.cuda.mem_get_info(self.device)
            sx, sy = torch.empty_like(x), torch.empty_like(y)
            sx.copy_(x)
            sy.copy_(y)
            try:
                segs, loss = self._capture_segments(sx, sy, optimizer, reducer, metrics)   # records, does not execute
            except Exception as e:
                print("unetsulc_b200: CUDA-graph capture failed (%s); continuing without graphs" % e)
                self.use_cuda_graph = False
                return self._eager_step(x, y, optimizer, reducer, metrics)
            stage = dict(x=torch.empty_like(sx), y=torch.empty_like(sy), free_ev=None, loss_ev=None,
                         loss_host=torch.empty(2, dtype=torch.float32).pin_memory())
            ent = cache[key] = (segs, sx, sy, loss, stage)
        else:
            segs, sx, sy, loss, stage = ent
            if x.is_cuda:
                sx.copy_(x, non_blocking=True)
                sy.copy_(y, non_blocking=True)
            else:
                cs = self.__dict__.get("_copy_stream")
                if cs is None:
                    cs = self.__dict__["_copy_stream"] = torch.cuda.Stream(device=self.device)
                cur = torch.cuda.current_stream()
                with torch.cuda.stream(cs):
                    if stage["free_ev"] is not None:      # the previous step has copied the staging buffers out
                        cs.wait_event(stage["free_ev"])
                    stage["x"].copy_(x, non_blocking=True)
                    stage["y"].copy_(y, non_blocking=True)
                    staged = torch.cuda.Event()
                    staged.record()
                cur.wait_event(staged)
                sx.copy_(stage["x"], non_blocking=True)   # stream order: after the previous replay's last read of sx
                sy.copy_(stage["y"], non_blocking=True)
                stage["free_ev"] = torch.cuda.Event()
                stage["free_ev"].record()
        dbg = os.environ.get("B2_DEBUG_DP") == "1"
        for k, (g, actions) in enumerate(ent[0]):
            if dbg:
                print("[b2 dp-graph] replay segment %d/%d then %r" % (k, len(ent[0]), actions), file=sys.stderr,
                      flush=True)
            g.replay()
            for action in actions:
                if os.environ.get("B2_DP_GRAPH_SYNC") == "1":   # debugging aid: no compute / collective concurrency
                    torch.cuda.synchronize()
                if action[0] == "reduce":
                    reducer._launch(action[1])
                elif action[0] == "loss":
                    if read_loss:                         # early read-back: the backward pass keeps running
                        stage["loss_host"].copy_(ent[3], non_blocking=True)
                        stage["loss_ev"] = torch.cuda.Event()
                        stage["loss_ev"].record()
                        self.__dict__["_pending_loss"] = stage
                else:
                    reducer.finish()
        # the replayed SGD changed the fp32 masters behind PyTorch's back: bump their version counters so that eager
        # paths (validation, labeling, state_dict consumers) re-pack the bf16 weights
        for p in self.model.ordered_parameters():
            if p.requires_grad:
                torch.autograd.graph.increment_version(p)
        return ent[3]

    def _take_loss(self, loss):
        """the step's loss as a Python float: from the pinned early read-back when there is one, else a D2H read"""
        pend = self.__dict__.pop("_pending_loss", None)
        if pend is not None:
            pend["loss_ev"].synchronize()
            return float(pend["loss_host"][0])
        return float(loss[0].item())

    def train_step_device(self, x, y, optimizer, reducer=None):
        """One training step on DEVICE tensors, no host synchronisation.  Returns the [2] loss tensor (mean, sum)."""
        self.model.train()
        if self.use_cuda_graph:
            return self._graphed_step(x, y, optimizer, reducer)
        return self._eager_step(x, y, optimizer, reducer)

    def train_step(self, inputs, labels, optimizer, reducer=None):
        """One training step from HOST tensors (pinned memory recommended): H2D copy, fused forward + loss +
        backward, gradient all-reduce when data parallel, fused SGD.  Returns the loss as a Python float (one D2H
        read), i.e. what the reference's batch loop does per batch (training.py:198-215)."""
        if self.use_cuda_graph and not inputs.is_cuda and not labels.is_cuda and labels.dtype == torch.int64:
            # graph replay, software-pipelined: the loss is read back as soon as the head has run, so this call returns
            # while the backward pass is still on the GPU and the next call's H2D copies overlap it
            self.model.train()
            return self._take_loss(self._graphed_step(inputs, labels, optimizer, reducer, read_loss=True))
        x = inputs.to(self.device, non_blocking=True)
        y = labels.to(self.device, non_blocking=True)
        loss = self.train_step_device(x, y, optimizer, reducer)
        return float(loss[0].item())

    @staticmethod
    def _iter_batches(loader, rank, world, pad):
        """Batches of `loader` for this rank as (inputs, labels, weight).  One rank: the DataLoader as is.  Data
        parallel over subjects (SURVEY §8(e)): batch b goes to rank b % world; the random draws of the other ranks'
        subjects are consumed so that every rank follows the seeded sequence of a single-process run; when the number
        of batches is not a multiple of `world` and `pad` is set, the ranks without a batch re-run their last batch
        with weight 0, so that every rank issues the same collectives."""
        if world == 1:
            for inputs, labels in loader:
                yield inputs, labels, 1.0
            return
        import random
        ds = loader.dataset
        bs = loader.batch_size or 1
        n = len(ds)
        n_batches = (n + bs - 1) // bs
        # ownership and step count come from parallel.shard_subjects: batch b -> rank b % world, every rank the same
        # number of steps (weight 0 = padding step)
        plan = parallel.shard_subjects(range(n_batches), rank, world)
        owned = {b for b, wgt in plan if wgt > 0}
        last = None
        for step in range(len(plan)):
            mine = None
            for r in range(world):
                b = step * world + r
                idx = range(b * bs, min((b + 1) * bs, n)) if b < n_batches else ()
                if r == rank and len(idx):
                    assert b in owned
                    items = [ds[i] for i in idx]
                    mine = (torch.stack([it[0] for it in items]), torch.stack([it[1] for it in items]))
                elif hasattr(ds, "consume_draws"):
                    for i in idx:
                        ds.consume_draws(i)
            if mine is not None:
                last = mine
                yield mine[0], mine[1], 1.0
            elif pad:
                if last is None:   # fewer batches than ranks: any real sample will do (its draws are rolled back)
                    st, nst = random.getstate(), np.random.get_state()
                    item = ds[0]
                    random.setstate(st)
                    np.random.set_state(nst)
                    last = (item[0].unsqueeze(0), item[1].unsqueeze(0))
                yield last[0], last[1], 0.0

    def _run_phase(self, phase, loader, optimizer, reducer, before_step=None):
        """One pass over `loader`.  Returns (epoch_loss, epoch_acc).  Losses and ESI counters stay on the device
        until the end of the phase (one D2H read per phase instead of three per batch, training.py:215-217)."""
        train = phase == 'train'
        self.model.train() if train else self.model.eval()
        rank, world = self._dist()
        cuda = self.device.type == "cuda"
        metrics = self._step_metrics()
        metrics["counts"].zero_()
        metrics["loss"].zero_()
        if cuda:
            torch.cuda.synchronize(self.device)
        t0 = time.time()
        steps = 0
        for inputs, labels, weight in self._iter_batches(loader, rank, world, pad=train):
            inputs = inputs.to(self.device, non_blocking=True)
            labels = labels.to(self.device, non_blocking=True)
            if train:
                if before_step is not None:
                    before_step()
                want_loss = self.step_callback is not None and weight > 0
                if self.use_cuda_graph and cuda and weight == 1.0:
                    loss = self._graphed_step(inputs, labels, optimizer, reducer, metrics, read_loss=want_loss)
                else:
                    loss = self._eager_step(inputs, labels, optimizer, reducer, metrics, loss_scale=weight)
                if want_loss:
                    self.step_callback(phase, steps, self._take_loss(loss))
            elif weight > 0:
                with torch.no_grad():
                    loss, preds = self.model.loss_and_preds(inputs, labels)
                ops.step_metrics(labels, preds, metrics["n_classes"], metrics["counts"], loss.reshape(1),
                                 float(inputs.size(0)), metrics["loss"])
            steps += 1
        total = len(loader.dataset)
        if cuda:
            ops.check_oob(self.device)       # samples built on the device report out-of-volume points here
        loss_sum, n_seen = (float(v) for v in metrics["loss"].cpu())          # the phase's one D2H read
        counts, loss_total, _ = parallel.allreduce_metrics(metrics["counts"].clone(), loss_sum, int(round(n_seen)))
        self.timings.setdefault(phase, []).append({"seconds": time.time() - t0, "steps": steps})
        epoch_loss = loss_total / total
        epoch_acc = 1 - esi_from_counts(counts, [self.dict_sulci[ss] for ss in self.sslist])
        return epoch_loss, epoch_acc

    def _fit(self, lr, momentum, num_epochs, trainloader, valloader, patience, save_results, num_training,
             tb_dir, before_step=None, after_epoch=None):
        """Epoch loop shared by full training and transfer learning.  `after_epoch(epoch, val_loss, state)` may
        change state['lr'] / request a new optimiser (LR division, fine-tuning switch).  Returns elapsed seconds."""
        _, world = self._dist()
        ordered = self.model.ordered_parameters()
        state = {'lr': lr, 'optimizer': SGD(ordered, lr=lr, momentum=momentum, weight_decay=0)}
        # data parallel: the reducer first broadcasts rank 0's parameters (every process initialised its own network)
        reducer = parallel.BucketedGradReducer(self.model) if world > 1 else None
        writer = _summary_writer(tb_dir) if save_results else None
        es_stop = EarlyStopping(patience=patience['early_stopping']) if 'early_stopping' in patience else None

        print('training...')
        since = time.time()
        best_wts = copy.deepcopy(self.model.state_dict())
        best_acc, best_epoch = 0., 0
        for epoch in range(num_epochs):
            print('Epoch {}/{}'.format(epoch, num_epochs - 1))
            print('-' * 10)
            t0 = time.time()
            for phase in ('train', 'val'):
                loader = trainloader if phase == 'train' else valloader
                epoch_loss, epoch_acc = self._run_phase(phase, loader, state['optimizer'], reducer, before_step)
                print('{} Loss: {:.4f} Acc: {:.4f}'.format(phase, epoch_loss, epoch_acc))
                if save_results:
                    if writer is not None:
                        writer.add_scalar('Loss/' + phase, epoch_loss, epoch)
                        writer.add_scalar('Accuracy/' + phase, epoch_acc, epoch)
                    if epoch == 0:
                        self.results['epoch_loss_' + phase].append([epoch_loss])
                        self.results['epoch_acc_' + phase].append([epoch_acc])
                    else:
                        self.results['epoch_loss_' + phase][num_training].append(epoch_loss)
                        self.results['epoch_acc_' + phase][num_training].append(epoch_acc)
                if phase == 'val' and epoch_acc > best_acc:
                    best_acc, best_epoch = epoch_acc, epoch
                    best_wts = copy.deepcopy(self.model.state_dict())
            # epoch_loss is now the VAL loss (CE of the softmax outputs, as in the reference)
            if after_epoch is not None:
                after_epoch(epoch, epoch_loss, state)
                if state.pop('new_optimizer', False):   # a rebuilt optimiser starts with empty momentum buffers
                    state['optimizer'] = SGD(ordered, lr=state['lr'], momentum=momentum)
            if es_stop is not None:
                es_stop(epoch_loss, self.model)
                if es_stop.early_stop:
                    print("Early stopping")
                    break
            print('Epoch took %i s.' % (time.time() - t0))
            print('\n')
        elapsed = time.time() - since
        print('Training complete in {:.0f}m {:.0f}s'.format(elapsed // 60, elapsed % 60))
        print('Best val Acc: {:4f}, Epoch {}'.format(best_acc, best_epoch))
        if save_results:
            self.results['best_acc'].append(best_acc)
            self.results['best_epoch'].append(best_epoch)
            self.results['duration'].append(elapsed)
            if writer is not None:
                writer.close()
        if reducer is not None:
            self.model.grad_ready_hook = None
        # the captured steps of this training reference its optimiser and buckets: release them (and their pools)
        self.__dict__.pop("_graphs", None)
        self.__dict__.pop("_graph_seen", None)
        self.model.load_state_dict(best_wts)
        return elapsed
