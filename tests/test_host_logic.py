"""CPU: host-side mirror of the reference interface (no compute kernels are called)."""
import copy
import io
import json
import os
import random
import contextlib

import numpy as np
import pytest
import torch
import torch.nn as nn

import unetsulc_b200
from unetsulc_b200 import dataset as ds_mod
from unetsulc_b200 import early_stopping as es_mod
from unetsulc_b200 import parallel, stats
from unetsulc_b200.pattern_class import UnetPatternSulciLabelling, make_head
from unetsulc_b200.training import UnetTrainingSulciLabelling
from unetsulc_b200.transfer_learning import UnetTransferSulciLabelling
from tests import harness

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_plateau_trackers_match_reference_traces():
    """DivideLr / FineTunning decisions equal those of the reference's own classes (fixture generated from
    /root/reference/divide_lr.py and fine_tunning.py)."""
    g = json.load(open(os.path.join(G, "plateau_traces.json")))
    for key, trace in g["traces"].items():
        parts = key.split("/")
        seq = g["loss_sequences"][parts[1]]
        patience = int(parts[2][1:])
        with contextlib.redirect_stdout(io.StringIO()):
            if parts[0] == "divide_lr":
                t = es_mod.DivideLr(patience=patience, repeat=int(parts[3][1:]))
                got = []
                for v in seq:
                    t(v, None)
                    got.append([t.divide_lr, t.stop, t.counter])
            else:
                t = es_mod.FineTunning(patience=patience)
                got = []
                for v in seq:
                    t(v, None)
                    got.append([t.ft_start, t.stop, t.counter])
        assert got == trace, key


def test_early_stopping_rule():
    with contextlib.redirect_stdout(io.StringIO()):
        e = es_mod.EarlyStopping(patience=2)
        for v, want in [(1.0, False), (0.9, False), (0.95, False), (0.96, True), (0.5, True)]:
            e(v, None)
            assert e.early_stop == want


def test_sulci_dataset_matches_reference_volumes():
    """Same volumes / labels as the reference's SulciDataset for seeded draws (incl. rotation augmentation)."""
    g = np.load(os.path.join(G, "dataset_cases.npz"))
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=2, shape=(12, 14, 10), n_classes=5, seed=3)
    dict_sulci = {s: i for i, s in enumerate(sslist)}
    files = sorted(bck2)
    for train in (False, True):
        random.seed(11); np.random.seed(11)
        d = ds_mod.SulciDataset(files, dict(dict_sulci), train=train, dict_bck2=bck2, dict_names=names)
        for i in range(len(files)):
            for rep in range(2 if train else 1):
                x, y = d[i]
                assert x.dtype == torch.float32 and y.dtype == torch.int64
                assert np.array_equal(x.numpy().astype(np.uint8), g["x_train%d_s%d_r%d" % (train, i, rep)])
                assert np.array_equal(y.numpy().astype(np.int16), g["y_train%d_s%d_r%d" % (train, i, rep)])
    d = ds_mod.SulciDataset(files, dict(dict_sulci), train=False, dict_bck2=bck2, dict_names=names,
                            img_size=[16, 16, 16])
    x, y = d[0]
    assert np.array_equal(x.numpy().astype(np.uint8), g["x_fixed"])
    assert np.array_equal(y.numpy().astype(np.int16), g["y_fixed"])


def test_unet3d_module_surface_matches_what_the_reference_uses():
    from oracle.unet3d_ref import UNet3DRef
    m = unetsulc_b200.UNet3D(1, 56, final_sigmoid=False, interpolate=True, dropout=0., conv_layer_order='crg',
                             init_channel_number=64)
    ref = UNet3DRef(1, 56)
    assert list(m.state_dict().keys()) == list(ref.state_dict().keys())
    assert [tuple(v.shape) for v in m.state_dict().values()] == [tuple(v.shape) for v in ref.state_dict().values()]
    ref.load_state_dict(m.state_dict())                       # loads into the reference layout unchanged
    m.load_state_dict(ref.state_dict())
    # prefix freezing (transfer_learning.py:330-335)
    names = [n for n, _ in m.named_parameters()]
    assert sum(n.startswith('final_conv') for n in names) == 2
    assert sum(n.startswith('decoders.2') for n in names) == 6
    # head replaced after construction (pattern_class.py:364) and deepcopy (transfer_learning.py:159)
    m.final_conv = nn.Conv3d(64, 7, 1)
    m2 = copy.deepcopy(m)
    assert m2.final_conv.out_channels == 7 and m2 is not m
    assert len(list(m2.parameters())) == 44
    assert len(m.ordered_parameters()) == 44
    # hard errors instead of silent fallbacks
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 1, 8, 8, 8))
    for kw in (dict(in_channels=2), dict(conv_layer_order='cr'), dict(interpolate=False), dict(final_sigmoid=True),
               dict(init_channel_number=16)):
        args = dict(in_channels=1, out_channels=5)
        args.update(kw)
        with pytest.raises(ValueError):
            unetsulc_b200.UNet3D(**args)


def test_api_classes_keep_reference_constructor_and_results_layout(tmp_path):
    bck2, names, sslist = harness.synthetic_cohort()
    with contextlib.redirect_stdout(io.StringIO()):
        t = UnetTrainingSulciLabelling(sorted(bck2), 'L', cuda=-1, working_path=str(tmp_path),
                                       dict_model={'name': 'm'}, dict_names=names, dict_bck2=bck2,
                                       sulci_side_list=sslist)
    golden = json.load(open(os.path.join(G, "reference_training.json")))
    for k in golden:
        if k not in ('state_dict_keys',):
            assert k in t.results or k in ('duration',), k
    assert t.sslist == [s for s in sslist if not s.startswith('unknown')]
    assert t.dict_sulci['background'] == -1 and t.device.type == 'cpu'
    assert t.num_filter == 64 and t.conv_layer_order == 'crg' and t.interpolate is True
    with contextlib.redirect_stdout(io.StringIO()):
        t.load_network()
        assert isinstance(t.model, unetsulc_b200.UNet3D)
        t.save_model(name='m_cv0'); t.save_results(); t.save_data('cohort'); t.save_params(best_threshold=100, name='m_cv0')
    assert os.path.exists(tmp_path / 'models' / 'm' / 'm_cv0_model.mdsm')
    assert os.path.exists(tmp_path / 'results' / 'm_results.json')
    assert os.path.exists(tmp_path / 'data' / 'cohort_data.json')
    params = json.load(open(tmp_path / 'models' / 'm' / 'm_cv0_params.json'))
    assert params['cutting_threshold'] == 100 and params['dict_model']['out_channels'] == len(sslist)
    sd = torch.load(tmp_path / 'models' / 'm' / 'm_cv0_model.mdsm', map_location='cpu')
    assert list(sd.keys()) == golden['state_dict_keys']
    # transfer class: new-style signature, default layer lists
    with contextlib.redirect_stdout(io.StringIO()):
        tr = UnetTransferSulciLabelling(sorted(bck2), 'L', cuda=-1, working_path=str(tmp_path), dict_model={},
                                        dict_trained_model={'out_channels': len(sslist),
                                                            'model_file': str(tmp_path / 'models' / 'm' / 'm_cv0_model.mdsm')},
                                        dict_names=names, dict_bck2=bck2, sulci_side_list=sslist[:4])
        tr.load_model()
    assert tr.training_layers == ['final_conv'] and tr.fine_tunning_layers == ['decoders.2', 'decoders.1', 'decoders.0']
    assert tr.model.final_conv.out_channels == 4
    tr._apply_freeze_mask()
    assert [n for n, p in tr.model.named_parameters() if p.requires_grad] == ['final_conv.weight', 'final_conv.bias']
    assert isinstance(make_head(64, 10, 3), nn.Sequential)


def test_learning_without_data_returns_1(tmp_path):
    with contextlib.redirect_stdout(io.StringIO()):
        t = UnetTrainingSulciLabelling([], 'L', working_path=str(tmp_path))
        assert t.learning(1e-2, 0.9, 1, [], []) == 1        # reference prints an error and returns 1


def test_esi_score_host_signature():
    assert stats.esi_score([0, 1, 2, 2], [0, 1, 1, 2], [0, 1, 2]) == pytest.approx(2 / 8)
    assert stats.esi_score(['a', 'b'], ['a', 'a'], ['a', 'b']) == pytest.approx(2 / 4)
    c = np.array([[5, 0], [1, 2], [3, 0]])
    assert stats.esi_from_counts(c, [0]) == pytest.approx(4 / 14)


def test_shard_subjects():
    assert parallel.shard_subjects(list(range(5)), 0, 2) == [(0, 1.0), (2, 1.0), (4, 1.0)]
    assert parallel.shard_subjects(list(range(5)), 1, 2) == [(1, 1.0), (3, 1.0), (4, 0.0)]
    assert parallel.shard_subjects([], 0, 4) == []


def test_reference_host_code_runs_unmodified_on_the_boundary(tmp_path):
    """The reference's own training.py (unmodified) driven through the deepsulci import boundary with the oracle:
    must reproduce the committed trace (skipped unless UNETSULC_REFERENCE names a checkout of the reference)."""
    if not harness.reference_available():
        pytest.skip("no checkout of the reference: set UNETSULC_REFERENCE")
    from oracle.unet3d_ref import UNet3DRef
    method = harness.run_reference_training(str(tmp_path), UNet3DRef, n_epochs=2,
                                            patience={'divide_lr': 1, 'early_stopping': 3})
    golden = json.load(open(os.path.join(G, "reference_training.json")))
    for k in ('epoch_loss_train', 'epoch_loss_val', 'epoch_acc_train', 'epoch_acc_val', 'best_acc'):
        assert np.allclose(np.asarray(method.results[k], dtype=float), np.asarray(golden[k], dtype=float),
                           rtol=2e-3, atol=1e-4), k
    assert method.results['divide_lr_epoch'] == golden['divide_lr_epoch']
    assert method.results['best_epoch'] == golden['best_epoch']


def test_num_conv_chain_head_composes_exactly():
    """A chain of 1x1x1 convs without activations (reference pattern_class.py:357-363) is one affine map: the composed
    (W, b) the head kernels use reproduces the sequential application, and autograd reaches every link."""
    import torch.nn.functional as F
    from unetsulc_b200.pattern_class import make_head
    torch.manual_seed(3)
    m = unetsulc_b200.UNet3D(1, 56)
    m.final_conv = make_head(64, 56, 3)
    assert [c.out_channels for c in m.final_conv] == [61, 59, 56]
    hw, hb = m._head_effective()
    assert tuple(hw.shape) == (56, 64, 1, 1, 1) and tuple(hb.shape) == (56,)
    x = torch.randn(2, 64, 3, 4, 5)
    want = m.final_conv(x)
    got = F.conv3d(x, hw, hb)
    assert torch.allclose(got, want, rtol=1e-4, atol=1e-5)
    got.sum().backward()
    assert all(p.grad is not None and p.grad.abs().sum() > 0 for p in m.head_parameters())
    assert len(m.ordered_parameters()) == 42 + 6
    # state_dict round trip with the chain (keys final_conv.0.weight ...)
    m2 = unetsulc_b200.UNet3D(1, 56)
    m2.final_conv = make_head(64, 56, 3)
    m2.load_state_dict(m.state_dict())
    assert "final_conv.2.bias" in m.state_dict()


def test_gradient_buckets_cover_a_chain_head():
    """the bucketed reducer's flat buffers follow ordered_parameters(), also with a num_conv > 1 head (42 + 2n
    tensors): every head tensor lands in bucket 0, views alias the flat buffers, slots are 16-byte aligned"""
    from unetsulc_b200 import parallel
    from unetsulc_b200.pattern_class import make_head
    m = unetsulc_b200.UNet3D(1, 56)
    m.final_conv = make_head(64, 56, 2)
    red = parallel.BucketedGradReducer(m)
    params = m.ordered_parameters()
    assert len(params) == 46 and len(red.outs()) == 46
    assert sum(p.numel() for p in params) <= sum(f.numel() for f in red.flat)
    for i, (p, v, (b, off, n)) in enumerate(zip(params, red.outs(), red.slot)):
        assert v.shape == p.shape and n == p.numel() and off % 4 == 0
        assert b == (0 if i >= 42 else parallel._BUCKET_OF_LAYER[i // 3])
        v.fill_(float(i))
        assert float(red.flat[b][off]) == float(i)
    items = parallel.shard_subjects(list(range(5)), 1, 2)
    assert items == [(1, 1.0), (3, 1.0), (4, 0.0)]


def test_two_limb_statistics_accumulator_is_exact_and_order_independent():
    """numpy mirror of stat_atomic_add / stat_read (csrc/common.h): an fp32 partial sum splits into rint(p) +
    fraction * 2^32 (two int64 limbs) — exactly for |p| >= 2^-9, within 2^-33 otherwise; integer adds commute, so any
    arrival order gives the same bits and the total equals the fp64 sum of the partials."""
    rng = np.random.RandomState(0)
    p = np.concatenate([rng.randn(4096).astype(np.float32) * s for s in (1e-3, 1.0, 1e3, 1e6, 3e9)])
    hi = np.rint(p).astype(np.float32)                     # rintf
    lo = np.rint((p - hi).astype(np.float32) * np.float32(4294967296.0)).astype(np.int64)   # __float2ll_rn
    hi = hi.astype(np.int64)
    back = hi.astype(np.float64) + lo.astype(np.float64) / 4294967296.0
    p64 = p.astype(np.float64)
    assert np.all(np.abs(back - p64) <= 2.0 ** -33)
    big = np.abs(p64) >= 2.0 ** -9
    assert np.array_equal(back[big], p64[big])              # exact decomposition above 2^-9
    perm = rng.permutation(p.size)
    assert hi.sum() == hi[perm].sum() and lo.sum() == lo[perm].sum()
    total = float(hi.sum()) + float(lo.sum()) / 4294967296.0
    ref = float(np.sum(p.astype(np.float64)))
    assert abs(total - ref) <= p.size * 2.0 ** -33 + 1e-12 * abs(ref)


def test_data_parallel_batches_uneven_cohort_and_seeded_draws():
    """Data parallel over subjects (SURVEY §8(e)): every rank runs ceil(batches / world) steps (the tail is padded
    with a zero-weight repeat, ADVICE r1), the union of the weight-1 batches is the cohort, and every rank's samples
    are exactly the ones a single-process run draws (the other ranks' random draws are consumed, not skipped)."""
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=5, shape=(12, 14, 10), n_classes=5, seed=3)
    dict_sulci = {s: i for i, s in enumerate(sslist)}
    files = sorted(bck2)

    def make():
        random.seed(21); np.random.seed(21)
        ds = ds_mod.SulciDataset(files, dict(dict_sulci), train=True, dict_bck2=bck2, dict_names=names)
        return torch.utils.data.DataLoader(ds, batch_size=1, shuffle=False, num_workers=0)

    single = [(x.clone(), y.clone()) for x, y, w in UnetPatternSulciLabelling._iter_batches(make(), 0, 1, True)]
    assert len(single) == 5
    for world in (2, 3, 4, 8):
        seen = {}
        for rank in range(world):
            got = list(UnetPatternSulciLabelling._iter_batches(make(), rank, world, True))
            assert len(got) == -(-5 // world), (world, rank, len(got))     # same number of steps on every rank
            real = [(x, y) for x, y, w in got if w == 1.0]
            assert all(w in (0.0, 1.0) for _, _, w in got)
            assert len(real) == len(range(rank, 5, world))
            for k, (x, y) in zip(range(rank, 5, world), real):
                assert torch.equal(x, single[k][0]) and torch.equal(y, single[k][1]), (world, rank, k)
                seen[k] = True
            for x, y, w in got:                   # padding steps carry a real (labelled) sample
                assert (y >= 0).any()
            # validation never pads
            assert len(list(UnetPatternSulciLabelling._iter_batches(make(), rank, world, False))) == len(real)
        assert sorted(seen) == list(range(5))


def test_item_size_follows_the_same_draws_as_getitem():
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=3, shape=(12, 14, 10), n_classes=5, seed=3)
    dict_sulci = {s: i for i, s in enumerate(sslist)}
    files = sorted(bck2)
    random.seed(5); np.random.seed(5)
    d = ds_mod.SulciDataset(files, dict(dict_sulci), train=True, dict_bck2=bck2, dict_names=names)
    shapes = [tuple(d[i][0].shape[1:]) for i in range(3)]
    random.seed(5); np.random.seed(5)
    assert [d.item_size(i) for i in range(3)] == shapes
    random.seed(5); np.random.seed(5)
    for i in range(3):
        d.consume_draws(i)
    a = (random.random(), np.random.rand())
    random.seed(5); np.random.seed(5)
    for i in range(3):
        d[i]
    assert a == (random.random(), np.random.rand())


def test_workspace_regrowth_retires_instead_of_freeing():
    """A captured CUDA graph keeps the address of the workspace it recorded (ADVICE r1): regrowing a workspace must
    not free the old buffer."""
    from unetsulc_b200 import ops
    a = ops.Workspace.get(1 << 20, "cpu", "t_regrow")
    b = ops.Workspace.get(4 << 20, "cpu", "t_regrow")
    assert b.numel() >= 4 << 20 and any(r is a for r in ops.Workspace._retired)
    assert ops.Workspace.get(1 << 20, "cpu", "t_regrow") is b
