"""CPU: U-Nets whose 14 trunk convolutions carry a bias (the 58-key checkpoint layout) — parameter layout against the
oracle, load_state_dict in every direction, the gradient plumbing's per-layer stride, prefix freezing and the API
classes' .mdsm / _params.json round trips."""
import json
import os

import pytest
import torch

import unetsulc_b200
from oracle import unet3d_ref
from oracle.unet3d_ref import UNet3DRef

TRUNK = ["%s.%d.double_conv.conv%d" % (part, j, k)
         for part, n in (("encoders", 4), ("decoders", 3)) for j in range(n) for k in (1, 2)]
BIAS_KEYS = [t + ".bias" for t in TRUNK]


@pytest.fixture
def biased_oracle(monkeypatch):
    monkeypatch.setattr(unet3d_ref, "CONV_BIAS_WHEN_NORM", True)

    def make(f, seed=0):
        torch.manual_seed(seed)
        ref = UNet3DRef(1, 56, init_channel_number=f)
        with torch.no_grad():   # non-zero biases of both signs
            for k, v in ref.state_dict().items():
                if k in BIAS_KEYS:
                    v.copy_(torch.randn_like(v) * 0.1)
        return ref
    return make


@pytest.mark.parametrize("f, nparams", [(64, 16323832), (32, 4083864)])
def test_biased_layout_matches_the_oracle(biased_oracle, f, nparams):
    ref = biased_oracle(f)
    ours = unetsulc_b200.UNet3D(1, 56, init_channel_number=f, conv_bias=True)
    assert ours.conv_bias and ours.trunk_stride() == 4
    rs, os_ = ref.state_dict(), ours.state_dict()
    assert len(rs) == 58 and list(rs) == list(os_)
    for k in rs:
        assert rs[k].shape == os_[k].shape, k
    assert sum(p.numel() for p in ours.parameters()) == nparams
    assert sum(p.numel() for p in ref.parameters()) == nparams
    assert len(ours.ordered_parameters()) == 58
    # trunk_parameters() order: (w, b, gamma, beta) per layer, the state_dict order
    names = {id(p): n for n, p in ours.named_parameters()}
    want = [t + s for t in TRUNK for s in (".weight", ".bias")]
    got = [names[id(p)] for p in ours.trunk_parameters()]
    assert got[0::4] == want[0::2] and got[1::4] == want[1::2]
    assert all(n.endswith("norm1.weight") or n.endswith("norm2.weight") for n in got[2::4])
    assert all(n.endswith("norm1.bias") or n.endswith("norm2.bias") for n in got[3::4])


def test_ordered_parameters_with_a_chain_head():
    from unetsulc_b200.pattern_class import make_head
    for n in (1, 2, 3):
        m = unetsulc_b200.UNet3D(1, 56, conv_bias=True)
        m.final_conv = make_head(64, 56, n)
        assert len(m.ordered_parameters()) == 56 + 2 * n


def test_load_state_dict_in_every_direction(biased_oracle):
    ref = biased_oracle(64, seed=1)
    sd = ref.state_dict()
    # bias-free model + biased checkpoint: becomes biased, bit for bit
    ours = unetsulc_b200.UNet3D(1, 56)
    assert not ours.conv_bias and len(ours.ordered_parameters()) == 44
    ours.load_state_dict(sd)
    assert ours.conv_bias and len(ours.ordered_parameters()) == 58
    for k, v in ours.state_dict().items():
        assert torch.equal(v, sd[k]), k
    for k in BIAS_KEYS:
        p = dict(ours.named_parameters())[k]
        assert isinstance(p, torch.nn.Parameter) and p.dtype == torch.float32 and p.requires_grad
    # back into the oracle
    back = UNet3DRef(1, 56)
    back.load_state_dict(ours.state_dict())
    for k, v in sd.items():
        assert torch.equal(v, back.state_dict()[k]), k
    # biased model + 44-key checkpoint: becomes bias-free
    torch.manual_seed(2)
    plain_sd = unetsulc_b200.UNet3D(1, 56).state_dict()
    assert len(plain_sd) == 44
    ours.load_state_dict(plain_sd)
    assert not ours.conv_bias and len(ours.state_dict()) == 44 and len(ours.ordered_parameters()) == 44
    for k, v in ours.state_dict().items():
        assert torch.equal(v, plain_sd[k]), k
    assert ours._layers()[0].conv.bias is None


def test_partial_bias_set_is_refused(biased_oracle):
    sd = dict(biased_oracle(64).state_dict())
    missing = BIAS_KEYS[5]
    del sd[missing]
    ours = unetsulc_b200.UNet3D(1, 56)
    with pytest.raises(RuntimeError, match=missing.replace(".", r"\.")):
        ours.load_state_dict(sd)
    assert not ours.conv_bias


def test_layout_switch_rebuilds_the_layer_cache():
    m = unetsulc_b200.UNet3D(1, 56)
    L0 = m._layers()
    m.set_conv_bias(True)
    L1 = m._layers()
    assert L1 is not L0 and all(l.conv.bias is not None for l in L1)
    assert len(m.trunk_parameters()) == 56
    m.set_conv_bias(False)
    assert all(l.conv.bias is None for l in m._layers()) and len(m.trunk_parameters()) == 42


def test_gradient_buckets_cover_a_biased_model():
    from unetsulc_b200 import parallel
    from unetsulc_b200.pattern_class import make_head
    for n in (1, 2):
        m = unetsulc_b200.UNet3D(1, 56, conv_bias=True)
        m.final_conv = make_head(64, 56, n)
        red = parallel.BucketedGradReducer(m)
        params = m.ordered_parameters()
        assert len(red.outs()) == len(params) == 56 + 2 * n
        assert sum(p.numel() for p in params) <= sum(f.numel() for f in red.flat)
        seen = set()
        for i, (p, v, (b, off, cnt)) in enumerate(zip(params, red.outs(), red.slot)):
            layer = parallel.layer_of_param(i, 4)
            assert layer == (14 if i >= 56 else i // 4)
            assert v.shape == p.shape and cnt == p.numel() and off % 4 == 0
            assert b == parallel._BUCKET_OF_LAYER[layer]
            assert (b, off) not in seen
            seen.add((b, off))
            v.fill_(float(i))
            assert float(red.flat[b][off]) == float(i)
        # every conv bias maps to its own layer
        names = {id(p): nm for nm, p in m.named_parameters()}
        for i, p in enumerate(params[:56]):
            if names[id(p)].endswith("conv1.bias") or names[id(p)].endswith("conv2.bias"):
                assert TRUNK[parallel.layer_of_param(i, 4)] + ".bias" == names[id(p)]


def test_prefix_freezing_covers_the_biases(tmp_path):
    from unetsulc_b200.transfer_learning import UnetTransferSulciLabelling
    t = UnetTransferSulciLabelling.__new__(UnetTransferSulciLabelling)
    t.model = unetsulc_b200.UNet3D(1, 56, conv_bias=True)
    for layers in (['final_conv'], ['final_conv', 'decoders.2', 'decoders.1', 'decoders.0']):
        t.training_layers = layers
        t._apply_freeze_mask()
        for name, p in t.model.named_parameters():
            assert p.requires_grad == any(name.startswith(l) for l in layers), name
        trainable = {n for n, p in t.model.named_parameters() if p.requires_grad}
        for k in BIAS_KEYS:
            assert (k in trainable) == k.startswith(tuple(layers))


def _api(tmp_path, dict_model):
    from unetsulc_b200.training import UnetTrainingSulciLabelling
    return UnetTrainingSulciLabelling(graphs=[], hemi='L', cuda=-1, working_path=str(tmp_path), dict_model=dict_model,
                                      sulci_side_list=['S.C._left', 'unknown'], dict_names={}, dict_bck2={})


@pytest.mark.parametrize("biased", [False, True])
def test_mdsm_and_params_json_round_trip(tmp_path, biased):
    dm = {'name': 'm', 'num_filter': 32}
    if biased:
        dm['conv_bias'] = True
    t = _api(tmp_path, dm)
    t.load_network()
    assert t.model.conv_bias == biased
    torch.manual_seed(5)
    with torch.no_grad():
        for p in t.model.parameters():
            p.copy_(torch.randn_like(p))
    want = {k: v.clone() for k, v in t.model.state_dict().items()}
    t.save_model()
    t.save_params()
    params = json.load(open(os.path.join(str(tmp_path), 'models', 'm_params.json')))
    assert ('conv_bias' in params['dict_model']) == biased
    if biased:
        assert params['dict_model']['conv_bias'] is True
    # a fresh object built without the key follows the checkpoint's layout
    t2 = _api(tmp_path / "other", {'name': 'm2'})
    d = dict(params['dict_model'])
    d.pop('conv_bias', None)
    d['init_channel_number'] = 32
    t2.load_saved_model(d)
    assert t2.model.conv_bias == biased
    got = t2.model.state_dict()
    assert list(got) == list(want)
    for k, v in want.items():
        assert torch.equal(got[k], v), k


def test_sgd_takes_58_tensors():
    from unetsulc_b200.optim import SGD
    m = unetsulc_b200.UNet3D(1, 56, conv_bias=True)
    opt = SGD(m.ordered_parameters(), lr=1e-2, momentum=0.9)
    assert len(opt.params) == 58
