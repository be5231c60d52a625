"""CPU: the 32-filter network (init_channel_number=32) — parameter layout against the oracle, the widths that stay
errors, and the weight-gradient plans of its 13 tensor-core layers."""
import pytest
import torch

import unetsulc_b200
from oracle.unet3d_ref import UNet3DRef

# (Cin, Cout, level) of the 13 3x3x3 convs of UNet3D(1, 56, init_channel_number=32) behind encoders.0.conv1
F32_LAYERS = [
    (16, 32, 0),                  # encoders.0.conv2
    (32, 32, 1), (32, 64, 1),     # encoders.1
    (64, 64, 2), (64, 128, 2),    # encoders.2
    (128, 128, 3), (128, 256, 3),  # encoders.3
    (384, 128, 2), (128, 128, 2),  # decoders.0
    (192, 64, 1), (64, 64, 1),    # decoders.1
    (96, 32, 0), (32, 32, 0),     # decoders.2
]


def test_width32_matches_the_oracle_layout():
    ref = UNet3DRef(1, 56, init_channel_number=32)
    ours = unetsulc_b200.UNet3D(1, 56, init_channel_number=32)
    assert ours.num_groups == 16 and ours.init_channel_number == 32
    rs, os_ = ref.state_dict(), ours.state_dict()
    assert list(rs) == list(os_)
    for k in rs:
        assert rs[k].shape == os_[k].shape, k
    assert sum(p.numel() for p in ours.parameters()) == 4082696
    assert len(ours.ordered_parameters()) == 44
    convs = [(l.cin, l.cout) for l in ours._layers()]
    assert convs == [(1, 16)] + [(ci, co) for ci, co, _ in F32_LAYERS]
    # load_state_dict both ways, bit for bit
    torch.manual_seed(3)
    ref2 = UNet3DRef(1, 56, init_channel_number=32)
    ours.load_state_dict(ref2.state_dict())
    back = UNet3DRef(1, 56, init_channel_number=32)
    back.load_state_dict(ours.state_dict())
    for k, v in ref2.state_dict().items():
        assert torch.equal(v, back.state_dict()[k]), k


@pytest.mark.parametrize("f", [16, 48, 128])
def test_other_widths_stay_errors(f):
    with pytest.raises(ValueError, match="32 or 64"):
        unetsulc_b200.UNet3D(1, 56, init_channel_number=f)


def test_wgrad_plans_of_the_width32_layers():
    """Every f = 32 layer has a weight-gradient plan at the 96 x 112 x 96 box (levels halve it); the plans of the f = 64
    layers and the Cin = 48 refusal are pinned in test_capi.py."""
    from unetsulc_b200 import _lib
    import __graft_entry__ as ge
    ge.build()
    lib = _lib.load()
    dims = [(96, 112, 96), (48, 56, 48), (24, 28, 24), (12, 14, 12)]
    for cin, cout, lvl in F32_LAYERS:
        nbytes = lib.b2_conv3d_wgrad_workspace_bytes(1, *dims[lvl], cin, cout)
        assert nbytes > 0 and nbytes % (27 * cin * cout * 4) == 0, (cin, cout, lvl, nbytes)
    assert lib.b2_conv3d_first_wgrad_workspace_bytes(16) == 592 * 27 * 16 * 4
    for cin, cout in ((8, 32), (24, 32), (48, 32), (32, 16), (32, 48)):
        assert lib.b2_conv3d_wgrad_workspace_bytes(1, 8, 8, 8, cin, cout) == -1, (cin, cout)
