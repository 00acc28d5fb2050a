"""SwiGLU MLP on the host: timm's ``GluMlp`` / ``SwiGLUPacked`` layout, the torch forward, ``mlp_layer`` validation,
the train.py flags and the C prototypes.  No GPU needed."""
import functools
import re

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import train
from vit_rpe_rope_b200 import VisionTransformer, _lib
from vit_rpe_rope_b200.models.vit import Block, GluMlp, Mlp, SwiGLUPacked

TINY = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=2, num_heads=3)


def test_swiglu_packed_is_timms_partial():
    assert isinstance(SwiGLUPacked, functools.partial) and SwiGLUPacked.func is GluMlp
    assert SwiGLUPacked.keywords == dict(act_layer=nn.SiLU, gate_last=False)


def test_glu_mlp_attributes_and_shapes():
    m = SwiGLUPacked(in_features=64, hidden_features=96, out_features=48)
    assert [n for n, _ in m.named_children()] == ["fc1", "act", "drop1", "norm", "fc2", "drop2"]
    assert type(m.act) is nn.SiLU and type(m.norm) is nn.Identity and m.gate_last is False
    assert tuple(m.fc1.weight.shape) == (96, 64) and tuple(m.fc1.bias.shape) == (96,)
    assert tuple(m.fc2.weight.shape) == (48, 48) and tuple(m.fc2.bias.shape) == (48,)
    assert list(m.state_dict()) == ["fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias"]
    d = GluMlp(64)
    assert type(d.act) is nn.Sigmoid and d.gate_last is True and d.fc2.in_features == 32


def test_glu_mlp_odd_width_asserts():
    with pytest.raises(AssertionError):
        GluMlp(64, hidden_features=97)


@pytest.mark.parametrize("gate_last", [False, True])
def test_glu_mlp_forward_is_the_torch_restatement(gate_last):
    torch.manual_seed(0)
    m = GluMlp(32, hidden_features=48, act_layer=nn.SiLU, gate_last=gate_last).eval()
    x = torch.randn(5, 7, 32)
    h = F.linear(x, m.fc1.weight, m.fc1.bias)
    x1, x2 = h[..., :24], h[..., 24:]
    a = x1 * F.silu(x2) if gate_last else F.silu(x1) * x2
    want = F.linear(a, m.fc2.weight, m.fc2.bias)
    assert torch.equal(m(x), want)


def test_model_state_dict_keys_and_shapes():
    model = VisionTransformer(**TINY, mlp_ratio=5.33334, mlp_layer=SwiGLUPacked)
    sd = model.state_dict()
    assert tuple(sd["blocks.0.mlp.fc1.weight"].shape) == (1024, 192)
    assert tuple(sd["blocks.0.mlp.fc1.bias"].shape) == (1024,)
    assert tuple(sd["blocks.1.mlp.fc2.weight"].shape) == (192, 512)
    assert tuple(sd["blocks.1.mlp.fc2.bias"].shape) == (192,)
    gelu = VisionTransformer(**TINY)
    assert list(sd) == list(gelu.state_dict())  # the same keys as the GELU model, in the same order
    assert all(isinstance(b.mlp, GluMlp) for b in model.blocks)


def test_construction_is_deterministic_and_initialised_like_every_linear():
    torch.manual_seed(3)
    a = VisionTransformer(**TINY, mlp_ratio=5.33334, mlp_layer=SwiGLUPacked)
    torch.manual_seed(3)
    b = VisionTransformer(**TINY, mlp_ratio=5.33334, mlp_layer=SwiGLUPacked)
    for (n, p), (_, q) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(p, q), n
    fc1 = a.blocks[0].mlp.fc1
    assert torch.equal(fc1.bias, torch.zeros_like(fc1.bias))
    assert abs(fc1.weight.std().item() - 0.02) < 1e-3  # trunc_normal_(std=0.02), not nn.Linear's default


def test_mlp_layer_validation():
    for bad in (nn.Linear, "swiglu", functools.partial(Mlp), None):
        with pytest.raises(ValueError):
            VisionTransformer(**TINY, mlp_layer=bad)
        with pytest.raises(ValueError):
            Block(64, 2, mlp_layer=bad)
    Block(64, 2, mlp_layer=GluMlp)  # the class itself is a factory too
    assert type(Block(64, 2).mlp) is Mlp


def test_train_flags():
    args = train.get_args(["--mlp_layer", "swiglu", "--mlp_ratio", "5.33334"])
    assert args.mlp_layer == "swiglu" and args.mlp_ratio == pytest.approx(5.33334)
    args = train.get_args([])
    assert args.mlp_layer == "mlp" and args.mlp_ratio == 4.0
    with pytest.raises(SystemExit):
        train.get_args(["--mlp_layer", "geglu"])


def test_c_prototypes_are_declared():
    header = open(_lib.HEADER_PATH).read()
    for name in ("vrr_gemm_swiglu", "vrr_gemm_swiglu_bwd"):
        assert re.search(rf"\bint {name}\(", header) and name in _lib.SIGNATURES
