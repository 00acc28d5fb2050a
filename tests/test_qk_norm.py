"""QK-norm without a device: the modules and state_dict, seeded construction, the reference's positional signatures, the
norm layers the fused kernel refuses, the C entry points' argument checks, the data-parallel buckets and the flag."""
import ctypes
import os

import pytest
import torch
import torch.nn as nn

import train
from vit_rpe_rope_b200 import _lib
from vit_rpe_rope_b200.dp import BucketedDataParallel
from vit_rpe_rope_b200.models.vit import Attention, Block, VisionTransformer

KW = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=64, depth=3, num_heads=2)
DH = KW["embed_dim"] // KW["num_heads"]
MODES = ["none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed"]


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.load()


def _buf():
    buf = ctypes.create_string_buffer(256)
    return buf, ctypes.cast(buf, ctypes.c_void_p)


def test_modules_and_init():
    a = Attention(64, num_heads=2, qk_norm=True)
    for m in (a.q_norm, a.k_norm):
        assert type(m) is nn.LayerNorm and tuple(m.normalized_shape) == (32,) and m.eps == 1e-5
        assert torch.equal(m.weight, torch.ones(32)) and torch.equal(m.bias, torch.zeros(32))
    off = Attention(64, num_heads=2)
    assert type(off.q_norm) is nn.Identity and type(off.k_norm) is nn.Identity
    # Block hands its own norm_layer to the attention, as timm does
    blk = Block(64, 2, norm_layer=lambda d: nn.LayerNorm(d, eps=1e-6), qk_norm=True)
    assert blk.attn.q_norm.eps == 1e-6 and blk.attn.k_norm.eps == 1e-6 and blk.norm1.eps == 1e-6


@pytest.mark.parametrize("mode", MODES)
def test_qk_norm_adds_exactly_the_norm_tensors(mode):
    plain = VisionTransformer(**KW, pos_encoding=mode).state_dict()
    qk = VisionTransformer(**KW, pos_encoding=mode, qk_norm=True).state_dict()
    want = {f"blocks.{i}.attn.{n}_norm.{p}" for i in range(KW["depth"]) for n in "qk" for p in ("weight", "bias")}
    assert set(qk) - set(plain) == want and set(plain) <= set(qk)
    for k in want:
        assert qk[k].shape == (DH,) and qk[k].dtype == torch.float32
        assert torch.equal(qk[k], torch.ones(DH) if k.endswith("weight") else torch.zeros(DH))
    assert list(VisionTransformer(**KW, pos_encoding=mode, qk_norm=False).state_dict()) == list(plain)


@pytest.mark.parametrize("mode", ["absolute", "rope-mixed"])
def test_qk_norm_leaves_the_seeded_initial_weights_alone(mode):
    kw = dict(KW, pos_encoding=mode, reg_tokens=2, init_values=1e-5)
    torch.manual_seed(5)
    a = VisionTransformer(**kw).state_dict()
    after_plain = torch.get_rng_state()
    torch.manual_seed(5)
    b = VisionTransformer(**kw, qk_norm=True).state_dict()
    assert torch.equal(torch.get_rng_state(), after_plain)  # construction draws no random numbers of its own
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_reference_positional_signatures():
    a = Attention(64, 2, False, 0., 0.1)
    assert a.num_heads == 2 and a.proj_drop.p == 0.1 and type(a.q_norm) is nn.Identity
    blk = Block(64, 2, 4., False, 0.1, 0., 0.05, nn.GELU, nn.LayerNorm)
    assert blk.mlp.fc1.out_features == 256 and type(blk.attn.k_norm) is nn.Identity
    vit = VisionTransformer(32, 4, 3, 10, 64, 2, 2, 4., "rope-mixed", 100.0, 3, True)
    assert vit.head_dim == 32 and type(vit.blocks[0].attn.q_norm) is nn.Identity


class _RMSNorm(nn.Module):
    def __init__(self, d, eps=1e-6):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(d))
        self.eps = eps

    def forward(self, x):
        return x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + self.eps) * self.weight


@pytest.mark.parametrize("norm_layer", [_RMSNorm, lambda d: nn.LayerNorm(d, elementwise_affine=False),
                                        lambda d: nn.LayerNorm(d, bias=False)], ids=["rmsnorm", "no-affine", "no-bias"])
def test_other_norm_layers_raise(norm_layer):
    with pytest.raises(NotImplementedError, match="qk_norm"):
        Attention(64, num_heads=2, qk_norm=True, norm_layer=norm_layer)
    with pytest.raises(NotImplementedError, match="qk_norm"):
        Block(64, 2, norm_layer=norm_layer, qk_norm=True)
    Block(64, 2, norm_layer=norm_layer)  # without qk_norm the norm layer is the block's own business


def _fwd(lib, p, qn=(1, 1, 1, 1), saved=(1, 1), eps=1e-5):
    g = [p if f else None for f in qn]
    s = [p if f else None for f in saved]
    return lib.vrr_qkv_rope_norm_fwd(p, p, p, p, None, p, 2, 17, 128, 2, 1, _lib.ROPE_AXIAL, _lib.VRR_BF16, *g, eps, *s, None)


def _bwd(lib, p, qn=(1, 1, 1, 1), grads=(1, 1, 1, 1), cs=(1, 1)):
    g = [p if f else None for f in qn]
    d = [p if f else None for f in grads]
    c = [p if f else None for f in cs]
    return lib.vrr_qkv_rope_norm_bwd(p, p, p, p, p, *g, p, *c, *d, 2, 17, 128, 2, 1, _lib.ROPE_AXIAL, _lib.VRR_BF16, None)


def test_c_abi_rejects_inconsistent_pointer_sets(lib):
    _, p = _buf()
    for qn in [(0, 1, 1, 1), (1, 1, 1, 0), (0, 0, 0, 0)]:
        assert _fwd(lib, p, qn=qn) == -1 and "required" in _lib.last_error()
        assert _bwd(lib, p, qn=qn) == -1 and "required" in _lib.last_error()
    for saved in [(1, 0), (0, 1)]:
        assert _fwd(lib, p, saved=saved) == -1 and "qk_pre" in _lib.last_error()
    assert _fwd(lib, p, eps=-1.0) == -1
    for grads in [(1, 0, 1, 1), (0, 0, 0, 1), (1, 1, 1, 0)]:
        assert _bwd(lib, p, grads=grads) == -1 and "d_qn_w" in _lib.last_error()
    assert _bwd(lib, p, cs=(1, 0)) == -1 and "d_cos" in _lib.last_error()
    assert lib.vrr_qkv_rope_norm_fwd(p, p, p, p, None, p, 2, 17, 128, 2, 0, _lib.ROPE_AXIAL, _lib.VRR_BF16, p, p, p, p,
                                     1e-5, p, p, None) == -1  # n_prefix 0


def test_c_abi_valid_sets_reach_the_device_check(lib):
    if torch.cuda.is_available():
        pytest.skip("checks the CPU-only failure mode")
    _, p = _buf()
    assert _fwd(lib, p) == -3 and _fwd(lib, p, saved=(0, 0)) == -3
    assert _bwd(lib, p) == -3 and _bwd(lib, p, grads=(0, 0, 0, 0), cs=(0, 0)) == -3


def test_norm_parameters_go_to_the_normal_buckets():
    m = VisionTransformer(**KW, pos_encoding="rope-mixed", qk_norm=True)
    late = BucketedDataParallel._late_parameter_ids(m)
    for b in m.blocks:
        for t in (b.attn.q_norm.weight, b.attn.q_norm.bias, b.attn.k_norm.weight, b.attn.k_norm.bias):
            assert id(t) not in late


def test_train_flag():
    assert train.get_args([]).qk_norm is False
    assert train.get_args(["--qk_norm"]).qk_norm is True
