"""Register tokens without a device: the prefix-aware C entry points' argument checks, the constructor, the state_dict,
the data-parallel bucket and the training flag."""
import ctypes
import os

import pytest
import torch

import train
from vit_rpe_rope_b200 import _lib, ops
from vit_rpe_rope_b200.dp import BucketedDataParallel
from vit_rpe_rope_b200.models.vit import VisionTransformer

KW = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=64, depth=3, num_heads=2)


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.load()


def _buf():
    buf = ctypes.create_string_buffer(256)
    return buf, ctypes.cast(buf, ctypes.c_void_p)


@pytest.mark.parametrize("n_prefix", [0, -1, 66])
def test_qkv_entry_points_reject_n_prefix_outside_1_to_N(lib, n_prefix):
    _, p = _buf()
    N = 65
    rc = lib.vrr_qkv_rope_fwd_prefix(p, p, p, p, None, p, 2, N, 128, 2, n_prefix, _lib.ROPE_AXIAL, _lib.VRR_F32, None)
    assert rc == -1 and "n_prefix" in _lib.last_error()
    rc = lib.vrr_qkv_rope_bwd_prefix(p, p, p, p, p, None, None, 2, N, 128, 2, n_prefix, _lib.ROPE_AXIAL, _lib.VRR_F32, None)
    assert rc == -1 and "n_prefix" in _lib.last_error()


@pytest.mark.parametrize("n_prefix", [0, -3, 1 << 30])
def test_patch_embed_entry_points_reject_bad_n_prefix(lib, n_prefix):
    _, p = _buf()
    rc = lib.vrr_patch_embed_fwd_prefix(p, p, p, p, n_prefix, None, p, None, 0, 2, 3, 32, 32, 4, 64, _lib.VRR_F32,
                                        _lib.VRR_F32, _lib.VRR_F32, None)
    assert rc == -1 and "n_prefix" in _lib.last_error()
    rc = lib.vrr_patch_embed_bwd_prefix(p, p, None, p, p, n_prefix, None, 2, 3, 32, 32, 4, 64, _lib.VRR_F32,
                                        _lib.VRR_F32, _lib.VRR_F32, None)
    assert rc == -1 and "n_prefix" in _lib.last_error()


def test_valid_n_prefix_reaches_the_device_check(lib):
    """n_prefix = N is accepted (no patch row is rotated); without an sm_100 device the call then fails loudly."""
    if torch.cuda.is_available():
        pytest.skip("checks the CPU-only failure mode")
    _, p = _buf()
    assert lib.vrr_qkv_rope_fwd_prefix(p, p, p, p, None, p, 2, 65, 128, 2, 65, _lib.ROPE_AXIAL, _lib.VRR_F32, None) == -3
    assert lib.vrr_patch_embed_fwd_prefix(p, p, p, p, 5, None, p, None, 0, 2, 3, 32, 32, 4, 64, _lib.VRR_F32,
                                          _lib.VRR_F32, _lib.VRR_F32, None) == -3


def test_rope_table_rows_follow_n_prefix():
    cos = torch.zeros(60, 16)
    assert ops._rope_args(cos, cos, 2, 65, 32, n_prefix=5) == _lib.ROPE_AXIAL
    # a table sized for another prefix count is an error, never reinterpreted
    with pytest.raises(RuntimeError, match="does not broadcast"):
        ops._rope_args(cos, cos, 2, 65, 32)
    mixed = torch.zeros(2, 64, 16)
    assert ops._rope_args(mixed, mixed, 2, 65, 32) == _lib.ROPE_MIXED
    with pytest.raises(RuntimeError, match="does not broadcast"):
        ops._rope_args(mixed, mixed, 2, 65, 32, n_prefix=2)


@pytest.mark.parametrize("mode", ["none", "absolute", "rope-axial", "rope-mixed"])
def test_state_dict_keys_and_prefix_attributes(mode):
    plain = VisionTransformer(**KW, pos_encoding=mode)
    zero = VisionTransformer(**KW, pos_encoding=mode, reg_tokens=0)
    four = VisionTransformer(**KW, pos_encoding=mode, reg_tokens=4)
    assert list(zero.state_dict()) == list(plain.state_dict())
    assert not hasattr(zero, "reg_token") and zero.num_prefix_tokens == 1
    assert set(four.state_dict()) - set(plain.state_dict()) == {"reg_token"}
    assert four.reg_token.shape == (1, 4, KW["embed_dim"]) and four.num_prefix_tokens == 5
    assert all(b.attn.num_prefix_tokens == 5 for b in four.blocks)
    assert all(b.attn.num_prefix_tokens == 1 for b in zero.blocks)


@pytest.mark.parametrize("mode", ["absolute", "rope-mixed"])
def test_registers_leave_the_seeded_initial_weights_alone(mode):
    torch.manual_seed(11)
    a = VisionTransformer(**KW, pos_encoding=mode).state_dict()
    torch.manual_seed(11)
    b = VisionTransformer(**KW, pos_encoding=mode, reg_tokens=4).state_dict()
    for k in a:
        assert torch.equal(a[k], b[k]), k
    r = b["reg_token"]
    assert r.abs().max() < 1e-5 and r.std() > 0  # timm: normal_(std=1e-6)


@pytest.mark.parametrize("mode", ["relative", "polynomial"])
def test_bias_modes_reject_registers(mode):
    with pytest.raises(ValueError, match="reg_tokens"):
        VisionTransformer(**KW, pos_encoding=mode, reg_tokens=1)
    VisionTransformer(**KW, pos_encoding=mode, reg_tokens=0)


def test_negative_reg_tokens_raise():
    with pytest.raises(ValueError, match="reg_tokens"):
        VisionTransformer(**KW, pos_encoding="none", reg_tokens=-1)


def test_reg_token_gradient_goes_to_the_late_bucket():
    m = VisionTransformer(**KW, pos_encoding="rope-mixed", reg_tokens=4)
    late = BucketedDataParallel._late_parameter_ids(m)
    assert id(m.reg_token) in late and id(m.cls_token) in late
    assert id(m.blocks[0].attn.qkv.weight) not in late


def test_train_flag():
    assert train.get_args([]).reg_tokens == 0
    assert train.get_args(["--reg_tokens", "4"]).reg_tokens == 4
