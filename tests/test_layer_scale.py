"""LayerScale without a device: the constructor, the state_dict, seeded construction, the C entry points' argument
checks, the data-parallel buckets and the training flag."""
import ctypes
import os

import pytest
import torch
import torch.nn as nn

import train
from vit_rpe_rope_b200 import _lib
from vit_rpe_rope_b200.dp import BucketedDataParallel
from vit_rpe_rope_b200.models.vit import Block, LayerScale, VisionTransformer

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


@pytest.mark.parametrize("init_values", [None, 0, 0.0])
def test_no_layer_scale_keeps_the_state_dict(init_values):
    plain = VisionTransformer(**KW, pos_encoding="rope-mixed")
    off = VisionTransformer(**KW, pos_encoding="rope-mixed", init_values=init_values)
    assert list(off.state_dict()) == list(plain.state_dict())
    assert all(type(b.ls1) is nn.Identity and type(b.ls2) is nn.Identity for b in off.blocks)


@pytest.mark.parametrize("mode", ["none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed"])
def test_layer_scale_adds_exactly_the_gammas(mode):
    plain = VisionTransformer(**KW, pos_encoding=mode).state_dict()
    ls = VisionTransformer(**KW, pos_encoding=mode, init_values=1e-5).state_dict()
    want = {f"blocks.{i}.ls{j}.gamma" for i in range(KW["depth"]) for j in (1, 2)}
    assert set(ls) - set(plain) == want and set(plain) <= set(ls)
    for k in want:
        assert ls[k].shape == (KW["embed_dim"],) and ls[k].dtype == torch.float32
        assert torch.equal(ls[k], torch.full((KW["embed_dim"],), 1e-5))


@pytest.mark.parametrize("mode", ["absolute", "rope-mixed"])
def test_layer_scale_leaves_the_seeded_initial_weights_alone(mode):
    torch.manual_seed(5)
    a = VisionTransformer(**KW, pos_encoding=mode, reg_tokens=2).state_dict()
    torch.manual_seed(5)
    b = VisionTransformer(**KW, pos_encoding=mode, reg_tokens=2, init_values=1e-5).state_dict()
    for k in a:
        assert torch.equal(a[k], b[k]), k
    # and construction draws no random numbers of its own: the generator ends where it ends without LayerScale
    torch.manual_seed(5)
    VisionTransformer(**KW, pos_encoding=mode, reg_tokens=2)
    after_plain = torch.get_rng_state()
    torch.manual_seed(5)
    VisionTransformer(**KW, pos_encoding=mode, reg_tokens=2, init_values=1e-5)
    assert torch.equal(torch.get_rng_state(), after_plain)


def test_block_and_layer_scale_semantics():
    blk = Block(64, 2, init_values=0.5)
    assert isinstance(blk.ls1, LayerScale) and isinstance(blk.ls2, LayerScale)
    assert [n for n, _ in blk.ls1.named_parameters()] == ["gamma"]
    x = torch.randn(3, 64)
    with torch.no_grad():
        blk.ls1.gamma.uniform_(0.25, 1.0)
    assert torch.equal(blk.ls1(x), x * blk.ls1.gamma)
    # a 16-bit branch times the fp32 parameter gives an fp32 result (timm under autocast)
    assert blk.ls1(x.bfloat16()).dtype == torch.float32


def test_ls_bwd_rejects_d_ls_without_ls_or_branch(lib):
    _, p = _buf()
    M, E = 8, 128
    for ls, branch in [(None, p), (p, None), (None, None)]:
        rc = lib.vrr_add_layernorm_ls_bwd(p, None, p, p, p, p, p, p, p, p, M, E, _lib.VRR_F32, _lib.VRR_F32, None,
                                          ls, branch, p, None)
        assert rc == -1 and "d_ls" in _lib.last_error(), (ls, branch)


def test_ls_entry_points_reach_the_device_check(lib):
    """Valid arguments (d_ls NULL, or with ls and branch; ls NULL) pass the argument checks; without an sm_100 device
    the call then fails loudly."""
    if torch.cuda.is_available():
        pytest.skip("checks the CPU-only failure mode")
    _, p = _buf()
    M, E = 8, 128
    for ls, branch, d_ls in [(p, p, p), (p, None, None), (None, None, None)]:
        rc = lib.vrr_add_layernorm_ls_bwd(p, None, p, p, p, p, p, p, p, p, M, E, _lib.VRR_F32, _lib.VRR_F32, None,
                                          ls, branch, d_ls, None)
        assert rc == -3
    for ls in (p, None):
        rc = lib.vrr_add_layernorm_ls_fwd(p, p, p, p, p, p, p, p, M, E, 1e-5, _lib.VRR_F32, _lib.VRR_F32, None, ls, None)
        assert rc == -3


def test_gammas_go_to_the_normal_buckets():
    m = VisionTransformer(**KW, pos_encoding="rope-mixed", init_values=1e-5)
    late = BucketedDataParallel._late_parameter_ids(m)
    for b in m.blocks:
        assert id(b.ls1.gamma) not in late and id(b.ls2.gamma) not in late


def test_train_flag():
    assert train.get_args([]).init_values is None
    assert train.get_args(["--init_values", "1e-5"]).init_values == 1e-5
