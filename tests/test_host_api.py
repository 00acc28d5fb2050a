"""Host-side mirror of the reference module API (CPU: construction, tables, state_dict, errors)."""
import ast
import os

import numpy as np
import pytest
import torch

from oracle import make_golden, tables_np as T
from vit_rpe_rope_b200 import models
from vit_rpe_rope_b200.models import positional_encoding as PE
from vit_rpe_rope_b200.models.rope_utils import reshape_for_broadcast
from vit_rpe_rope_b200.models.vit import Attention, VisionTransformer

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
MODES = ("none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed")


@pytest.fixture(scope="module")
def tables():
    return np.load(os.path.join(GOLDEN, "tables.npz"))


def test_module_surface():
    for name in ("Attention", "Block", "VisionTransformer", "NoPositionalEncoding", "AbsolutePositionalEncoding",
                 "RelativePositionalEncoding", "PolynomialRPE", "RoPEAxial", "RoPEMixed", "apply_rotary_emb",
                 "reshape_for_broadcast"):
        assert hasattr(models, name), name
    m = VisionTransformer(pos_encoding="rope-mixed")
    for attr in ("pos_embed", "blocks", "patch_embed", "cls_token", "norm", "head", "num_patches", "head_dim",
                 "num_heads", "patch_size", "embed_dim", "pos_encoding_type", "use_rope", "use_pos_embed_in_forward"):
        assert hasattr(m, attr), attr
    assert m.use_rope and not m.use_pos_embed_in_forward and m.num_patches == 64 and m.head_dim == 32


def test_unknown_mode_raises_value_error():
    with pytest.raises(ValueError, match="Unknown positional encoding type"):
        VisionTransformer(pos_encoding="bogus")


def test_reshape_for_broadcast_contract():
    tgt = torch.zeros(2, 3, 5, 8)
    assert reshape_for_broadcast(torch.zeros(5, 4), tgt).shape == (1, 1, 5, 4)
    assert reshape_for_broadcast(torch.zeros(3, 5, 4), tgt).shape == (1, 3, 5, 4)
    with pytest.raises(ValueError, match="Unexpected tensor shapes"):
        reshape_for_broadcast(torch.zeros(4), tgt)


def test_cpu_tensors_fail_loudly():
    m = VisionTransformer(pos_encoding="none", depth=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 3, 32, 32))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        models.apply_rotary_emb(torch.zeros(1, 1, 4, 8), torch.zeros(1, 1, 4, 8), torch.ones(4, 4), torch.zeros(4, 4))


def test_unsupported_ctor_options_raise():
    with pytest.raises(NotImplementedError):
        Attention(64, qkv_bias=True)
    with pytest.raises(NotImplementedError):
        Attention(64, attn_drop=0.1)


@pytest.mark.parametrize("length", [17, 65])
def test_relative_index_buffer_bit_exact(tables, length):
    m = PE.RelativePositionalEncoding(length - 1, num_heads=2)
    assert m.relative_position_index.dtype == torch.int64
    assert np.array_equal(m.relative_position_index.numpy(), tables[f"rel_index_L{length}"])
    assert m.get_bias().shape == (2, length, length)


def test_relative_get_bias_matches_golden(tables):
    m = PE.RelativePositionalEncoding(64, num_heads=6)
    with torch.no_grad():
        m.relative_position_bias_table.copy_(torch.from_numpy(tables["rel_table_H6_L65"]))
    assert np.array_equal(m.get_bias().detach().numpy(), tables["rel_bias_H6_L65"])


@pytest.mark.parametrize("g", [8, 14])
def test_axial_coordinates_bit_exact(tables, g):
    tx, ty = PE.RoPEAxial(32).init_t_xy(g, g, "cpu")
    assert np.array_equal(tx.numpy(), tables[f"t_x_g{g}"]) and np.array_equal(ty.numpy(), tables[f"t_y_g{g}"])
    tx2, ty2 = PE.RoPEMixed(32, 6).init_t_xy(g, g, "cpu")
    assert torch.equal(tx, tx2) and torch.equal(ty, ty2)


@pytest.mark.parametrize("dim", [16, 32, 64])
def test_axial_tables_bit_exact(tables, dim):
    m = PE.RoPEAxial(dim=dim, theta=100.0)
    assert np.array_equal(m.inv_freq.numpy(), tables[f"axial_inv_freq_D{dim}"])
    for n in (16, 64, 196):
        c, s = m.get_freqs_cis(n, "cpu")
        assert np.array_equal(c.numpy(), tables[f"axial_cos_D{dim}_N{n}"])
        assert np.array_equal(s.numpy(), tables[f"axial_sin_D{dim}_N{n}"])


@pytest.mark.parametrize("dim,heads", [(32, 6), (64, 12), (16, 2)])
def test_mixed_tables_bit_exact_including_scramble(tables, dim, heads):
    m = PE.RoPEMixed(dim=dim, num_heads=heads, theta=100.0)
    with torch.no_grad():
        m.freqs.copy_(torch.from_numpy(tables[f"mixed_freqs_D{dim}_H{heads}"]))
    for n in (16, 64, 196):
        c, s = m.get_freqs_cis(n, "cpu")
        assert c.shape == (heads, n, dim // 2) and c.dtype == torch.float32
        assert np.array_equal(c.detach().numpy(), tables[f"mixed_cos_D{dim}_H{heads}_N{n}"])
        assert np.array_equal(s.detach().numpy(), tables[f"mixed_sin_D{dim}_H{heads}_N{n}"])
    # closed form of the scramble (oracle) agrees too
    c_np, _ = T.mixed_cos_sin(tables[f"mixed_freqs_D{dim}_H{heads}"], 64)
    np.testing.assert_allclose(m.get_freqs_cis(64, "cpu")[0].detach().numpy(), c_np, atol=5e-7)


@pytest.mark.parametrize("shared", [True, False])
def test_poly_bias_matches_golden(tables, shared):
    tag = f"{'shared' if shared else 'perhead'}_N64_H6"
    m = PE.PolynomialRPE(64, degree=3, num_heads=6, shared_across_heads=shared)
    with torch.no_grad():
        m.coefficients.copy_(torch.from_numpy(tables[f"poly_coef_{tag}"]))
    got = m.get_bias().detach().numpy()
    np.testing.assert_allclose(got, tables[f"poly_bias_{tag}"], rtol=1e-6, atol=1e-7)
    assert np.array_equal(m.l1_distance().numpy(), T.poly_l1_distance(64))


def test_absolute_forward_is_in_place_and_skips_cls():
    m = PE.AbsolutePositionalEncoding(8, max_len=50)
    x = torch.zeros(2, 5, 8)
    y = m(x)
    assert y is x and torch.all(x[:, 0] == 0) and torch.equal(x[0, 1:], m.pos_embed[0, :4].detach())


@pytest.mark.parametrize("mode", MODES)
def test_state_dict_contract_vs_golden(mode):
    tag = mode.replace("-", "_")
    z = np.load(os.path.join(GOLDEN, f"model_{tag}.npz"))
    kw = eval(str(z["kwargs"]))  # noqa: S307 - fixture written by oracle/make_golden.py
    m = VisionTransformer(**kw)
    want = {k[3:]: z[k] for k in z.files if k.startswith("sd.")}
    got = m.state_dict()
    assert list(got.keys()) == list(want.keys())
    for k in want:
        assert tuple(got[k].shape) == tuple(want[k].shape), k
    m.load_state_dict({k: torch.from_numpy(v) for k, v in want.items()}, strict=True)
    # the PE module is ONE shared module: parameters() dedups it (train.py:195)
    n_pe = sum(1 for n, _ in m.named_parameters() if "pos_encoding" in n)
    assert n_pe == 0


@pytest.mark.parametrize("mode", MODES)
def test_seeded_construction_matches_reference_bit_for_bit(mode):
    """Same RNG consumption order as the reference constructor -> identical initial weights.  The fixture's
    state_dict is the reference's model built and perturbed by the same seeded recipe; the perturbation draws
    in named_parameters() order, so that order must match the reference's too."""
    tag = mode.replace("-", "_")
    z = np.load(os.path.join(GOLDEN, f"model_{tag}.npz"))
    kw = ast.literal_eval(str(z["kwargs"]))
    mine = make_golden.seeded_model(VisionTransformer, kw, tag)
    want = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    got = mine.state_dict()
    assert list(got.keys()) == list(want.keys())
    for k in want:
        assert got[k].dtype == want[k].dtype and torch.equal(got[k], want[k]), k
    mine.load_state_dict(want, strict=True)
