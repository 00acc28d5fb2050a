"""Pin the oracle (oracle/) against the fixtures generated from the unmodified reference
(tests/golden/, made by oracle/make_golden.py).  CPU only."""
import ast
import os

import numpy as np
import pytest
import torch

from oracle import attention_np as A
from oracle import tables_np as T, vit_torch as V

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
MODEL_TAGS = ["none", "absolute", "relative", "polynomial", "polynomial_perhead", "rope_axial", "rope_mixed"]
ATTN_TAGS = [t for t in MODEL_TAGS if t != "absolute"]


@pytest.fixture(scope="module")
def tables():
    return np.load(os.path.join(GOLDEN, "tables.npz"))


# ----------------------------------------------------------------------------- tables

@pytest.mark.parametrize("length", [17, 65])
def test_relative_index_bit_exact(tables, length):
    want = tables[f"rel_index_L{length}"]
    got = T.relative_position_index(length)
    assert got.dtype == np.int64 and want.dtype == np.int64
    assert np.array_equal(got, want)
    # Toeplitz structure: constant along diagonals, range [0, 2L-2]
    assert got.min() == 0 and got.max() == 2 * length - 2


def test_relative_bias_gather(tables):
    got = T.relative_bias(tables["rel_table_H6_L65"], 65)
    assert np.array_equal(got, tables["rel_bias_H6_L65"])


@pytest.mark.parametrize("g", [8, 14])
def test_grid_coords_bit_exact(tables, g):
    tx, ty = T.grid_coords(g, g)
    assert np.array_equal(tx, tables[f"t_x_g{g}"]) and np.array_equal(ty, tables[f"t_y_g{g}"])
    assert tx.dtype == np.float32


@pytest.mark.parametrize("dim", [16, 32, 64])
def test_axial_tables(tables, dim):
    inv = T.axial_inv_freq(dim, 100.0)
    np.testing.assert_allclose(inv, tables[f"axial_inv_freq_D{dim}"], rtol=2e-7, atol=0)
    for n in (16, 64, 196):
        c, s = T.axial_cos_sin(n, tables[f"axial_inv_freq_D{dim}"])
        np.testing.assert_allclose(c, tables[f"axial_cos_D{dim}_N{n}"], rtol=0, atol=3e-7)
        np.testing.assert_allclose(s, tables[f"axial_sin_D{dim}_N{n}"], rtol=0, atol=3e-7)


@pytest.mark.parametrize("dim,heads", [(32, 6), (64, 12), (16, 2)])
def test_mixed_tables_scramble(tables, dim, heads):
    freqs = tables[f"mixed_freqs_D{dim}_H{heads}"]
    for n in (16, 64, 196):
        c, s = T.mixed_cos_sin(freqs, n)
        # angles reach ~30 rad; fp32 libm cos/sin agree to a few 1e-7 absolute
        np.testing.assert_allclose(c, tables[f"mixed_cos_D{dim}_H{heads}_N{n}"], rtol=0, atol=5e-7)
        np.testing.assert_allclose(s, tables[f"mixed_sin_D{dim}_H{heads}_N{n}"], rtol=0, atol=5e-7)
    hs, ps = T.mixed_scramble(heads, 64)
    flat = np.arange(heads * 64).reshape(64, heads).T  # [h', n'] -> n'*H + h'
    assert np.array_equal(hs * 64 + ps, flat)


def test_mixed_init_freqs_structure(tables):
    """freqs[0] = mag*[cos a, cos(pi/2+a)], freqs[1] = mag*[sin a, sin(pi/2+a)] per head."""
    freqs = tables["mixed_freqs_D32_H6"].astype(np.float64)
    q = 8
    ang = np.arctan2(freqs[1, :, 0], freqs[0, :, 0])
    want = T.mixed_init_freqs(32, 6, 100.0, ang)
    np.testing.assert_allclose(freqs, want, rtol=0, atol=1e-6)
    assert freqs.shape == (2, 6, 2 * q)


@pytest.mark.parametrize("tag,heads,npatch", [("shared_N64_H6", 6, 64), ("perhead_N64_H6", 6, 64),
                                               ("shared_N16_H2", 2, 16), ("perhead_N16_H2", 2, 16)])
def test_poly_bias(tables, tag, heads, npatch):
    got = T.poly_bias(tables[f"poly_coef_{tag}"], npatch, heads)
    want = tables[f"poly_bias_{tag}"]
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)
    assert np.all(got[:, 0, :] == 0) and np.all(got[:, :, 0] == 0)  # cls row / column


def test_poly_distance_is_l1_on_transposed_raster():
    d = T.poly_l1_distance(16)
    assert d[0, 1] == 1 and d[0, 4] == 1 and d[0, 5] == 2 and d[0, 15] == 6
    assert np.array_equal(d, d.T) and d.dtype == np.int64


# ----------------------------------------------------------------------------- attention core

def _split_qkv(x, w, heads):
    b, n, e = x.shape
    qkv = (x @ w.T).reshape(b, n, 3, heads, e // heads).transpose(2, 0, 3, 1, 4)
    return qkv[0], qkv[1], qkv[2]


def _attn_bias(tag, z, heads, n):
    if tag == "relative":
        return T.relative_bias(z["sd.pos_encoding.relative_position_bias_table"].astype(np.float64), n)
    if tag.startswith("polynomial"):
        return T.poly_bias(z["sd.pos_encoding.coefficients"], n - 1, heads).astype(np.float64)
    return None


@pytest.mark.parametrize("tag", ATTN_TAGS)
def test_attention_np_forward_backward(tag):
    z = np.load(os.path.join(GOLDEN, f"attn_{tag}.npz"))
    heads = 3
    x = z["x"].astype(np.float64)
    wqkv, wproj, bproj = (z["sd.qkv.weight"].astype(np.float64), z["sd.proj.weight"].astype(np.float64),
                          z["sd.proj.bias"].astype(np.float64))
    b, n, e = x.shape
    q, k, v = _split_qkv(x, wqkv, heads)
    scale = (e // heads) ** -0.5
    cos = z["cos"] if "cos" in z else None
    sin = z["sin"] if "sin" in z else None
    bias = _attn_bias(tag, z, heads, n)
    o, _, _, _ = A.attention_forward(q, k, v, scale, bias, cos, sin)
    y = o @ wproj.T + bproj
    np.testing.assert_allclose(y, z["y"], rtol=0, atol=2e-6)

    d_o = z["dy"].astype(np.float64) @ wproj
    g = A.attention_backward(d_o, q, k, v, scale, bias, cos, sin)
    dqkv = np.stack([g["dq"], g["dk"], g["dv"]]).transpose(1, 3, 0, 2, 4).reshape(b, n, 3 * e)
    np.testing.assert_allclose(dqkv @ wqkv, z["dx"], rtol=0, atol=3e-6)
    dw = np.einsum("bnk,bne->ke", dqkv, x)
    np.testing.assert_allclose(dw, z["grad.qkv.weight"], rtol=0, atol=2e-5)
    if tag == "relative":
        dt = A.dtable_from_dbias(g["dbias"])
        np.testing.assert_allclose(dt, z["grad.pos_encoding.relative_position_bias_table"], rtol=0, atol=3e-6)
    if tag.startswith("polynomial"):
        dc = A.dcoef_from_dbias(g["dbias"], 3, shared=(tag == "polynomial"))
        want = z["grad.pos_encoding.coefficients"]
        np.testing.assert_allclose(dc, want, rtol=2e-5, atol=1e-5 * np.abs(want).max())
    if tag == "rope_mixed":
        # chain dcos/dsin through cos/sin(phase) and the scramble into dfreqs (SURVEY row A18)
        freqs = z["sd.pos_encoding.freqs"]
        ang = T.mixed_angles(freqs, n - 1).astype(np.float64)
        dphi = -np.sin(ang) * g["dcos"] + np.cos(ang) * g["dsin"]
        hs, ps = T.mixed_scramble(heads, n - 1)
        tx, ty = T.grid_coords(8, 8)
        df = np.zeros((2, heads, e // heads // 2))
        np.add.at(df[0], hs, tx[ps][..., None] * dphi)
        np.add.at(df[1], hs, ty[ps][..., None] * dphi)
        want = z["grad.pos_encoding.freqs"]
        np.testing.assert_allclose(df, want, rtol=0, atol=2e-5 * max(1.0, np.abs(want).max()))


# ----------------------------------------------------------------------------- whole model

def _load_model(tag):
    z = np.load(os.path.join(GOLDEN, f"model_{tag}.npz"))
    kw = ast.literal_eval(str(z["kwargs"]))
    cfg = V.VitConfig(**kw)
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    return z, cfg, sd


@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_vit_torch_matches_golden(tag):
    z, cfg, sd = _load_model(tag)
    torch.set_num_threads(1)
    p = V.params_from_state_dict(sd)
    logits = V.forward(cfg, p, torch.from_numpy(z["images"]))
    loss = torch.nn.functional.cross_entropy(logits, torch.from_numpy(z["labels"]))
    loss.backward()
    np.testing.assert_allclose(logits.detach().numpy(), z["logits"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(loss.item(), float(z["loss"]), rtol=0, atol=1e-6)
    for k in z.files:
        if not k.startswith("grad."):
            continue
        name = k[5:]
        if ".attn.pos_encoding." in name:
            continue
        g = p[name].grad
        assert g is not None, name
        want = z[k]
        np.testing.assert_allclose(g.numpy(), want, rtol=0, atol=1e-6 + 1e-5 * np.abs(want).max(), err_msg=name)


@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_state_dict_key_contract(tag):
    """SURVEY.md row B3: PE keys are duplicated under every block for the shared-module modes."""
    z, cfg, sd = _load_model(tag)
    dup = [k for k in sd if ".attn.pos_encoding." in k]
    if cfg.pos_encoding in ("none", "absolute"):
        assert not dup
    else:
        pe_keys = [k for k in sd if k.startswith("pos_embed.")]
        assert len(dup) == cfg.depth * len(pe_keys)
        for k in dup:
            assert torch.equal(sd[k], sd["pos_embed." + k.split(".attn.pos_encoding.")[1]])
    fresh = V.init_state_dict(cfg)
    assert set(fresh) == set(V.canonical_keys(sd))
    for k, v in fresh.items():
        assert tuple(v.shape) == tuple(sd[k].shape), k


@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_vit_torch_bit_exact_vs_reference_golden(tag):
    """Same torch ops in the same order as the reference: its stored logits, loss and every parameter
    gradient come out bit for bit (single-threaded CPU fp32)."""
    z, cfg, sd = _load_model(tag)
    torch.set_num_threads(1)
    p = V.params_from_state_dict(sd)
    logits = V.forward(cfg, p, torch.from_numpy(z["images"]))
    loss = torch.nn.functional.cross_entropy(logits, torch.from_numpy(z["labels"]))
    loss.backward()
    assert np.array_equal(logits.detach().numpy(), z["logits"])
    assert np.array_equal(loss.detach().numpy(), z["loss"])
    for k in z.files:
        if k.startswith("grad.") and ".attn.pos_encoding." not in k:
            assert np.array_equal(p[k[5:]].grad.numpy(), z[k]), k


def test_oracle_error_behaviour():
    """The reference's error contract (SURVEY.md rows B4, A8), restated by the oracle: an unknown positional
    encoding and a cos / sin table of the wrong rank raise ValueError."""
    with pytest.raises(ValueError):
        V.init_state_dict(V.VitConfig(pos_encoding="bogus"))
    with pytest.raises(ValueError):
        V.expand_cs(torch.zeros(4))
