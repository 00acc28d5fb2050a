"""Generate ``tests/golden/*.npz`` by running the UNMODIFIED reference (build container only).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

    python -m oracle.make_golden            # from the repo root; needs /root/reference

The reference ships no golden vectors of its own (SURVEY.md section 4), so these fixtures
- outputs of the reference itself on seeded inputs, CPU fp32 - are what pins the
oracle and, through it, the CUDA kernels.  Three families:

* ``tables.npz``          index / coordinate / frequency / bias tables of the PE modules;
* ``attn_<mode>.npz``     one ``Attention`` module (with its PE module) at ViT-Tiny token
                          geometry: inputs, weights, output, all gradients;
* ``model_<mode>.npz``    a small ``VisionTransformer``: state_dict, images, labels, logits,
                          loss and every parameter gradient.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import live_reference  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
MODES = ("none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed")


def _np(t):
    return t.detach().cpu().numpy()


def make_tables(pe):
    out = {}
    for length in (17, 65):
        m = pe.RelativePositionalEncoding(length - 1, num_heads=2)
        out[f"rel_index_L{length}"] = _np(m.relative_position_index)
    torch.manual_seed(11)
    m = pe.RelativePositionalEncoding(64, num_heads=6)
    out["rel_table_H6_L65"] = _np(m.relative_position_bias_table)
    out["rel_bias_H6_L65"] = _np(m.get_bias())

    for g in (8, 14):
        ax = pe.RoPEAxial(dim=32, theta=100.0)
        tx, ty = ax.init_t_xy(g, g, "cpu")
        out[f"t_x_g{g}"], out[f"t_y_g{g}"] = _np(tx), _np(ty)
    for dim in (16, 32, 64):
        ax = pe.RoPEAxial(dim=dim, theta=100.0)
        out[f"axial_inv_freq_D{dim}"] = _np(ax.inv_freq)
        for n in (16, 64, 196):
            c, s = ax.get_freqs_cis(n, "cpu")
            out[f"axial_cos_D{dim}_N{n}"], out[f"axial_sin_D{dim}_N{n}"] = _np(c), _np(s)

    torch.manual_seed(12)
    for (dim, heads) in ((32, 6), (64, 12), (16, 2)):
        mx = pe.RoPEMixed(dim=dim, num_heads=heads, theta=100.0)
        out[f"mixed_freqs_D{dim}_H{heads}"] = _np(mx.freqs)
        for n in (16, 64, 196):
            c, s = mx.get_freqs_cis(n, "cpu")
            out[f"mixed_cos_D{dim}_H{heads}_N{n}"] = _np(c)
            out[f"mixed_sin_D{dim}_H{heads}_N{n}"] = _np(s)

    torch.manual_seed(13)
    for shared in (True, False):
        for (npatch, heads) in ((64, 6), (16, 2)):
            po = pe.PolynomialRPE(npatch, degree=3, num_heads=heads, shared_across_heads=shared)
            tag = f"{'shared' if shared else 'perhead'}_N{npatch}_H{heads}"
            out[f"poly_coef_{tag}"] = _np(po.coefficients)
            out[f"poly_bias_{tag}"] = _np(po.get_bias())
    np.savez_compressed(os.path.join(GOLDEN, "tables.npz"), **out)
    return len(out)


def _pe_module(pe, mode, num_patches, heads, head_dim, embed, shared=True):
    if mode == "relative":
        return pe.RelativePositionalEncoding(num_patches, heads)
    if mode == "polynomial":
        return pe.PolynomialRPE(num_patches, degree=3, num_heads=heads, shared_across_heads=shared)
    if mode == "rope-axial":
        return pe.RoPEAxial(dim=head_dim, theta=100.0)
    if mode == "rope-mixed":
        return pe.RoPEMixed(dim=head_dim, num_heads=heads, theta=100.0)
    return pe.NoPositionalEncoding()


def make_attention(vit, pe, mode, tag, shared=True):
    """One Attention module at ViT-Tiny token geometry (65 tokens, head_dim 32), 3 heads."""
    b, n, heads, dh = 2, 65, 3, 32
    e = heads * dh
    torch.manual_seed(100 + len(tag))
    attn = vit.Attention(e, num_heads=heads)
    for lin in (attn.qkv, attn.proj):
        torch.nn.init.normal_(lin.weight, std=0.08)
    torch.nn.init.normal_(attn.proj.bias, std=0.05)
    mod = _pe_module(pe, mode, n - 1, heads, dh, e, shared)
    # make the learnable PE tensors large enough to matter numerically
    with torch.no_grad():
        for p_ in mod.parameters():
            if mode in ("relative", "polynomial"):
                p_.mul_(4.0 if mode == "relative" else 0.25)
    attn.set_pos_encoding(mod)
    x = torch.randn(b, n, e, requires_grad=True)
    freqs_cis = mod.get_freqs_cis(n - 1, "cpu") if mode.startswith("rope") else None
    y = attn(x, freqs_cis=freqs_cis)
    w = torch.randn(b, n, e)
    (y * w).sum().backward()
    out = {"x": _np(x), "y": _np(y), "dy": _np(w), "dx": _np(x.grad)}
    for k, v in attn.state_dict().items():
        out["sd." + k] = _np(v)
    for k, p_ in attn.named_parameters():
        out["grad." + k] = _np(p_.grad)
    if freqs_cis is not None:
        out["cos"], out["sin"] = _np(freqs_cis[0]), _np(freqs_cis[1])
    np.savez_compressed(os.path.join(GOLDEN, f"attn_{tag}.npz"), **out)


def seeded_model(ctor, kw, tag):
    """``ctor(**kw)`` under the seed of ``model_<tag>.npz``, then perturbed in place.  Run with the
    reference's ``VisionTransformer`` it makes the fixture's state_dict; run with the product's, the
    same RNG order must give the same tensors (tests/test_host_api.py)."""
    torch.manual_seed(200 + len(tag))
    model = ctor(**kw)
    with torch.no_grad():  # cls_token / biases are zero-initialised: perturb so their paths are live
        for name, p_ in model.named_parameters():
            if name == "cls_token" or name.endswith(".bias"):
                p_.add_(0.05 * torch.randn_like(p_))
            if name.endswith("coefficients"):
                p_.mul_(0.25)
            if name.endswith("relative_position_bias_table"):
                p_.mul_(4.0)
    return model


def make_model(vit, mode, tag, shared=True):
    kw = dict(img_size=16, patch_size=4, in_chans=3, num_classes=5, embed_dim=32, depth=2,
              num_heads=2, pos_encoding=mode, rope_theta=100.0, poly_degree=3,
              poly_shared_heads=shared)
    model = seeded_model(vit.VisionTransformer, kw, tag)
    images = torch.randn(3, 3, 16, 16)
    labels = torch.tensor([1, 4, 0])
    logits = model(images)
    loss = torch.nn.CrossEntropyLoss()(logits, labels)
    loss.backward()
    out = {"images": _np(images), "labels": _np(labels), "logits": _np(logits), "loss": _np(loss)}
    for k, v in model.state_dict().items():
        out["sd." + k] = _np(v)
    for k, p_ in model.named_parameters():  # named_parameters dedups the shared PE parameter
        out["grad." + k] = _np(p_.grad)
    out["kwargs"] = np.array(repr(kw))
    np.savez_compressed(os.path.join(GOLDEN, f"model_{tag}.npz"), **out)


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(1)
    vit, pe, _ = live_reference.load()
    n = make_tables(pe)
    print(f"tables.npz: {n} arrays")
    for mode in MODES:
        tag = mode.replace("-", "_")
        if mode != "absolute":  # absolute PE acts outside Attention (vit.py:257-258)
            make_attention(vit, pe, mode, tag)
        make_model(vit, mode, tag)
    make_attention(vit, pe, "polynomial", "polynomial_perhead", shared=False)
    make_model(vit, "polynomial", "polynomial_perhead", shared=False)
    total = sum(os.path.getsize(os.path.join(GOLDEN, f)) for f in os.listdir(GOLDEN))
    print(f"golden fixtures: {len(os.listdir(GOLDEN))} files, {total / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
