"""torch fp32 restatement of the whole reference model (CPU reference / CPU baseline).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  Citations are relative
to ``/root/reference``.  The model is written functionally over a plain dict of
tensors that uses the reference's ``state_dict`` key names (SURVEY.md row B3),
so weights move between the reference, this oracle and the product model with
``state_dict()`` / ``load_state_dict()`` alone.  It issues the same torch ops in
the same order as the reference's eager path, so it reproduces the reference's
stored outputs bit for bit (checked in ``tests/test_oracle_golden.py``), and it
is what ``bench.py --impl reference`` and the ``cpu_baseline`` leg time.
"""
import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F


@dataclass
class VitConfig:
    """Constructor arguments of ``VisionTransformer`` - models/vit.py:148-151."""
    img_size: int = 32
    patch_size: int = 4
    in_chans: int = 3
    num_classes: int = 10
    embed_dim: int = 192
    depth: int = 6
    num_heads: int = 6
    mlp_ratio: float = 4.0
    pos_encoding: str = "absolute"
    rope_theta: float = 100.0
    poly_degree: int = 3
    poly_shared_heads: bool = True

    @property
    def head_dim(self):
        return self.embed_dim // self.num_heads

    @property
    def num_patches(self):
        return (self.img_size // self.patch_size) ** 2


MODES = ("none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed")


# --------------------------------------------------------------------------- tables

def grid_coords(h, w, device=None):
    """models/positional_encoding.py:198-214 / :292-311."""
    t = torch.arange(h * w, device=device, dtype=torch.float32)
    return (t % w).float(), torch.div(t, w, rounding_mode="floor").float()


def axial_cos_sin(inv_freq, num_patches):
    """models/positional_encoding.py:216-245."""
    g = int(math.sqrt(num_patches))
    t_x, t_y = grid_coords(g, g, inv_freq.device)
    ang = torch.cat([torch.outer(t_x, inv_freq), torch.outer(t_y, inv_freq)], dim=-1)
    return torch.cos(ang), torch.sin(ang)


def mixed_cos_sin(freqs, num_patches):
    """models/positional_encoding.py:313-351 including the ``view`` scramble (:341-342)."""
    num_heads = freqs.shape[1]
    g = int(math.sqrt(num_patches))
    t_x, t_y = grid_coords(g, g, freqs.device)
    with torch.autocast("cuda", enabled=False):
        fx = t_x.unsqueeze(-1) @ freqs[0].unsqueeze(-2)  # broadcasts to [H, N, D/2]
        fy = t_y.unsqueeze(-1) @ freqs[1].unsqueeze(-2)
        fx = fx.view(num_patches, num_heads, -1).permute(1, 0, 2)
        fy = fy.view(num_patches, num_heads, -1).permute(1, 0, 2)
        ang = fx + fy
        return torch.cos(ang), torch.sin(ang)


def relative_bias(table, index):
    """models/positional_encoding.py:82-95."""
    return table[:, index]


def poly_bias(coefficients, num_patches, num_heads, shared):
    """models/positional_encoding.py:127-171."""
    g = int(math.sqrt(num_patches))
    dev = coefficients.device
    ys = torch.arange(g, device=dev).repeat(g)
    xs = torch.arange(g, device=dev).repeat_interleave(g)
    dist = (ys[:, None] - ys[None, :]).abs() + (xs[:, None] - xs[None, :]).abs()
    degree = coefficients.shape[-1] - 1
    feats = torch.stack([dist.float().pow(k) for k in range(degree + 1)], dim=-1)
    if shared:
        core = (feats @ coefficients).unsqueeze(0).expand(num_heads, -1, -1)
    else:
        core = torch.zeros(num_heads, num_patches, num_patches, device=dev)
        for h in range(num_heads):
            core[h] = feats @ coefficients[h]
    full = torch.zeros(num_heads, num_patches + 1, num_patches + 1, device=dev)
    full[:, 1:, 1:] = core
    return full


def rotate_half_pair(q, k, cos, sin):
    """models/rope_utils.py:3-37."""
    half = q.shape[-1] // 2
    q1, q2 = q[..., :half], q[..., half:]
    k1, k2 = k[..., :half], k[..., half:]
    q_out = torch.cat([q1 * cos - q2 * sin, q1 * sin + q2 * cos], dim=-1)
    k_out = torch.cat([k1 * cos - k2 * sin, k1 * sin + k2 * cos], dim=-1)
    return q_out, k_out


def expand_cs(t):
    """models/rope_utils.py:39-66."""
    if t.ndim == 3:
        return t.unsqueeze(0)
    if t.ndim == 2:
        return t.unsqueeze(0).unsqueeze(0)
    raise ValueError(f"Unexpected tensor shapes: {t.shape}")


# --------------------------------------------------------------------------- model

def attention(cfg, p, prefix, x, pe_prefix, rope):
    """``Attention.forward`` - models/vit.py:43-94."""
    b, n, c = x.shape
    h, dh = cfg.num_heads, cfg.head_dim
    qkv = F.linear(x, p[prefix + "qkv.weight"]).reshape(b, n, 3, h, dh).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    scale = dh ** -0.5
    if rope is not None:
        cos, sin = expand_cs(rope[0]), expand_cs(rope[1])
        q_rest, k_rest = rotate_half_pair(q[:, :, 1:], k[:, :, 1:], cos, sin)
        q = torch.cat([q[:, :, :1], q_rest], dim=2)
        k = torch.cat([k[:, :, :1], k_rest], dim=2)
        att = (q @ k.transpose(-2, -1)) * scale
    else:
        att = (q @ k.transpose(-2, -1)) * scale
        if cfg.pos_encoding == "relative":
            att = att + relative_bias(p[pe_prefix + "relative_position_bias_table"],
                                      p[pe_prefix + "relative_position_index"])
        elif cfg.pos_encoding == "polynomial":
            att = att + poly_bias(p[pe_prefix + "coefficients"], cfg.num_patches, h,
                                  cfg.poly_shared_heads)
    att = att.softmax(dim=-1)
    out = (att @ v).transpose(1, 2).reshape(b, n, c)
    return F.linear(out, p[prefix + "proj.weight"], p[prefix + "proj.bias"])


def block(cfg, p, i, x, rope):
    """``Block.forward`` - models/vit.py:120-125 (+ timm ``Mlp``, exact-erf GELU)."""
    pre = f"blocks.{i}."
    e = cfg.embed_dim
    y = F.layer_norm(x, (e,), p[pre + "norm1.weight"], p[pre + "norm1.bias"], 1e-5)
    x = x + attention(cfg, p, pre + "attn.", y, "pos_embed.", rope)
    y = F.layer_norm(x, (e,), p[pre + "norm2.weight"], p[pre + "norm2.bias"], 1e-5)
    y = F.linear(y, p[pre + "mlp.fc1.weight"], p[pre + "mlp.fc1.bias"])
    y = F.gelu(y)
    y = F.linear(y, p[pre + "mlp.fc2.weight"], p[pre + "mlp.fc2.bias"])
    return x + y


def forward_features(cfg, p, images):
    """``VisionTransformer.forward_features`` - models/vit.py:235-271."""
    b, _, hh, ww = images.shape
    x = F.conv2d(images, p["patch_embed.weight"], p["patch_embed.bias"], stride=cfg.patch_size)
    gh, gw = hh // cfg.patch_size, ww // cfg.patch_size
    x = x.flatten(2).transpose(1, 2)
    x = torch.cat((p["cls_token"].expand(b, -1, -1), x), dim=1)
    if cfg.pos_encoding == "absolute":
        # in-place slice add of models/positional_encoding.py:37-40
        x[:, 1:] = x[:, 1:] + p["pos_embed.pos_embed"][:, : x.size(1) - 1]
    rope = None
    if cfg.pos_encoding == "rope-axial":
        rope = axial_cos_sin(p["pos_embed.inv_freq"], gh * gw)
    elif cfg.pos_encoding == "rope-mixed":
        rope = mixed_cos_sin(p["pos_embed.freqs"], gh * gw)
    for i in range(cfg.depth):
        x = block(cfg, p, i, x, rope)
    return x


def forward(cfg, p, images):
    """``VisionTransformer.forward`` - models/vit.py:273-285."""
    x = forward_features(cfg, p, images)
    x = F.layer_norm(x, (cfg.embed_dim,), p["norm.weight"], p["norm.bias"], 1e-5)
    return F.linear(x[:, 0], p["head.weight"], p["head.bias"])


# --------------------------------------------------------------------------- parameters

def canonical_keys(state_dict):
    """Drop the per-block duplicates ``blocks.{i}.attn.pos_encoding.*`` (SURVEY.md row B3):
    they alias ``pos_embed.*`` (one shared module assigned into every block, vit.py:98,205-207)."""
    return {k: v for k, v in state_dict.items() if ".attn.pos_encoding." not in k}


def params_from_state_dict(state_dict, requires_grad=True, dtype=torch.float32, device="cpu"):
    """Leaf tensors for :func:`forward` from a reference-format ``state_dict``."""
    out = {}
    for k, v in canonical_keys(state_dict).items():
        t = v.detach().clone().to(device)
        if t.is_floating_point():
            t = t.to(dtype)
            # buffers (inv_freq) need no grad; everything else is a parameter
            t.requires_grad_(requires_grad and not k.endswith("inv_freq"))
        out[k] = t
    return out


def init_state_dict(cfg: VitConfig, seed: int = 0):
    """Random-init weights with the reference's shapes and init scales (vit.py:214-233,
    positional_encoding.py:35,64,117,271-290).  RNG *order* is not reproduced - parity tests
    always move weights by ``state_dict``; this exists so the GPU box (which has no reference)
    can still build a correctly-shaped, sensibly-scaled model."""
    g = torch.Generator().manual_seed(seed)
    e, h, dh, hid = cfg.embed_dim, cfg.num_heads, cfg.head_dim, int(cfg.embed_dim * cfg.mlp_ratio)

    def tn(*shape, std=0.02):
        t = torch.empty(*shape)
        torch.nn.init.trunc_normal_(t, std=std, generator=g)
        return t

    sd = {"cls_token": torch.zeros(1, 1, e)}
    fan_out = e * cfg.patch_size * cfg.patch_size
    sd["patch_embed.weight"] = torch.randn(e, cfg.in_chans, cfg.patch_size, cfg.patch_size,
                                           generator=g) * math.sqrt(2.0 / fan_out)
    sd["patch_embed.bias"] = torch.zeros(e)
    pe = cfg.pos_encoding
    if pe == "absolute":
        sd["pos_embed.pos_embed"] = tn(1, 5000, e)
    elif pe == "relative":
        length = cfg.num_patches + 1
        sd["pos_embed.relative_position_bias_table"] = tn(h, 2 * length - 1)
        pos = torch.arange(length)
        sd["pos_embed.relative_position_index"] = (pos[:, None] - pos[None, :] + length - 1).clamp(0, 2 * length - 2)
    elif pe == "polynomial":
        sd["pos_embed.coefficients"] = tn(cfg.poly_degree + 1) if cfg.poly_shared_heads else tn(h, cfg.poly_degree + 1)
    elif pe == "rope-axial":
        q = dh // 4
        sd["pos_embed.inv_freq"] = 1.0 / (cfg.rope_theta ** (torch.arange(0, q, dtype=torch.float) / q))
    elif pe == "rope-mixed":
        mag = 1 / (cfg.rope_theta ** (torch.arange(0, dh, 4)[: dh // 4].float() / dh))
        fx, fy = [], []
        for _ in range(h):
            a = torch.rand(1, generator=g) * 2 * torch.pi
            fx.append(torch.cat([mag * torch.cos(a), mag * torch.cos(torch.pi / 2 + a)], dim=-1))
            fy.append(torch.cat([mag * torch.sin(a), mag * torch.sin(torch.pi / 2 + a)], dim=-1))
        sd["pos_embed.freqs"] = torch.stack([torch.stack(fx), torch.stack(fy)], dim=0)
    elif pe != "none":
        raise ValueError(f"Unknown positional encoding type: {pe}")
    for i in range(cfg.depth):
        b = f"blocks.{i}."
        sd[b + "norm1.weight"], sd[b + "norm1.bias"] = torch.ones(e), torch.zeros(e)
        sd[b + "attn.qkv.weight"] = tn(3 * e, e)
        sd[b + "attn.proj.weight"], sd[b + "attn.proj.bias"] = tn(e, e), torch.zeros(e)
        sd[b + "norm2.weight"], sd[b + "norm2.bias"] = torch.ones(e), torch.zeros(e)
        sd[b + "mlp.fc1.weight"], sd[b + "mlp.fc1.bias"] = tn(hid, e), torch.zeros(hid)
        sd[b + "mlp.fc2.weight"], sd[b + "mlp.fc2.bias"] = tn(e, hid), torch.zeros(e)
    sd["norm.weight"], sd["norm.bias"] = torch.ones(e), torch.zeros(e)
    sd["head.weight"], sd["head.bias"] = tn(cfg.num_classes, e), torch.zeros(cfg.num_classes)
    return sd


def train_step(cfg, params, opt, images, labels):
    """One step of ``train.py:108-116``: zero_grad -> forward -> CE -> backward -> AdamW.step."""
    opt.zero_grad()
    logits = forward(cfg, params, images)
    loss = F.cross_entropy(logits, labels)
    loss.backward()
    opt.step()
    return loss
