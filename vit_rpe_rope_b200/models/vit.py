"""Vision Transformer: drop-in for ``models/vit.py`` of the reference, running the attention hot
path on the sm_100a kernels of ``libvrr_b200``.

``Attention`` / ``Block`` / ``VisionTransformer`` keep the reference's constructor and ``forward``
signatures, attribute names, sub-module names (hence ``state_dict`` keys, including the per-block
``attn.pos_encoding.*`` duplicates of the shared PE module) and RNG consumption order at
construction (citations: /root/reference/models/vit.py).  What changes is underneath:

* patch embedding + cls concat + absolute add      -> one unfold+GEMM kernel   (vit.py:248-258)
* qkv Linear + head split + RoPE + cls re-concat    -> one GEMM with RoPE epilogue (vit.py:47-68)
* QK^T, scale, RPE / Poly-RPE bias, softmax, PV, merge -> one fused attention kernel (vit.py:71-88)

LayerNorm (fused with the residual adds), the output projection, the MLP (bias + GELU in the fc1 GEMM epilogue)
and the head run library kernels too (SURVEY.md section 8(f) N1): the forward and backward contain no cuBLAS
GEMM.  CUDA sm_100 only: CPU inputs raise; there is no fallback path.

Regularisers of a ViT training recipe (``VisionTransformer(drop_rate, drop_path_rate)``, timm's names): inside the
fused block loop, proj_drop / drop2 and stochastic depth are applied by the add+LayerNorm kernels that read the
branch anyway, and drop1 by fc1's GELU epilogue, all from one Philox key drawn per training forward.

Register tokens (``VisionTransformer(reg_tokens=R)``, timm's name; DINOv2-with-registers, DINOv3): R learnable tokens
between the cls token and the patches, ``[cls, reg_0 .. reg_{R-1}, patch_0 ..]``.  Like the cls token they get no
absolute position embedding and are never rotated; the patch-embedding kernel writes them and the QKV+RoPE epilogue
skips them (``num_prefix_tokens = 1 + R``).

LayerScale (``VisionTransformer(init_values=)``, timm's name; DeiT III, DINOv2, DINOv3): a learnable per-channel
``gamma`` multiplies each residual branch before it is added.  Inside the fused block loop the add+LayerNorm kernels
apply it in fp32 as they read the branch and reduce its gradient in the same backward pass.

SwiGLU MLP (``VisionTransformer(mlp_layer=SwiGLUPacked)``, timm's ``GluMlp`` / ``SwiGLUPacked``; EVA-02, DINOv3):
``fc2(silu(x W_g + b_g) * (x W_v + b_v))`` with the gate and value rows packed in ``fc1``.  fc1's GEMM pairs each gate
column with its value column and applies SiLU, the product and drop1 in its epilogue; fc2's dX GEMM applies the
backward.

QK-norm (``VisionTransformer(qk_norm=True)``, timm's name; ViT-22B): a LayerNorm over each head's channels of q and
of k before RoPE, against attention-logit growth in low-precision training.  The QKV GEMM's epilogue normalises and
then rotates; the RoPE backward kernel takes the LayerNorm backward and the q_norm / k_norm gradients.
"""
import functools

import torch
import torch.nn as nn

from .. import _lib, ops
from .positional_encoding import (AbsolutePositionalEncoding, NoPositionalEncoding, PolynomialRPE,
                                  RelativePositionalEncoding, RoPEAxial, RoPEMixed)


def drop_path(x, drop_prob: float = 0., training: bool = False, scale_by_keep: bool = True):
    """timm's stochastic depth on its own (torch ops): each sample of the batch is kept with probability
    1 - drop_prob and scaled by 1 / (1 - drop_prob)."""
    if drop_prob == 0. or not training:
        return x
    keep_prob = 1 - drop_prob
    shape = (x.shape[0],) + (1,) * (x.ndim - 1)
    random_tensor = x.new_empty(shape).bernoulli_(keep_prob)
    if keep_prob > 0.0 and scale_by_keep:
        random_tensor.div_(keep_prob)
    return x * random_tensor


class DropPath(nn.Module):
    """Stochastic depth per sample (timm.layers.DropPath).  Inside ``VisionTransformer``'s fused block loop the
    decision is taken by the add+LayerNorm kernels instead (same probability and scale, Philox draws)."""

    def __init__(self, drop_prob: float = 0., scale_by_keep: bool = True):
        super().__init__()
        self.drop_prob = drop_prob
        self.scale_by_keep = scale_by_keep

    def forward(self, x):
        return drop_path(x, self.drop_prob, self.training, self.scale_by_keep)

    def extra_repr(self):
        return f'drop_prob={round(self.drop_prob, 3):0.3f}'


def _drop_p(m):
    return m.p if isinstance(m, nn.Dropout) else 0.


def _gamma(ls):
    return ls.gamma if isinstance(ls, LayerScale) else None


class LayerScale(nn.Module):
    """``x * gamma`` with ``gamma = init_values * ones(dim)`` (timm.layers.LayerScale without ``inplace``).  Inside
    ``VisionTransformer``'s fused block loop the product is taken by the add+LayerNorm kernels instead."""

    def __init__(self, dim, init_values=1e-5):
        super().__init__()
        self.gamma = nn.Parameter(init_values * torch.ones(dim))

    def forward(self, x):
        return x * self.gamma


class Mlp(nn.Module):
    """fc1 -> GELU -> fc2 with timm's parameter names (the reference takes it from timm, vit.py:9,118).  In training
    mode drop1 runs in fc1's GEMM epilogue (a Philox key drawn per call) and drop2 as ``nn.Dropout``."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.):
        super().__init__()
        hidden_features = hidden_features or in_features
        out_features = out_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.drop1 = nn.Dropout(drop)
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop2 = nn.Dropout(drop)

    def forward(self, x):
        drop1 = None
        if self.training and _drop_p(self.drop1) > 0 and x.is_cuda:
            drop1 = (_drop_p(self.drop1), 0., 1, 0, ops.new_seed(x.device))
        return self.drop2(self._branch(x, drop1))

    def _branch(self, x, drop1=None):
        """fc2(drop1(gelu(fc1(x)))) without drop2; ``drop1``: the dropout site of fc1's epilogue (training), or None."""
        if ops.can_fuse_mlp(x, self):
            dt = ops.compute_dtype(x)
            return ops.mlp(x, self.fc1, self.fc2, ops.lp_weight(self.fc1.weight, dt), ops.lp_weight(self.fc2.weight, dt),
                           drop1)
        return self.fc2(self.drop1(self.act(self.fc1(x))))


class GluMlp(nn.Module):
    """Gated MLP with timm's names and layout (timm.layers.GluMlp without ``use_conv``): fc1 is ``hidden_features``
    wide (even), its output is split into halves ``x1, x2`` and ``act(x1) * x2`` (or ``x1 * act(x2)`` with
    ``gate_last``) feeds fc2 (``hidden_features // 2`` -> out).  ``SwiGLUPacked`` (SiLU on the first half) runs fc1,
    the gate and the product in one GEMM epilogue on CUDA, with drop1 there as in ``Mlp``; other configurations run
    this module's torch forward."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.Sigmoid, norm_layer=None,
                 bias=True, drop=0., gate_last=True):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        assert hidden_features % 2 == 0
        bias = bias if isinstance(bias, (tuple, list)) else (bias, bias)
        drop_probs = drop if isinstance(drop, (tuple, list)) else (drop, drop)
        self.chunk_dim = -1
        self.gate_last = gate_last  # use second half of width for gate
        self.fc1 = nn.Linear(in_features, hidden_features, bias=bias[0])
        self.act = act_layer()
        self.drop1 = nn.Dropout(drop_probs[0])
        self.norm = norm_layer(hidden_features // 2) if norm_layer is not None else nn.Identity()
        self.fc2 = nn.Linear(hidden_features // 2, out_features, bias=bias[1])
        self.drop2 = nn.Dropout(drop_probs[1])

    def forward(self, x):
        drop1 = None
        if self.training and _drop_p(self.drop1) > 0 and x.is_cuda:
            drop1 = (_drop_p(self.drop1), 0., 1, 0, ops.new_seed(x.device))
        return self.drop2(self._branch(x, drop1))

    def _branch(self, x, drop1=None):
        """fc2(norm(drop1(gate(fc1(x))))) without drop2; ``drop1``: the dropout site of fc1's epilogue, or None."""
        if ops.can_fuse_swiglu(x, self):
            dt = ops.compute_dtype(x)
            return ops.swiglu_mlp(x, self.fc1, self.fc2, ops.lp_weight(self.fc1.weight, dt),
                                  ops.lp_weight(self.fc2.weight, dt), drop1)
        x1, x2 = self.fc1(x).chunk(2, dim=self.chunk_dim)
        x = x1 * self.act(x2) if self.gate_last else self.act(x1) * x2
        return self.fc2(self.norm(self.drop1(x)))


SwiGLUPacked = functools.partial(GluMlp, act_layer=nn.SiLU, gate_last=False)


def _is_glu_factory(layer):
    return ((isinstance(layer, type) and issubclass(layer, GluMlp))
            or (isinstance(layer, functools.partial) and isinstance(layer.func, type) and issubclass(layer.func, GluMlp)))


class Attention(nn.Module):
    """Multi-head self-attention (reference vit.py:14-98) on the fused kernels.  ``qk_norm`` (timm's name) adds
    ``q_norm`` / ``k_norm = norm_layer(head_dim)``, applied to every q / k head row before RoPE inside the QKV GEMM's
    epilogue; the kernel implements an affine ``nn.LayerNorm``, so any other ``norm_layer`` raises
    NotImplementedError.  Without it both are ``nn.Identity``."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, attn_drop=0., proj_drop=0., qk_norm=False,
                 norm_layer=nn.LayerNorm):
        super().__init__()
        if qkv_bias:
            raise NotImplementedError("qkv_bias=True is never used by the reference (vit.py:110,200) and the "
                                      "fused QKV+RoPE kernel has no bias term")
        if attn_drop != 0.:
            raise NotImplementedError("attention dropout is structurally 0 in the reference (vit.py:110,200); "
                                      "the fused attention kernel has no dropout")
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.q_norm = norm_layer(self.head_dim) if qk_norm else nn.Identity()
        self.k_norm = norm_layer(self.head_dim) if qk_norm else nn.Identity()
        if qk_norm:
            ops.check_qk_norm(self.q_norm, self.k_norm, self.head_dim)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        self.pos_encoding = None
        self.num_prefix_tokens = 1  # leading tokens RoPE leaves alone (cls + registers; VisionTransformer sets it)

    def forward(self, x, freqs_cis=None):
        return self.proj_drop(self._branch(x, freqs_cis))

    def _branch(self, x, freqs_cis=None):
        """The attention output before proj_drop (the fused block loop applies it in the next add+LayerNorm)."""
        pe = self.pos_encoding
        cos = sin = None
        bias_mode, bias_param, bias_grid = _lib.BIAS_NONE, None, 0
        if isinstance(pe, (RoPEAxial, RoPEMixed)) and freqs_cis is not None:
            cos, sin = freqs_cis  # rotary branch: no additive bias (vit.py:51-71)
        elif isinstance(pe, RelativePositionalEncoding):
            bias_mode, bias_param = _lib.BIAS_TABLE, pe.relative_position_bias_table
        elif isinstance(pe, PolynomialRPE):
            bias_mode, bias_param, bias_grid = _lib.BIAS_POLY, pe.coefficients, pe.grid_size
        dt = ops.compute_dtype(x)
        qk = (None, None) if type(self.q_norm) is nn.Identity and type(self.k_norm) is nn.Identity else (self.q_norm,
                                                                                                      self.k_norm)
        planes = ops.qkv_rope(x, self.qkv.weight, cos, sin, self.num_heads, ops.lp_weight(self.qkv.weight, dt),
                              self.num_prefix_tokens, *qk)
        out = ops.fused_attention(planes, self.scale, bias_mode, bias_param, bias_grid)
        return ops.linear(out, self.proj, ops.lp_weight(self.proj.weight, dt))

    def set_pos_encoding(self, pos_encoding):
        self.pos_encoding = pos_encoding  # registers the shared PE module as a child (state_dict dups)


class Block(nn.Module):
    """Pre-LN transformer block (reference vit.py:100-129); ``init_values`` adds timm's LayerScale ``ls1`` / ``ls2``
    (None or 0: none, the reference's block).  ``mlp_layer``: ``Mlp`` (default) or a ``GluMlp`` factory such as
    ``SwiGLUPacked``, built with ``hidden_features = int(dim * mlp_ratio)`` (fc1's width) as timm does.  ``qk_norm``:
    QK-norm in the attention, with this block's ``norm_layer``."""

    def __init__(self, dim, num_heads, mlp_ratio=4., qkv_bias=False, drop=0., attn_drop=0.,
                 drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm, init_values=None, mlp_layer=Mlp,
                 qk_norm=False):
        super().__init__()
        if mlp_layer is not Mlp and not _is_glu_factory(mlp_layer):
            raise ValueError(f"mlp_layer must be Mlp or a GluMlp factory (e.g. SwiGLUPacked), got {mlp_layer!r}")
        self.norm1 = norm_layer(dim)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias, attn_drop=attn_drop, proj_drop=drop,
                              qk_norm=qk_norm, norm_layer=norm_layer)
        self.ls1 = LayerScale(dim, init_values) if init_values else nn.Identity()
        self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.norm2 = norm_layer(dim)
        if mlp_layer is Mlp:
            self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)
        else:
            self.mlp = mlp_layer(in_features=dim, hidden_features=int(dim * mlp_ratio), drop=drop)
        self.ls2 = LayerScale(dim, init_values) if init_values else nn.Identity()

    def forward(self, x, freqs_cis=None):
        x = x + self.drop_path(self.ls1(self.attn(ops.layer_norm(x, self.norm1), freqs_cis=freqs_cis)))
        x = x + self.drop_path(self.ls2(self.mlp(ops.layer_norm(x, self.norm2))))
        return x

    def set_pos_encoding(self, pos_encoding):
        self.attn.set_pos_encoding(pos_encoding)


class VisionTransformer(nn.Module):
    """ViT with selectable positional encoding (reference vit.py:131-285).

    ``pos_encoding`` is one of ``none | absolute | relative | polynomial | rope-axial | rope-mixed``;
    anything else raises ``ValueError`` (vit.py:196).  ``drop_rate`` is every block's proj_drop / Mlp dropout,
    ``drop_path_rate`` the stochastic-depth rate of the last block (timm's rule: block i of d gets
    ``linspace(0, drop_path_rate, d)[i]``); both default to 0, the reference's values.

    ``reg_tokens`` adds that many register tokens after the cls token (parameter ``reg_token`` [1, R, E], present
    only when R > 0, initialised ``normal_(std=1e-6)`` as timm does, drawn after every other parameter so the rest of
    a seeded model is unchanged).  The relative and polynomial biases are defined against a single cls token and
    raise ``ValueError`` with registers.

    ``init_values`` gives every block LayerScale (``blocks.{i}.ls1.gamma`` / ``ls2.gamma`` [E], filled with the value;
    no random numbers are drawn); None or 0, the default, means none.

    ``mlp_layer`` is every block's MLP: ``Mlp`` (default) or a ``GluMlp`` factory; ``SwiGLUPacked`` with
    ``mlp_ratio = 16 / 3`` matches the GELU MLP's parameters and FLOPs (fc1 ``E -> 2H``, fc2 ``H -> E``).

    ``qk_norm`` gives every attention QK-norm (``blocks.{i}.attn.q_norm`` / ``k_norm``, ``nn.LayerNorm(head_dim)``
    initialised to ones / zeros; no random numbers are drawn).
    """

    def __init__(self, img_size=32, patch_size=4, in_chans=3, num_classes=10,
                 embed_dim=192, depth=6, num_heads=6, mlp_ratio=4.,
                 pos_encoding='absolute', rope_theta=100.0,
                 poly_degree=3, poly_shared_heads=True, drop_rate=0., drop_path_rate=0., reg_tokens=0,
                 init_values=None, mlp_layer=Mlp, qk_norm=False):
        super().__init__()
        if mlp_layer is not Mlp and not _is_glu_factory(mlp_layer):
            raise ValueError(f"mlp_layer must be Mlp or a GluMlp factory (e.g. SwiGLUPacked), got {mlp_layer!r}")
        if reg_tokens < 0:
            raise ValueError(f"reg_tokens must be >= 0, got {reg_tokens}")
        if reg_tokens > 0 and pos_encoding in ('relative', 'polynomial'):
            raise ValueError(f"reg_tokens > 0 is not supported with pos_encoding={pos_encoding!r}: its attention bias "
                             "is defined against a single cls token")
        self.num_classes = num_classes
        self.embed_dim = embed_dim
        self.patch_size = patch_size
        self.pos_encoding_type = pos_encoding
        self.head_dim = embed_dim // num_heads
        self.num_heads = num_heads
        self.num_patches = (img_size // patch_size) ** 2
        self.num_reg_tokens = reg_tokens
        self.num_prefix_tokens = 1 + reg_tokens

        # parameter holder for the patch projection; the forward pass runs the unfold+GEMM kernel
        self.patch_embed = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))

        self.use_pos_embed_in_forward = pos_encoding == 'absolute'
        self.use_rope = pos_encoding in ('rope-axial', 'rope-mixed')
        if pos_encoding == 'absolute':
            self.pos_embed = AbsolutePositionalEncoding(embed_dim)
        elif pos_encoding == 'relative':
            self.pos_embed = RelativePositionalEncoding(self.num_patches, num_heads)
        elif pos_encoding == 'polynomial':
            self.pos_embed = PolynomialRPE(self.num_patches, degree=poly_degree, num_heads=num_heads,
                                           shared_across_heads=poly_shared_heads)
        elif pos_encoding == 'rope-axial':
            self.pos_embed = RoPEAxial(dim=self.head_dim, theta=rope_theta)
        elif pos_encoding == 'rope-mixed':
            self.pos_embed = RoPEMixed(dim=self.head_dim, num_heads=num_heads, theta=rope_theta)
        elif pos_encoding == 'none':
            self.pos_embed = NoPositionalEncoding()
        else:
            raise ValueError(f"Unknown positional encoding type: {pos_encoding}")

        dpr = [r.item() for r in torch.linspace(0, drop_path_rate, depth)]  # draws no random numbers
        self.blocks = nn.ModuleList([Block(embed_dim, num_heads, mlp_ratio, drop=drop_rate, drop_path=dpr[i],
                                           init_values=init_values, mlp_layer=mlp_layer, qk_norm=qk_norm)
                                     for i in range(depth)])
        if not self.use_pos_embed_in_forward:
            for blk in self.blocks:
                blk.set_pos_encoding(self.pos_embed)  # one shared module, referenced by every block
        for blk in self.blocks:
            blk.attn.num_prefix_tokens = self.num_prefix_tokens

        self.norm = nn.LayerNorm(embed_dim)
        self.head = nn.Linear(embed_dim, num_classes)
        self.apply(self._init_weights)
        if reg_tokens > 0:  # drawn last: every other tensor matches a model built with the same seed and no registers
            self.reg_token = nn.Parameter(torch.zeros(1, reg_tokens, embed_dim))
            nn.init.normal_(self.reg_token, std=1e-6)

    def _init_weights(self, m):
        """Same initialisers as the reference (vit.py:216-233); PE parameters are left alone."""
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=0.02)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)
        elif isinstance(m, nn.Conv2d):
            nn.init.kaiming_normal_(m.weight, mode='fan_out', nonlinearity='relu')
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)

    def forward_features(self, x):
        """[B, C, H, W] -> [B, N, E] with N = (H/P)(W/P) + num_prefix_tokens taken from the input (vit.py:235-271)."""
        x, m, drop, ls = self._features(x)
        if m is None:
            return x
        if drop is not None:
            m = m.float() * ops.branch_factor(drop, *m.shape)
        if ls is not None:
            m = m.float() * ls
        return x + m

    def _drop_sites(self, x):
        """Per block (attention branch, fc1's activation, MLP branch): the dropout sites of one training forward, all
        keyed by one seed drawn here, or None where a rate is 0.  Sites 3i, 3i+1, 3i+2 of block i."""
        rates = []
        for blk in self.blocks:
            pp = blk.drop_path.drop_prob if isinstance(blk.drop_path, DropPath) else 0.
            rates.append((_drop_p(blk.attn.proj_drop), pp, _drop_p(blk.mlp.drop1), _drop_p(blk.mlp.drop2)))
        if not self.training or not any(any(r) for r in rates):
            return None
        seed = ops.new_seed(x.device)
        self._drop_seed = seed  # the key of the last training forward (tests replay its masks)
        N = x.shape[1]
        site = lambda p, pp, i: (p, pp, N, i, seed) if (p > 0 or pp > 0) else None
        return [(site(pa, pp, 3 * i), site(p1, 0., 3 * i + 1), site(p2, pp, 3 * i + 2))
                for i, (pa, pp, p1, p2) in enumerate(rates)]

    def _features(self, x):
        """The token stream before the LAST residual add, that add's branch, its dropout site and its LayerScale gamma
        (or the finished stream, None, None, None): ``forward`` only needs the cls row of the sum."""
        B, C, H, W = x.shape
        h, w = H // self.patch_size, W // self.patch_size
        if x.is_cuda:  # one multi-tensor refresh of the 16-bit weight copies per forward (no-op in fp32)
            ops.refresh_lp_weights(self._gemm_weights(), ops.compute_dtype(x))
        abs_table = self.pos_embed.pos_embed if self.use_pos_embed_in_forward else None
        # (under autocast the token stream comes back fp32, like the reference's cat with the fp32 cls token)
        prefix = self.cls_token if self.num_reg_tokens == 0 else torch.cat((self.cls_token, self.reg_token), 1)
        x = ops.patch_embed(x, self.patch_embed.weight, self.patch_embed.bias, prefix, abs_table, self.patch_size)

        freqs_cis = None
        if self.use_rope:
            freqs_cis = self.pos_embed.get_freqs_cis(h * w, x.device)  # once per forward, all blocks
        if not self._fusable(x):
            for blk in self.blocks:
                x = blk(x, freqs_cis=freqs_cis)
            return x, None, None, None
        # Same arithmetic as the loop above (vit.py:120-125 per block), with every residual add fused with
        # the LayerNorm that follows it - also across block boundaries:
        #   x = x + drop_path(ls1(proj_drop(attn(norm1(x)))));  x = x + drop_path(ls2(drop2(mlp(norm2(x)))))
        blocks = self.blocks
        sites = self._drop_sites(x)
        y = ops.layer_norm(x, blocks[0].norm1)
        m = d_mlp = None
        for i, blk in enumerate(blocks):
            d_attn, d_fc1, d_mlp = sites[i] if sites is not None else (None, None, None)
            x, y = ops.add_layer_norm(x, blk.attn._branch(y, freqs_cis=freqs_cis), blk.norm2, drop=d_attn,
                                      ls=_gamma(blk.ls1))
            m = blk.mlp._branch(y, d_fc1)
            if i + 1 < len(blocks):
                x, y = ops.add_layer_norm(x, m, blocks[i + 1].norm1, drop=d_mlp, ls=_gamma(blk.ls2))
        return x, m, d_mlp, _gamma(blocks[-1].ls2)

    def _gemm_weights(self):
        ws = [self.head.weight]
        for blk in self.blocks:
            ws += [blk.attn.qkv.weight, blk.attn.proj.weight]
            if isinstance(blk.mlp, (Mlp, GluMlp)):
                ws += [blk.mlp.fc1.weight, blk.mlp.fc2.weight]
        return ws

    def _fusable(self, x):
        return len(self.blocks) > 0 and all(
            type(blk) is Block and type(blk.drop_path) in (nn.Identity, DropPath) and type(blk.mlp) in (Mlp, GluMlp)
            and type(blk.ls1) in (nn.Identity, LayerScale) and type(blk.ls2) in (nn.Identity, LayerScale)
            and type(blk.attn.proj_drop) is nn.Dropout and type(blk.mlp.drop2) is nn.Dropout
            and ops.can_fuse_add_layer_norm(x, blk.norm1) and ops.can_fuse_add_layer_norm(x, blk.norm2)
            for blk in self.blocks)

    def forward(self, x):
        x, m, drop, ls = self._features(x)
        # LayerNorm is per token and only the cls token reaches the head (vit.py:284-285): the last residual
        # add and the final norm of that row alone give identical logits and gradients (with dropout: the factors
        # of token rows b*N; with LayerScale: then times gamma - the same arithmetic as forward_features)
        if m is None:
            cls = x[:, 0]
        elif drop is None and ls is None:
            cls = x[:, 0] + m[:, 0]
        else:
            b = m[:, 0]
            if drop is not None:
                b = b.float() * ops.branch_factor(drop, *m.shape, cls_only=True)[:, 0]
            if ls is not None:
                b = b.float() * ls
            cls = x[:, 0] + b
        y = ops.layer_norm(cls, self.norm)
        return ops.linear(y, self.head, ops.lp_weight(self.head.weight, ops.compute_dtype(y)))
