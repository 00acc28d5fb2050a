"""Dropout and stochastic depth without a device: the Philox restatement, the constructor arguments and the flags."""
import numpy as np
import pytest
import torch

import train
from oracle import philox_np
from vit_rpe_rope_b200.models.vit import Block, DropPath, VisionTransformer


@pytest.mark.parametrize("counter,key,want", [
    ([0, 0, 0, 0], (0, 0), [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, (0xffffffff, 0xffffffff), [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], (0xa4093822, 0x299f31d0),
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
])
def test_philox_known_answers(counter, key, want):
    """Random123's known-answer vectors for philox4x32-10 (counter words, key words -> output)."""
    got = philox_np.philox4x32_10(np.array([counter], dtype=np.uint32), key)[0]
    assert [int(v) for v in got] == want


def test_mask_layout_and_rates():
    m = philox_np.element_mask(0x0123456789abcdef, 5, 0.25, 40, 64)
    assert m.shape == (40, 64) and abs(m.mean() - 0.75) < 0.02
    # element (m, n) is half (n & 1) of word (n % 8) >> 1 of group (m E + n) / 8
    r = philox_np.philox4x32_10(np.array([[3 * 64 // 8 + 1, 0, 5, 0]], dtype=np.uint32), (0x89abcdef, 0x01234567))[0]
    t = philox_np.threshold(0.25)
    want = [((int(r[j >> 1]) >> (16 * (j & 1))) & 0xFFFF) < t for j in range(8)]
    assert list(m[3, 8:16]) == want
    assert philox_np.threshold(0.0) == 65536 and philox_np.element_mask(1, 0, 0.0, 2, 8).all()
    f = philox_np.factor(7, 1, 0.1, 0.2, 4, 16, 8)
    kp = philox_np.path_mask(7, 1, 0.2, 4)
    assert (f[~np.repeat(kp, 4)] == 0).all()
    assert set(np.unique(f)) <= {np.float32(0), philox_np.scale(0.1, 0.2)}


KW = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=64, depth=4, num_heads=2,
          pos_encoding="rope-mixed")


def test_rates_leave_the_initial_weights_and_keys_alone():
    torch.manual_seed(3)
    a = VisionTransformer(**KW).state_dict()
    torch.manual_seed(3)
    b = VisionTransformer(**KW, drop_rate=0.1, drop_path_rate=0.1).state_dict()
    assert list(a) == list(b)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_per_block_rates_follow_timm():
    m = VisionTransformer(**KW, drop_rate=0.1, drop_path_rate=0.3)
    want = torch.linspace(0, 0.3, KW["depth"])
    assert isinstance(m.blocks[0].drop_path, torch.nn.Identity)
    for i, blk in enumerate(m.blocks[1:], 1):
        assert isinstance(blk.drop_path, DropPath) and blk.drop_path.drop_prob == pytest.approx(want[i].item())
    for blk in m.blocks:
        assert blk.attn.proj_drop.p == 0.1 and blk.mlp.drop1.p == 0.1 and blk.mlp.drop2.p == 0.1
    plain = VisionTransformer(**KW)
    assert all(isinstance(b.drop_path, torch.nn.Identity) and b.mlp.drop1.p == 0.0 for b in plain.blocks)


def test_drop_path_module_has_timm_attributes():
    d = DropPath(0.2)
    assert d.drop_prob == 0.2 and d.scale_by_keep is True and "0.200" in repr(d)
    x = torch.randn(64, 3, 5)
    d.eval()
    assert d(x) is x
    d.train()
    torch.manual_seed(0)
    y = d(x)
    kept = (y.reshape(64, -1) != 0).all(1)
    assert ((y.reshape(64, -1) != 0).any(1) == kept).all() and 0 < int(kept.sum()) < 64
    assert torch.allclose(y[kept], x[kept] / 0.8)
    assert isinstance(Block(32, 2, drop_path=0.1).drop_path, DropPath)
    with pytest.raises(NotImplementedError):
        Block(32, 2, attn_drop=0.1)


def test_train_flags():
    a = train.get_args([])
    assert a.drop_rate == 0.0 and a.drop_path_rate == 0.0
    a = train.get_args(["--drop_rate", "0.1", "--drop_path_rate", "0.2"])
    assert a.drop_rate == 0.1 and a.drop_path_rate == 0.2
