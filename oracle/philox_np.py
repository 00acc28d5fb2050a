"""numpy restatement of the dropout / stochastic-depth decisions of include/vrr.h (``vrr_drop_desc``).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random
numbers: as easy as 1, 2, 3", SC'11; the constants of Random123), vectorised over counters.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(counter, key):
    """counter: uint32 array [..., 4]; key: (k0, k1).  Returns uint32 [..., 4]."""
    c = np.asarray(counter, dtype=np.uint64)
    c0, c1, c2, c3 = c[..., 0], c[..., 1], c[..., 2], c[..., 3]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for r in range(10):
        if r:
            k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & _MASK32,
                          (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & _MASK32)
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def threshold(p):
    """Keep threshold of a probability as the library forms it from the fp32 value: round((1 - p) * 65536)."""
    return int(np.rint((1.0 - float(np.float32(p))) * 65536.0))


def split_seed(seed):
    """64-bit key (int, possibly negative as torch.int64 stores it) -> (low word, high word)."""
    s = int(seed) & 0xFFFFFFFFFFFFFFFF
    return s & 0xFFFFFFFF, s >> 32


def element_mask(seed, site, p, M, E):
    """keep [M, E] bool of element dropout at ``site`` (E % 8 == 0)."""
    assert E % 8 == 0
    g = np.arange(M * E // 8, dtype=np.uint64)
    ctr = np.stack([g & _MASK32, g >> np.uint64(32), np.full_like(g, site & 0xFFFFFFFF), np.zeros_like(g)], axis=-1)
    r = philox4x32_10(ctr, split_seed(seed))                       # [groups, 4]
    halves = np.stack([r & 0xFFFF, r >> 16], axis=-1).reshape(-1, 8)  # element j of a group: word j >> 1, half j & 1
    return (halves < threshold(p)).reshape(M, E)


def path_mask(seed, site, p_path, images):
    """keep [images] bool of stochastic depth at ``site``."""
    b = np.arange(images, dtype=np.uint64)
    ctr = np.stack([b, np.zeros_like(b), np.full_like(b, site & 0xFFFFFFFF), np.ones_like(b)], axis=-1)
    r = philox4x32_10(ctr, split_seed(seed))
    return (r[:, 0] & 0xFFFF) < threshold(p_path)


def scale(p, p_path):
    """s = (1 / (1 - p)) * (1 / (1 - p_path)) in fp32."""
    one = np.float32(1)
    return (one / (one - np.float32(p))) * (one / (one - np.float32(p_path)))


def factor(seed, site, p, p_path, rows_per_sample, M, E):
    """f [M, E] float32 = keep * keep_path(m // rows_per_sample) * s."""
    f = np.full((M, E), scale(p, p_path), dtype=np.float32)
    if p > 0:
        f *= element_mask(seed, site, p, M, E)
    if p_path > 0:
        kp = path_mask(seed, site, p_path, -(-M // rows_per_sample))
        f *= kp[np.arange(M) // rows_per_sample][:, None]
    return f
