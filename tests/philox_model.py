"""numpy model of the seeded noise of csrc/noise.cu (tests only).

Philox4x32-10 (Salmon et al., SC'11; Random123's constants and key schedule), vectorised over counters, and the full
mapping (seed, c, t) -> normal: key = the seed's 32-bit halves, counter = (t >> 2, c, draw, 0), Box-Muller on the
four words, frame t taking normal t & 3.  The uniforms are the kernel's exact fp32 values; the transcendental part is
evaluated in float64, so the model is the exact value of the kernel's formula."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: uint32-valued array [..., 4], key: [..., 2] (broadcast); returns uint32 [..., 4]."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (ctr[..., i] for i in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(W0)) & MASK
            k1 = (k1 + np.uint64(W1)) & MASK
        p0, p1 = M0 * c0, M1 * c2                      # < 2^64: exact in uint64
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & MASK, p1 & MASK, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & MASK, \
            p0 & MASK
    return np.stack([c0, c1, c2, c3], -1).astype(np.uint32)


def unit_open(w):
    """The kernel's uniforms: odd multiples of 2^-24, as fp32 (exact)."""
    return (((np.asarray(w, np.uint32) >> 8) | 1).astype(np.float64) * 2.0 ** -24).astype(np.float32)


def seeded_normal(seed: int, C: int, T: int, draw: int = 0) -> np.ndarray:
    """float64 [C, T]: the exact value of the kernel's formula for one item (seed taken modulo 2^64)."""
    seed &= (1 << 64) - 1
    G = (T + 3) // 4
    g, c = np.meshgrid(np.arange(G, dtype=np.uint64), np.arange(C, dtype=np.uint64))
    ctr = np.stack([g, c, np.full_like(g, draw), np.zeros_like(g)], -1)
    w = philox4x32_10(ctr, np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64))
    u = unit_open(w).astype(np.float64)
    r0, r1 = np.sqrt(-2 * np.log(u[..., 0])), np.sqrt(-2 * np.log(u[..., 2]))
    a0, a1 = 2 * np.pi * u[..., 1], 2 * np.pi * u[..., 3]
    n = np.stack([r0 * np.cos(a0), r0 * np.sin(a0), r1 * np.cos(a1), r1 * np.sin(a1)], -1)   # [C, G, 4]
    return n.reshape(C, 4 * G)[:, :T]
