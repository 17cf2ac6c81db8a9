"""numpy reference of the acting noise of grl_gaussian_act (geometry_rl_b200/csrc/grl_act.cu): Philox4x32-10 and the
Box-Muller mapping documented there, vectorised over samples and components."""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """ctr: uint64 array [..., 4] of 32-bit words, key: [..., 2] -> [..., 4] output words (uint64 holding 32 bits)."""
    c = [np.asarray(ctr[..., i], dtype=np.uint64) for i in range(4)]
    k0, k1 = np.asarray(key[..., 0], dtype=np.uint64), np.asarray(key[..., 1], dtype=np.uint64)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c[0], np.uint64(M1) * c[2]  # 32 x 32 -> 64 bit, no overflow
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & np.uint64(MASK), p1 & np.uint64(MASK),
             ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & np.uint64(MASK), p0 & np.uint64(MASK)]
        k0, k1 = (k0 + np.uint64(W0)) & np.uint64(MASK), (k1 + np.uint64(W1)) & np.uint64(MASK)
    return np.stack(c, axis=-1)


def uniform(words):
    """u = (x + 0.5) 2^-32, exactly representable in fp64, in (0, 1)."""
    return (words.astype(np.float64) + 0.5) * 2.0 ** -32


def box_muller(words):
    """[..., 4] Philox words of one block -> the block's 4 normals (fp64)."""
    u = uniform(words)
    r01, r23 = np.sqrt(-2.0 * np.log(u[..., 0])), np.sqrt(-2.0 * np.log(u[..., 2]))
    t01, t23 = 2.0 * np.pi * u[..., 1], 2.0 * np.pi * u[..., 3]
    return np.stack([r01 * np.cos(t01), r01 * np.sin(t01), r23 * np.cos(t23), r23 * np.sin(t23)], axis=-1)


def act_eps(seed: int, call: int, batch: int, k: int, rank: int = 0):
    """The [batch, k] standard normals grl_gaussian_act draws for state {seed, call} (fp32, like the kernel's output).
    key = (seed low word, seed high word ^ rank), counter = (block, sample, call low word, call high word)."""
    seed &= (1 << 64) - 1
    call &= (1 << 64) - 1
    nblk = (k + 3) // 4
    s, q = np.meshgrid(np.arange(batch, dtype=np.uint64), np.arange(nblk, dtype=np.uint64), indexing="ij")
    ctr = np.stack([q, s, np.full_like(s, call & MASK), np.full_like(s, call >> 32)], axis=-1)
    key = np.broadcast_to(np.array([seed & MASK, (seed >> 32) ^ rank], dtype=np.uint64), s.shape + (2,))
    z = box_muller(philox4x32_10(ctr, key)).reshape(batch, nblk * 4)[:, :k]
    return z.astype(np.float32)
