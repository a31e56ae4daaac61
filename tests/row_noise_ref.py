"""numpy restatement of the keyed row noise of ``k_row_noise`` (DESIGN.md 4.8), shared by the CPU and GPU tests:
Philox4x32-10 on exact integers, the exact uniform mapping, Box-Muller in float64."""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = 0xFFFFFFFF

# Random123 kat_vectors for philox4x32_10: (counter, key, output)
KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((MASK32,) * 4, (MASK32, MASK32), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Elementwise over arrays (or scalars) of uint32 values; returns four uint64 arrays holding uint32 words."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK32 for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0), np.uint64(k1)
    m0, m1, mask = np.uint64(M0), np.uint64(M1), np.uint64(MASK32)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & mask, p1 & mask, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & mask, \
            p0 & mask
        k0, k1 = (k0 + np.uint64(W0)) & mask, (k1 + np.uint64(W1)) & mask
    return c0, c1, c2, c3


def uniform(x):
    """(2 (x >> 9) + 1) 2^-24, exact in float64 (and float32)."""
    x = np.asarray(x, dtype=np.uint64)
    return ((x >> np.uint64(9)) * np.uint64(2) + np.uint64(1)).astype(np.float64) * 2.0 ** -24


def row_noise(seed, draw, T):
    """float64 noise of one row: seed (int, taken mod 2^64), draw index, length T."""
    seed = int(seed) & ((1 << 64) - 1)
    j = np.arange((T + 3) // 4, dtype=np.uint64)
    x0, x1, x2, x3 = philox4x32_10(j, draw, 0, 0, seed & MASK32, seed >> 32)
    out = np.empty((j.size, 4))
    for q, (a, b) in enumerate(((x0, x1), (x2, x3))):
        r = np.sqrt(-2.0 * np.log(uniform(a)))
        th = 2.0 * np.pi * uniform(b)
        out[:, 2 * q] = r * np.cos(th)
        out[:, 2 * q + 1] = r * np.sin(th)
    return out.reshape(-1)[:T]
