"""numpy oracle of the seeded sampling noise (include/cesm_b200.h, "Seeded sampling noise"): Philox4x32-10
(Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011; the Random123 constants) and Box-Muller in
float64.  Element e of field f in draw d is word e & 3 of Philox(counter = (e >> 2, d, f_lo, f_hi), key = seed), and
the word pairs (w0, w1), (w2, w3) give (r cos(2 pi u_b), r sin(2 pi u_b)) with r = sqrt(-2 log u_a)."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)
X_T_DRAW = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """ctr: four uint32 arrays (broadcastable), key: (k0, k1) ints -> four uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & MASK for x in np.broadcast_arrays(*ctr)]
    k0, k1 = int(key[0]), int(key[1])
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return [x.astype(np.uint32) for x in c]


def uniform(w):
    """uint32 words -> float64 u = ((w >> 9) + 0.5) 2^-23: 24 significant bits, so the kernel's fp32 value is the
    same number, and it lies in (0, 1)."""
    return ((np.asarray(w, dtype=np.uint32) >> np.uint32(9)).astype(np.float64) + 0.5) * 2.0 ** -23


def field_normal(seed: int, field: int, draw: int, per: int) -> np.ndarray:
    """The `per` float64 normals of one field in one draw."""
    q = np.arange((per + 3) // 4, dtype=np.uint64)
    f = int(field)
    w = philox4x32_10((q, draw, f & 0xFFFFFFFF, f >> 32), (seed & 0xFFFFFFFF, seed >> 32))
    u = [uniform(x) for x in w]
    r01, r23 = np.sqrt(-2.0 * np.log(u[0])), np.sqrt(-2.0 * np.log(u[2]))
    z = np.stack([r01 * np.cos(2 * np.pi * u[1]), r01 * np.sin(2 * np.pi * u[1]),
                  r23 * np.cos(2 * np.pi * u[3]), r23 * np.sin(2 * np.pi * u[3])], axis=1)
    return z.reshape(-1)[:per]
