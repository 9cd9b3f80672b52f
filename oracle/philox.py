"""Philox4x32-10 counter-based RNG + Box-Muller, numpy restatement of the in-kernel noise generator.

TEST INFRASTRUCTURE -- not product code.  The reference draws all noise with torch's CPU generator
(solver.py:381, xi = randn(K, d, N+1)), which cannot be reproduced on a GPU; the B200 path instead keys a
counter-based generator on the GLOBAL path index so that results are independent of the sharding (SURVEY.md
section 8e).  The integer part is pinned by the Random123 known-answer vectors (tests/test_philox.py); the
float part (Box-Muller) is compared with the device dump ``pspde_philox_dump`` to 1e-5 absolute.

Counter layout (include/pspde.h):  ctr = (k_global, n, j // 4, offset),  key = (seed_lo, seed_hi);
the four 32-bit outputs give the normals for components 4*(j//4) .. 4*(j//4)+3 of xi_{n+1}.
"""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: (..., 4) uint32, key: (..., 2) uint32 (broadcastable). Returns (..., 4) uint32."""
    c = [np.asarray(ctr[..., i], dtype=np.uint32) for i in range(4)]
    k0 = np.asarray(key[..., 0], dtype=np.uint32)
    k1 = np.asarray(key[..., 1], dtype=np.uint32)
    with np.errstate(over="ignore"):
        for r in range(10):
            p0 = M0 * c[0].astype(np.uint64)
            p1 = M1 * c[2].astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & MASK).astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & MASK).astype(np.uint32)
            c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
            if r < 9:
                k0 = (k0 + W0).astype(np.uint32)
                k1 = (k1 + W1).astype(np.uint32)
    return np.stack(c, axis=-1)


def box_muller(r):
    """(..., 4) uint32 -> (..., 4) float32 standard normals; u = ((r >> 8) + 0.5) * 2^-24 in (0, 1)."""
    u = ((r >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
    out = np.empty(r.shape, np.float32)
    for a in (0, 2):
        rad = np.sqrt(np.float32(-2.0) * np.log(u[..., a]))
        ang = np.float32(2 * np.pi) * u[..., a + 1]
        out[..., a] = rad * np.cos(ang)
        out[..., a + 1] = rad * np.sin(ang)
    return out


def normals(seed, offset, k_global, n, d):
    """xi_{n+1}[k, :d] for an array of global path indices k_global and a scalar step n. Returns (len(k), d)."""
    k_global = np.asarray(k_global, dtype=np.uint32)
    nb = (d + 3) // 4
    ctr = np.empty((k_global.size, nb, 4), np.uint32)
    ctr[..., 0] = k_global[:, None]
    ctr[..., 1] = np.uint32(n)
    ctr[..., 2] = np.arange(nb, dtype=np.uint32)[None, :]
    ctr[..., 3] = np.uint32(offset & 0xFFFFFFFF)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    z = box_muller(philox4x32_10(ctr, key))
    return z.reshape(k_global.size, nb * 4)[:, :d]


def u01(r):
    """uint32 -> float32 uniform in (0, 1), as in csrc/philox.cuh."""
    return ((r >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)


def ball_and_time(seed, offset, k_offset, K, d, radius, T):
    """Restatement of diffusion_sample_kernel (csrc/diffusion_kernels.cuh): X_0 uniform in the ball of radius R (the
    normals of counters (k, 0xFFFFFFFF, jb, offset), normalised, times R u_0^(1/d)) and t_0 = u_1 T in [0, T), where
    (u_0, u_1) are the first two uniforms of counter (k, 0xFFFFFFFE, 0, offset).  float64 from the float32 draws."""
    ks = np.arange(k_offset, k_offset + K)
    z = normals(seed, offset, ks, 0xFFFFFFFF, d).astype(np.float64)
    ctr = np.zeros((K, 4), np.uint32)
    ctr[:, 0], ctr[:, 1], ctr[:, 3] = ks, 0xFFFFFFFE, offset & 0xFFFFFFFF
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    u = u01(philox4x32_10(ctr, key)).astype(np.float64)
    scale = radius / np.sqrt((z ** 2).sum(1)) * u[:, 0] ** (1.0 / d)
    return z * scale[:, None], u[:, 1] * T


def xi_tensor(seed, offset, k_offset, K, d, N):
    """Reference-layout noise tensor (K, d, N+1); slice 0 is unused by the reference and left zero."""
    xi = np.zeros((K, d, N + 1), np.float32)
    ks = np.arange(k_offset, k_offset + K)
    for n in range(N):
        xi[:, :, n + 1] = normals(seed, offset, ks, n, d)
    return xi
