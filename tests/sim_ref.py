"""numpy restatement of the noise of pp_simulate_batch (kernels.cuh philox4x32_10 / sim_uniform / box_muller).

Philox4x32-10 (Salmon, Moraes, Dror and Shaw 2011, the Random123 constants) in uint64 arithmetic, the uint32 ->
float32 uniform mapping in float32 arithmetic (bit for bit the device's), and Box-Muller in float64 on those
uniforms: the device evaluates it in float32 (accurate logf, sqrtf, sincospif), which the tests bound by
Z_REL * r with r = sqrt(-2 ln u0).
"""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF
# |z_device - z_ref| <= Z_REL r: logf and sincospif within 2 ulp, sqrtf and the product correctly rounded (about
# 2.5 2^-23 r), with a factor 2 to spare
Z_REL = 2.0 ** -20


def philox4x32_10(ctr, key):
    """ctr: 4 uint32 arrays (broadcast together), key: 2 uint32 -> 4 uint32 arrays"""
    c0, c1, c2, c3 = [np.asarray(c, dtype=np.uint64) & MASK for c in ctr]
    k0, k1 = [np.uint64(int(k) & MASK) for k in key]
    for i in range(10):
        if i:
            k0 = np.uint64((int(k0) + W0) & MASK)
            k1 = np.uint64((int(k1) + W1) & MASK)
        p0 = np.uint64(M0) * c0
        p1 = np.uint64(M1) * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & np.uint64(MASK)
        hi1, lo1 = p1 >> np.uint64(32), p1 & np.uint64(MASK)
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
    return [c.astype(np.uint32) for c in (c0, c1, c2, c3)]


def uniform(x):
    """u = f32((x >> 8) 2^-24 + 2^-25), float32 arithmetic as on the device"""
    m = (np.asarray(x, dtype=np.uint32) >> np.uint32(8)).astype(np.float32)
    return m * np.float32(2.0 ** -24) + np.float32(2.0 ** -25)


def box_muller(a, b):
    """(z0, z1, r) in float64 from the uniforms of two uint32 arrays"""
    u0 = uniform(a).astype(np.float64)
    u1 = uniform(b).astype(np.float64)
    r = np.sqrt(-2.0 * np.log(u0))
    return r * np.cos(2.0 * np.pi * u1), r * np.sin(2.0 * np.pi * u1), r


def noise(seed, s_global, nchan, nbin):
    """(z, r) [len(s_global), nchan, nbin]: the standard normal draws of bins 0..nbin-1 of every channel of the given
    global subint indices, and the Box-Muller radius each draw came with"""
    s = np.asarray(s_global, dtype=np.uint64)[:, None, None]
    n = np.arange(nchan, dtype=np.uint64)[None, :, None]
    q = np.arange((nbin + 3) // 4, dtype=np.uint64)[None, None, :]
    x = philox4x32_10((q + 0 * n + 0 * s, n + 0 * q + 0 * s, s & np.uint64(MASK), s >> np.uint64(32)),
                      (int(seed) & MASK, (int(seed) >> 32) & MASK))
    z0, z1, r01 = box_muller(x[0], x[1])
    z2, z3, r23 = box_muller(x[2], x[3])
    z = np.stack([z0, z1, z2, z3], axis=-1).reshape(z0.shape[:2] + (-1,))[..., :nbin]
    r = np.stack([r01, r01, r23, r23], axis=-1).reshape(z0.shape[:2] + (-1,))[..., :nbin]
    return z, r
