"""Restatement of the random-walk drift step (csrc/obe_device.cuh: obe_drift_normals, ObeDrift) for the tests.

The drift normals reuse the Philox4x32-10 + float32 Box-Muller arithmetic of obe_oracle.device_normals with their own
counter word and key, so that they share nothing with the Liu-West jitter of the same engine seed.
"""
import numpy as np

from oracle.obe_oracle import _u24, philox4x32_10

DRIFT_CTR = 0x40000000
DRIFT_KEY = 0x9E3779B97F4A7C15


def drift_normals(n, d, seed, epoch, slot_begin=0):
    """(n, d) standard normals of particle slots slot_begin .. slot_begin+n-1 as the drift pass draws them: the
    per-slot layout of device_normals -- call c gives coordinates 4c .. 4c+3 -- with ctr = (slot_lo, slot_hi,
    0x40000000 | c, epoch) and key = seed ^ 0x9E3779B97F4A7C15.  Same accuracy caveat as device_normals (float32
    rounding, ~1e-6)."""
    i = np.arange(n, dtype=np.uint64) + np.uint64(slot_begin)
    ilo = (i & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    ihi = (i >> np.uint64(32)).astype(np.uint32)
    key = (int(seed) ^ DRIFT_KEY) & 0xFFFFFFFFFFFFFFFF
    z = np.empty((n, d))
    for c in range((d + 3) // 4):
        x = philox4x32_10(ilo, ihi, np.uint32(DRIFT_CTR | c), np.uint32(epoch), key & 0xFFFFFFFF, key >> 32)
        for h in range(2):
            if 4 * c + 2 * h < d:
                rad = np.sqrt(np.float32(-2.0) * np.log(_u24(x[2 * h])))
                ang = np.float32(2.0) * _u24(x[2 * h + 1]).astype(np.float64) * np.pi
                z[:, 4 * c + 2 * h] = (rad * np.cos(ang).astype(np.float32)).astype(np.float64)
                if 4 * c + 2 * h + 1 < d:
                    z[:, 4 * c + 2 * h + 1] = (rad * np.sin(ang).astype(np.float32)).astype(np.float64)
    return z


def drift_step(particles, factor, z, mask_le=0, mask_lt=0):
    """x + F z per particle (particles (d, n), z (n, d)); a particle whose step would break a constraint mask (bit j
    of mask_le: x_j <= 0, of mask_lt: x_j < 0) keeps its position.  Returns (moved, accepted)."""
    moved = particles + np.asarray(factor) @ z.T
    bad = np.zeros(particles.shape[1], dtype=bool)
    for j in range(particles.shape[0]):
        if (mask_le >> j) & 1:
            bad |= moved[j] <= 0.0
        if (mask_lt >> j) & 1:
            bad |= moved[j] < 0.0
    moved[:, bad] = particles[:, bad]
    return moved, ~bad
