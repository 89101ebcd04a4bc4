"""Restatement of the batched engines' random-walk drift (csrc/obe_device.cuh: ObeBDrift; csrc/obe_b200.cu:
k_btruth_drift) for the tests.

The particle drift of instance b is the single engine's keying (oracle/drift.py) with the instance in the high slot
word.  The walk of the simulator's true parameters draws the same float32 Box-Muller normals per instance with its own
counter word and key, so that it shares nothing with the particle drift, the Liu-West jitter or the simulator noise.
"""
import numpy as np

from oracle.drift import drift_normals
from oracle.obe_oracle import _u24, philox4x32_10

TRUTH_CTR = 0x50000000
TRUTH_KEY = 0xD1B54A32D192ED03


def batched_drift_normals(n, d, seed, step, instance):
    """(n, d) normals of slots 0 .. n-1 of instance ``instance`` in drift step ``step`` of a batched engine: the single
    engine's keying with the instance in the high slot word, ctr = (i, b, 0x40000000 | c, step)."""
    return drift_normals(n, d, seed, step, slot_begin=int(instance) << 32)


def truth_normals(n_instances, d, seed, step):
    """(B, d) normals of the batched simulator's truth walk in step ``step``: the per-slot layout of drift_normals with
    ctr = (b_lo, b_hi, 0x50000000 | c, step) and key = seed ^ 0xD1B54A32D192ED03 (float32 rounding, ~1e-6)."""
    b = np.arange(n_instances, dtype=np.uint64)
    blo = (b & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    bhi = (b >> np.uint64(32)).astype(np.uint32)
    key = (int(seed) ^ TRUTH_KEY) & 0xFFFFFFFFFFFFFFFF
    z = np.empty((n_instances, d))
    for c in range((d + 3) // 4):
        x = philox4x32_10(blo, bhi, np.uint32(TRUTH_CTR | c), np.uint32(step), key & 0xFFFFFFFF, key >> 32)
        for h in range(2):
            if 4 * c + 2 * h < d:
                rad = np.sqrt(np.float32(-2.0) * np.log(_u24(x[2 * h])))
                ang = np.float32(2.0) * _u24(x[2 * h + 1]).astype(np.float64) * np.pi
                z[:, 4 * c + 2 * h] = (rad * np.cos(ang).astype(np.float32)).astype(np.float64)
                if 4 * c + 2 * h + 1 < d:
                    z[:, 4 * c + 2 * h + 1] = (rad * np.sin(ang).astype(np.float32)).astype(np.float64)
    return z


def truth_walk(truth, factors, seed, steps, first_step=1):
    """The (B, npm) truths after ``steps`` random-walk steps numbered first_step, first_step+1, ...: each adds F_b z_b
    with ``factors`` one (npm, npm) F for all instances or (B, npm, npm) per instance."""
    x = np.array(truth, dtype=np.float64)
    f = np.asarray(factors, dtype=np.float64)
    fb = np.broadcast_to(f, (x.shape[0],) + f.shape[-2:])
    for k in range(first_step, first_step + steps):
        z = truth_normals(x.shape[0], x.shape[1], seed, k)
        x = x + np.einsum('bjk,bk->bj', fb, z)
    return x
