"""CPU oracle for the device random-number stream (Philox4x32-10 + Box-Muller).

TEST INFRASTRUCTURE ONLY (see oracle/flow.py header for who may import this).

The reference draws from torch's global CPU generator (sampler.py:310,334,377,412) which cannot
be reproduced on a GPU; north_star replaces it by a counter-based Philox stream keyed per chain.
This module is the executable specification of that stream (documented in DESIGN.md):
  key     = (seed & 0xffffffff, seed >> 32)
  counter = (j, step, chain, tag)   tag 0: proposal normals, 1: accept uniform, 2: start latents,
                                    3: jitter of the flow-fitting data (step = epoch, chain = position in the epoch)
  normals for dims 4j..4j+3 come from the four outputs of counter word j (two Box-Muller pairs)
Pinned by the Random123 known-answer vectors in tests/test_oracle_philox.py.
"""
import numpy as np

M0 = np.uint64(0xD2511F53)
M1 = np.uint64(0xCD9E8D57)
W0 = 0x9E3779B9
W1 = 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)
TAG_NORMAL, TAG_UNIFORM, TAG_INIT, TAG_TRAIN = 0, 1, 2, 3
TWO_M24 = np.float32(1.0 / 16777216.0)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """All arguments broadcastable unsigned 32-bit values; returns 4 uint32 arrays."""
    c0, c1, c2, c3 = [np.asarray(c, dtype=np.uint64) & MASK for c in (c0, c1, c2, c3)]
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = int(k0) & 0xFFFFFFFF
    k1 = int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0
        p1 = M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0)), lo1, (hi0 ^ c3 ^ np.uint64(k1)), lo0
        k0 = (k0 + W0) & 0xFFFFFFFF
        k1 = (k1 + W1) & 0xFFFFFFFF
    return [c.astype(np.uint32) for c in (c0, c1, c2, c3)]


def _box_muller(ra, rb):
    u1 = ((ra >> np.uint32(8)).astype(np.float32) + np.float32(1.0)) * TWO_M24       # (0, 1]
    u2 = (rb >> np.uint32(8)).astype(np.float32) * TWO_M24                            # [0, 1)
    rad = np.sqrt(np.float32(-2.0) * np.log(u1)).astype(np.float32)
    ang = ((u2 - np.float32(0.5)) * np.float32(6.283185307179586)).astype(np.float32)      # [-pi, pi)
    return (rad * np.cos(ang)).astype(np.float32), (rad * np.sin(ang)).astype(np.float32)


def normals(seed, step, chains, d, tag=TAG_NORMAL):
    """float32 (len(chains), d) standard normals for one step."""
    chains = np.asarray(chains, dtype=np.uint64)
    nblk = (d + 3) // 4
    j = np.arange(nblk, dtype=np.uint64)[None, :]
    r = philox4x32_10(j, step, chains[:, None], tag, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    n0, n1 = _box_muller(r[0], r[1])
    n2, n3 = _box_muller(r[2], r[3])
    out = np.stack([n0, n1, n2, n3], axis=-1).reshape(len(chains), nblk * 4)
    return np.ascontiguousarray(out[:, :d])


def uniforms(seed, step, chains):
    """float32 (len(chains),) in [0,1) for the accept test of one step."""
    chains = np.asarray(chains, dtype=np.uint64)
    r = philox4x32_10(0, step, chains, TAG_UNIFORM, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return (r[0] >> np.uint32(8)).astype(np.float32) * TWO_M24


class PhiloxNoise(object):
    """Noise provider for oracle.mcmc.mcmc_sample mirroring the device stream."""

    def __init__(self, seed, chain_offset=0, step_offset=0):
        self.seed, self.chain_offset, self.step_offset = int(seed), int(chain_offset), int(step_offset)

    def normal(self, step, n, d):
        return normals(self.seed, self.step_offset + step, self.chain_offset + np.arange(n), d)

    def uniform(self, step, n):
        return uniforms(self.seed, self.step_offset + step, self.chain_offset + np.arange(n))
