"""Oracle (test infrastructure): numpy restatement of the normals that `tg_solve_kernel` (csrc/tridiag.cu) draws
when no `debug_z` is injected.  It has no reference counterpart (the reference draws with numpy's generator): it
pins the device stream to its own specification, so that a tile, a thread, a pair or a counter word out of place
shows up element by element.

Stream of one chain, element i (0-based):
  group = i // 18 (the 18 consecutive elements of one solve thread), j = i % 18, pair c = j // 2;
  Philox4x32-10 block = group * 5 + c // 2, words (x, y) for even c and (z, w) for odd c (block 4 uses (x, y) only);
  element j takes the first normal of its pair when j is even, the second when j is odd.
  counter = (sweep lo, sweep hi ^ (block >> 20) * 0x9E3779B9, chain_offset + chain, site << 20 | block & 0xFFFFF),
  key = (seed lo, seed hi).
Pair (w1, w2) with w1 >= 2^12 (`normal_pair_f32`): U = w1 truncated to its 24 leading bits, times 2^-32,
  r = sqrt(-2 ln U), theta = int32(w2) * 2 pi 2^-32, (z0, z1) = r (cos theta, sin theta).  The device evaluates lg2,
  sqrt, sin and cos on the fp32 special-function unit, so it agrees with this fp64 evaluation within `tolerance`,
  not bit for bit:
    angle   sin / cos.approx have absolute error <= 2^-20.5, and theta is rounded to fp32: r * 1.1e-6 at most;
    radius  e2 = -2 ln U = (j + 1 - lg2(m)) * 2 ln 2 carries the absolute error of lg2.approx (<= 2^-22.6) times
            2 ln 2, about 2.2e-7, and r = sqrt(e2) turns it into |dr| <= 2.2e-7 / (2 r).  Near U = 1 the radius is
            small and this term dominates: at r = 5e-4 (U = 1 - 1.2e-7, about one pair in 8e6) it is 2e-4.
  The bar is 2e-5 + 2^-21 / r: 2e-5 covers the angle term (r <= 5.3 on this path) and the fp32 roundings, 2^-21 / r
  is the radius term with a factor of four to spare.  It still fails a swapped pair, a repeated or shifted stream and
  a wrong counter word, which move z by O(1) almost everywhere.
Pair with w1 < 2^12 (`normal_pair_f32_slow`, probability 2^-20): a second block with key (k0 ^ 0x5A1C0DE5, k1 + 1)
  supplies 32 more radius bits and the angle's low word; the pair is `normal_from` in fp64, modelled by
  tools/rng_model.py, and agrees with the device to about 1e-15 (bar 1e-9).
"""

import math

import numpy as np

from tools import rng_model

M32 = np.uint64(0xFFFFFFFF)
PHILOX_M = (np.uint64(0xD2511F53), np.uint64(0xCD9E8D57))
PHILOX_W = (np.uint64(0x9E3779B9), np.uint64(0xBB67AE85))
TG_K = 18                  # elements per solve thread (one "group")
BLOCKS_PER_GROUP = 5       # Philox blocks per group: four normals per block, the last block half used
TILE = 128 * TG_K          # elements per solve tile
REDO_BELOW = 1 << 12       # radius words below this are redone in fp64
FAST_ABS, FAST_RAD = 2e-5, 2.0 ** -21   # device vs model on fp32-assisted pairs: FAST_ABS + FAST_RAD / r
REDO_ABS = 1e-9                         # device vs model on fp64 redo pairs
SLOW_KEY_XOR = 0x5A1C0DE5


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al. 2011) on broadcastable uint32 arrays: ctr = (c0, c1, c2, c3), key = (k0, k1).
    Returns the four output words as uint32 arrays."""
    x, y, z, w = (np.asarray(c, dtype=np.uint64) for c in ctr)
    k0, k1 = (np.asarray(k, dtype=np.uint64) for k in key)
    for _ in range(10):
        p0 = PHILOX_M[0] * x
        p1 = PHILOX_M[1] * z
        x, y, z, w = (p1 >> np.uint64(32)) ^ y ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ w ^ k1, p0 & M32
        k0 = (k0 + PHILOX_W[0]) & M32
        k1 = (k1 + PHILOX_W[1]) & M32
    return tuple(np.asarray(v, dtype=np.uint32) for v in (x, y, z, w))


def normal_counter(sweep, gchain, site, block):
    """Counter words of Philox block `block` (uint64 array) of global chain `gchain` (`normal_counter`)."""
    sweep = int(sweep) & 0xFFFFFFFFFFFFFFFF
    block = np.asarray(block, dtype=np.uint64)
    spill = ((block >> np.uint64(20)) * PHILOX_W[0]) & M32
    c0 = np.full(block.shape, sweep & 0xFFFFFFFF, dtype=np.uint64)
    c1 = np.uint64(sweep >> 32) ^ spill
    c2 = np.full(block.shape, int(gchain) & 0xFFFFFFFF, dtype=np.uint64)
    c3 = ((np.uint64(int(site)) << np.uint64(20)) | (block & np.uint64(0xFFFFF))) & M32
    return c0, c1, c2, c3


def seed_key(seed):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)


def element_pair(i):
    """Philox block, half (0: words x, y; 1: words z, w) and position in the pair (0: z0, 1: z1) of element(s) i."""
    i = np.asarray(i, dtype=np.int64)
    group, j = np.divmod(i, TG_K)
    c = j // 2
    return group * BLOCKS_PER_GROUP + c // 2, c & 1, j & 1


def fast_pair(w1, w2):
    """`normal_pair_f32` evaluated in fp64: the pair the device draws from (w1, w2) when w1 >= 2^12."""
    w1 = np.asarray(w1, dtype=np.uint64)
    nbits = np.floor(np.log2(np.maximum(w1, np.uint64(1)).astype(np.float64))).astype(np.int64) + 1
    drop = np.maximum(nbits - 24, 0).astype(np.uint64)
    u = ((w1 >> drop) << drop).astype(np.float64) * 2.0 ** -32
    with np.errstate(divide="ignore"):
        r = np.sqrt(-2.0 * np.log(u))
    theta = np.asarray(w2, dtype=np.uint32).view(np.int32).astype(np.float64) * (2.0 * math.pi * 2.0 ** -32)
    return r * np.cos(theta), r * np.sin(theta)


def slow_pair(seed, sweep, gchain, site, block, half):
    """`normal_pair_f32_slow` for pair `half` of block(s) `block`: fp64 `normal_from` on 64 radius bits."""
    block = np.asarray(block, dtype=np.uint64)
    half = np.asarray(half, dtype=bool)
    k0, k1 = seed_key(seed)
    ctr = normal_counter(sweep, gchain, site, block)
    b = philox4x32_10(ctr, (k0, k1))
    b2 = philox4x32_10(ctr, (k0 ^ np.uint64(SLOW_KEY_XOR), (k1 + np.uint64(1)) & M32))
    w1 = np.where(half, b[2], b[0]).astype(np.uint64)
    w2 = np.where(half, b[3], b[1]).astype(np.uint64)
    r = (w1 << np.uint64(32)) | np.where(half, b2[2], b2[0]).astype(np.uint64)
    a = (w2 << np.uint64(32)) | np.where(half, b2[3], b2[1]).astype(np.uint64)
    z0, z1, *_ = rng_model.normal_pair(r, a, fast=False)
    return z0, z1


def tolerance(r, redo):
    """Largest |device - model| of a normal whose pair has radius r (module docstring)."""
    with np.errstate(divide="ignore"):
        return np.where(redo, REDO_ABS, FAST_ABS + FAST_RAD / r)


def pair_words(seed, sweep, gchain, site, n_groups):
    """Radius and angle words of every pair of the first `n_groups` groups: two uint32 arrays [n_groups, 9]."""
    blocks = np.arange(n_groups * BLOCKS_PER_GROUP, dtype=np.uint64)
    x, y, z, w = philox4x32_10(normal_counter(sweep, gchain, site, blocks), seed_key(seed))
    w1 = np.stack([x, z], axis=1).reshape(n_groups, 2 * BLOCKS_PER_GROUP)[:, : TG_K // 2]
    w2 = np.stack([y, w], axis=1).reshape(n_groups, 2 * BLOCKS_PER_GROUP)[:, : TG_K // 2]
    return w1, w2


def chain_normals(seed, sweep, gchain, site, n):
    """The n normals of one chain's draw and, per element, whether its pair took the fp64 redo path and how far the
    device's value may be from the model's (`tolerance`)."""
    n_groups = -(-int(n) // TG_K)
    w1, w2 = pair_words(seed, sweep, gchain, site, n_groups)
    z0, z1 = fast_pair(w1, w2)
    redo = w1 < REDO_BELOW
    if redo.any():
        g, c = np.nonzero(redo)
        s0, s1 = slow_pair(seed, sweep, gchain, site, g * BLOCKS_PER_GROUP + c // 2, c & 1)
        z0[g, c], z1[g, c] = s0, s1
    tol = np.repeat(tolerance(np.hypot(z0, z1), redo), 2, axis=1).reshape(-1)[:n]
    z = np.stack([z0, z1], axis=2).reshape(n_groups, TG_K)
    return z.reshape(-1)[:n], np.repeat(redo, 2, axis=1).reshape(-1)[:n], tol


def normals_at(seed, sweep, gchain, site, idx):
    """Normals of the elements `idx` of one chain (any order, any size), whether each is on a redone pair, and the
    tolerance of each."""
    block, half, pos = element_pair(idx)
    b = philox4x32_10(normal_counter(sweep, gchain, site, block.astype(np.uint64)), seed_key(seed))
    w1 = np.where(half == 1, b[2], b[0])
    w2 = np.where(half == 1, b[3], b[1])
    z0, z1 = fast_pair(w1, w2)
    redo = w1 < REDO_BELOW
    if redo.any():
        s0, s1 = slow_pair(seed, sweep, gchain, site, block[redo], half[redo] == 1)
        z0[redo], z1[redo] = s0, s1
    return np.where(pos == 1, z1, z0), redo, tolerance(np.hypot(z0, z1), redo)
