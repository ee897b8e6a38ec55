"""CPU checks of oracle/tridiag_stream.py, the numpy restatement of the solve kernel's normals: Philox4x32-10
against the Random123 known-answer vectors, the counter spill beyond block 2^20, the element -> block map, and the
split between the fp32 fast pair and the fp64 redo."""

import numpy as np
import pytest

from oracle import tridiag_stream as ts


@pytest.mark.parametrize("ctr,key,out", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox4x32_10_known_answers(ctr, key, out):
    assert tuple(int(v) for v in ts.philox4x32_10(ctr, key)) == out
    # the same block among others in one vectorised call
    c = [np.array([v, 7, v], dtype=np.uint32) for v in ctr]
    got = ts.philox4x32_10(c, key)
    assert [int(w[0]) for w in got] == list(out) and [int(w[2]) for w in got] == list(out)


def test_counter_spill_beyond_block_2_20():
    blocks = np.array([(1 << 20) - 1, 1 << 20, 1 << 21, 0, 1], dtype=np.uint64)
    c = np.stack(ts.normal_counter(5 + (3 << 32), 11, 7, blocks), axis=1)
    assert len({tuple(r) for r in c}) == len(blocks)
    # below 2^20 the second word is the sweep's high word; block 2^20 wraps word 3 to block 0 and moves word 1
    assert c[0, 1] == 3 and c[3, 1] == 3 and c[1, 3] == c[3, 3] == 7 << 20
    assert c[1, 1] == 3 ^ 0x9E3779B9 and c[2, 1] == 3 ^ ((2 * 0x9E3779B9) & 0xFFFFFFFF)
    assert list(c[:, 2]) == [11] * 5 and list(c[:, 0]) == [5] * 5
    # the first spilled block is block 1 of group 209,715: its first element is 3,774,874
    assert 209_715 * ts.BLOCKS_PER_GROUP + 1 == 1 << 20
    blk, half, pos = ts.element_pair(np.array([3_774_873, 3_774_874]))
    assert list(blk) == [(1 << 20) - 1, 1 << 20] and list(half) == [1, 0] and list(pos) == [1, 0]


def test_element_map_and_whole_chain_agree():
    i = np.arange(40)
    blk, half, pos = ts.element_pair(i)
    # group 0: blocks 0-4, (x, y) (z, w) per block, block 4 only (x, y); group 1 starts at block 5
    assert list(blk[:18]) == [0] * 4 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 2 and blk[18] == 5
    assert list(half[:8]) == [0, 0, 1, 1, 0, 0, 1, 1] and half[16] == 0 and list(pos[:4]) == [0, 1, 0, 1]
    z, redo, tol = ts.chain_normals(3, 2, 1, 5, 5000)
    idx = np.random.default_rng(0).permutation(5000)
    z2, redo2, tol2 = ts.normals_at(3, 2, 1, 5, idx)
    np.testing.assert_array_equal(z2, z[idx])
    np.testing.assert_array_equal(redo2, redo[idx])
    np.testing.assert_array_equal(tol2, tol[idx])
    # block k of a group: its words (x, y) are elements 4k, 4k+1, (z, w) elements 4k+2, 4k+3
    x, y, zz, w = ts.philox4x32_10(ts.normal_counter(2, 1, 5, np.array([5 * 7 + 2], dtype=np.uint64)), ts.seed_key(3))
    a0, a1 = ts.fast_pair(x, y)
    b0, b1 = ts.fast_pair(zz, w)
    np.testing.assert_array_equal(z[7 * 18 + 8: 7 * 18 + 12], [a0[0], a1[0], b0[0], b1[0]])


def test_fast_pair_radius_and_angle():
    w1 = np.array([1 << 12, 0xFFFFFFFF, 0x12345678, (1 << 31) + 1], dtype=np.uint32)
    w2 = np.array([0, 1 << 30, 0x80000000, 0xFFFFFFFF], dtype=np.uint32)
    z0, z1 = ts.fast_pair(w1, w2)
    u = np.array([2.0 ** -20, 0xFFFFFF00 / 2.0 ** 32, 0x12345660 / 2.0 ** 32, 2.0 ** -1])   # 24 leading bits kept
    r = np.sqrt(-2 * np.log(u))
    th = np.array([0.0, np.pi / 2, -np.pi, -2 * np.pi / 2.0 ** 32])
    np.testing.assert_allclose(z0, r * np.cos(th), rtol=1e-15, atol=1e-15)
    np.testing.assert_allclose(z1, r * np.sin(th), rtol=1e-15, atol=1e-15)
    assert np.all(r <= 5.3)


def test_redo_split_follows_radius_word():
    """A pair is redone exactly when its radius word is below 2^12; the redone values are normal_from on the 64-bit
    radius word, so they differ from what the fast pair would give for the same words."""
    seed, sweep, gchain, site = 9, 0, 0, 1
    n_groups = 400_000
    w1, w2 = ts.pair_words(seed, sweep, gchain, site, n_groups)
    z, redo, tol = ts.chain_normals(seed, sweep, gchain, site, n_groups * ts.TG_K)
    expect = np.repeat(w1 < ts.REDO_BELOW, 2, axis=1).reshape(-1)
    np.testing.assert_array_equal(redo, expect)
    assert 1 <= redo.sum() // 2 <= 20       # 3.6e6 pairs x 2^-20
    g, c = np.nonzero(w1 < ts.REDO_BELOW)
    f0, f1 = ts.fast_pair(w1[g, c], w2[g, c])
    s0, s1 = ts.slow_pair(seed, sweep, gchain, site, g * ts.BLOCKS_PER_GROUP + c // 2, c & 1)
    zz = z.reshape(n_groups, ts.TG_K)
    np.testing.assert_array_equal(zz[g, 2 * c], s0)
    np.testing.assert_array_equal(zz[g, 2 * c + 1], s1)
    assert np.all(np.abs(f0 - s0) + np.abs(f1 - s1) > 1e-9)
    # the radius is exact beyond the fast path's 24 bits: -2 ln U from the full 64-bit word
    assert np.all(np.hypot(s0, s1) > 5.0)
    assert np.all(tol[redo] == ts.REDO_ABS)


def test_fast_pair_tolerance_follows_radius():
    """The fast-pair bar widens as 2^-21 / r near U = 1, where fp32 lg2 error dominates the radius, and is at most
    2e-5 plus 4.8e-7 for radii of 1 and above."""
    w1 = np.array([0xFFFFFFFF, 0xF0000000, 1 << 31, 1 << 20], dtype=np.uint32)
    z0, z1 = ts.fast_pair(w1, np.zeros(4, dtype=np.uint32))
    r = np.hypot(z0, z1)
    tol = ts.tolerance(r, np.zeros(4, dtype=bool))
    assert r[0] < 4e-4 and tol[0] > 1e-3                 # U = 1 - 2^-24: the smallest fast radius
    assert np.all(tol[2:] <= ts.FAST_ABS + 2.0 ** -21)  # r >= 1.17
