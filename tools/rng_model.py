#!/usr/bin/env python
"""numpy model of `normal_from` in tridiag.cu: the fp64 Box-Muller pair built from the omc_logtab.cuh table, a
degree-7 log series, Taylor sin / cos and the swap and sign bits.  The solve kernel's fp32-assisted generator uses it
only to redo the pairs whose radius word is below 2^12 (oracle/tridiag_stream.py restates the whole stream on top of
it).  Run as a script, it checks the log / sincos approximations against libm and the output distribution against
N(0,1)."""
import math
import os
import re

import numpy as np

_LOGTAB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "openmcmc_b200", "csrc", "omc_logtab.cuh")
tab = []
for line in open(_LOGTAB):
    m = re.findall(r"0x[0-9a-f.]+p[-+]?\d+", line)
    if len(m) == 2:
        tab.append((float.fromhex(m[0]), float.fromhex(m[1])))
tab = np.array(tab)
LN2 = math.log(2.0)
SC = [(-1) ** k / math.factorial(2 * k + 1) for k in range(8)]
CC = [(-1) ** k / math.factorial(2 * k) for k in range(9)]
LC = [(-1) ** (k + 1) / k for k in range(1, 8)]


def horner(cs, x):
    r = np.full_like(x, cs[-1])
    for c in cs[-2::-1]:
        r = r * x + c
    return r


def clz64(r):
    j = np.full(r.shape, 64, dtype=np.int64)
    x = r.copy()
    n = np.zeros(r.shape, dtype=np.int64)
    for s in (32, 16, 8, 4, 2, 1):
        hi = x >> np.uint64(64 - s)
        z = hi == 0
        n = np.where(z, n + s, n)
        x = np.where(z, x << np.uint64(s), x)
    return np.where(r == 0, 64, n)


def normal_pair(r, a, fast=True):
    """normal_from on the 64-bit radius word r and angle word a = (w << 32) | z.  fast=False is normal_from as
    normal_pair_f32_slow calls it: r = (w1 << 32) | the second block's word, every bit of r below its leading one
    feeds the mantissa.  fast=True is the earlier all-fp64 pair generator, which took the 52 low bits of r as the
    mantissa unless its high word had 12 or more leading zeros; no kernel runs it now."""
    j = clz64(r)
    sh = np.where(j >= 63, np.uint64(0), r << np.minimum(j + 1, 63).astype(np.uint64))
    mb = sh >> np.uint64(12)
    if fast:
        slow = (r >> np.uint64(32)) < np.uint64(1 << 20)
        mb_fast = r & np.uint64((1 << 52) - 1)          # low 20 bits of y : x
        mb = np.where(slow, mb, mb_fast)
    idx = (mb >> np.uint64(45)).astype(np.int64)
    m = (np.uint64(0x3FF0000000000000) | mb).view(np.float64)
    rr = m * tab[idx, 0] - 1.0
    p = rr * horner(LC, rr)
    lnm = tab[idx, 1] + p
    E = (j + 1) * LN2 - lnm
    rad = np.sqrt(2 * E + 2.0 ** -47)
    f = (np.uint64(0x3FF0000000000000) | (a & np.uint64((1 << 52) - 1))).view(np.float64) - 1.0   # low 20 of w : z
    bits = ((a >> np.uint64(52)) & np.uint64(7)).astype(np.int64)
    phi = f * (math.pi / 4)
    x2 = phi * phi
    s = phi * horner(SC, x2)
    c = horner(CC, x2)
    s, c = np.where(bits & 1, c, s), np.where(bits & 1, s, c)
    z0 = rad * c * np.where(bits & 2, -1.0, 1.0)
    z1 = rad * s * np.where(bits & 4, -1.0, 1.0)
    # exact reference of E
    U = m * np.exp2(-(j + 1).astype(np.float64))
    return z0, z1, E, -np.log(U), (phi, s, c, bits)


if __name__ == "__main__":
    from scipy import stats

    rng = np.random.default_rng(1)
    N = 4_000_000
    r = rng.integers(0, 2 ** 64, size=N, dtype=np.uint64)
    a = rng.integers(0, 2 ** 64, size=N, dtype=np.uint64)
    z0, z1, E, Eref, (phi, s, c, bits) = normal_pair(r, a)
    print("max |E - (-ln U)|:", np.max(np.abs(E - Eref)), " rel:", np.max(np.abs(E - Eref) / Eref))
    z = np.concatenate([z0, z1])
    print("mean %.5f sd %.5f skew %.5f kurt %.5f" % (z.mean(), z.std(), stats.skew(z), stats.kurtosis(z)))
    print("KS p:", stats.kstest(z[::4], "norm").pvalue, " corr(z0,z1): %.5f" % np.corrcoef(z0, z1)[0, 1])
    print("corr(z0^2,z1^2): %.5f" % np.corrcoef(z0 ** 2, z1 ** 2)[0, 1])
    ang = np.arctan2(z1, z0)
    print("angle KS p:", stats.kstest((ang[::4] + np.pi) / (2 * np.pi), "uniform").pvalue)
