"""Lane-level numpy model of csrc/dense_warp.cu (one warp per chain, Q in registers as 8x8 tiles in the DMMA
accumulator layout).  Every array below has a leading axis of 32 lanes; `shfl(v, src)` is __shfl_sync with a per-lane
source; the tile product is written out as the m8n8k4 fragment contraction.  Checked against numpy's Cholesky: run

    python tools/gen/warp_chol_model.py
"""
import numpy as np

LANES = np.arange(32)
G, KQ = LANES >> 2, LANES & 3


def shfl(v, src):
    return v[np.broadcast_to(src, (32,))]


def rowfrag(t):
    """C-layout tile (t[:, 0], t[:, 1] = elements [g][2kq], [g][2kq+1]) -> (f0, f1) with f_s = element [g][4s + kq]."""
    out = []
    for s in range(2):
        src = 4 * G + 2 * s + (KQ >> 1)
        v0, v1 = shfl(t[:, 0], src), shfl(t[:, 1], src)
        out.append(np.where(KQ & 1, v1, v0))
    return out


def dmma(c, a, b):
    """c[g][2kq + e] += sum_k a(lane (g, k)) * b(lane (n = 2kq + e, k)) -- one m8n8k4 step."""
    A = np.zeros((8, 4))
    B = np.zeros((4, 8))
    A[G, KQ] = a
    B[KQ, G] = b
    P = A @ B
    c = c.copy()
    c[:, 0] += P[G, 2 * KQ]
    c[:, 1] += P[G, 2 * KQ + 1]
    return c


def run(Q, b, z, PB, dmma_panel=False):
    p = Q.shape[0]
    n = 8 * PB
    Qp, bp, zp = np.eye(n), np.zeros(n), np.zeros(n)
    Qp[:p, :p], bp[:p], zp[:p] = Q, b, z
    T = {}
    for i in range(PB):
        for j in range(i + 1):
            T[i, j] = np.stack([Qp[8 * i + G, 8 * j + 2 * KQ], Qp[8 * i + G, 8 * j + 2 * KQ + 1]], axis=1)
    w = [bp[8 * i + G].copy() for i in range(PB)]
    for k in range(PB):
        # dmma_panel: the column operations of the 8 pivot stages run on the diagonal tile and on an identity tile E only
        # (E becomes L_kk^-T); the tiles below the diagonal are then L(i,k) = T(i,k) E on the tensor pipe, and the
        # right-hand side follows as w_i -= L(i,k) w_k
        E = np.stack([(G == 2 * KQ).astype(float), (G == 2 * KQ + 1).astype(float)], axis=1)
        rows = range(k, k + 1) if dmma_panel else range(k, PB)
        for jj in range(8):
            reg, own = jj & 1, KQ == (jj >> 1)
            piv = shfl(T[k, k][:, reg], 4 * jj + (jj >> 1))
            assert np.all(piv > 0)
            rd = 1.0 / np.sqrt(piv)
            for i in rows:
                T[i, k][:, reg] = np.where(own, T[i, k][:, reg] * rd, T[i, k][:, reg])
            if dmma_panel:
                E[:, reg] = np.where(own, E[:, reg] * rd, E[:, reg])
            wc = shfl(w[k], 4 * jj) * rd
            w[k] = np.where(G == jj, wc, w[k])
            lc0 = np.where(2 * KQ > jj, shfl(T[k, k][:, reg], 4 * (2 * KQ) + (jj >> 1)), 0.0)
            lc1 = np.where(2 * KQ + 1 > jj, shfl(T[k, k][:, reg], 4 * (2 * KQ + 1) + (jj >> 1)), 0.0)
            for i in rows:
                lg = shfl(T[i, k][:, reg], 4 * G + (jj >> 1))
                T[i, k][:, 0] -= lg * lc0
                T[i, k][:, 1] -= lg * lc1
                if i == k:
                    w[k] = np.where(G > jj, w[k] - lg * wc, w[k])
                else:
                    w[i] = w[i] - lg * wc
            if dmma_panel:
                le = shfl(E[:, reg], 4 * G + (jj >> 1))
                E[:, 0] -= le * lc0
                E[:, 1] -= le * lc1
            # 1 / L_cc replaces L_cc on the diagonal (nothing reads L_cc again; the backward solve wants the reciprocal)
            T[k, k][:, reg] = np.where(own & (G == jj), rd, T[k, k][:, reg])
        if dmma_panel and k + 1 < PB:
            # B fragments of E: lane (g, kq), step s needs E[4s + kq][g], held by lane (4s + kq, g >> 1), register g & 1
            Bf = []
            for s in range(2):
                src = 4 * (4 * s + KQ) + (G >> 1)
                Bf.append(np.where(G & 1, shfl(E[:, 1], src), shfl(E[:, 0], src)))
            wk0, wk1 = shfl(w[k], 4 * (2 * KQ)), shfl(w[k], 4 * (2 * KQ + 1))
            for i in range(k + 1, PB):
                A = rowfrag(T[i, k])
                c = np.zeros((32, 2))
                for s in range(2):
                    c = dmma(c, A[s], Bf[s])
                T[i, k] = c
                t = c[:, 0] * wk0 + c[:, 1] * wk1
                t = t + shfl(t, LANES ^ 1)
                t = t + shfl(t, LANES ^ 2)
                w[i] = w[i] - t
        R = {i: rowfrag(T[i, k]) for i in range(k + 1, PB)}
        for j in range(k + 1, PB):
            for i in range(j, PB):
                c = T[i, j]
                for s in range(2):
                    c = dmma(c, -R[i][s], R[j][s])
                T[i, j] = c
    # ---- r = w + z in column layout, partial accumulators over g
    zpad = np.concatenate([zp, np.zeros(64)])     # lanes with g >= PB own no element
    zmine = np.stack([zpad[8 * G + 2 * KQ], zpad[8 * G + 2 * KQ + 1]], axis=1)
    racc = {}
    for tc in range(PB):
        for r in range(2):
            wcol = shfl(w[tc], 4 * (2 * KQ + r))
            zcol = shfl(zmine[:, r], 4 * tc + KQ)
            racc[tc, r] = np.where(G == 0, wcol + zcol, 0.0)
    x = np.zeros(n)
    for j in range(PB - 1, -1, -1):
        v = []
        for r in range(2):
            t = racc[j, r].copy()
            for m in (4, 8, 16):
                t = t + shfl(t, LANES ^ m)
            v.append(t)
        for c in range(7, -1, -1):
            lrow = [shfl(T[j, j][:, r], 4 * c + KQ) for r in range(2)]     # L_jj[c][2kq + r] (the diagonal holds 1/L_cc)
            own = v[c & 1] * lrow[c & 1]
            xc = shfl(own, 4 * G + (c >> 1))
            v[c & 1] = np.where(KQ == (c >> 1), xc, v[c & 1])
            for r in range(2):
                v[r] = np.where(2 * KQ + r < c, v[r] - lrow[r] * xc, v[r])
        for r in range(2):
            x[8 * j + 2 * KQ + r] = v[r]
        a0, a1 = shfl(v[0], 4 * G + (G >> 1)), shfl(v[1], 4 * G + (G >> 1))
        xg = np.where(G & 1, a1, a0)
        for tc in range(j):
            for r in range(2):
                racc[tc, r] = racc[tc, r] - T[j, tc][:, r] * xg
    return x[:p]


def tile_matrix(T, PB):
    """Accumulator-layout tiles {(i, j): [32, 2]} -> the dense 8PB x 8PB matrix (absent tiles are zero)."""
    M = np.zeros((8 * PB, 8 * PB))
    for (i, j), t in T.items():
        for r in range(2):
            M[8 * i + G, 8 * j + 2 * KQ + r] = t[:, r]
    return M


def factor_diag(D, E, wk):
    """The 8 pivot stages of a diagonal tile D (accumulator layout) with E (identity on entry -> L_kk^-T) and the
    right-hand side block wk riding along, as csrc/dense_warp.cu's factor_diag.  Returns (Lk, E, wk), Lk the factor
    L_kk (lower triangle)."""
    D, E, wk = D.copy(), E.copy(), wk.copy()
    Lk = np.zeros((8, 8))
    for jj in range(8):
        reg, jq = jj & 1, jj >> 1
        own = KQ == jq
        piv = shfl(D[:, reg], 4 * jj + jq)
        assert np.all(piv > 0)
        rd = 1.0 / np.sqrt(piv)
        D[:, reg] = np.where(own, D[:, reg] * rd, D[:, reg])
        E[:, reg] = np.where(own, E[:, reg] * rd, E[:, reg])
        wc = shfl(wk, 4 * jj) * rd
        wk = np.where(G == jj, wc, wk)
        lc0 = np.where(2 * KQ > jj, shfl(D[:, reg], 8 * KQ + jq), 0.0)
        lc1 = np.where(2 * KQ + 1 > jj, shfl(D[:, reg], 8 * KQ + 4 + jq), 0.0)
        lg, le = shfl(D[:, reg], 4 * G + jq), shfl(E[:, reg], 4 * G + jq)
        Lk[G[KQ == 0], jj] = lg[KQ == 0]
        D[:, 0] -= lg * lc0
        D[:, 1] -= lg * lc1
        wk = np.where(G > jj, wk - lg * wc, wk)
        E[:, 0] -= le * lc0
        E[:, 1] -= le * lc1
    return np.tril(Lk), E, wk


def run_left(Q, b, z, PB):
    """The left-looking kernel (nn_left_draw_kernel): block column k accumulated from the finished columns on the
    tensor pipe, the pivot stages on the diagonal tile only with an identity tile E riding along (E -> L_kk^-T), the
    panel L(i,k) = C(i,k) E by two m8n8k4 steps, w[i] -= L(i,k) w[k] as a lane-local mat-vec and a quad reduction,
    L_kk^-1 kept in place of L_kk, and the backward solve x_j = L_jj^-T v_j as a mat-vec per block.  The products
    take a tile's k index as k = 2kq + s in step s, so every operand fragment is a lane's own accumulator element
    [g][2kq + s] (no re-layout), except E's, which is E[2kq + s][g] by shuffle.
    Returns (x, L, Linv): L the factor (lower block triangle, diagonal blocks included), Linv its diagonal blocks'
    inverses as a block-diagonal matrix."""
    p = Q.shape[0]
    n = 8 * PB
    Qp, bp, zp = np.eye(n), np.zeros(n), np.zeros(n)
    Qp[:p, :p], bp[:p], zp[:p] = Q, b, z
    L, Lkk, Inv = {}, {}, {}
    w = [bp[8 * i + G].copy() for i in range(PB)]
    for k in range(PB):
        # the products from zero, block column k of Q added once at the end
        C = {i: np.zeros((32, 2)) for i in range(k, PB)}
        for j in range(k):
            for i in range(k, PB):
                for s in range(2):
                    C[i] = dmma(C[i], -L[i, j][:, s], L[k, j][:, s])
        for i in range(k, PB):
            C[i] = C[i] + np.stack([Qp[8 * i + G, 8 * k + 2 * KQ], Qp[8 * i + G, 8 * k + 2 * KQ + 1]], axis=1)
        E = np.stack([(G == 2 * KQ).astype(float), (G == 2 * KQ + 1).astype(float)], axis=1)
        Lkk[k], E, w[k] = factor_diag(C[k], E, w[k])
        Inv[k] = E
        # B fragments of E: lane (g, kq), step s needs E[2kq + s][g], held by lane (2kq + s, g >> 1), register g & 1
        Bf = []
        for s in range(2):
            src = 4 * (2 * KQ + s) + (G >> 1)
            Bf.append(np.where(G & 1, shfl(E[:, 1], src), shfl(E[:, 0], src)))
        wk0, wk1 = shfl(w[k], 8 * KQ), shfl(w[k], 8 * KQ + 4)
        for i in range(k + 1, PB):
            c = np.zeros((32, 2))
            for s in range(2):
                c = dmma(c, C[i][:, s], Bf[s])
            L[i, k] = c
            t = c[:, 0] * wk0 + c[:, 1] * wk1
            t = t + shfl(t, LANES ^ 1)
            t = t + shfl(t, LANES ^ 2)
            w[i] = w[i] - t
    # ---- backward solve: racc as in run(); per block a reduction over g, then x[8j + g] = sum_r Linv[r][g] v[r]
    zpad = np.concatenate([zp, np.zeros(64)])
    zmine = np.stack([zpad[8 * G + 2 * KQ], zpad[8 * G + 2 * KQ + 1]], axis=1)
    racc = {}
    for tc in range(PB):
        for r in range(2):
            racc[tc, r] = np.where(G == 0, shfl(w[tc], 4 * (2 * KQ + r)) + shfl(zmine[:, r], 4 * tc + KQ), 0.0)
    x = np.zeros(n)
    for j in range(PB - 1, -1, -1):
        v = []
        for r in range(2):
            t = racc[j, r].copy()
            for m in (4, 8, 16):
                t = t + shfl(t, LANES ^ m)
            v.append(t)
        xg = Inv[j][:, 0] * v[0] + Inv[j][:, 1] * v[1]      # E[g][2kq + r] = L_jj^-1[2kq + r][g]
        xg = xg + shfl(xg, LANES ^ 1)
        xg = xg + shfl(xg, LANES ^ 2)
        x[8 * j + G] = xg
        for tc in range(j):
            for r in range(2):
                racc[tc, r] = racc[tc, r] - L[j, tc][:, r] * xg
    Lfull = tile_matrix(L, PB)
    for k in range(PB):
        Lfull[8 * k:8 * k + 8, 8 * k:8 * k + 8] = Lkk[k]
    Linv = tile_matrix({(k, k): Inv[k] for k in range(PB)}, PB).T
    return x[:p], np.tril(Lfull)[:p, :p], Linv[:p, :p]


if __name__ == "__main__":
    rng = np.random.default_rng(0)
    for p in (64, 40, 33, 8, 3, 57):
        PB = (p + 7) // 8
        A = rng.standard_normal((p, 3 * p + 5))
        Q = A @ A.T + np.eye(p)
        b, z = rng.standard_normal(p), rng.standard_normal(p)
        L = np.linalg.cholesky(Q)
        ref = np.linalg.solve(Q, b) + np.linalg.solve(L.T, z)
        got = run(Q, b, z, PB)
        got2 = run(Q, b, z, PB, dmma_panel=True)
        got3 = run_left(Q, b, z, PB)[0]
        print(p, *(np.max(np.abs(x - ref)) / np.max(np.abs(ref)) for x in (got, got2, got3)))
