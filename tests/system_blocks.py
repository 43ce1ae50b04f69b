"""Block-wise comparison of reduced systems (S, b and the per-dof vectors) with the oracle's.

A tolerance relative to max|S| says little about the bias and gravity parts of S: their entries are 1e-9 .. 1e-5 of
the largest pose entry, so a global check at 1e-9 passes whatever they hold.  Here the reduced dofs are split into
per-knot pose blocks (6), per-knot gyroscope- and accelerometer-bias blocks (3 each) and the gravity block (2); every
block of S is held to a tolerance relative to its OWN largest entry, and every entry the reference has as exactly zero
(gyro x accel bias, unequal bias components, pose blocks outside the band) must be exactly zero.
"""
import numpy as np

TOL = 1e-9
CS_FLOOR = 1e-7
KINDS = ("pose", "gyro_bias", "accel_bias", "gravity")


def rel_err(a, b):
    """max |a - b| / max |b| (the global measure; blind to blocks far below max |b|)."""
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-300))


class DofLayout:
    """Reduced-system dof order: 6 K pose | 3 Kbg gyroscope bias | 3 Kba accelerometer bias | 2 gravity."""

    def __init__(self, K, Kbg, Kba):
        self.K, self.Kbg, self.Kba = K, Kbg, Kba
        sizes = [6] * K + [3] * Kbg + [3] * Kba + [2]
        self.kind = np.array([0] * K + [1] * Kbg + [2] * Kba + [3])
        self.knot = np.concatenate([np.arange(K), np.arange(Kbg), np.arange(Kba), [0]])
        self.starts = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.intp)
        self.n = int(np.sum(sizes))
        self.kind_of_dof = np.repeat(self.kind, sizes)

    @classmethod
    def of(cls, win):
        return cls(win.knots.shape[0], win.gyro_bias.shape[0], win.accel_bias.shape[0])

    def name(self, i):
        return f"{KINDS[self.kind[i]]} {self.knot[i]}" if self.kind[i] < 3 else "gravity"

    def block_max(self, M):
        """max |M| over every (row block, column block) pair."""
        A = np.maximum.reduceat(np.abs(M), self.starts, axis=0)
        return np.maximum.reduceat(A, self.starts, axis=1)


def matrix_mismatches(got, ref, lay, tol=TOL, tols=None, zeros=None):
    """Every block of `got` whose max deviation from `ref` exceeds tol x that block's scale, and every entry that is
    non-zero where `ref` is exactly zero (or where `zeros` is set: the structural zeros when `ref` is itself a device
    run, whose sums can cancel to an exact zero by chance).  tols: {(kind_a, kind_b): tol} for a block family that needs
    its own bound.  Returns human-readable findings (empty list: the matrices agree).

    A block's scale is its own max |ref|, but not less than CS_FLOOR x sqrt(max|ref_ii| max|ref_jj|) of the diagonal
    blocks it couples: a symmetric positive semi-definite S has |S_ij| <= sqrt(S_ii S_jj), and the rounding of the sums
    (J^T J, the Schur complement) that make S_ij scales with their terms, bounded so, not with a near-cancelled result
    (band-edge fill-in blocks 1e-11 of the diagonal, B-spline edge weights)."""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape == (lay.n, lay.n), (got.shape, ref.shape, lay.n)
    out = []
    zero = (ref == 0) if zeros is None else np.asarray(zeros)
    bad_zero = zero & (got != 0)
    if bad_zero.any():
        rows, cols = np.nonzero(bad_zero)
        blocks = sorted({(int(np.searchsorted(lay.starts, r, side="right") - 1), int(np.searchsorted(lay.starts, c, side="right") - 1))
                         for r, c in zip(rows[:2000], cols[:2000])})
        for bi, bj in blocks[:20]:
            out.append(f"S[{lay.name(bi)}, {lay.name(bj)}]: non-zero where the reference is exactly zero")
    err = lay.block_max(np.where(zero, 0.0, got - ref))
    scale = lay.block_max(ref)
    d = np.diag(scale)
    scale = np.maximum(scale, CS_FLOOR * np.sqrt(np.outer(d, d)))
    limit = np.full(err.shape, float(tol))
    for (ka, kb), t in (tols or {}).items():
        a, b = KINDS.index(ka), KINDS.index(kb)
        sel = (lay.kind[:, None] == a) & (lay.kind[None, :] == b) | (lay.kind[:, None] == b) & (lay.kind[None, :] == a)
        limit[sel] = t
    bad = (scale > 0) & (err > limit * scale)
    for bi, bj in zip(*np.nonzero(bad)):
        if bi >= bj:
            out.append(f"S[{lay.name(bi)}, {lay.name(bj)}]: max err {err[bi, bj]:.3e} = {err[bi, bj] / scale[bi, bj]:.3e} of the block's max "
                       f"{scale[bi, bj]:.3e} (limit {limit[bi, bj]:.0e})")
    return out


def vector_mismatches(got, ref, lay, name, tol=TOL):
    """Per dof family (pose, gyro bias, accel bias, gravity): max |got - ref| <= tol x max |ref| of that family; exact
    zeros of `ref` stay exact zeros."""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape == (lay.n,), (got.shape, ref.shape)
    out = []
    for k, kind in enumerate(KINDS):
        sel = lay.kind_of_dof == k
        g, r = got[sel], ref[sel]
        if np.any((r == 0) & (g != 0)):
            out.append(f"{name}[{kind}]: non-zero where the reference is exactly zero")
        scale = np.abs(r).max() if r.size else 0.0
        err = np.abs(g - r).max() if r.size else 0.0
        if err > tol * scale:
            out.append(f"{name}[{kind}]: max err {err:.3e} = {err / (scale + 1e-300):.3e} of the family's max {scale:.3e} (limit {tol:.0e})")
    return out


def assert_system_close(S, b, S_ref, b_ref, lay, tol=TOL, tols=None):
    found = matrix_mismatches(S, S_ref, lay, tol, tols) + vector_mismatches(b, b_ref, lay, "b", tol)
    assert not found, "\n".join(found)


def oracle_packed(packed, n):
    """oracle OracleWindow.build_packed(): undamped, unmasked S (after the landmark Schur complement), b = -g + Schur part,
    diag(J^T J), g and the cost."""
    S = packed[: n * n].reshape(n, n)
    b, diagH, g = (packed[n * n + i * n: n * n + (i + 1) * n] for i in range(3))
    return dict(S=S, b=b, diagH=diagH, g=g, cost=float(packed[n * n + 3 * n]))


def sys_layout(K, beta, m):
    """hb200_types.cuh sys_layout(): offsets (in doubles) of the device's packed band-only system."""
    h, np_ = 6 + 6 * beta, 6 * K
    n = np_ + m
    oA = K * h * 6
    oC = oA + m * np_
    ob = (oC + m * m + 1) & ~1
    oD = (ob + n + 1) & ~1
    og = (oD + n + 1) & ~1
    os_ = (og + n + 1) & ~1
    return dict(h=h, np=np_, n=n, m=m, oA=oA, oC=oC, ob=ob, oD=oD, og=og, os=os_, total=os_ + 8)


def device_packed(buf, K, beta, m):
    """Decode the device's packed system (hb200_system_device_ptr) into dense symmetric S and the oracle's vectors:
    P [K][h][6] band columns (lower), A [m][6K] arrow rows, C [m][m] corner (lower), b = Schur part, diagH, g, scal.
    The device rhs is b - g (densify_kernel); returned as "b" so that it compares with the oracle's b."""
    L = sys_layout(K, beta, m)
    buf = np.asarray(buf, dtype=np.float64)
    assert buf.size == L["total"], (buf.size, L["total"])
    n, np_, h = L["n"], L["np"], L["h"]
    low = np.zeros((n, n))
    P = buf[: K * h * 6].reshape(K, h, 6)
    for c in range(K):
        rows = 6 * c + np.arange(h)
        keep = rows < np_
        low[rows[keep], 6 * c: 6 * c + 6] = P[c, keep]
    low[np_:, :np_] = buf[L["oA"]: L["oA"] + m * np_].reshape(m, np_)
    low[np_:, np_:] = buf[L["oC"]: L["oC"] + m * m].reshape(m, m)
    low = np.tril(low)
    S = low + np.tril(low, -1).T
    b_schur = buf[L["ob"]: L["ob"] + n]
    g = buf[L["og"]: L["og"] + n]
    return dict(S=S, b=b_schur - g, b_schur=b_schur.copy(), diagH=buf[L["oD"]: L["oD"] + n].copy(), g=g.copy(), cost=float(buf[L["os"]]))


def packed_mismatches(got, ref, lay, tol=TOL, tols=None, cost_tol=1e-10, zeros=None, vec_tol=None):
    """Device packed system (device_packed) against the oracle's (oracle_packed) or another device run's."""
    out = matrix_mismatches(got["S"], ref["S"], lay, tol, tols, zeros)
    for key in ("b", "diagH", "g"):
        out += vector_mismatches(got[key], ref[key], lay, key, tol if vec_tol is None else vec_tol)
    if abs(got["cost"] - ref["cost"]) > cost_tol * abs(ref["cost"]):
        out.append(f"cost {got['cost']!r} vs {ref['cost']!r}")
    return out
