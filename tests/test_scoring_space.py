"""The oracle under scoring other than BLOSUM62 (CPU only): asymmetric substitution matrices over 1..64-letter alphabets,
a dyadic matrix at the finest grid the integer kernels accept, a tie-heavy scoring and free gaps.  Every GPU comparison
of tests/test_gpu_scoring_space.py is against the oracle, so the oracle is first anchored here to an independent float64
dynamic program of the same alignment model.  The scoring generators live here and are shared with the GPU file."""
import numpy as np
import pytest

from util import po, MODES, MODE_NAMES

NONLOCAL = [po.GLOBAL_LOCAL, po.GLOBAL, po.LOCAL_GLOBAL, po.SEMI_LOCAL]
# the transposed problem: template and query trade places, so free deletions and free insertions trade places too
SWAPPED_MODE = {po.GLOBAL: po.GLOBAL, po.SEMI_LOCAL: po.SEMI_LOCAL, po.LOCAL: po.LOCAL,
                po.GLOBAL_LOCAL: po.LOCAL_GLOBAL, po.LOCAL_GLOBAL: po.GLOBAL_LOCAL}
ALPHABET_SIZES = [1, 2, 4, 20, 31, 32, 33, 64]


# ---- scoring generators ----

def asym_matrix(A, seed, lo=-9, hi=9):
    """Seeded integer matrix with entries in [lo, hi]; for A > 1 it is asymmetric and sub[0, A-1] != sub[A-1, 0], so a
    query/template swap in any lookup changes the score of a pair that contains both end codes."""
    rng = np.random.default_rng(seed)
    sub = rng.integers(lo, hi + 1, (A, A)).astype(np.float32)
    if A > 1:
        sub[0, A - 1], sub[A - 1, 0] = hi, lo
        assert not np.array_equal(sub, sub.T)
    return sub


def extreme_matrix(A=20, seed=7):
    """Integer matrix whose entries reach +127 and -127 (the int8 profile range at s = 0), placed asymmetrically."""
    sub = asym_matrix(A, seed, -127, 127)
    sub[0, A - 1], sub[A - 1, 0] = 127, -127
    sub[1, 1] = 127
    return sub


def dyadic_matrix(A, seed):
    """Entries k/256 with |k| <= 127 and odd k present: the grid 2^-8 is the smallest one that holds it."""
    rng = np.random.default_rng(seed)
    k = rng.integers(-127, 128, (A, A))
    k[0, A - 1], k[A - 1, 0] = 127, -125
    return (k / 256.0).astype(np.float32)


def tie_matrix(A=4):
    """+1 on the diagonal, -1 elsewhere: with gi = ge = 1 and low-entropy sequences nearly every cell has several
    equal predecessors, so the tie rules ("first maximum in scan order") decide every traceback pointer."""
    return (2 * np.eye(A) - 1).astype(np.float32)


def seq(rng, L, A):
    """Random codes over 0..A-1 that contain both 0 and A-1 (as far as the length allows)."""
    s = rng.integers(0, A, L).astype(np.uint8)
    if L >= 2:
        i, j = rng.choice(L, 2, replace=False)
        s[i], s[j] = 0, A - 1
    elif L == 1:
        s[0] = rng.choice([0, A - 1])
    return s


def low_entropy_seq(rng, L, A=4):
    """Runs of one or two letters: many equal-scoring alignments."""
    out = []
    while len(out) < L:
        a = int(rng.integers(0, A))
        out += [a] * int(rng.integers(1, 6))
        if rng.random() < 0.5:
            out += [a, (a + 1) % A] * int(rng.integers(1, 3))
    return np.array(out[:L], np.uint8)


def scorings():
    """(name, sub, gi, ge) of every scoring the CPU anchor covers; all of them lie on a dyadic grid."""
    out = []
    for A in ALPHABET_SIZES:
        out.append(("asym%d" % A, asym_matrix(A, 1000 + A), 7.0, 2.0))
    out.append(("extreme127", extreme_matrix(), 40.0, 3.0))
    out.append(("dyadic8", dyadic_matrix(20, 5), 3.0 + 1 / 256.0, 0.5 + 3 / 256.0))
    out.append(("ties", tie_matrix(), 1.0, 1.0))
    out.append(("zero_gap", asym_matrix(4, 77), 0.0, 0.0))
    return out


# ---- an independent float64 dynamic program of the reference's alignment model ----

def gotoh_optimum(q, t, sub, gi, ge, at):
    """Forward optimum of the reference's model in float64: an alignment is a path (0,0) -> matched cells -> (Lq+1,Lt+1)
    whose every step advances both indices and skips residues of at most ONE sequence (a deletion skips template
    residues, an insertion query residues; no deletion is adjacent to an insertion).  A gap of length n costs
    gi + ge*(n-1), and nothing where the align type frees that end (tests/test_gpu_parity.py::_rescore,
    aasubalib.h:27-77).  Affine running maxima instead of the oracle's scans; LOCAL returns the Smith-Waterman maximum
    over matched cells (every path may start and end anywhere)."""
    q, t = np.asarray(q, np.int64), np.asarray(t, np.int64)
    sub = np.asarray(sub, np.float64)
    Lq, Lt = len(q), len(t)
    local = at == po.LOCAL
    delfree = at in (po.LOCAL, po.SEMI_LOCAL, po.LOCAL_GLOBAL)
    insfree = at in (po.LOCAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL)
    NEG = -np.inf
    # M[i, j]: best path from (0,0) ending with q[i-1] matched to t[j-1]; row/column 0 hold only the start (0,0)
    M = np.full((Lq + 1, Lt + 1), NEG)
    M[0, 0] = 0.0
    col_acc = np.full(Lt + 1, NEG)  # max over rows r <= i-2 of M[r, j] + ge*r (insertions ending in column j+1)
    cols = np.arange(Lt + 1, dtype=np.float64)

    def pen(n):
        return gi + ge * (n - 1)

    for i in range(1, Lq + 1):
        P = M[i - 1]
        if i >= 2:
            col_acc = np.maximum(col_acc, M[i - 2] + ge * (i - 2))
        best = np.full(Lt + 1, NEG)
        best[1:] = P[:-1]                                                     # diagonal
        # deletion (i-1,k) -> (i,j), k <= j-2, length j-1-k: prefix maximum of P[k] + ge*k
        acc = np.maximum.accumulate(P + ge * cols)
        best[2:] = np.maximum(best[2:], acc[:-2] - (gi + ge * (cols[2:] - 2)))
        if delfree:                                                           # from (0,0): free leading deletion
            best[2:] = np.maximum(best[2:], P[0])
        # insertion (r,j-1) -> (i,j), r <= i-2, length i-1-r
        if i >= 2:
            best[1:] = np.maximum(best[1:], col_acc[:-1] - (gi + ge * (i - 2)))
            if insfree and Lt:
                best[1] = max(best[1], M[0, 0])
        if local:
            best = np.maximum(best, 0.0)                                      # a local path starts anywhere
        row = sub[q[i - 1], t] + best[1:]
        M[i, 1:] = np.maximum(row, 0.0) if local else row
    if local:
        return float(M[1:, 1:].max()) if Lq and Lt else 0.0
    # the final cell (Lq+1, Lt+1), similarity 0: from the last matched cell, or across one end gap
    cand = [M[Lq, Lt]] if (Lq and Lt) or (not Lq and not Lt) else []
    if Lt:   # deletion of t[k+1..Lt] after (Lq, k)
        src = [(0.0, 0)] if Lq == 0 else [(M[Lq, k], k) for k in range(1, Lt)]
        cand += [v - (0.0 if delfree else pen(Lt - k)) for v, k in src]
    if Lq:   # insertion of q[r+1..Lq] after (r, Lt)
        src = [(0.0, 0)] if Lt == 0 else [(M[r, Lt], r) for r in range(1, Lq)]
        cand += [v - (0.0 if insfree else pen(Lq - r)) for v, r in src]
    return float(max(cand))


def oracle_optimum(O, q, t):
    F = O.fill(q, t, po.FWD, True, fast=True)[0]
    if O.align_type == po.LOCAL:
        return float(F[1:-1, 1:-1].max()) if len(q) and len(t) else 0.0
    return float(F[-1, -1])


def _pairs(rng, A, n, maxlen, low_entropy=False):
    for k in range(n):
        Lq, Lt = int(rng.integers(0, maxlen)), int(rng.integers(0, maxlen))
        if k < 4:
            Lq, Lt = [(0, 0), (0, 5), (6, 0), (1, 1)][k]
        if low_entropy:
            yield low_entropy_seq(rng, Lq, A), low_entropy_seq(rng, Lt, A)
        else:
            yield seq(rng, Lq, A), seq(rng, Lt, A)


def test_generators_cover_the_scoring_space():
    # what the GPU tests rely on: asymmetry, the int8 extremes, the 2^-8 grid, both end codes in every sequence
    rng = np.random.default_rng(0)
    for A in ALPHABET_SIZES[1:]:
        sub = asym_matrix(A, A)
        assert sub.shape == (A, A) and sub[0, A - 1] != sub[A - 1, 0]
        s = seq(rng, 10, A)
        assert 0 in s and A - 1 in s
    x = extreme_matrix()
    assert x.max() == 127 and x.min() == -127 and x[0, -1] != x[-1, 0]
    d = dyadic_matrix(20, 5) * 256
    assert np.array_equal(d, np.round(d)) and np.abs(d).max() <= 127 and (np.round(d).astype(int) % 2).any()
    assert np.array_equal(tie_matrix(), tie_matrix().T)


@pytest.mark.parametrize("at", MODES, ids=[MODE_NAMES[m] for m in MODES])
def test_oracle_optimum_equals_float64_gotoh(at):
    # the oracle's fill (fp32, literal reference scans) against the float64 affine recurrence: every value on these
    # grids is exact in both, so the optima must be equal
    rng = np.random.default_rng(300 + at)
    n = 0
    for name, sub, gi, ge in scorings():
        O = po.Oracle(sub, gi, ge, at)
        A = sub.shape[0]
        for q, t in _pairs(rng, A, 30, 28, low_entropy=(name == "ties")):
            want = gotoh_optimum(q, t, sub, gi, ge, at)
            got = oracle_optimum(O, q, t)
            assert got == want, (name, MODE_NAMES[at], len(q), len(t), got, want)
            n += 1
    assert n >= 360


@pytest.mark.parametrize("at", MODES, ids=[MODE_NAMES[m] for m in MODES])
def test_oracle_optimum_is_invariant_under_transposition(at):
    # optimum(q, t, sub, mode) == optimum(t, q, sub^T, mode'), GLOBAL_LOCAL <-> LOCAL_GLOBAL: a pure property of the
    # model, which an orientation mistake in the oracle would break for every asymmetric matrix
    rng = np.random.default_rng(400 + at)
    for name, sub, gi, ge in scorings():
        O = po.Oracle(sub, gi, ge, at)
        OT = po.Oracle(np.ascontiguousarray(sub.T), gi, ge, SWAPPED_MODE[at])
        for q, t in _pairs(rng, sub.shape[0], 20, 40, low_entropy=(name == "ties")):
            assert oracle_optimum(O, q, t) == oracle_optimum(OT, t, q), (name, len(q), len(t))


def test_float64_gotoh_sees_the_orientation():
    # the anchor itself is not symmetric in q and t: with an asymmetric matrix, swapping the lookup changes optima
    rng = np.random.default_rng(9)
    sub = asym_matrix(20, 1020)
    diff = 0
    for _ in range(40):
        q, t = seq(rng, 12, 20), seq(rng, 15, 20)
        diff += gotoh_optimum(q, t, sub, 7, 2, po.GLOBAL) != gotoh_optimum(q, t, sub.T, 7, 2, po.GLOBAL)
    assert diff >= 20
