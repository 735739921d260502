"""Sub-rectangle fills of the oracle (build_subdpm, dpmatrix.h:319-353) under scoring other than BLOSUM62 (CPU only).
tests/test_gpu_subrect.py compares the GPU's rectangle fills with orc_fill_sub bit for bit; this file anchors
orc_fill_sub itself:
  * its final score against an independent float64 dynamic program of the rectangle model (rect_optimum), in all five
    modes and both directions;
  * transposition: the rectangle (a, b, c, d) on (q, t, sub, mode) scores as (b, a, d, c) on (t, q, sub^T, mode');
  * window invariance: a rectangle inside long sequences fills exactly like the shifted rectangle on a short window cut
    around it.  The long-sequence GPU test relies on it, because the oracle cannot hold a 30 000 x 30 000 matrix.
The rectangle kinds (rect_kinds) are shared with the GPU file."""
import numpy as np
import pytest

from util import po, MODES, MODE_NAMES
from test_scoring_space import SWAPPED_MODE, scorings, seq, low_entropy_seq

MODE_IDS = [MODE_NAMES[m] for m in MODES]


# ---- rectangle kinds ----

def rect_kinds(rng, Lq, Lt, h=(2, 12), w=(2, 14)):
    """(name, (q1_end, t1_end, q2_beg, t2_beg)) of every rectangle kind, matrix indices (0 = Head, L+1 = Tail), in a
    pair of lengths Lq, Lt >= 40: the whole matrix (all four borders); each border touched alone; strictly interior;
    degenerate in rows, in columns and in both; one interior cell; 31, 32 and 33 interior columns.  h / w bound the
    interior rows / columns of the random kinds."""
    assert Lq >= 40 and Lt >= 40

    def span(L, n, head=False, tail=False):  # anchors (lo, hi) with n interior positions, touching Head / Tail on request
        if head:
            return 0, n + 1
        if tail:
            return L - n, L + 1
        lo = int(rng.integers(1, L - n))   # lo >= 1 and hi = lo + n + 1 <= L: both anchors are residues
        return lo, lo + n + 1

    def hq():
        return int(rng.integers(h[0], h[1] + 1))

    def wt():
        return int(rng.integers(w[0], w[1] + 1))

    out = [("whole", (0, 0, Lq + 1, Lt + 1))]
    for name, qh, qt, th, tt in (("q_head", 1, 0, 0, 0), ("t_head", 0, 0, 1, 0), ("q_tail", 0, 1, 0, 0),
                                 ("t_tail", 0, 0, 0, 1)):
        q1, q2 = span(Lq, hq(), qh, qt)
        t1, t2 = span(Lt, wt(), th, tt)
        out.append((name, (q1, t1, q2, t2)))
    for name, nq, nt in (("interior", hq(), wt()), ("degenerate_rows", 0, wt()), ("degenerate_cols", hq(), 0),
                         ("degenerate_both", 0, 0), ("one_cell", 1, 1), ("cols31", hq(), 31), ("cols32", hq(), 32),
                         ("cols33", hq(), 33)):
        q1, q2 = span(Lq, nq)
        t1, t2 = span(Lt, nt)
        out.append((name, (q1, t1, q2, t2)))
    return out


# ---- an independent float64 dynamic program of the rectangle model ----

def rect_optimum(q, t, sub, gi, ge, at, rect):
    """Forward score of the final anchor (q2_beg, t2_beg) of rect = (q1_end, t1_end, q2_beg, t2_beg), float64.

    A path runs from the start anchor (score 0) through matched interior cells to the end anchor; every step advances
    both indices and skips residues of at most one sequence.  The end anchor adds its similarity unless it lies on the
    Tail row or column (the similarity matrix is 0 there).  A gap of length n costs gi + ge*(n-1), and nothing where
    the mode frees that end AND its lower end is the Head (index 0) or its upper end is the Tail (Lq+1 / Lt+1): only
    gaps leaving a start anchor on row / column 0 or entering an end anchor on the last row / column can be free.  A
    rectangle without interior rows or columns takes one forced gap from anchor to anchor, never clamped.

    LOCAL (the reference clamps every cell at 0, dpmatrix.h:580): a cell of flow row >= 2 and flow column >= 2 is
    Smith-Waterman's -- a path may also start there, with nothing before it -- but a cell of the first flow row or
    column is reached from the start anchor only, across the gap it leaves (free only at the Head), and keeps
    max(0, that score).  The final cell is max(0, its best predecessor + its similarity).  Computed with affine
    running maxima, not with the oracle's scans."""
    q, t = np.asarray(q, np.int64), np.asarray(t, np.int64)
    sub = np.asarray(sub, np.float64)
    Lq, Lt = len(q), len(t)
    q1, t1, q2, t2 = [int(x) for x in rect]
    nq, nt = q2 - q1, t2 - t1                      # flow index of the final cell
    local = at == po.LOCAL
    delfree = at in (po.LOCAL, po.SEMI_LOCAL, po.LOCAL_GLOBAL)
    insfree = at in (po.LOCAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL)
    NEG = -np.inf

    def pen(n):
        return gi + ge * (np.asarray(n, np.float64) - 1)

    simf = 0.0 if q2 == Lq + 1 or t2 == Lt + 1 else float(sub[q[q2 - 1], t[t2 - 1]])
    if nq == 1 or nt == 1:
        if nq == 1:
            n, free = nt - 1, delfree and (t1 == 0 or t2 == Lt + 1)
        else:
            n, free = nq - 1, insfree and (q1 == 0 or q2 == Lq + 1)
        return (0.0 if n == 0 or free else -float(pen(n))) + simf
    Iq, It = nq - 1, nt - 1                        # interior rows / columns
    S = sub[q[q1:q1 + Iq]][:, t[t1:t1 + It]]       # S[a-1, b-1]: similarity of flow cell (a, b)
    # M[a, b]: best path to the interior flow cell (a, b); row and column 0 hold only the start anchor (0, 0)
    M = np.full((Iq + 1, It + 1), NEG)
    M[0, 0] = 0.0
    cols = np.arange(It + 1, dtype=np.float64)
    col_acc = np.full(It + 1, NEG)                 # max over interior rows r <= a-2 of M[r, j] + ge*r
    for a in range(1, Iq + 1):
        P = M[a - 1]
        best = np.full(It + 1, NEG)
        best[1:] = P[:-1]                                                     # diagonal (from the anchor into (1,1))
        if a == 1:   # from the anchor: deletion of the template residues 1..b-1 of the rectangle
            best[2:] = 0.0 if (delfree and t1 == 0) else -pen(cols[2:] - 1)
        else:        # deletion (a-1, k) -> (a, b), 1 <= k <= b-2, length b-1-k
            acc = np.maximum.accumulate(P + ge * cols)
            best[2:] = np.maximum(best[2:], acc[:-2] - (gi + ge * (cols[2:] - 2)))
            # insertion from the anchor into column 1, length a-1
            best[1] = max(best[1], 0.0 if (insfree and q1 == 0) else -float(pen(a - 1)))
            if a >= 3:   # insertion (r, b-1) -> (a, b), 1 <= r <= a-2, length a-1-r
                col_acc = np.maximum(col_acc, M[a - 2] + ge * (a - 2))
                best[2:] = np.maximum(best[2:], col_acc[1:-1] - (gi + ge * (a - 2)))
            if local:
                best[2:] = np.maximum(best[2:], 0.0)                          # Smith-Waterman start
        row = S[a - 1] + best[1:]
        M[a, 1:] = np.maximum(row, 0.0) if local else row
    cand = [M[Iq, It]]
    endd = 0.0 if (delfree and t2 == Lt + 1) else None
    endi = 0.0 if (insfree and q2 == Lq + 1) else None
    for k in range(1, It):      # deletion (Iq, k) -> end anchor, length It-k
        cand.append(M[Iq, k] - (endd if endd is not None else float(pen(It - k))))
    for r in range(1, Iq):      # insertion (r, It) -> end anchor, length Iq-r
        cand.append(M[r, It] - (endi if endi is not None else float(pen(Iq - r))))
    s = max(cand) + simf
    return max(s, 0.0) if local else s


def reversed_rect(Lq, Lt, rect):
    """The rectangle of the reversed sequences whose forward fill is the reverse fill of rect."""
    q1, t1, q2, t2 = rect
    return (Lq + 1 - q2, Lt + 1 - t2, Lq + 1 - q1, Lt + 1 - t1)


def window(L, lo, hi):
    """Cut of a sequence of length L around the anchors lo < hi of one axis: it starts with the residue of lo (which
    becomes index 1), or at the Head when lo is the Head, and ends with the residue of hi, or runs to the Tail when hi
    is the Tail.  Returns (offset, end): the window is s[offset:end], and matrix index i becomes i - offset."""
    off = lo - 1 if lo >= 1 else 0
    return off, min(hi, L)


def window_case(q, t, rect):
    """(q window, t window, shifted rect, (row offset, column offset)) of rect on (q, t)."""
    q1, t1, q2, t2 = [int(x) for x in rect]
    oq, qe = window(len(q), q1, q2)
    ot, te = window(len(t), t1, t2)
    return q[oq:qe], t[ot:te], (q1 - oq, t1 - ot, q2 - oq, t2 - ot), (oq, ot)


def _cases(rng, A, name, n=2, L=(40, 70)):
    """Pairs of sequences long enough for every rectangle kind (low-entropy ones for the tie scoring)."""
    for _ in range(n):
        Lq, Lt = int(rng.integers(*L)), int(rng.integers(L[0] + 6, L[1] + 6))
        if name == "ties":
            yield low_entropy_seq(rng, Lq, A), low_entropy_seq(rng, Lt, A)
        else:
            yield seq(rng, Lq, A), seq(rng, Lt, A)


def test_rect_kinds_are_what_they_say():
    rng = np.random.default_rng(1)
    for _ in range(50):
        Lq, Lt = int(rng.integers(40, 90)), int(rng.integers(40, 90))
        kinds = dict(rect_kinds(rng, Lq, Lt))
        for name, (q1, t1, q2, t2) in kinds.items():
            assert 0 <= q1 < q2 <= Lq + 1 and 0 <= t1 < t2 <= Lt + 1, name
            touches = (q1 == 0, t1 == 0, q2 == Lq + 1, t2 == Lt + 1)
            want = {"whole": (1, 1, 1, 1), "q_head": (1, 0, 0, 0), "t_head": (0, 1, 0, 0), "q_tail": (0, 0, 1, 0),
                    "t_tail": (0, 0, 0, 1)}.get(name, (0, 0, 0, 0))
            assert touches == tuple(bool(x) for x in want), name
        assert kinds["degenerate_rows"][2] - kinds["degenerate_rows"][0] == 1
        assert kinds["degenerate_cols"][3] - kinds["degenerate_cols"][1] == 1
        assert kinds["one_cell"][2] - kinds["one_cell"][0] == 2 and kinds["one_cell"][3] - kinds["one_cell"][1] == 2
        for w in (31, 32, 33):
            assert kinds["cols%d" % w][3] - kinds["cols%d" % w][1] - 1 == w


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_rectangle_score_equals_float64_model(at):
    # orc_fill_sub's final score against rect_optimum, forward; the reverse score at (q1_end, t1_end) against the model
    # on the reversed sequences (the reverse fill is the forward fill of the mirrored problem).  Every value on these
    # grids is exact in fp32 and float64, so the scores must be equal.
    rng = np.random.default_rng(500 + at)
    n = 0
    for name, sub, gi, ge in scorings():
        O = po.Oracle(sub, gi, ge, at)
        A = sub.shape[0]
        for q, t in _cases(rng, A, name):
            for kind, rect in rect_kinds(rng, len(q), len(t)):
                S = O.fill_sub(q, t, rect, po.FWD)[0]
                want = rect_optimum(q, t, sub, gi, ge, at, rect)
                assert S[rect[2], rect[3]] == want, (name, MODE_NAMES[at], kind, rect, S[rect[2], rect[3]], want)
                R = O.fill_sub(q, t, rect, po.REV)[0]
                want = rect_optimum(q[::-1], t[::-1], sub, gi, ge, at, reversed_rect(len(q), len(t), rect))
                assert R[rect[0], rect[1]] == want, (name, MODE_NAMES[at], kind, rect, "rev", R[rect[0], rect[1]], want)
                n += 1
    assert n >= 12 * 2 * 13


def test_float64_rect_model_sees_the_anchors():
    # the model is not blind to what it is meant to check: the end anchor's similarity (an asymmetric lookup), and a
    # gap that is free only at the Head / Tail
    from test_scoring_space import asym_matrix
    rng = np.random.default_rng(4)
    sub = asym_matrix(20, 1020)
    diff_sub = diff_free = 0
    for _ in range(40):
        q, t = seq(rng, 50, 20), seq(rng, 55, 20)
        rect = (3, 5, 20, 30)
        diff_sub += rect_optimum(q, t, sub, 7, 2, po.GLOBAL, rect) != rect_optimum(q, t, sub.T.copy(), 7, 2, po.GLOBAL,
                                                                                   rect)
        r2 = (0, 5, 20, 30)
        diff_free += rect_optimum(q, t, sub, 7, 2, po.SEMI_LOCAL, r2) != rect_optimum(q, t, sub, 7, 2, po.GLOBAL, r2)
    assert diff_sub >= 20 and diff_free >= 10


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_rectangle_is_invariant_under_transposition(at):
    # the whole forward and reverse score matrices: rect (a, b, c, d) on (q, t, sub, mode) is the transpose of
    # (b, a, d, c) on (t, q, sub^T, mode'), GLOBAL_LOCAL <-> LOCAL_GLOBAL.  Every cell takes the max of the same fp32
    # candidate values, so the scores agree bit for bit (the predecessors may differ on ties: the scan order changes).
    rng = np.random.default_rng(600 + at)
    for name, sub, gi, ge in scorings():
        O = po.Oracle(sub, gi, ge, at)
        OT = po.Oracle(np.ascontiguousarray(sub.T), gi, ge, SWAPPED_MODE[at])
        for q, t in _cases(rng, sub.shape[0], name, n=1):
            for kind, (a, b, c, d) in rect_kinds(rng, len(q), len(t)):
                for di in (po.FWD, po.REV):
                    S = O.fill_sub(q, t, (a, b, c, d), di)[0]
                    ST = OT.fill_sub(t, q, (b, a, d, c), di)[0]
                    assert np.array_equal(S, ST.T), (name, MODE_NAMES[at], kind, di)


def _shifted(P, off):
    return np.where(P >= 0, P - off, P)


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_rectangle_fill_is_invariant_under_windowing(at):
    # a rectangle inside sequences of up to ~400 residues fills exactly like the shifted rectangle on the window cut
    # around it (window_case): scores equal, predecessors equal after the index shift, in both directions.  The reverse
    # fill reproduces the reference's opt_j bug (REPRO_REV_BUG: the final cell of the global reverse fill records the
    # matrix column t2_beg - 1 for a left-column winner); that column moves with the window, so the invariance holds
    # there too and the long-sequence GPU test checks both directions in full.
    rng = np.random.default_rng(700 + at)
    for name, sub, gi, ge in scorings():
        O = po.Oracle(sub, gi, ge, at)
        A = sub.shape[0]
        for _ in range(2):
            Lq, Lt = int(rng.integers(200, 400)), int(rng.integers(200, 400))
            if name == "ties":
                q, t = low_entropy_seq(rng, Lq, A), low_entropy_seq(rng, Lt, A)
            else:
                q, t = seq(rng, Lq, A), seq(rng, Lt, A)
            for kind, rect in rect_kinds(rng, Lq, Lt, h=(2, 30), w=(2, 40)):
                if kind == "whole":
                    continue   # the window is the whole pair
                wq, wt, wrect, (oq, ot) = window_case(q, t, rect)
                q1, t1, q2, t2 = rect
                for di in (po.FWD, po.REV):
                    S, PQ, PT = O.fill_sub(q, t, rect, di)
                    WS, WQ, WT = O.fill_sub(wq, wt, wrect, di)
                    inside = (slice(q1, q2 + 1), slice(t1, t2 + 1))
                    winside = (slice(q1 - oq, q2 - oq + 1), slice(t1 - ot, t2 - ot + 1))
                    tag = (name, MODE_NAMES[at], kind, rect, di)
                    assert np.array_equal(S[inside], WS[winside]), tag
                    assert np.array_equal(PQ[inside], _shifted(WQ[winside], -oq)), tag
                    assert np.array_equal(PT[inside], _shifted(WT[winside], -ot)), tag
                    # outside the rectangle every cell keeps the DPCell defaults, in both fills
                    for X, Y, Z, ins in ((S, PQ, PT, inside), (WS, WQ, WT, winside)):
                        m = np.ones(X.shape, bool)
                        m[ins] = False
                        assert not X[m].any() and (Y[m] == -1).all() and (Z[m] == -1).all(), tag
