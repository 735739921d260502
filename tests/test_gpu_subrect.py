"""GPU sub-rectangle fills (run with -m gpu on a B200): aadp_fill_subpair, aadp_fill_subpair_batch and aadp_fill_pair_general
with a rectangle, against the oracle's build_subdpm (orc_fill_sub) under asymmetric matrices over 1..64-letter alphabets,
the scoring limits of tests/test_scoring_space.py and a scoring off the dyadic grid.  Every comparison is bit-exact.

Sub-rectangles run on their own path: always the exact fp32 kernels (the record-list kernel frec_fill_kernel, or
general_fill_kernel), the end anchor's similarity read from the substitution table (an asymmetric lookup no whole-matrix
fill makes), end gaps free only where an anchor is the real Head or Tail, and for batches compact storage, per-item
final scores and subali_trace_kernel.  The rectangle alone picks the kernel and its shared memory: a loop of a
30 000-residue pair fills like any other loop, and an item's result does not depend on the chunk it shares.
tests/test_subrect_scoring.py anchors orc_fill_sub to a float64 model of the rectangle and proves the window
invariance the long-sequence test relies on."""
import numpy as np
import pytest

from util import po, MODES, MODE_NAMES, assert_matrix_equal, subali_walk
from test_scoring_space import (ALPHABET_SIZES, SWAPPED_MODE, asym_matrix, extreme_matrix, dyadic_matrix, tie_matrix,
                                seq, low_entropy_seq)
from test_subrect_scoring import rect_kinds, window_case
from test_gpu_scoring_space import kernels, new_ctx, float_matrix

pytestmark = pytest.mark.gpu

MODE_IDS = [MODE_NAMES[m] for m in MODES]
DIRS = ((1, po.FWD, "fwd"), (2, po.REV, "rev"))   # (aadp direction, oracle direction, tag); AADP_FWD = 1, AADP_REV = 2


def subrect_scorings():
    """(name, sub, gi, ge): asymmetric matrices for every alphabet size, the SPECIAL scorings and one off-grid matrix."""
    out = [("asym%d" % A, asym_matrix(A, 1000 + A), 7.0, 2.0) for A in ALPHABET_SIZES]
    out.append(("extreme127", extreme_matrix(), 40.0, 3.0))
    out.append(("dyadic8", dyadic_matrix(20, 5), 3.0 + 1 / 256.0, 0.5 + 3 / 256.0))
    out.append(("ties", tie_matrix(), 1.0, 1.0))
    out.append(("zero_gap", asym_matrix(4, 77), 0.0, 0.0))
    out.append(("float473", float_matrix(20, 6020), 4.73, 0.34))
    return out


def seqs_for(rng, name, A, *lengths):
    return [low_entropy_seq(rng, L, A) if name == "ties" else seq(rng, L, A) for L in lengths]


def fill_kernels(names):
    return [n for n in names if n.startswith(("frec_fill_kernel", "general_fill_kernel"))]


def expected_kernel(records, rects):
    """The kernel a launch of these rectangles is meant to run on: the record-list kernel while every rectangle has at
    most 2048 interior columns and fewer than 32000 interior rows and columns (WIDE beyond 1024 columns), else the
    general kernel.  Returns (kernel name prefix, wide)."""
    r = np.asarray(rects).reshape(-1, 4)
    nt = int((r[:, 3] - r[:, 1] - 1).max())
    nq = int((r[:, 2] - r[:, 0] - 1).max())
    if records and nt <= 2048 and max(nq, nt) < 32000:
        return "frec_fill_kernel", nt > 1024
    return "general_fill_kernel", False


def assert_kernel(names, records, rects, tag):
    fk = fill_kernels(names)
    want, wide = expected_kernel(records, rects)
    assert fk and all(n.startswith(want) for n in fk), (tag, fk, want)
    if want == "frec_fill_kernel":
        assert all(("WIDE=1" in n) == wide for n in fk), (tag, fk, wide)


def check_subpair(c, q, t, rect, want, records, tag):
    """fill_subpair in both directions against the oracle's (score, prev_q, prev_t) in want[direction]."""
    for d, od, nm in DIRS:
        (s, pq, pt), names = kernels(c, lambda: c.fill_subpair(q, t, rect, d))
        ws, wq, wt = want[od]
        assert_matrix_equal("%s %s score" % (tag, nm), s, ws)
        assert_matrix_equal("%s %s prev_q" % (tag, nm), pq, wq)
        assert_matrix_equal("%s %s prev_t" % (tag, nm), pt, wt)
        assert_kernel(names, records, rect, tag)


def oracle_sub(O, q, t, rect):
    return {od: O.fill_sub(q, t, tuple(int(x) for x in rect), od) for _, od, _ in DIRS}


# ---- 2a. fill_subpair: every scoring, every mode, every rectangle kind, both kernels ----

@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_fill_subpair_scorings_and_rect_kinds(at):
    ctxs = {1: new_ctx(general_records=1), 0: new_ctx(general_records=0)}
    try:
        rng = np.random.default_rng(800 + at)
        for name, sub, gi, ge in subrect_scorings():
            A = sub.shape[0]
            O = po.Oracle(sub, gi, ge, at)
            for c in ctxs.values():
                c.set_scoring(sub, gi, ge, at)
            q, t = seqs_for(rng, name, A, int(rng.integers(40, 70)), int(rng.integers(46, 76)))
            for kind, rect in rect_kinds(rng, len(q), len(t)):
                want = oracle_sub(O, q, t, rect)
                for records, c in ctxs.items():
                    check_subpair(c, q, t, rect, want, records, "%s %s %s rec%d" % (name, MODE_NAMES[at], kind, records))
            # a rectangle of more than 96 rows and columns, where the general kernel prunes its scans: pruned and
            # unpruned both equal the oracle
            q, t = seqs_for(rng, name, A, 140, 150)
            rect = (int(rng.integers(1, 20)), int(rng.integers(1, 20)), 120 + int(rng.integers(0, 20)),
                    130 + int(rng.integers(0, 20)))
            want = oracle_sub(O, q, t, rect)
            for prune in (1, 0):
                ctxs[0].set_option("general_prune", prune)
                check_subpair(ctxs[0], q, t, rect, want, 0, "%s %s prune%d" % (name, MODE_NAMES[at], prune))
            ctxs[0].set_option("general_prune", 1)
            check_subpair(ctxs[1], q, t, rect, want, 1, "%s %s large" % (name, MODE_NAMES[at]))
    finally:
        for c in ctxs.values():
            c.close()


# ---- 2b. width edges: key columns per lane, the 2048-column limit, the general kernel's column loop ----

@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_fill_subpair_width_edges(at):
    sub = asym_matrix(64, 1064)
    gi, ge = 7.0, 2.0
    O = po.Oracle(sub, gi, ge, at)
    rng = np.random.default_rng(900 + at)
    ctxs = {1: new_ctx(general_records=1), 0: new_ctx(general_records=0)}
    try:
        for c in ctxs.values():
            c.set_scoring(sub, gi, ge, at)
        cases = []
        q, t = seq(rng, 16, 64), seq(rng, 1300, 64)
        for w in (511, 512, 513, 1024, 1025, 1100):   # threads of the general kernel loop over columns beyond 512;
            t1 = int(rng.integers(1, 1300 - w - 1))     # the record-list kernel goes WIDE beyond 1024
            cases.append(("w%d" % w, q, t, (2, t1, 14, t1 + w + 1)))
        cases.append(("w1100_q_head_t_tail", q, t, (0, 1300 - 1100, 9, 1301)))
        for Lt in (2048, 2049):
            q, t = seq(rng, 10, 64), seq(rng, Lt, 64)
            cases.append(("t%d_whole" % Lt, q, t, (0, 0, 11, Lt + 1)))               # general beyond 2048 columns
            cases.append(("t%d_loop" % Lt, q, t, (3, 1000, 9, 1021)))                # a loop: record-list, narrow
            cases.append(("t%d_2048cols" % Lt, q, t, (2, Lt - 2048, 8, Lt + 1)))     # the widest record-list rectangle
            cases.append(("t%d_head" % Lt, q, t, (0, 0, 5, 40)))
        for kind, q, t, rect in cases:
            want = oracle_sub(O, q, t, rect)
            for records, c in ctxs.items():
                check_subpair(c, q, t, rect, want, records, "%s %s rec%d" % (kind, MODE_NAMES[at], records))
        # the selection these cases are meant to exercise
        assert expected_kernel(1, (0, 0, 11, 2050)) == ("general_fill_kernel", False)
        assert expected_kernel(1, (3, 1000, 9, 1021)) == ("frec_fill_kernel", False)
        assert expected_kernel(1, (2, 1, 8, 2050)) == ("frec_fill_kernel", True)
        assert expected_kernel(1, (2, 0, 14, 1025)) == ("frec_fill_kernel", False)
        assert expected_kernel(1, (2, 0, 14, 1026)) == ("frec_fill_kernel", True)
    finally:
        for c in ctxs.values():
            c.close()


# ---- 2c. fill_pair_general with a rectangle: the similarity-override path of the reference patch ----

@pytest.mark.parametrize("records", [1, 0], ids=["records", "scans"])
def test_fill_pair_general_rectangles(records):
    sub = float_matrix(20, 6120)
    gi, ge = 4.73, 0.34
    rng = np.random.default_rng(1000 + records)
    c = new_ctx(general_records=records)
    try:
        for at in MODES:
            O = po.Oracle(sub, gi, ge, at)
            q, t = seq(rng, int(rng.integers(40, 60)), 20), seq(rng, int(rng.integers(46, 66)), 20)
            sim = O.sim(q, t)
            for kind, rect in rect_kinds(rng, len(q), len(t)):
                for d, od, nm in DIRS:
                    (s, pq, pt), names = kernels(c, lambda: c.fill_pair_general(sim, gi, ge, at, d, rect))
                    ws, wq, wt = O.fill_sub(q, t, rect, od)
                    tag = "%s %s %s" % (MODE_NAMES[at], kind, nm)
                    assert_matrix_equal(tag + " score", s, ws)
                    assert_matrix_equal(tag + " prev_q", pq, wq)
                    assert_matrix_equal(tag + " prev_t", pt, wt)
                    assert_kernel(names, records, rect, tag)
        # a position-specific similarity no substitution table can produce: the rectangle on it equals the transposed
        # rectangle on its transpose in the swapped mode, every score cell (the predecessors may differ on ties)
        for at in MODES:
            Lq, Lt = 57, 63
            sim = np.zeros((Lq + 2, Lt + 2), np.float32)
            sim[1:-1, 1:-1] = np.round(rng.normal(0, 4, (Lq, Lt)) * 64) / 64 + rng.integers(-3, 4, (Lq, Lt)) * 0.01
            for kind, (a1, b1, a2, b2) in rect_kinds(rng, Lq, Lt):
                for d, _, nm in DIRS:
                    s = c.fill_pair_general(sim, gi, ge, at, d, (a1, b1, a2, b2))[0]
                    sT = c.fill_pair_general(np.ascontiguousarray(sim.T), gi, ge, SWAPPED_MODE[at], d, (b1, a1, b2, a2))[0]
                    assert_matrix_equal("%s %s %s transposed" % (MODE_NAMES[at], kind, nm), s, sT.T)
    finally:
        c.close()


# ---- 2d / 2e. fill_subpair_batch: every mode, mixed batches, chunking, alone vs batched, transposition ----

def mixed_batch(rng, name, A):
    """Sequences and items of a mixed loop batch: several items on one pair, items with item_q == item_t, empty
    sequences with whole-matrix rectangles, every rectangle kind (degenerate ones and each border included), and loops
    in a 2100-residue template next to a whole matrix on it (more than 2048 columns: the general kernel)."""
    L = [int(x) for x in rng.integers(40, 90, 4)]
    seqs = seqs_for(rng, name, A, *L) + [np.zeros(0, np.uint8)] + seqs_for(rng, name, A, 12, 2100)
    E, S12, BIG = 4, 5, 6
    items = []
    for qi, ti in ((0, 1), (0, 1), (2, 2), (3, 0), (1, 3)):   # (0, 1) twice: two kinds lists on one pair
        items += [(qi, ti, r) for _, r in rect_kinds(rng, L[qi], L[ti])]
    items += [(E, 1, (0, 0, 1, L[1] + 1)), (2, E, (0, 0, L[2] + 1, 1)), (E, E, (0, 0, 1, 1))]
    items += [(0, BIG, (5, 300, 20, 330)), (0, BIG, (0, 0, 9, 25)), (1, BIG, (L[1] - 9, 2080, L[1] + 1, 2101)),
              (S12, BIG, (0, 0, 13, 2101)), (S12, BIG, (3, 1000, 10, 1040))]
    order = rng.permutation(len(items))
    items = [items[k] for k in order]
    iq = np.array([x[0] for x in items], np.int32)
    it = np.array([x[1] for x in items], np.int32)
    rects = np.array([x[2] for x in items], np.int32)
    return seqs, iq, it, rects


def run_batch(c, seqs, iq, it, rects, direction, want_alignments=True):
    import alignment_algos_b200 as a
    res, off = a.Context.pack(seqs)
    return kernels(c, lambda: c.fill_subpair_batch(res, off, iq, it, rects, direction, want_alignments))


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("scoring", ["asym20", "asym64", "ties"])
def test_fill_subpair_batch_vs_oracle(scoring, at):
    import alignment_algos_b200 as a
    sub, gi, ge = {"asym20": (asym_matrix(20, 1020), 7.0, 2.0), "asym64": (asym_matrix(64, 1064), 7.0, 2.0),
                   "ties": (tie_matrix(), 1.0, 1.0)}[scoring]
    A = sub.shape[0]
    rng = np.random.default_rng(1100 + 7 * at + A)
    seqs, iq, it, rects = mixed_batch(rng, scoring, A)
    n = len(iq)
    O = po.Oracle(sub, gi, ge, at)
    c = new_ctx()
    try:
        c.set_scoring(sub, gi, ge, at)
        (score, aoff, pairs, n_out, st), names = run_batch(c, seqs, iq, it, rects, a.FWD)
        assert_kernel(names, 1, rects, "batch")   # the 2100-column whole matrix puts the whole launch on the general kernel
        assert any(n.startswith("subali_trace_kernel") for n in names)
        (rscore, _, _, _, _), _ = run_batch(c, seqs, iq, it, rects, a.REV)
        for k in range(n):
            q, t, rect = seqs[iq[k]], seqs[it[k]], tuple(int(x) for x in rects[k])
            tag = "%s %s item %d %s" % (scoring, MODE_NAMES[at], k, rect)
            ws, wq, wt = O.fill_sub(q, t, rect, po.FWD)
            wst, wpairs, wscore = subali_walk(ws, wq, wt, rect)
            assert aoff[k + 1] - aoff[k] == rect[2] - rect[0] + 1, tag
            assert st[k] == wst and score[k] == wscore, (tag, st[k], wst, score[k], wscore)
            assert n_out[k] == len(wpairs), tag
            assert_matrix_equal(tag + " pairs", pairs[aoff[k]:aoff[k] + n_out[k]], wpairs)
            assert rscore[k] == O.fill_sub(q, t, rect, po.REV)[0][rect[0], rect[1]], tag
        # score only equals traced; a chunked run equals an unchunked one
        (sonly, _, _, _, _), _ = run_batch(c, seqs, iq, it, rects, a.FWD, want_alignments=False)
        assert_matrix_equal("score-only", sonly, score)
        c.set_option("general_budget_mcells", 1)
        (s2, _, p2, n2, st2), _ = run_batch(c, seqs, iq, it, rects, a.FWD)
        c.set_option("general_budget_mcells", 1000)
        assert_matrix_equal("chunked score", s2, score)
        assert_matrix_equal("chunked pairs", p2, pairs)
        assert_matrix_equal("chunked n", n2, n_out)
        assert_matrix_equal("chunked status", st2, st)
        # each item alone, on the kernel its own rectangle picks, equals the item inside the batch
        for k in range(n):
            sl = slice(k, k + 1)
            (s1, o1, p1, n1, st1), names = run_batch(c, seqs, iq[sl], it[sl], rects[sl], a.FWD)
            assert_kernel(names, 1, rects[sl], "item %d alone" % k)
            assert s1[0] == score[k] and n1[0] == n_out[k] and st1[0] == st[k], k
            assert_matrix_equal("item %d alone pairs" % k, p1[:n1[0]], pairs[aoff[k]:aoff[k] + n_out[k]])
            (r1, _, _, _, _), _ = run_batch(c, seqs, iq[sl], it[sl], rects[sl], a.REV)
            assert r1[0] == rscore[k], k
        # 2e. transposition: item_q / item_t swapped, anchors swapped, sub^T, swapped mode -- the same scores
        c.set_scoring(np.ascontiguousarray(sub.T), gi, ge, SWAPPED_MODE[at])
        rT = np.ascontiguousarray(rects[:, [1, 0, 3, 2]])
        for d, want in ((a.FWD, score), (a.REV, rscore)):
            (sT, _, _, _, _), _ = run_batch(c, seqs, it, iq, rT, d, want_alignments=False)
            assert_matrix_equal("transposed %d" % d, sT, want)
    finally:
        c.close()


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_fill_subpair_batch_chunks_change_nothing(at):
    # a batch of more than 3 M compact cells: with general_budget_mcells 1 it runs in several launches, and its chunk
    # with the 2100-column whole matrix runs on the general kernel, the others on the record-list kernel.  Chunked,
    # unchunked and every item alone give the same scores, alignments and status.
    import alignment_algos_b200 as a
    sub = asym_matrix(20, 1020)
    rng = np.random.default_rng(1200 + at)
    seqs = [seq(rng, L, 20) for L in (900, 950, 1000)] + [seq(rng, 12, 20), seq(rng, 2100, 20)]
    items = []
    for k in range(50):
        qi, ti = int(rng.integers(0, 3)), int(rng.integers(0, 3))
        q1, t1 = int(rng.integers(0, 500)), int(rng.integers(0, 500))
        items.append((qi, ti, (q1, t1, q1 + int(rng.integers(250, 350)), t1 + int(rng.integers(250, 350)))))
    items += [(3, 4, (0, 0, 13, 2101)), (3, 4, (2, 7, 11, 60)), (0, 4, (100, 2000, 140, 2101))]
    items += [(qi, ti, r) for qi, ti in ((0, 1), (2, 2)) for _, r in rect_kinds(rng, len(seqs[qi]), len(seqs[ti]))]
    iq = np.array([x[0] for x in items], np.int32)
    it = np.array([x[1] for x in items], np.int32)
    rects = np.array([x[2] for x in items], np.int32)
    cells = ((rects[:, 2] - rects[:, 0] + 1) * (rects[:, 3] - rects[:, 1] + 1)).sum()
    assert cells > 3_000_000
    c = new_ctx()
    try:
        c.set_scoring(sub, 4.73, 0.34, at)
        full, names = run_batch(c, seqs, iq, it, rects, a.FWD)
        assert len(fill_kernels(names)) == 1 and fill_kernels(names)[0].startswith("general_fill_kernel")
        c.set_option("general_budget_mcells", 1)
        chunked, names = run_batch(c, seqs, iq, it, rects, a.FWD)
        fk = fill_kernels(names)
        assert len(fk) >= 3 and any(n.startswith("general_fill_kernel") for n in fk) and \
            any(n.startswith("frec_fill_kernel") for n in fk), fk
        for x, y, nm in zip(chunked, full, ("score", "ali_off", "pairs", "n_out", "status")):
            assert_matrix_equal("chunked " + nm, x, y)
        rchunk, _ = run_batch(c, seqs, iq, it, rects, a.REV)
        c.set_option("general_budget_mcells", 1000)
        rfull, _ = run_batch(c, seqs, iq, it, rects, a.REV)
        assert_matrix_equal("chunked rev", rchunk[0], rfull[0])
        score, aoff, pairs, n_out, st = full
        for k in range(len(iq)):
            sl = slice(k, k + 1)
            (s1, _, p1, n1, st1), _ = run_batch(c, seqs, iq[sl], it[sl], rects[sl], a.FWD)
            assert s1[0] == score[k] and n1[0] == n_out[k] and st1[0] == st[k], k
            assert_matrix_equal("item %d alone" % k, p1[:n1[0]], pairs[aoff[k]:aoff[k] + n_out[k]])
        # the oracle on the items that are cheap for it
        O = po.Oracle(sub, 4.73, 0.34, at)
        for k in range(50, len(iq)):
            q, t, rect = seqs[iq[k]], seqs[it[k]], tuple(int(x) for x in rects[k])
            if (rect[2] - rect[0]) * (rect[3] - rect[1]) * (rect[2] - rect[0] + rect[3] - rect[1]) > 1e8:
                continue
            wst, wpairs, wscore = subali_walk(*O.fill_sub(q, t, rect, po.FWD), rect)
            assert st[k] == wst and score[k] == wscore, k
            assert_matrix_equal("item %d vs oracle" % k, pairs[aoff[k]:aoff[k] + n_out[k]], wpairs)
    finally:
        c.close()


# ---- 2f. loops in long sequences: only the rectangles live on the device ----

def long_loop_batch(rng, A):
    """Sequences of 18 000, 19 000, 30 000 and 30 000 residues and ~300 loops on pairs of them: small interior loops,
    loops on the Head and on the Tail, degenerate loops and one loop of 1500 columns."""
    seqs = [seq(rng, L, A) for L in (18000, 19000, 30000, 30000)]
    pairs = [(0, 1), (1, 0), (2, 3), (3, 2), (2, 2), (1, 3), (0, 2)]
    items = []
    for k in range(280):
        qi, ti = pairs[k % len(pairs)]
        Lq, Lt = len(seqs[qi]), len(seqs[ti])
        hq, wt = int(rng.integers(0, 26)), int(rng.integers(0, 26))
        kind = k % 10
        q1 = 0 if kind == 1 else (Lq - hq if kind == 2 else int(rng.integers(1, Lq - hq)))
        t1 = 0 if kind in (1, 3) else (Lt - wt if kind in (2, 4) else int(rng.integers(1, Lt - wt)))
        if kind == 5:
            hq = 0          # degenerate in rows
        if kind == 6:
            wt = 0          # degenerate in columns
        items.append((qi, ti, (q1, t1, q1 + hq + 1, t1 + wt + 1)))
    items.append((2, 3, (15000, 9000, 15012, 10501)))      # 1500 interior columns
    items.append((1, 2, (0, 0, 1, 1)))                     # Head to the first residues, degenerate both ways
    items.append((3, 0, (30000, 18000, 30001, 18001)))     # last residues to the Tail
    iq = np.array([x[0] for x in items], np.int32)
    it = np.array([x[1] for x in items], np.int32)
    rects = np.array([x[2] for x in items], np.int32)
    return seqs, iq, it, rects


@pytest.mark.parametrize("records", [1, 0], ids=["records", "scans"])
def test_loops_in_long_sequences(records):
    import alignment_algos_b200 as a
    sub = float_matrix(20, 6020)
    gi, ge = 4.73, 0.34
    rng = np.random.default_rng(1300 + records)
    seqs, iq, it, rects = long_loop_batch(rng, 20)
    c = new_ctx(general_records=records)
    try:
        for at in MODES:
            c.set_scoring(sub, gi, ge, at)
            O = po.Oracle(sub, gi, ge, at)
            (score, aoff, pairs, n_out, st), names = run_batch(c, seqs, iq, it, rects, a.FWD)
            assert_kernel(names, records, rects, "long")
            (rscore, _, _, _, _), _ = run_batch(c, seqs, iq, it, rects, a.REV)
            for k in range(len(iq)):
                wq, wt, wrect, (oq, ot) = window_case(seqs[iq[k]], seqs[it[k]], rects[k])
                tag = "%s item %d %s" % (MODE_NAMES[at], k, tuple(rects[k]))
                wst, wpairs, wscore = subali_walk(*O.fill_sub(wq, wt, wrect, po.FWD), wrect)
                assert st[k] == wst and score[k] == wscore, (tag, st[k], wst, score[k], wscore)
                assert_matrix_equal(tag + " pairs", pairs[aoff[k]:aoff[k] + n_out[k]], wpairs + np.array([oq, ot], np.int32))
                assert rscore[k] == O.fill_sub(wq, wt, wrect, po.REV)[0][wrect[0], wrect[1]], tag
    finally:
        c.close()
