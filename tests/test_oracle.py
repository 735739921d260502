"""CPU tests: pin the C restatement (oracle/aadp_oracle.c) against the real reference's results and the
committed golden vectors, and check the domain properties the GPU tests rely on."""
import numpy as np

from util import po, MODES, ReferenceResults, golden_cases, golden_case, rand_pair, assert_matrix_equal


def test_oracle_matches_golden(golden):
    sub = golden["sub"]
    for name in golden_cases(golden):
        q, t, gi, ge, at = golden_case(golden, name)
        O = po.Oracle(sub, gi, ge, at)
        for d, tag in ((po.FWD, "fwd"), (po.REV, "rev")):
            for fast in (False, True):
                s, pq, pt = O.fill(q, t, d, True, fast)
                assert_matrix_equal(name + tag + ".score", s, golden[name + "." + tag + ".score"])
                assert_matrix_equal(name + tag + ".pq", pq, golden[name + "." + tag + ".pq"].astype(np.int32))
                assert_matrix_equal(name + tag + ".pt", pt, golden[name + "." + tag + ".pt"].astype(np.int32))
            rc, pairs, sc = O.optimal(s, pq, pt, d)
            want_rc = int(golden[name + "." + tag + ".opt_rc"][0])
            assert (rc != 0) == (want_rc != 0), name + tag
            if rc == 0:
                assert_matrix_equal(name + tag + ".opt", pairs, golden[name + "." + tag + ".opt_pairs"].astype(np.int32))
                assert sc == golden[name + "." + tag + ".opt_score"][0]


def test_revbug_case_b5(golden):
    # SURVEY.md App. B.5: global rev cell (0,0) gets traceback (5,4) where (5,1) would be right
    name = "b5_revbug"
    q, t, gi, ge, at = golden_case(golden, name)
    assert golden[name + ".rev.pq"][0, 0] == 5 and golden[name + ".rev.pt"][0, 0] == 4
    O = po.Oracle(golden["sub"], gi, ge, at)
    _, pq, pt = O.fill(q, t, po.REV, True)
    assert (pq[0, 0], pt[0, 0]) == (5, 4)
    _, pq, pt = O.fill(q, t, po.REV, False)
    assert (pq[0, 0], pt[0, 0]) == (5, 1)


def test_oracle_matches_reference_random(blosum):
    _, M = blosum
    ref = ReferenceResults("test_oracle.py::test_oracle_matches_reference_random")
    rng = np.random.default_rng(7)
    cells = 0
    for gi, ge in [(12, 1), (3, 1), (2, 2), (10.5, 0.25), (1, 0)]:
        for at in MODES:
            O = po.Oracle(M, gi, ge, at)
            for trial in range(6):
                Lq, Lt = int(rng.integers(0, 36)), int(rng.integers(0, 36))
                q, t = rand_pair(rng, Lq, Lt, 24)
                for d in (po.FWD, po.REV):
                    case = "fill %s %s %d %dx%d" % (gi, ge, at, Lq, Lt)
                    for fast in (False, True):
                        s, pq, pt = O.fill(q, t, d, True, fast)
                        ref.check(case, s, pq, pt)
                        cells += s.size
                    if at == po.LOCAL and (Lq == 0 or Lt == 0):
                        continue  # optimal.h:100 reads getCell(-1,-1) here: undefined behaviour in the reference
                    rc, pairs, sc = O.optimal(s, pq, pt, d)
                    ref.check("optimal of " + case, rc != 0, *((pairs, sc) if rc == 0 else ()))
    ref.close()
    assert cells > 100000


def test_fwd_end_equals_rev_start(blosum):
    # SURVEY.md §4: F[last][last] == R[0][0] for every non-local mode (both are the optimum)
    _, M = blosum
    rng = np.random.default_rng(11)
    for at in MODES:
        O = po.Oracle(M, 12, 1, at)
        for _ in range(5):
            q, t = rand_pair(rng, int(rng.integers(1, 60)), int(rng.integers(1, 60)))
            F = O.fill(q, t, po.FWD, fast=True)[0]
            R = O.fill(q, t, po.REV, fast=True)[0]
            if at != po.LOCAL:
                assert F[-1, -1] == R[0, 0]


def test_ucw_union_equals_mask_golden(golden):
    # SURVEY.md §0.9 / App. B.4: union of cells over all UCW alignments == {F+R-sim > thr}
    sub = golden["sub"]
    n_checked = 0
    for name in golden_cases(golden):
        for dr in (5, 20):
            key = "%s.ucw%02d" % (name, dr)
            if key + ".union" not in golden:
                continue
            q, t, gi, ge, at = golden_case(golden, name)
            O = po.Oracle(sub, gi, ge, at)
            F = golden[name + ".fwd.score"]
            R = golden[name + ".rev.score"]
            sim = O.sim(q, t)
            thr = O.threshold(float(F[-1, -1]), dr / 100.0)
            assert thr == golden[key + ".thr"][0]
            mask, cnt = O.nearopt_mask(F, R, sim, thr)
            union = np.unpackbits(golden[key + ".union"])[: F.size].reshape(F.shape)
            interior = np.zeros_like(union)
            interior[1:-1, 1:-1] = union[1:-1, 1:-1]
            assert_matrix_equal(key + " mask vs reference UCW union", mask, interior)
            # the restated branching agrees with the reference enumerator on cells and count
            mark, n = O.ucw_cells(q, t, F, sim, thr)
            assert n == int(golden[key + ".n"][0])
            assert_matrix_equal(key + " restated UCW", mark, union)
            n_checked += 1
    assert n_checked >= 8


def test_threshold_formula():
    O = po.Oracle(np.zeros((2, 2), np.float32), 1, 1, po.GLOBAL)
    for opt, dr in [(100.0, 0.01), (5.0, 0.01), (-20.0, 0.2), (0.0, 0.5), (483.0, 0.2)]:
        want = np.float32(min(np.float32(np.float32(1.0) - np.float32(dr)) * np.float32(opt),
                              np.float32(opt) - np.float32(0.1)))
        assert O.threshold(opt, dr) == want


def test_oracle_literal_fill_matches_float_golden(golden_float):
    # non-dyadic scoring (reference defaults 4.73 / 0.34, scaled matrix): only the literal O(n^3)
    # restatement is exact there; it must reproduce every rounding of the real reference
    g = golden_float
    for name in golden_cases(g):
        q, t, gi, ge, at = golden_case(g, name)
        O = po.Oracle(g["sub." + str(g[name + ".sub"])], gi, ge, at)
        for d, tag in ((po.FWD, "fwd"), (po.REV, "rev")):
            s, pq, pt = O.fill(q, t, d, True, False)
            assert_matrix_equal(name + tag + ".score", s, g[name + "." + tag + ".score"])
            assert_matrix_equal(name + tag + ".pq", pq, g[name + "." + tag + ".pq"].astype(np.int32))
            assert_matrix_equal(name + tag + ".pt", pt, g[name + "." + tag + ".pt"].astype(np.int32))


def test_record_list_fill_is_the_literal_fill(golden_float, blosum):
    # orc_fill_rec (the CPU model of the GPU's record-list kernel, csrc/aadp_frec.cuh) against the reference's golden
    # float vectors and against the literal O(n^3) restatement: default penalties, a scaled matrix, integer scoring
    # (exact key ties everywhere), zero gap extension; all align types, both directions; related and random pairs
    g = golden_float
    for name in golden_cases(g):
        q, t, gi, ge, at = golden_case(g, name)
        O = po.Oracle(g["sub." + str(g[name + ".sub"])], gi, ge, at)
        for d, tag in ((po.FWD, "fwd"), (po.REV, "rev")):
            s, pq, pt, _ = O.fill_rec(q, t, d, True)
            assert_matrix_equal(name + tag + ".score", s, g[name + "." + tag + ".score"])
            assert_matrix_equal(name + tag + ".pq", pq, g[name + "." + tag + ".pq"].astype(np.int32))
            assert_matrix_equal(name + tag + ".pt", pt, g[name + "." + tag + ".pt"].astype(np.int32))
    _, M = blosum
    rng = np.random.default_rng(77)
    visited = cells = 0
    for gi, ge, scale in ((4.73, 0.34, 1.0), (12.0, 1.0, 1.0), (3.3, 0.7, 0.37), (0.5, 0.0, 0.1)):
        Ms = (M.astype(np.float32) * np.float32(scale)).astype(np.float32)
        for at in (po.SEMI_LOCAL, po.GLOBAL, po.LOCAL, po.GLOBAL_LOCAL, po.LOCAL_GLOBAL):
            O = po.Oracle(Ms, gi, ge, at)
            for related in (0, 1):
                Lq, Lt = (int(x) for x in rng.integers(1, 140, 2))
                q = rng.integers(0, 20, Lq).astype(np.uint8)
                t = rng.integers(0, 20, Lt).astype(np.uint8)
                n = min(Lq, Lt) - 6
                if related and n > 10:
                    t[3:3 + n] = q[2:2 + n]
                    idx = rng.integers(3, 3 + n, n // 4)
                    t[idx] = rng.integers(0, 20, len(idx))
                for d in (po.FWD, po.REV):
                    want = O.fill(q, t, d, True)
                    s, pq, pt, st = O.fill_rec(q, t, d, True)
                    assert_matrix_equal("rec score", s, want[0])
                    assert_matrix_equal("rec pq", pq, want[1])
                    assert_matrix_equal("rec pt", pt, want[2])
                    cells += st[0]
                    visited += st[1] + st[2]
    assert visited < 4 * cells  # output-sensitive: a few candidates per cell, not a scan
    # benchmark-sized pairs (C3 shape), related and repetitive: long groups of noise-tied leaders
    for at, kind in ((po.SEMI_LOCAL, "related"), (po.GLOBAL, "related"), (po.LOCAL, "repeat"), (po.SEMI_LOCAL, "repeat")):
        O = po.Oracle(M.astype(np.float32), 4.73, 0.34, at)
        Lq, Lt = 330, 410
        if kind == "repeat":
            q = np.resize(rng.integers(0, 20, 3).astype(np.uint8), Lq)
            t = np.resize(rng.integers(0, 20, 2).astype(np.uint8), Lt)
        else:
            q = rng.integers(0, 20, Lq).astype(np.uint8)
            t = rng.integers(0, 20, Lt).astype(np.uint8)
            t[20:320] = q[10:310]
            idx = rng.integers(20, 320, 75)
            t[idx] = rng.integers(0, 20, len(idx))
        for d in (po.FWD, po.REV):
            want = O.fill(q, t, d, True)
            s_, pq_, pt_, _ = O.fill_rec(q, t, d, True)
            assert_matrix_equal("rec score (large)", s_, want[0])
            assert_matrix_equal("rec pq (large)", pq_, want[1])
            assert_matrix_equal("rec pt (large)", pt_, want[2])


def test_oracle_sub_rectangle_fill_matches_golden(golden_sub):
    # build_subdpm (dpmatrix.h:319-353): anchors inside the matrix, at the Head / Tail, degenerate rectangles
    g = golden_sub
    for name in golden_cases(g):
        q, t, gi, ge, at = golden_case(g, name)
        O = po.Oracle(g["sub"], gi, ge, at)
        for d, tag in ((po.FWD, "fwd"), (po.REV, "rev")):
            s, pq, pt = O.fill_sub(q, t, g[name + ".rect"], d)
            assert_matrix_equal(name + tag + ".score", s, g[name + "." + tag + ".score"])
            assert_matrix_equal(name + tag + ".pq", pq, g[name + "." + tag + ".pq"].astype(np.int32))
            assert_matrix_equal(name + tag + ".pt", pt, g[name + "." + tag + ".pt"].astype(np.int32))


def test_oracle_sub_rectangle_fill_matches_reference_random(blosum):
    _, M = blosum
    ref = ReferenceResults("test_oracle.py::test_oracle_sub_rectangle_fill_matches_reference_random")
    rng = np.random.default_rng(17)
    for gi, ge in [(12, 1), (4.73, 0.34)]:
        for at in MODES:
            O = po.Oracle(M, gi, ge, at)
            for trial in range(12):
                Lq, Lt = int(rng.integers(1, 30)), int(rng.integers(1, 30))
                q, t = rand_pair(rng, Lq, Lt)
                q0 = int(rng.integers(0, Lq + 1)); q1 = int(rng.integers(q0 + 1, Lq + 2))
                t0 = int(rng.integers(0, Lt + 1)); t1 = int(rng.integers(t0 + 1, Lt + 2))
                for d in (po.FWD, po.REV):
                    s, pq, pt = O.fill_sub(q, t, (q0, t0, q1, t1), d)
                    ref.check("fill_sub %s %d %dx%d" % (gi, at, Lq, Lt), s, pq, pt)
    ref.close()


def test_oracle_tabulated_gap_fill_matches_golden(golden_tab):
    # position-dependent gap models (hmap_eval.h:63-117 / gn2_eval.h:99-158 shaped) through the table-driven fill
    g = golden_tab
    for name in golden_cases(g):
        for d, tag in ((po.FWD, "fwd"), (po.REV, "rev")):
            s, pq, pt = po.Oracle.fill_tab(g[name + ".sim"], g[name + ".del"], g[name + ".ins"], int(g[name + ".local"]), d)
            assert_matrix_equal(name + tag + ".score", s, g[name + "." + tag + ".score"])
            assert_matrix_equal(name + tag + ".pq", pq, g[name + "." + tag + ".pq"].astype(np.int32))
            assert_matrix_equal(name + tag + ".pt", pt, g[name + "." + tag + ".pt"].astype(np.int32))


def test_oracle_tabulated_gap_fill_matches_reference_random(blosum):
    ref = ReferenceResults("test_oracle.py::test_oracle_tabulated_gap_fill_matches_reference_random")
    rng = np.random.default_rng(29)
    for at in MODES:
        for gen in (po.hmap_like_tables, po.gn2_like_tables):
            for trial in range(4):
                Lq, Lt = int(rng.integers(0, 45)), int(rng.integers(0, 45))
                sim, dt, it = gen(rng, Lq, Lt, at)
                for d in (po.FWD, po.REV):
                    got = po.Oracle.fill_tab(sim, dt, it, at == po.LOCAL, d)
                    ref.check("fill_tab %d %dx%d" % (at, Lq, Lt), *got)
    # tables tabulated from the affine AASubstitutionEval model reproduce the ordinary reference fill
    _, M = blosum
    for at in MODES:
        gi, ge = 4.73, 0.34
        O = po.Oracle(M, gi, ge, at)
        q, t = rand_pair(rng, 27, 22)
        sz1, sz2 = len(q) + 2, len(t) + 2
        dt = np.zeros((sz2, sz2), np.float32)
        it = np.zeros((sz1 - 1, sz2), np.float32)
        f32 = np.float32
        pen = lambda ln: f32(f32(gi) + f32(f32(ge) * f32(ln - 1)))
        dfree = at in (po.LOCAL, po.SEMI_LOCAL, po.LOCAL_GLOBAL)
        ifree = at in (po.LOCAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL)
        for t1 in range(sz2):
            for t2 in range(t1 + 2, sz2):
                dt[t1, t2] = 0 if (dfree and (t1 == 0 or t2 == sz2 - 1)) else pen(t2 - t1 - 1)
        for ln in range(1, sz1 - 1):
            for t2 in range(1, sz2):
                it[ln, t2] = 0 if (ifree and (t2 == 1 or t2 == sz2 - 1)) else pen(ln)
        for d in (po.FWD, po.REV):
            got = po.Oracle.fill_tab(O.sim(q, t), dt, it, at == po.LOCAL, d)
            ref.check("affine-as-table %d" % at, *got)
    ref.close()


def _canon(alis):
    return sorted((s, tuple(map(tuple, p))) for s, p in alis)


def _canon_arrays(alis):
    return [(s, np.array(p, np.int64).reshape(-1, 2)) for s, p in _canon(alis)]


def test_oracle_ucw_enumeration_matches_reference(blosum):
    # orc_ucw_enumerate == UnconstrainedNearOptimal::enumerate (ucw.h:63-191): same alignments, same fp32 scores
    # (the reference sorts its set at the end, so the comparison is on canonically sorted lists)
    _, M = blosum
    ref = ReferenceResults("test_oracle.py::test_oracle_ucw_enumeration_matches_reference")
    rng = np.random.default_rng(4)
    total = 0
    for at in (po.GLOBAL_LOCAL, po.GLOBAL, po.LOCAL_GLOBAL, po.SEMI_LOCAL):
        for gi, ge in ((12, 1), (3, 1)):
            O = po.Oracle(M, gi, ge, at)
            for Lq, Lt, delta in ((20, 25, 0.3), (30, 30, 0.2), (12, 40, 0.5), (0, 4, 0.1), (5, 1, 0.1)):
                q = rng.integers(0, 20, Lq).astype(np.uint8)
                t = q.copy() if Lq == Lt else rng.integers(0, 20, Lt).astype(np.uint8)
                t[::4] = rng.integers(0, 20, len(t[::4]))
                F, _, _ = O.fill(q, t, po.FWD, True, fast=True)
                thr = O.threshold(float(F[-1, -1]), delta)
                st, alis = O.ucw_enumerate(q, t, F, O.sim(q, t), thr, 100000)
                assert st == 0
                ref.check("ucw %d %s %dx%d" % (at, gi, Lq, Lt), _canon_arrays(alis))
                total += len(alis)
    ref.close()
    assert total > 2000


def test_oracle_constrained_enumeration_matches_reference(blosum):
    # orc_cno_enumerate == ConstrainedNearOptimal::enumerate (cw.h:60-284) for all-true, striped, random and all-false
    # SuboptFlags; integer and default float scoring
    _, M = blosum
    ref = ReferenceResults("test_oracle.py::test_oracle_constrained_enumeration_matches_reference")
    rng = np.random.default_rng(12)
    total = 0
    for at in (po.GLOBAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL):
        for gi, ge in ((3, 1), (4.73, 0.34)):
            O = po.Oracle(M, gi, ge, at)
            for Lq, Lt, delta in ((30, 30, 0.25), (12, 40, 0.5), (33, 33, 0.2), (1, 4, 0.2), (0, 3, 0.2)):
                q = rng.integers(0, 20, Lq).astype(np.uint8)
                t = q.copy() if Lq == Lt else rng.integers(0, 20, Lt).astype(np.uint8)
                t[::4] = rng.integers(0, 20, len(t[::4]))
                F, pq, pt = O.fill(q, t, po.FWD, True, fast=False)
                thr = O.threshold(float(F[-1, -1]), delta)
                for flags in (None, (np.arange(Lt + 2) // 5) % 2, rng.integers(0, 2, Lt + 2), np.zeros(Lt + 2, int)):
                    st, alis = O.cno_enumerate(q, t, F, O.sim(q, t), thr, pq, pt, flags, 100000)
                    assert st == 0
                    ref.check("cno %d %s %dx%d" % (at, gi, Lq, Lt), _canon_arrays(alis))
                    total += len(alis)
    ref.close()
    assert total > 1000


def test_oracle_user_limit_truncation_matches_reference(blosum):
    # ucw.h:72 hard-codes user_limit = 100000; beyond it every further branch() forces the optimal path (ucw.h:115-126).
    # A 26 x 26 related pair at delta 0.5 has 251972 near-optimal alignments; the reference returns 100075.
    _, M = blosum
    ref = ReferenceResults("test_oracle.py::test_oracle_user_limit_truncation_matches_reference")
    rng = np.random.default_rng(21)
    L = 26
    q = rng.integers(0, 20, L).astype(np.uint8)
    t = q.copy()
    t[::3] = rng.integers(0, 20, len(t[::3]))
    O = po.Oracle(M, 3, 1, po.SEMI_LOCAL)
    F, pq, pt = O.fill(q, t, po.FWD, True, fast=False)
    thr = O.threshold(float(F[-1, -1]), 0.5)
    st, alis = O.ucw_enumerate(q, t, F, O.sim(q, t), thr, 300000, pq, pt)
    assert st == 0 and len(alis) > 100000
    ref.check("truncated ucw", len(alis), _canon_arrays(alis))
    ref.close()
    st, full = O.ucw_enumerate(q, t, F, O.sim(q, t), thr, 300000, pq, pt, user_limit=10 ** 9)
    assert len(full) > 2 * len(alis)
