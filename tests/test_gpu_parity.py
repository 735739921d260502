"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against
the oracle on the same seeded inputs and against the golden vectors of the real reference.
Bit-exact bar: scores, traceback pointers and near-optimal cell sets for integer scoring."""
import numpy as np
import pytest

from util import po, MODES, MODE_NAMES, golden_cases, golden_case, rand_pair, assert_matrix_equal, subali_walk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["packed", "int32"])
def ctx(request):
    # every parity test runs twice: through the packed int16x2 kernels (where a pair qualifies)
    # and with the int32 kernels forced
    import alignment_algos_b200 as a
    c = a.Context(0)
    c.set_option("packed", 1 if request.param == "packed" else 0)
    yield c
    c.close()


def _check_pair(ctx, O, q, t, tag, mask_dr=None):
    import alignment_algos_b200 as a
    out = ctx.fill_pair(q, t, a.BOTH, delta_ratio=(mask_dr if mask_dr is not None else -1.0))
    for d, nm in ((po.FWD, "fwd"), (po.REV, "rev")):
        s, pq, pt = O.fill(q, t, d, True, fast=True)
        assert_matrix_equal(tag + " score_" + nm, out["score_" + nm], s)
        assert_matrix_equal(tag + " prevq_" + nm, out["prevq_" + nm], pq)
        assert_matrix_equal(tag + " prevt_" + nm, out["prevt_" + nm], pt)
    if mask_dr is not None:
        F = O.fill(q, t, po.FWD, True, fast=True)[0]
        R = O.fill(q, t, po.REV, True, fast=True)[0]
        thr = O.threshold(float(F[-1, -1]), mask_dr)
        mask, _ = O.nearopt_mask(F, R, O.sim(q, t), thr)
        assert out["threshold"] == thr
        assert_matrix_equal(tag + " nearopt", out["nearopt"], mask)


def test_golden_vectors_of_the_reference(ctx, golden):
    import alignment_algos_b200 as a
    sub = golden["sub"]
    for name in golden_cases(golden):
        q, t, gi, ge, at = golden_case(golden, name)
        ctx.set_scoring(sub, gi, ge, at)
        out = ctx.fill_pair(q, t, a.BOTH)
        for nm in ("fwd", "rev"):
            assert_matrix_equal(name + " score_" + nm, out["score_" + nm], golden[name + "." + nm + ".score"])
            assert_matrix_equal(name + " pq_" + nm, out["prevq_" + nm], golden[name + "." + nm + ".pq"].astype(np.int32))
            assert_matrix_equal(name + " pt_" + nm, out["prevt_" + nm], golden[name + "." + nm + ".pt"].astype(np.int32))


def test_golden_ucw_union_equals_gpu_mask(ctx, golden):
    import alignment_algos_b200 as a
    sub = golden["sub"]
    n = 0
    for name in golden_cases(golden):
        for dr in (5, 20):
            key = "%s.ucw%02d" % (name, dr)
            if key + ".union" not in golden:
                continue
            q, t, gi, ge, at = golden_case(golden, name)
            ctx.set_scoring(sub, gi, ge, at)
            out = ctx.fill_pair(q, t, a.BOTH, delta_ratio=dr / 100.0)
            shape = (len(q) + 2, len(t) + 2)
            union = np.unpackbits(golden[key + ".union"])[: shape[0] * shape[1]].reshape(shape)
            interior = np.zeros_like(union)
            interior[1:-1, 1:-1] = union[1:-1, 1:-1]
            assert out["threshold"] == golden[key + ".thr"][0]
            assert_matrix_equal(key, out["nearopt"], interior)
            n += 1
    assert n >= 8


@pytest.mark.parametrize("at", MODES, ids=[MODE_NAMES[m] for m in MODES])
def test_random_pairs_all_modes(ctx, blosum, at):
    _, M = blosum
    rng = np.random.default_rng(100 + at)
    for gi, ge in [(12, 1), (3, 1), (10.5, 0.25), (1, 0)]:
        ctx.set_scoring(M, gi, ge, at)
        O = po.Oracle(M, gi, ge, at)
        for _ in range(5):
            q, t = rand_pair(rng, int(rng.integers(0, 70)), int(rng.integers(0, 70)), 24)
            _check_pair(ctx, O, q, t, "at%d gi%s ge%s %dx%d" % (at, gi, ge, len(q), len(t)),
                        mask_dr=(0.1 if at != po.LOCAL and len(q) and len(t) else None))


@pytest.mark.parametrize("at", [po.GLOBAL, po.SEMI_LOCAL, po.LOCAL, po.GLOBAL_LOCAL],
                         ids=["global", "semi_local", "local", "global_local"])
def test_edge_lengths(ctx, blosum, at):
    # ragged / boundary sizes: empty, 1, lane-chunk edges (8,16), bucket edge (256/257), stripe edge (512/513)
    _, M = blosum
    ctx.set_scoring(M, 12, 1, at)
    O = po.Oracle(M, 12, 1, at)
    rng = np.random.default_rng(5)
    for Lq, Lt in [(0, 0), (0, 5), (5, 0), (1, 1), (1, 9), (9, 1), (2, 2), (3, 8), (8, 9), (17, 16), (5, 255),
                   (5, 256), (6, 257), (40, 300), (7, 512), (7, 513), (33, 1100), (300, 40)]:
        q, t = rand_pair(rng, Lq, Lt)
        _check_pair(ctx, O, q, t, "at%d %dx%d" % (at, Lq, Lt))


def test_config1_size_250(ctx, blosum):
    # BASELINE.json configs[0]: one pair of ~250-residue proteins, optimal + near-optimal cell set
    import alignment_algos_b200 as a
    alpha20, M20 = a.blosum62()
    from alignment_algos_b200 import synth
    seqs, pq, pt = synth.config("c1")
    for at in (po.SEMI_LOCAL, po.GLOBAL):
        ctx.set_scoring(M20, 12, 1, at)
        O = po.Oracle(M20, 12, 1, at)
        _check_pair(ctx, O, seqs[0], seqs[1], "c1 at%d" % at, mask_dr=0.01)


def test_batch_matches_oracle_and_properties(ctx):
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    alpha20, M20 = a.blosum62()
    seqs, pq, pt = synth.pair_workload(77, 600, 20, 330)
    res, off = a.Context.pack(seqs)
    for at in (po.SEMI_LOCAL, po.GLOBAL):
        ctx.set_scoring(M20, 12, 1, at)
        O = po.Oracle(M20, 12, 1, at)
        what = a.W_FWD | a.W_REV | a.W_TB | a.W_SCORES | a.W_MASK
        out = ctx.fill_batch(res, off, pq, pt, what, 0.01)
        # property over the whole batch: F(end) == R(0,0) (SURVEY.md §4)
        assert_matrix_equal("fwd==rev optimum", out["fwd_score"], out["rev_score"])
        assert ctx.last_launch_count() >= 3
        rng = np.random.default_rng(3)
        for p in rng.choice(len(pq), 24, replace=False):
            q, t = seqs[pq[p]], seqs[pt[p]]
            F, fq, ft = O.fill(q, t, po.FWD, True, fast=True)
            R, rq, rt = O.fill(q, t, po.REV, True, fast=True)
            assert out["fwd_score"][p] == F[-1, -1] and out["rev_score"][p] == R[0, 0]
            thr = O.threshold(float(F[-1, -1]), 0.01)
            mask, cnt = O.nearopt_mask(F, R, O.sim(q, t), thr)
            assert out["threshold"][p] == thr and out["nearopt_count"][p] == cnt
            got = ctx.fetch_pair(int(p), len(q), len(t), fwd=True, rev=True, mask=True)
            assert_matrix_equal("F", got["score_fwd"], F)
            assert_matrix_equal("R", got["score_rev"], R)
            assert_matrix_equal("fq", got["prevq_fwd"], fq)
            assert_matrix_equal("ft", got["prevt_fwd"], ft)
            assert_matrix_equal("rq", got["prevq_rev"], rq)
            assert_matrix_equal("rt", got["prevt_rev"], rt)
            assert_matrix_equal("mask", got["nearopt"], mask)
            # optimal alignment through the packed traceback (optimal.h:47-75)
            rc, pairs, sc = ctx.optimal(int(p), a.FWD, len(q), len(t))
            orc, opairs, osc = O.optimal(F, fq, ft, po.FWD)
            assert rc == orc == 0 and sc == osc
            assert_matrix_equal("optimal fwd", pairs, opairs)
            rc, pairs, sc = ctx.optimal(int(p), a.REV, len(q), len(t))
            orc, opairs, osc = O.optimal(R, rq, rt, po.REV)
            assert (rc != 0) == (orc != 0)
            if rc == 0:
                assert_matrix_equal("optimal rev", pairs, opairs)


def test_packed_local_batch_vs_oracle():
    # LOCAL alignments on the packed int16x2 kernels (LOC = 1: every candidate clamped at 0, dpmatrix.h:538-689 / 879-1030):
    # a batch of random and related pairs; final scores of every pair against the int32 kernels, full score and
    # predecessor matrices of a sample against the oracle, local optimal alignments (find_max + enumerate_local)
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    alpha20, M20 = a.blosum62()
    seqs, pq, pt = synth.pair_workload(79, 500, 20, 512)
    res, off = a.Context.pack(seqs)
    ctx = a.Context(0)
    ctx.set_scoring(M20, 12, 1, po.LOCAL)
    O = po.Oracle(M20, 12, 1, po.LOCAL)
    what = a.W_FWD | a.W_REV | a.W_TB | a.W_SCORES
    ctx.set_profiling(True)
    out = ctx.fill_batch(res, off, pq, pt, what)
    names = {n for n, _, _ in ctx.profile()}
    ctx.set_profiling(False)
    assert any("LOC=1" in n for n in names), names
    rng = np.random.default_rng(4)
    for p in rng.choice(len(pq), 16, replace=False):
        q, t = seqs[pq[p]], seqs[pt[p]]
        F, fq, ft = O.fill(q, t, po.FWD, True, fast=True)
        R, rq, rt = O.fill(q, t, po.REV, True, fast=True)
        assert out["fwd_score"][p] == F[-1, -1] and out["rev_score"][p] == R[0, 0]
        got = ctx.fetch_pair(int(p), len(q), len(t), fwd=True, rev=True, mask=False)
        assert_matrix_equal("F", got["score_fwd"], F)
        assert_matrix_equal("R", got["score_rev"], R)
        assert_matrix_equal("fq", got["prevq_fwd"], fq)
        assert_matrix_equal("ft", got["prevt_fwd"], ft)
        assert_matrix_equal("rq", got["prevq_rev"], rq)
        assert_matrix_equal("rt", got["prevt_rev"], rt)
        for d, (S, sq, st) in ((a.FWD, (F, fq, ft)), (a.REV, (R, rq, rt))):
            rc, pairs, sc = ctx.optimal(int(p), d, len(q), len(t))
            orc, opairs, osc = O.optimal(S, sq, st, po.FWD if d == a.FWD else po.REV)
            assert rc == orc == 0 and sc == osc
            assert_matrix_equal("local optimal", pairs, opairs)
    # every pair: the int32 kernels (packed path off) give the same final scores; score-only variant as well
    ctx.set_option("packed", 0)
    ref = ctx.fill_batch(res, off, pq, pt, what)
    ctx.set_option("packed", 1)
    so = ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV)
    for k in ("fwd_score", "rev_score"):
        assert_matrix_equal("int32 " + k, out[k], ref[k])
        assert_matrix_equal("score-only " + k, out[k], so[k])
    ctx.close()


def test_score_only_batch_equals_full_batch(ctx):
    # the score-only kernels (DPX viaddmax/vimax3 path) and the traceback kernels agree
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    alpha20, M20 = a.blosum62()
    seqs, pq, pt = synth.pair_workload(78, 3000, 100, 500)
    res, off = a.Context.pack(seqs)
    ctx.set_scoring(M20, 12, 1, po.SEMI_LOCAL)
    s0 = ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV)
    s1 = ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB)
    assert_matrix_equal("fwd", s0["fwd_score"], s1["fwd_score"])
    assert_matrix_equal("rev", s0["rev_score"], s1["rev_score"])
    assert_matrix_equal("fwd==rev", s0["fwd_score"], s0["rev_score"])
    O = po.Oracle(M20, 12, 1, po.SEMI_LOCAL)
    for p in (0, 17, 2999):
        F = O.fill(seqs[pq[p]], seqs[pt[p]], po.FWD, True, fast=True)[0]
        assert s0["fwd_score"][p] == F[-1, -1]


def test_errors_are_loud(ctx, blosum):
    import alignment_algos_b200 as a
    _, M = blosum
    with pytest.raises(a.AadpError):
        ctx.set_scoring(M, -1.0, 0.34, po.SEMI_LOCAL)  # negative gap penalty
    with pytest.raises(a.AadpError):
        ctx.set_scoring(M, 12, 1, 7)  # "Illegal gap style" (aasubalib.h:49)
    ctx.set_scoring(M, 12, 1, po.GLOBAL)
    with pytest.raises(a.AadpError):
        ctx.fill_pair(np.array([30], np.uint8), np.array([1], np.uint8))  # code outside the alphabet


@pytest.mark.parametrize("at", [po.GLOBAL, po.SEMI_LOCAL, po.LOCAL], ids=["global", "semi_local", "local"])
def test_long_pair_multi_cta_wavefront(blosum, at):
    # BASELINE.json configs[4] in miniature: one long pair filled by the multi-CTA wavefront kernel
    # (one CTA per 256-column stripe, both directions in one cooperative launch)
    import alignment_algos_b200 as a
    _, M = blosum
    c = a.Context(0)
    c.set_option("wave_min_cells", 1)
    c.set_scoring(M, 12, 1, at)
    O = po.Oracle(M, 12, 1, at)
    rng = np.random.default_rng(9)
    try:
        for Lq, Lt in [(40, 600), (700, 1300), (1500, 2100), (33, 513), (300, 4000)]:
            q, t = rand_pair(rng, Lq, Lt)
            _check_pair(c, O, q, t, "wave at%d %dx%d" % (at, Lq, Lt), mask_dr=(0.02 if at != po.LOCAL else None))
            names = set()
    finally:
        c.close()


def test_long_pair_uses_wave_kernel(blosum):
    import alignment_algos_b200 as a
    _, M = blosum
    c = a.Context(0)
    c.set_option("wave_min_cells", 1)
    c.set_scoring(M, 12, 1, po.GLOBAL)
    rng = np.random.default_rng(10)
    q, t = rand_pair(rng, 900, 1800)
    res, off = a.Context.pack([q, t])
    c.set_profiling(True)
    out = c.fill_batch(res, off, [0], [1], a.W_FWD | a.W_REV | a.W_TB)
    names = [n for n, ms, cells in c.profile()]
    c.close()
    assert any(n.startswith("wave_kernel") for n in names), names
    assert out["fwd_score"][0] == out["rev_score"][0]


def _rescore(O, q, t, pairs, sub, gi, ge, at):
    """Score of an alignment given as (q,t) index pairs incl. (0,0) and (last,last), with the
    evaluator's gap rules (aasubalib.h:27-77)."""
    sz1, sz2 = len(q) + 2, len(t) + 2
    delfree = at in (po.LOCAL, po.SEMI_LOCAL, po.LOCAL_GLOBAL)
    insfree = at in (po.LOCAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL)
    s = 0.0
    for (a0, b0), (a1, b1) in zip(pairs[:-1], pairs[1:]):
        dl, il = b1 - b0 - 1, a1 - a0 - 1
        assert a1 > a0 and b1 > b0 and (dl == 0 or il == 0), "not a valid alignment step"
        if dl >= 1 and not (delfree and (b0 == 0 or b1 == sz2 - 1)):
            s -= gi + ge * (dl - 1)
        if il >= 1 and not (insfree and (a0 == 0 or a1 == sz1 - 1)):
            s -= gi + ge * (il - 1)
        if 1 <= a1 <= len(q) and 1 <= b1 <= len(t):
            s += sub[q[a1 - 1], t[b1 - 1]]
    return s


def test_large_batch_size_independent_properties(ctx):
    # at sizes the oracle cannot sweep: (1) F(end) == R(0,0) for every pair, (2) the optimal alignment
    # decoded from the packed traceback is a valid alignment whose rescored value equals the fill's optimum,
    # in both directions, (3) every cell of that alignment is in the near-optimal set
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    alpha20, M20 = a.blosum62()
    seqs, pq, pt = synth.pair_workload(4242, 12000, 100, 500)
    res, off = a.Context.pack(seqs)
    for at in (po.SEMI_LOCAL, po.GLOBAL):
        ctx.set_scoring(M20, 12, 1, at)
        out = ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB | a.W_MASK, 0.01)
        assert_matrix_equal("fwd==rev optimum", out["fwd_score"], out["rev_score"])
        assert (out["nearopt_count"] >= 1).all()
        rng = np.random.default_rng(at)
        for p in rng.choice(len(pq), 40, replace=False):
            q, t = seqs[pq[p]], seqs[pt[p]]
            rc, pairs, sc = ctx.optimal(int(p), a.FWD, len(q), len(t))
            assert rc == 0 and sc == out["fwd_score"][p]
            assert tuple(pairs[0]) == (0, 0) and tuple(pairs[-1]) == (len(q) + 1, len(t) + 1)
            assert _rescore(None, q, t, [tuple(x) for x in pairs], M20, 12, 1, at) == sc
            got = ctx.fetch_pair(int(p), len(q), len(t), fwd=False, rev=False, tb=False, scores=False, mask=True)
            for (i, j) in pairs[1:-1]:
                assert got["nearopt"][i, j] == 1, "optimal cell missing from the near-optimal set"
            rc, rpairs, rsc = ctx.optimal(int(p), a.REV, len(q), len(t))
            if rc == 0:
                rp = [tuple(int(v) for v in x) for x in rpairs]
                # dpmatrix.h:868 (reproduced) can make the FIRST reverse step jump in both indices; that walk is
                # the reference's behaviour but not an alignment. Every other reverse walk must rescore exactly.
                first_ok = (rp[1][0] - rp[0][0] == 1) or (rp[1][1] - rp[0][1] == 1)
                if first_ok:
                    assert _rescore(None, q, t, rp, M20, 12, 1, at) == rsc
                else:
                    assert rp[1][1] == len(t), "only the :868 pattern may produce such a step"


def test_large_batch_enumeration_properties(ctx):
    # near-optimal enumeration at a size the oracle cannot sweep (8000 related pairs of 100-500 residues): every
    # alignment (1) is a valid alignment from (0,0) to (last,last) whose rescored value equals the returned score,
    # (2) scores above the pair's threshold, (3) lies inside the near-optimal cell set of the fused mask pass;
    # (4) the alignments of a pair are pairwise different and (5) the optimal alignment is among them;
    # (6) constrained enumeration with all flags set = the optimal alignment of every branch taken at the root
    import alignment_algos_b200 as a
    alpha20, M20 = a.blosum62()
    rng = np.random.default_rng(2027)
    seqs, pq, pt = [], [], []
    for k in range(8000):
        L = int(rng.integers(100, 501))
        s = rng.integers(0, 20, L).astype(np.uint8)
        m = s.copy()
        m[::9] = rng.integers(0, 20, len(m[::9]))
        cut = int(rng.integers(10, L - 10))
        seqs += [s, np.concatenate([m[:cut], m[cut + int(rng.integers(0, 3)):]])]
        pq.append(2 * k)
        pt.append(2 * k + 1)
    pq, pt = np.array(pq, np.int32), np.array(pt, np.int32)
    res, off = a.Context.pack(seqs)
    at, delta, K = po.SEMI_LOCAL, 0.01, 48
    ctx.set_scoring(M20, 12, 1, at)
    out = ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB | a.W_MASK, delta)
    got = ctx.near_optimal(np.arange(8000), delta, K)
    con = ctx.near_optimal(np.arange(0, 8000, 40), delta, K, constrained=True)
    n_multi = 0
    for p in range(8000):
        st, thr, alis = got[p]
        assert st in (0, 1) and len(alis) >= 1 and thr == out["threshold"][p]
        assert st == 0 or len(alis) == K
        n_multi += len(alis) > 1
        if p % 40:
            continue
        q, t = seqs[pq[p]], seqs[pt[p]]
        mask = ctx.fetch_pair(p, len(q), len(t), fwd=False, rev=False, tb=False, scores=False, mask=True)["nearopt"]
        rc, opt_pairs, opt_sc = ctx.optimal(p, a.FWD, len(q), len(t))
        seen = set()
        for sc, pairs in alis:
            pl = [tuple(int(v) for v in x) for x in pairs]
            assert pl[0] == (0, 0) and pl[-1] == (len(q) + 1, len(t) + 1)
            assert _rescore(None, q, t, pl, M20, 12, 1, at) == sc and sc > thr
            assert all(mask[i, j] == 1 for (i, j) in pl[1:-1])
            seen.add(tuple(pl))
        assert len(seen) == len(alis)
        assert tuple(tuple(int(v) for v in x) for x in opt_pairs) in seen or st == 1
        cst, cthr, calis = con[p // 40]
        assert cst == 0 and cthr == thr and 1 <= len(calis)
        for sc, pairs in calis:
            pl = [tuple(int(v) for v in x) for x in pairs]
            assert _rescore(None, q, t, pl, M20, 12, 1, at) == sc
    assert n_multi > 2000


@pytest.mark.parametrize("at", [po.GLOBAL, po.SEMI_LOCAL], ids=["global", "semi_local"])
def test_extreme_scores_near_the_packed_bound(ctx, blosum, at):
    # identical poly-W sequences (largest positive scores the packed int16 path accepts), all-mismatch
    # pairs (most negative), and mixtures; lengths at the packed limits
    alpha, M = blosum
    W, C, G = alpha.index("W"), alpha.index("C"), alpha.index("G")
    ctx.set_scoring(M, 12, 1, at)
    O = po.Oracle(M, 12, 1, at)
    rng = np.random.default_rng(3)
    cases = [(np.full(500, W), np.full(500, W)), (np.full(512, W), np.full(512, W)), (np.full(500, W), np.full(500, G)),
             (np.full(300, C), np.full(511, W)), (np.full(40, W), np.full(512, G)),
             (np.r_[np.full(200, W), rng.integers(0, 20, 100)], np.r_[rng.integers(0, 20, 150), np.full(300, W)])]
    for q, t in cases:
        _check_pair(ctx, O, q.astype(np.uint8), t.astype(np.uint8), "extreme at%d %dx%d" % (at, len(q), len(t)), mask_dr=0.01)


def test_half_unit_scoring_and_large_gaps(ctx, blosum):
    # dyadic (non-integer) grids and gap penalties near the packed path's limits
    _, M = blosum
    rng = np.random.default_rng(8)
    for gi, ge, at in [(10.5, 0.25, po.SEMI_LOCAL), (0.5, 0.5, po.GLOBAL), (40, 3, po.GLOBAL), (100, 0, po.SEMI_LOCAL),
                       (300, 10, po.GLOBAL_LOCAL)]:
        ctx.set_scoring(M, gi, ge, at)
        O = po.Oracle(M, gi, ge, at)
        for Lq, Lt in [(90, 130), (257, 31)]:
            q, t = rand_pair(rng, Lq, Lt)
            _check_pair(ctx, O, q, t, "gi%s ge%s at%d" % (gi, ge, at), mask_dr=0.05)


@pytest.mark.parametrize("at", [po.GLOBAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL, po.LOCAL],
                         ids=["global", "semi_local", "global_local", "local"])
def test_cross_scores_all_queries_vs_all_templates(ctx, at):
    # cross mode (one template profile shared by groups of query couples) against the oracle and against
    # the pair-list batch path; the lists mix eligible sequences with empty ones and templates > 512
    import alignment_algos_b200 as a
    alpha20, M20 = a.blosum62()
    rng = np.random.default_rng(41 + at)
    lens = list(rng.integers(1, 140, 37)) + [0, 1, 16, 17, 512, 513, 600, 33]
    seqs = [rng.integers(0, 20, int(L)).astype(np.uint8) for L in lens]
    res, off = a.Context.pack(seqs)
    q_ids = np.array([3, 0, 44, 38, 7, 37, 12, 5, 41, 9, 3, 20, 21, 22, 43], np.int32)   # repeats allowed, odd count
    t_ids = np.arange(len(seqs), dtype=np.int32)[::-1].copy()
    ctx.set_scoring(M20, 12, 1, at)
    got = ctx.cross_scores(res, off, q_ids, t_ids)
    O = po.Oracle(M20, 12, 1, at)
    want = np.zeros_like(got)
    for i, qs in enumerate(q_ids):
        for j, ts in enumerate(t_ids):
            want[i, j] = O.fill(seqs[qs], seqs[ts], po.FWD, False, fast=True)[0][-1, -1]
    assert_matrix_equal("cross scores", got, want)
    # the same rectangle as an explicit pair list
    pq = np.repeat(q_ids, len(t_ids)).astype(np.int32)
    pt = np.tile(t_ids, len(q_ids)).astype(np.int32)
    out = ctx.fill_batch(res, off, pq, pt, a.W_FWD)
    assert_matrix_equal("cross == pair list", got.reshape(-1), out["fwd_score"])


def test_cross_scores_block_properties(ctx):
    # larger rectangle: symmetry of semi_local/global scores under swapping roles (BLOSUM62 is symmetric),
    # block decomposition gives the same matrix, self-scores on the diagonal
    import alignment_algos_b200 as a
    import torch
    alpha20, M20 = a.blosum62()
    rng = np.random.default_rng(5)
    seqs = [rng.integers(0, 20, int(L)).astype(np.uint8) for L in rng.integers(100, 501, 300)]
    res, off = a.Context.pack(seqs)
    ids = np.arange(300, dtype=np.int32)
    ctx.set_scoring(M20, 12, 1, a.SEMI_LOCAL)
    full = ctx.cross_scores(res, off, ids, ids)
    assert_matrix_equal("symmetry", full, full.T)
    diag = np.array([sum(M20[x, x] for x in s) for s in seqs], np.float32)
    assert_matrix_equal("self score", np.diag(full), diag)
    ctx.upload_sequences(res, off)
    d = torch.zeros((100, 150), dtype=torch.float32, device="cuda")
    ctx.cross_run(ids[50:150], ids[150:300], d.data_ptr())
    ctx.synchronize()
    assert_matrix_equal("block", d.cpu().numpy(), full[50:150, 150:300])
    assert ctx.last_cross_cell_updates() == float(sum(len(s) for s in seqs[50:150])) * float(sum(len(s) for s in seqs[150:300]))


# ---- exact general-gap fp32 path: scoring that is not on a dyadic grid (reference defaults 4.73 / 0.34) ----

def test_float_golden_vectors_of_the_reference(golden_float):
    # bit-exact (0 ulp) scores, identical predecessors, identical optimal alignments
    import alignment_algos_b200 as a
    g = golden_float
    c = a.Context(0)
    for name in golden_cases(g):
        q, t, gi, ge, at = golden_case(g, name)
        c.set_scoring(g["sub." + str(g[name + ".sub"])], gi, ge, at)
        out = c.fill_pair(q, t, a.BOTH)
        for nm in ("fwd", "rev"):
            assert_matrix_equal(name + " score_" + nm, out["score_" + nm], g[name + "." + nm + ".score"])
            assert_matrix_equal(name + " pq_" + nm, out["prevq_" + nm], g[name + "." + nm + ".pq"].astype(np.int32))
            assert_matrix_equal(name + " pt_" + nm, out["prevt_" + nm], g[name + "." + nm + ".pt"].astype(np.int32))
        if at != po.LOCAL:
            res, off = a.Context.pack([q, t])
            c.fill_batch(res, off, [0], [1], a.W_FWD | a.W_REV)
            for d, nm in ((a.FWD, "fwd"), (a.REV, "rev")):
                rc, pairs, sc = c.optimal(0, d, len(q), len(t))
                want_rc = int(g[name + "." + nm + ".opt_rc"][0])
                assert (rc != 0) == (want_rc != 0), name + nm
                if rc == 0:
                    assert_matrix_equal(name + nm + ".opt", pairs, g[name + "." + nm + ".opt_pairs"].astype(np.int32))
                    assert sc == g[name + "." + nm + ".opt_score"][0]
    c.close()


def test_float_ucw_union_equals_gpu_mask(golden_float):
    import alignment_algos_b200 as a
    g = golden_float
    c = a.Context(0)
    n = 0
    for name in golden_cases(g):
        for dr in (5, 20):
            key = "%s.ucw%02d" % (name, dr)
            if key + ".union" not in g:
                continue
            q, t, gi, ge, at = golden_case(g, name)
            c.set_scoring(g["sub." + str(g[name + ".sub"])], gi, ge, at)
            out = c.fill_pair(q, t, a.BOTH, delta_ratio=dr / 100.0)
            shape = (len(q) + 2, len(t) + 2)
            union = np.unpackbits(g[key + ".union"])[: shape[0] * shape[1]].reshape(shape)
            interior = np.zeros_like(union)
            interior[1:-1, 1:-1] = union[1:-1, 1:-1]
            assert out["threshold"] == g[key + ".thr"][0]
            assert_matrix_equal(key, out["nearopt"], interior)
            n += 1
    assert n >= 6
    c.close()


@pytest.mark.parametrize("at", MODES, ids=[MODE_NAMES[m] for m in MODES])
def test_float_random_pairs_vs_literal_oracle(blosum, at):
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(900 + at)
    c = a.Context(0)
    c.set_scoring(M, 4.73, 0.34, at)
    O = po.Oracle(M, 4.73, 0.34, at)
    for Lq, Lt in [(0, 0), (0, 5), (4, 0), (1, 1), (2, 3), (33, 17), (64, 65), (120, 90), (5, 700)]:
        q, t = rand_pair(rng, Lq, Lt)
        out = c.fill_pair(q, t, a.BOTH, delta_ratio=0.05)
        F, fq, ft = O.fill(q, t, po.FWD, True, fast=False)
        R, rq, rt = O.fill(q, t, po.REV, True, fast=False)
        tag = "float at%d %dx%d " % (at, Lq, Lt)
        assert_matrix_equal(tag + "F", out["score_fwd"], F)
        assert_matrix_equal(tag + "R", out["score_rev"], R)
        assert_matrix_equal(tag + "fq", out["prevq_fwd"], fq)
        assert_matrix_equal(tag + "ft", out["prevt_fwd"], ft)
        assert_matrix_equal(tag + "rq", out["prevq_rev"], rq)
        assert_matrix_equal(tag + "rt", out["prevt_rev"], rt)
        thr = O.threshold(float(F[-1, -1]), 0.05)
        mask, _ = O.nearopt_mask(F, R, O.sim(q, t), thr)
        assert out["threshold"] == thr
        assert_matrix_equal(tag + "mask", out["nearopt"], mask)
    c.close()


def test_float_batch_scalars_and_forced_float_equals_integer_path(blosum):
    # (1) batches in exact-float mode: per-pair scalars against the literal oracle, chunked scratch;
    # (2) forcing the general-gap kernel on integer scoring gives exactly what the integer kernels give
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    _, M = blosum
    seqs, pq, pt = synth.pair_workload(11, 60, 5, 90)
    res, off = a.Context.pack(seqs)
    c = a.Context(0)
    c.set_option("general_budget_mcells", 1)  # forces several chunks
    c.set_scoring(M, 4.73, 0.34, po.SEMI_LOCAL)
    O = po.Oracle(M, 4.73, 0.34, po.SEMI_LOCAL)
    out = c.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_MASK, 0.02)
    for p in range(len(pq)):
        q, t = seqs[pq[p]], seqs[pt[p]]
        F = O.fill(q, t, po.FWD, True, fast=False)[0]
        R = O.fill(q, t, po.REV, True, fast=False)[0]
        thr = O.threshold(float(F[-1, -1]), 0.02)
        _, cnt = O.nearopt_mask(F, R, O.sim(q, t), thr)
        assert out["fwd_score"][p] == F[-1, -1] and out["rev_score"][p] == R[0, 0]
        assert out["threshold"][p] == thr and out["nearopt_count"][p] == cnt
    got = c.fetch_pair(7, len(seqs[pq[7]]), len(seqs[pt[7]]), fwd=True, rev=True, mask=True)
    F, fq, ft = O.fill(seqs[pq[7]], seqs[pt[7]], po.FWD, True, fast=False)
    assert_matrix_equal("fetch F", got["score_fwd"], F)
    assert_matrix_equal("fetch fq", got["prevq_fwd"], fq)
    c.set_option("exact_float", 1)
    c.set_scoring(M, 12, 1, po.GLOBAL)
    c2 = a.Context(0)
    c2.set_scoring(M, 12, 1, po.GLOBAL)
    o1 = c.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_MASK, 0.02)
    o2 = c2.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_MASK, 0.02)
    for k in ("fwd_score", "rev_score", "threshold", "nearopt_count"):
        assert_matrix_equal("forced float " + k, o1[k], o2[k])
    x1 = c.fill_pair(seqs[0], seqs[1], a.BOTH, delta_ratio=0.02)
    x2 = c2.fill_pair(seqs[0], seqs[1], a.BOTH, delta_ratio=0.02)
    for k in x1:
        if x1[k] is not None and k != "threshold":
            assert_matrix_equal("forced float pair " + k, x1[k], x2[k])
    # cross mode falls back to the general path in exact-float mode
    ids = np.arange(12, dtype=np.int32)
    assert_matrix_equal("cross float", c.cross_scores(res, off, ids, ids), c2.cross_scores(res, off, ids, ids))
    c.close()
    c2.close()


@pytest.mark.parametrize("at", [po.GLOBAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL, po.LOCAL_GLOBAL],
                         ids=["global", "semi_local", "global_local", "local_global"])
def test_gpu_traceback_of_whole_batch(ctx, at):
    # aadp_batch_optimal_all (one GPU thread per pair) against the per-pair host walk and the oracle
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    alpha20, M20 = a.blosum62()
    rng = np.random.default_rng(70 + at)
    seqs = [rng.integers(0, 20, int(L)).astype(np.uint8) for L in list(rng.integers(1, 200, 78)) + [0, 0, 530, 600]]
    pq = np.arange(0, len(seqs), 2, dtype=np.int32)
    pt = pq + 1
    res, off = a.Context.pack(seqs)
    ctx.set_scoring(M20, 3, 1, at)   # cheap gaps: alignments with many gaps
    O = po.Oracle(M20, 3, 1, at)
    ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB)
    for d, od in ((a.FWD, po.FWD), (a.REV, po.REV)):
        aoff, pairs, n, st = ctx.optimal_all(d, len(pq))
        for p in range(len(pq)):
            q, t = seqs[pq[p]], seqs[pt[p]]
            assert aoff[p + 1] - aoff[p] == len(q) + len(t) + 2
            rc, hp, sc = ctx.optimal(p, d, len(q), len(t))
            assert st[p] == rc, "pair %d dir %d status" % (p, d)
            assert_matrix_equal("pair %d dir %d" % (p, d), pairs[aoff[p]:aoff[p] + n[p]], hp)
            if p % 5 == 0:
                S, Q, T = O.fill(q, t, od, True, fast=True)
                orc, opairs, osc = O.optimal(S, Q, T, od)
                assert (orc != 0) == (st[p] != 0)
                if orc == 0:
                    assert_matrix_equal("oracle pair %d dir %d" % (p, d), pairs[aoff[p]:aoff[p] + n[p]], opairs)


def test_sub_rectangle_fill_golden_and_random(golden_sub, blosum):
    # aadp_fill_subpair == the reference's 9-argument constructor (build_subdpm, dpmatrix.h:319-353)
    import alignment_algos_b200 as a
    g = golden_sub
    c = a.Context(0)
    for name in golden_cases(g):
        q, t, gi, ge, at = golden_case(g, name)
        c.set_scoring(g["sub"], gi, ge, at)
        for d, tag in ((a.FWD, "fwd"), (a.REV, "rev")):
            s, pq, pt = c.fill_subpair(q, t, g[name + ".rect"], d)
            assert_matrix_equal(name + tag + ".score", s, g[name + "." + tag + ".score"])
            assert_matrix_equal(name + tag + ".pq", pq, g[name + "." + tag + ".pq"].astype(np.int32))
            assert_matrix_equal(name + tag + ".pt", pt, g[name + "." + tag + ".pt"].astype(np.int32))
    _, M = blosum
    rng = np.random.default_rng(23)
    for gi, ge, at in [(12, 1, po.SEMI_LOCAL), (4.73, 0.34, po.GLOBAL), (3, 1, po.LOCAL), (10.5, 0.25, po.GLOBAL_LOCAL)]:
        c.set_scoring(M, gi, ge, at)
        O = po.Oracle(M, gi, ge, at)
        for trial in range(10):
            Lq, Lt = int(rng.integers(1, 120)), int(rng.integers(1, 700 if trial == 0 else 120))
            q, t = rand_pair(rng, Lq, Lt)
            q0 = int(rng.integers(0, Lq + 1)); q1 = int(rng.integers(q0 + 1, Lq + 2))
            t0 = int(rng.integers(0, Lt + 1)); t1 = int(rng.integers(t0 + 1, Lt + 2))
            for d, od in ((a.FWD, po.FWD), (a.REV, po.REV)):
                s, pq, pt = c.fill_subpair(q, t, (q0, t0, q1, t1), d)
                ws, wq, wt = O.fill_sub(q, t, (q0, t0, q1, t1), od)
                assert_matrix_equal("sub score", s, ws)
                assert_matrix_equal("sub pq", pq, wq)
                assert_matrix_equal("sub pt", pt, wt)
        # the whole matrix as a rectangle is the ordinary fill
        q, t = rand_pair(rng, 40, 33)
        s, pq, pt = c.fill_subpair(q, t, (0, 0, 41, 34), a.FWD)
        out = c.fill_pair(q, t, a.FWD)
        assert_matrix_equal("full rect score", s, out["score_fwd"])
        assert_matrix_equal("full rect pq", pq, out["prevq_fwd"])
    with pytest.raises(a.AadpError):
        c.fill_subpair(q, t, (5, 5, 5, 9), a.FWD)  # "Illegal bounds building DPM"
    c.close()


def test_sub_rectangle_batch_golden_and_random(golden_sub, blosum):
    # aadp_fill_subpair_batch (row f4): many build_subdpm fills + Optimal_Subali tracebacks in one call, compact storage
    import alignment_algos_b200 as a
    g = golden_sub
    c = a.Context(0)
    groups = {}
    for name in golden_cases(g):
        q, t, gi, ge, at = golden_case(g, name)
        groups.setdefault((float(gi), float(ge), int(at), q.tobytes(), t.tobytes()), []).append(name)
    assert len(groups) >= 10
    for (gi, ge, at, _, _), names in groups.items():
        q, t, _, _, _ = golden_case(g, names[0])
        c.set_scoring(g["sub"], gi, ge, at)
        res, off = a.Context.pack([q, t])
        rects = np.array([g[n + ".rect"] for n in names], np.int32)
        iq, it = np.zeros(len(names), np.int32), np.ones(len(names), np.int32)
        score, aoff, pairs, n_out, st = c.fill_subpair_batch(res, off, iq, it, rects, a.FWD)
        rscore, _, _, _, _ = c.fill_subpair_batch(res, off, iq, it, rects, a.REV)
        for k, n in enumerate(names):
            wst, wpairs, wscore = subali_walk(g[n + ".fwd.score"], g[n + ".fwd.pq"], g[n + ".fwd.pt"], rects[k])
            assert aoff[k + 1] - aoff[k] == rects[k][2] - rects[k][0] + 1
            assert st[k] == wst, n
            assert score[k] == wscore, n
            assert_matrix_equal(n + " subali", pairs[aoff[k]:aoff[k] + n_out[k]], wpairs)
            assert rscore[k] == g[n + ".rev.score"][rects[k][0], rects[k][1]], n
    # random: several pairs, many loops each, chunked by a small scratch budget; oracle + the single-fill entry
    _, M = blosum
    rng = np.random.default_rng(31)
    for gi, ge, at in [(12, 1, po.SEMI_LOCAL), (4.73, 0.34, po.GLOBAL), (10.5, 0.25, po.GLOBAL_LOCAL)]:
        c.set_scoring(M, gi, ge, at)
        O = po.Oracle(M, gi, ge, at)
        seqs = [rng.integers(0, 20, int(L)).astype(np.uint8) for L in rng.integers(100, 300, 12)]
        res, off = a.Context.pack(seqs)
        n = 400
        iq = rng.integers(0, 12, n).astype(np.int32)
        it = rng.integers(0, 12, n).astype(np.int32)
        rects = np.zeros((n, 4), np.int32)
        for k in range(n):
            Lq, Lt = len(seqs[iq[k]]), len(seqs[it[k]])
            q0 = int(rng.integers(0, Lq + 1)); t0 = int(rng.integers(0, Lt + 1))
            rects[k] = (q0, t0, min(Lq + 1, q0 + int(rng.integers(1, 150))), min(Lt + 1, t0 + int(rng.integers(1, 150))))
        rects[0] = (0, 0, len(seqs[iq[0]]) + 1, len(seqs[it[0]]) + 1)   # a whole matrix among the loops
        c.set_option("general_budget_mcells", 1)
        score, aoff, pairs, n_out, st = c.fill_subpair_batch(res, off, iq, it, rects, a.FWD)
        c.set_option("general_budget_mcells", 400)
        score2, aoff2, pairs2, n2, st2 = c.fill_subpair_batch(res, off, iq, it, rects, a.FWD)
        assert_matrix_equal("chunked score", score, score2)
        assert_matrix_equal("chunked pairs", pairs, pairs2)
        assert_matrix_equal("chunked n", n_out, n2)
        sonly = c.fill_subpair_batch(res, off, iq, it, rects, a.FWD, want_alignments=False)[0]
        assert_matrix_equal("score-only", sonly, score)
        for k in list(range(0, n, 7)) + [n - 1]:
            q, t = seqs[iq[k]], seqs[it[k]]
            ws, wq, wt = O.fill_sub(q, t, tuple(int(x) for x in rects[k]), po.FWD)
            wst, wpairs, wscore = subali_walk(ws, wq, wt, rects[k])
            assert st[k] == wst and score[k] == wscore, k
            assert_matrix_equal("item %d subali" % k, pairs[aoff[k]:aoff[k] + n_out[k]], wpairs)
        s1, _, _ = c.fill_subpair(seqs[iq[5]], seqs[it[5]], rects[5], a.FWD)
        assert s1[rects[5][2], rects[5][3]] == score[5]
    with pytest.raises(a.AadpError):
        c.fill_subpair_batch(res, off, iq[:1], it[:1], np.array([[5, 5, 5, 9]], np.int32), a.FWD)
    z = c.fill_subpair_batch(res, off, iq[:0], it[:0], np.zeros((0, 4), np.int32), a.FWD)
    assert len(z[0]) == 0 and z[1][0] == 0
    c.close()


def test_tabulated_gap_model_golden_and_random(golden_tab):
    # aadp_fill_pair_tabulated (row f3): position-dependent gap penalties (hmap_eval.h:63-117 / gn2_eval.h:99-158 shaped)
    # through the exact general-gap kernel; golden = the REAL reference fill driven by a table-backed Evaluator
    import alignment_algos_b200 as a
    g = golden_tab
    c = a.Context(0)   # no aadp_set_scoring needed
    for name in golden_cases(g):
        for d, tag in ((a.FWD, "fwd"), (a.REV, "rev")):
            s, pq, pt = c.fill_pair_tabulated(g[name + ".sim"], g[name + ".del"], g[name + ".ins"], int(g[name + ".local"]), d)
            assert_matrix_equal(name + tag + ".score", s, g[name + "." + tag + ".score"])
            assert_matrix_equal(name + tag + ".pq", pq, g[name + "." + tag + ".pq"].astype(np.int32))
            assert_matrix_equal(name + tag + ".pt", pt, g[name + "." + tag + ".pt"].astype(np.int32))
    rng = np.random.default_rng(61)
    for at in (po.GLOBAL, po.SEMI_LOCAL, po.LOCAL):
        for gen, (Lq, Lt) in ((po.hmap_like_tables, (130, 97)), (po.gn2_like_tables, (64, 150)), (po.hmap_like_tables, (3, 600))):
            sim, dt, it = gen(rng, Lq, Lt, at)
            for d, od in ((a.FWD, po.FWD), (a.REV, po.REV)):
                got = c.fill_pair_tabulated(sim, dt, it, at == po.LOCAL, d)
                want = po.Oracle.fill_tab(sim, dt, it, at == po.LOCAL, od)
                for x, y, nm in zip(got, want, ("score", "pq", "pt")):
                    assert_matrix_equal("tab %s" % nm, x, y)
    # the affine model written as tables is the ordinary path (ties the table layout to aadp_fill_pair_general)
    sim, dt, it = po.hmap_like_tables(rng, 30, 41, po.GLOBAL)
    gi, ge = np.float32(4.73), np.float32(0.34)
    for t1 in range(43):
        for t2 in range(t1 + 2, 43):
            dt[t1, t2] = np.float32(gi + np.float32(ge * np.float32(t2 - t1 - 2)))
    for ln in range(1, 31):
        it[ln, 1:] = np.float32(gi + np.float32(ge * np.float32(ln - 1)))
    s1, q1, t1_ = c.fill_pair_tabulated(sim, dt, it, False, a.FWD)
    s2, q2, t2_ = c.fill_pair_general(sim, 4.73, 0.34, po.GLOBAL, a.FWD)
    assert_matrix_equal("affine tables score", s1, s2)
    assert_matrix_equal("affine tables pq", q1, q2)
    bad = dt.copy()
    bad[4, 5] = 1.0
    with pytest.raises(a.AadpError):
        c.fill_pair_tabulated(sim, bad, it, False, a.FWD)   # adjacent positions must cost nothing
    c.close()


def test_near_optimal_enumeration_on_gpu(blosum):
    # aadp_batch_near_optimal (row f1): UnconstrainedNearOptimal::enumerate (ucw.h:63-191) of listed pairs of a resident
    # batch, one warp per pair over the packed score blob.  Oracle = orc_ucw_enumerate (pinned to the reference in
    # tests/test_oracle.py): same alignments in the same depth-first order with bit-identical fp32 scores.
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(83)
    for gi, ge, at, delta in [(12, 1, po.SEMI_LOCAL, 0.08), (3, 1, po.GLOBAL, 0.12), (10.5, 0.25, po.GLOBAL_LOCAL, 0.2),
                              (3, 1, po.LOCAL_GLOBAL, 0.15)]:
        seqs = []
        for k in range(24):
            L = int(rng.integers(8, 70))
            s = rng.integers(0, 20, L).astype(np.uint8)
            seqs.append(s)
            m = s.copy()                      # a mutated copy: related pairs have many near-optimal alignments
            m[::5] = rng.integers(0, 20, len(m[::5]))
            seqs.append(np.concatenate([m[: L // 2], m[L // 2 + int(rng.integers(0, 3)):]]))
        seqs += [rng.integers(0, 20, L).astype(np.uint8) for L in (0, 1, 2, 530)]
        res, off = a.Context.pack(seqs)
        pq = np.array(list(range(0, 48, 2)) + [48, 49, 50, 3, 51, 6], np.int32)
        pt = np.array(list(range(1, 48, 2)) + [5, 49, 7, 48, 9, 51], np.int32)
        c = a.Context(0)
        c.set_scoring(M, gi, ge, at)
        what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK
        c.fill_batch(res, off, pq, pt, what, delta)
        K = 3000
        ids = np.arange(len(pq))[::-1].copy()          # any order, any subset
        got = c.near_optimal(ids, delta, K)
        O = po.Oracle(M, gi, ge, at)
        n_multi = 0
        for k, p in enumerate(ids):
            q, t = seqs[pq[p]], seqs[pt[p]]
            F, _, _ = O.fill(q, t, po.FWD, True, fast=True)
            thr = O.threshold(float(F[-1, -1]), delta)
            st, want = O.ucw_enumerate(q, t, F, O.sim(q, t), thr, K)
            gst, gthr, alis = got[k]
            assert gst == st, (p, gst, st)
            assert gthr == thr
            assert len(alis) == len(want), (p, len(alis), len(want))
            n_multi += len(alis) > 1
            for (gs, gp), (ws, wp) in zip(alis, want):
                assert gs == ws
                assert_matrix_equal("pair %d alignment" % p, gp, wp)
        assert n_multi >= 5
        # a budget smaller than the number of alignments: status 1 and the first K in depth-first order
        big = max(range(len(ids)), key=lambda k: len(got[k][2]))
        nbig = len(got[big][2])
        if nbig > 3:
            small = c.near_optimal(ids[big:big + 1], delta, nbig - 2)[0]
            assert small[0] == 1 and len(small[2]) == nbig - 2
            for (gs, gp), (ws, wp) in zip(small[2], got[big][2]):
                assert gs == ws and np.array_equal(gp, wp)
        c.close()
    # exact-float mode (scoring off the dyadic grid, the reference defaults): each listed pair is refilled by the exact
    # general-gap kernel and walked over its dense fp32 matrix, opt_path (ucw.h:194-236) included
    for gi, ge, at, delta in [(4.73, 0.34, po.GLOBAL, 0.1), (4.73, 0.34, po.SEMI_LOCAL, 0.06), (2.17, 0.61, po.GLOBAL_LOCAL, 0.15)]:
        c = a.Context(0)
        c.set_scoring(M, gi, ge, at)
        sel = np.array([0, 3, 7, 11, 24, 25, 27], np.int64)
        c.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_MASK, delta)
        got = c.near_optimal(sel, delta, 4000)
        O = po.Oracle(M, gi, ge, at)
        for k, p in enumerate(sel):
            q, t = seqs[pq[p]], seqs[pt[p]]
            F, fq, ft = O.fill(q, t, po.FWD, True, fast=False)
            thr = O.threshold(float(F[-1, -1]), delta)
            st, want = O.ucw_enumerate(q, t, F, O.sim(q, t), thr, 4000, fq, ft)
            gst, gthr, alis = got[k]
            assert (gst, gthr, len(alis)) == (st, thr, len(want)), (p, gst, st, len(alis), len(want))
            for (gs, gp), (ws, wp) in zip(alis, want):
                assert gs == ws
                assert_matrix_equal("float pair %d alignment" % p, gp, wp)
        c.close()
    c = a.Context(0)
    c.set_scoring(M, 3, 1, po.LOCAL)             # local alignments: loud refusal
    c.fill_batch(res, off, pq[:2], pt[:2], a.W_FWD | a.W_SCORES, 0.05)
    with pytest.raises(a.AadpError):
        c.near_optimal([0], 0.05, 10)
    c.close()


def test_constrained_near_optimal_enumeration_on_gpu(blosum):
    # aadp_batch_near_optimal_constrained: ConstrainedNearOptimal::enumerate (cw.h:60-284) -- branching only where the
    # SuboptFlag of the template position changes state, optimal predecessors (packed traceback) in between
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(91)
    for gi, ge, at, delta in [(3, 1, po.SEMI_LOCAL, 0.2), (12, 1, po.GLOBAL, 0.15), (4.73, 0.34, po.GLOBAL_LOCAL, 0.2)]:
        seqs = []
        for k in range(16):
            L = int(rng.integers(8, 60))
            s = rng.integers(0, 20, L).astype(np.uint8)
            m = s.copy()
            m[::4] = rng.integers(0, 20, len(m[::4]))
            seqs += [s, np.concatenate([m[: L // 2], m[L // 2 + int(rng.integers(0, 3)):]])]
        seqs += [rng.integers(0, 20, L).astype(np.uint8) for L in (0, 1, 520)]
        res, off = a.Context.pack(seqs)
        pq = np.array(list(range(0, 32, 2)) + [32, 33, 34, 5], np.int32)
        pt = np.array(list(range(1, 32, 2)) + [3, 33, 7, 34], np.int32)
        c = a.Context(0)
        c.set_scoring(M, gi, ge, at)
        c.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB | a.W_MASK, delta)
        ids = np.arange(len(pq))
        O = po.Oracle(M, gi, ge, at)
        total = 0
        for mode in ("all", "stripes", "random"):
            flags = []
            for p in ids:
                n = len(seqs[pt[p]]) + 2
                flags.append({"all": np.ones(n, np.uint8), "stripes": ((np.arange(n) // 4) % 2).astype(np.uint8),
                              "random": rng.integers(0, 2, n).astype(np.uint8)}[mode])
            got = c.near_optimal(ids, delta, 3000, subopt_flags=None if mode == "all" else flags, constrained=True)
            for k, p in enumerate(ids):
                q, t = seqs[pq[p]], seqs[pt[p]]
                F, fq, ft = O.fill(q, t, po.FWD, True, fast=(gi != 4.73))
                thr = O.threshold(float(F[-1, -1]), delta)
                st, want = O.cno_enumerate(q, t, F, O.sim(q, t), thr, fq, ft, flags[k], 3000)
                gst, gthr, alis = got[k]
                assert (gst, gthr, len(alis)) == (st, thr, len(want)), (mode, p, gst, st, len(alis), len(want))
                total += len(alis)
                for (gs, gp), (ws, wp) in zip(alis, want):
                    assert gs == ws
                    assert_matrix_equal("%s pair %d alignment" % (mode, p), gp, wp)
        assert total > 3 * len(ids)
        c.close()


def test_record_and_pruned_general_gap_kernels_change_nothing(blosum):
    # Three implementations of the exact fp32 fill must agree on every output, and with the oracle's literal scan:
    # the record-list kernel (aadp_frec.cuh, default), the pruned scans ("general_records" 0: prefix-maximum bound +
    # binary search) and the literal scans ("general_prune" 0 as well).  All align types incl. local, both directions,
    # whole matrices (short, wider than 512 columns, related pairs), sub-rectangles, and the batch scalars.
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(55)
    for gi, ge, at in [(4.73, 0.34, po.SEMI_LOCAL), (4.73, 0.34, po.LOCAL), (2.17, 0.61, po.GLOBAL), (0.9, 0.0, po.GLOBAL_LOCAL),
                       (12, 1, po.LOCAL_GLOBAL)]:
        cr, cp, cn = a.Context(0), a.Context(0), a.Context(0)
        for c, rec, prune in ((cr, 1, 1), (cp, 0, 1), (cn, 0, 0)):
            c.set_option("general_records", rec)
            c.set_option("general_prune", prune)
            c.set_option("exact_float", 1)
            c.set_scoring(M, gi, ge, at)
        O = po.Oracle(M, gi, ge, at)
        for Lq, Lt in [(2, 2), (3, 40), (61, 5), (1, 77), (97, 130), (150, 620), (333, 31), (300, 300), (40, 1500), (70, 2048), (4, 1), (1, 1), (33, 2), (2, 65)]:
            q, t = rand_pair(rng, Lq, Lt)
            if Lq == 97:
                t[:90] = q[:90]          # a related pair: the pruning bites hardest there
            if Lq == 300:
                t[10:290] = q[5:285]     # a related pair with mutations: groups of noise-tied leaders
                t[20:280:5] = rng.integers(0, 20, len(t[20:280:5]))
            y = cn.fill_pair(q, t, a.BOTH, delta_ratio=0.03)
            for tag, c in (("record", cr), ("prune", cp)):
                x = c.fill_pair(q, t, a.BOTH, delta_ratio=0.03)
                for key in x:
                    if x[key] is not None and key != "threshold":
                        assert_matrix_equal("%s %s" % (tag, key), x[key], y[key])
                assert x["threshold"] == y["threshold"]
            if Lq * Lt < 20000:
                for d, tag in ((po.FWD, "fwd"), (po.REV, "rev")):
                    ws, wq, wt = O.fill(q, t, d, True, fast=False)
                    assert_matrix_equal("oracle score", y["score_" + tag], ws)
                    assert_matrix_equal("oracle pq", y["prevq_" + tag], wq)
                    assert_matrix_equal("oracle pt", y["prevt_" + tag], wt)
            rect = (1, 0, Lq, Lt + 1) if Lq > 2 else (0, 0, Lq + 1, Lt + 1)
            for d in (a.FWD, a.REV):
                want = cn.fill_subpair(q, t, rect, d)
                for c in (cr, cp):
                    for u, v in zip(c.fill_subpair(q, t, rect, d), want):
                        assert_matrix_equal("sub-rectangle", u, v)
        seqs = [rng.integers(0, 20, int(L)).astype(np.uint8) for L in rng.integers(1, 200, 40)]
        res, off = a.Context.pack(seqs)
        pq, pt = rng.integers(0, 40, 300).astype(np.int32), rng.integers(0, 40, 300).astype(np.int32)
        what = a.W_FWD | a.W_REV | (0 if at == po.LOCAL else a.W_MASK)
        o2 = cn.fill_batch(res, off, pq, pt, what, 0.02)
        for c in (cr, cp):
            o1 = c.fill_batch(res, off, pq, pt, what, 0.02)
            for key in o1:
                if o1[key] is not None:
                    assert_matrix_equal("batch %s" % key, o1[key], o2[key])
        if at == po.SEMI_LOCAL:
            # the benchmark shape of the float-default line (bench.py --workload c3f): C3-shaped pairs, random and related
            from alignment_algos_b200 import synth
            sq, bq, bt = synth.pair_workload(1003, 384, 100, 500)
            sq = list(sq)
            for p in range(0, 384, 3):  # every third template becomes a mutated, shifted copy of its query
                qv = sq[bq[p]]
                tv = np.roll(qv.copy(), 3)
                idx = rng.integers(0, len(tv), len(tv) // 4)
                tv[idx] = rng.integers(0, 20, len(idx))
                sq[bt[p]] = tv
            r2, o2f = a.Context.pack(sq)
            w2 = a.W_FWD | a.W_REV | a.W_MASK
            want = cp.fill_batch(r2, o2f, bq, bt, w2, 0.01)
            got = cr.fill_batch(r2, o2f, bq, bt, w2, 0.01)
            for key in got:
                if got[key] is not None:
                    assert_matrix_equal("c3f batch %s" % key, got[key], want[key])
        for c in (cr, cp, cn):
            c.close()


def test_local_optimal_alignments_of_a_batch_on_gpu(blosum):
    # aadp_batch_optimal_all in LOCAL mode: find_max + enumerate_local (optimal.h:76-124, optimal_rev.h:79-131), one warp
    # per pair over the stored scores and the packed traceback
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(47)
    for gi, ge in [(12, 1), (3, 1), (10.5, 0.25)]:
        seqs = [rng.integers(0, 20, int(L)).astype(np.uint8) for L in rng.integers(1, 160, 60)]
        for k in range(0, 20, 2):      # related pairs: a shared core with different flanks
            core = rng.integers(0, 20, int(rng.integers(10, 60))).astype(np.uint8)
            seqs[k] = np.concatenate([rng.integers(0, 20, 7).astype(np.uint8), core, rng.integers(0, 20, 12).astype(np.uint8)])
            seqs[k + 1] = np.concatenate([rng.integers(0, 20, 15).astype(np.uint8), core, rng.integers(0, 20, 3).astype(np.uint8)])
        seqs += [np.zeros(0, np.uint8), rng.integers(0, 20, 600).astype(np.uint8)]
        res, off = a.Context.pack(seqs)
        pq = np.concatenate([np.arange(0, 20, 2), rng.integers(0, 62, 50)]).astype(np.int32)
        pt = np.concatenate([np.arange(1, 20, 2), rng.integers(0, 62, 50)]).astype(np.int32)
        c = a.Context(0)
        c.set_scoring(M, gi, ge, po.LOCAL)
        c.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB | a.W_SCORES)
        O = po.Oracle(M, gi, ge, po.LOCAL)
        for d, od in ((a.FWD, po.FWD), (a.REV, po.REV)):
            aoff, pairs, n, st = c.optimal_all(d, len(pq))
            for p in range(len(pq)):
                q, t = seqs[pq[p]], seqs[pt[p]]
                S, Q, T = O.fill(q, t, od, True, fast=True)
                orc, opairs, osc = O.optimal(S, Q, T, od)
                assert st[p] == 0 and orc == 0
                assert_matrix_equal("local pair %d dir %d" % (p, d), pairs[aoff[p]:aoff[p] + n[p]], opairs)
                if p % 7 == 0:    # the per-pair entry (host walk over the dense view) agrees
                    rc, hp, hs = c.optimal(p, d, len(q), len(t))
                    assert rc == 0 and hs == osc
                    assert_matrix_equal("local per-pair %d dir %d" % (p, d), hp, opairs)
        c.close()
    # exact-float mode, local: per-pair entry only
    c = a.Context(0)
    c.set_scoring(M, 4.73, 0.34, po.LOCAL)
    c.fill_batch(res, off, pq[:12], pt[:12], a.W_FWD | a.W_REV)
    O = po.Oracle(M, 4.73, 0.34, po.LOCAL)
    for p in range(12):
        q, t = seqs[pq[p]], seqs[pt[p]]
        for d, od in ((a.FWD, po.FWD), (a.REV, po.REV)):
            S, Q, T = O.fill(q, t, od, True, fast=False)
            orc, opairs, osc = O.optimal(S, Q, T, od)
            rc, hp, hs = c.optimal(p, d, len(q), len(t))
            assert rc == 0 and hs == osc
            assert_matrix_equal("float local per-pair %d dir %d" % (p, d), hp, opairs)
    c.close()


def test_batch_of_tabulated_pairs(golden_tab):
    # aadp_fill_batch_tabulated: many pairs with position-dependent gap tables in one call; golden = the real reference
    # fill driven by a table-backed Evaluator; optimal alignments = Optimal::enumerate over the reference matrices
    import alignment_algos_b200 as a
    g = golden_tab
    c = a.Context(0)
    for local in (0, 1):
        names = [n for n in golden_cases(g) if int(g[n + ".local"]) == local]
        sims, dels, inss = [g[n + ".sim"] for n in names], [g[n + ".del"] for n in names], [g[n + ".ins"] for n in names]
        c.set_option("general_budget_mcells", 1)     # several chunks
        fs, rs, aoff, pairs, n_out, st = c.fill_batch_tabulated(sims, dels, inss, bool(local), a.BOTH)
        c.set_option("general_budget_mcells", 400)
        fs2, rs2, _, pairs2, n2, st2 = c.fill_batch_tabulated(sims, dels, inss, bool(local), a.BOTH)
        assert_matrix_equal("chunked fwd", fs, fs2)
        assert_matrix_equal("chunked rev", rs, rs2)
        for k, n in enumerate(names):
            F = g[n + ".fwd.score"]
            assert fs[k] == F[-1, -1], n
            assert rs[k] == g[n + ".rev.score"][0, 0], n
            if not local:
                wst, wpairs, _ = subali_walk(F, g[n + ".fwd.pq"], g[n + ".fwd.pt"], (0, 0, F.shape[0] - 1, F.shape[1] - 1))
                assert st[k] == wst, n
                assert aoff[k + 1] - aoff[k] == F.shape[0]
                assert_matrix_equal(n + " optimal", pairs[aoff[k]:aoff[k] + n_out[k]], wpairs)
                assert_matrix_equal(n + " chunked optimal", pairs2[aoff[k]:aoff[k] + n2[k]], wpairs)
    # random larger items against the oracle, forward only
    rng = np.random.default_rng(77)
    items = [po.hmap_like_tables(rng, int(rng.integers(20, 140)), int(rng.integers(20, 140)), po.SEMI_LOCAL) for _ in range(40)]
    fs, rs, aoff, pairs, n_out, st = c.fill_batch_tabulated([x[0] for x in items], [x[1] for x in items], [x[2] for x in items],
                                                            False, a.FWD)
    assert rs is None
    for k in range(0, 40, 3):
        sim, dt, it = items[k]
        F, fq, ft = po.Oracle.fill_tab(sim, dt, it, False, po.FWD)
        wst, wpairs, _ = subali_walk(F, fq, ft, (0, 0, F.shape[0] - 1, F.shape[1] - 1))
        assert fs[k] == F[-1, -1] and st[k] == wst
        assert_matrix_equal("random item %d optimal" % k, pairs[aoff[k]:aoff[k] + n_out[k]], wpairs)
    z = c.fill_batch_tabulated([], [], [], False, a.BOTH)
    assert len(z[0]) == 0
    c.close()


def test_general_entry_with_similarity_matrix(blosum):
    # aadp_fill_pair_general: the fill from a host-built similarity matrix (any Evaluator) + affine gaps
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(77)
    c = a.Context(0)   # no aadp_set_scoring needed
    for gi, ge, at in [(12, 1, po.SEMI_LOCAL), (4.73, 0.34, po.GLOBAL), (2.5, 0.5, po.LOCAL), (7, 0.3, po.LOCAL_GLOBAL)]:
        O = po.Oracle(M, gi, ge, at)
        for Lq, Lt in [(0, 3), (1, 1), (17, 40), (90, 61)]:
            q, t = rand_pair(rng, Lq, Lt)
            sim = O.sim(q, t)
            for d, od in ((a.FWD, po.FWD), (a.REV, po.REV)):
                s, pq, pt = c.fill_pair_general(sim, gi, ge, at, d)
                ws, wq, wt = O.fill(q, t, od, True, fast=False)
                assert_matrix_equal("general score", s, ws)
                assert_matrix_equal("general pq", pq, wq)
                assert_matrix_equal("general pt", pt, wt)
    # a similarity matrix no substitution table could produce (position specific, like a profile evaluator):
    # symmetry check against the transposed problem with swapped free-end roles
    sim = rng.normal(0, 3, (42, 37)).astype(np.float32)
    sim[0, :] = sim[-1, :] = 0
    sim[:, 0] = sim[:, -1] = 0
    s1, _, _ = c.fill_pair_general(sim, 4.73, 0.34, po.GLOBAL, a.FWD)
    s2, _, _ = c.fill_pair_general(np.ascontiguousarray(sim.T), 4.73, 0.34, po.GLOBAL, a.FWD)
    assert s1[-1, -1] == s2[-1, -1]
    c.close()


def test_pipelined_fill_batch_equals_plain_path(blosum):
    # aadp_fill_batch pipelines large batches (residues in pieces on a copy stream, task list in chunks, forward
    # kernel of chunk k while the host schedules chunk k+1).  Same batch through the plain path (one chunk) and the
    # resident upload+run path must give identical scalars, matrices and alignments; the batch mixes packed pairs with
    # int32-path pairs (templates > 512) and shuffled pair order (chunks reference every residue piece).
    import alignment_algos_b200 as a
    import torch
    from alignment_algos_b200 import synth
    _, M = blosum
    rng = np.random.default_rng(99)
    seqs = synth.random_seqs(rng, 70000, 20, 90) + [rng.integers(0, 20, L).astype(np.uint8) for L in (530, 700, 0, 1)]
    n = 36000
    pq = rng.integers(0, 70000, n).astype(np.int32)
    pt = rng.integers(0, 70000, n).astype(np.int32)
    pt[::3000] = 70000 + (np.arange(len(pt[::3000])) % 4)   # int32-path / degenerate templates sprinkled in
    res, off = a.Context.pack(seqs)
    what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK | a.W_SCORES
    outs = []
    for chunks in (1, 2, 3):
        c = a.Context(0)
        c.set_option("pipeline_chunks", chunks)
        c.set_scoring(M, 12, 1, po.SEMI_LOCAL)
        out = c.fill_batch(res, off, pq, pt, what, 0.02)
        samp = [0, 1, 2999, 3000, 17777, n - 1]
        det = [c.fetch_pair(p, len(seqs[pq[p]]), len(seqs[pt[p]]), fwd=True, rev=True, mask=True) for p in samp]
        ali = [c.optimal(p, a.FWD, len(seqs[pq[p]]), len(seqs[pt[p]])) for p in samp]
        outs.append((out, det, ali))
        if chunks == 2:   # the resident path on the same context
            df = torch.zeros(n, dtype=torch.float32, device="cuda")
            c.upload_batch(res, off, pq, pt, what)
            c.run_batch(what, 0.02, d_fwd=df.data_ptr())
            c.synchronize()
            assert_matrix_equal("resident fwd", df.cpu().numpy(), out["fwd_score"])
        c.close()
    O = po.Oracle(M, 12, 1, po.SEMI_LOCAL)
    for p in (0, 3000, 6000, 17777):
        assert outs[0][0]["fwd_score"][p] == O.fill(seqs[pq[p]], seqs[pt[p]], po.FWD, fast=True)[0][-1, -1]
    for k in (1, 2):
        for key in ("fwd_score", "rev_score", "threshold", "nearopt_count"):
            assert_matrix_equal("chunks %s" % key, outs[k][0][key], outs[0][0][key])
        for d0, d1 in zip(outs[0][1], outs[k][1]):
            for key in d0:
                if d0[key] is not None:
                    assert_matrix_equal("chunks fetch " + key, d1[key], d0[key])
        for a0, a1 in zip(outs[0][2], outs[k][2]):
            assert a0[0] == a1[0] and a0[2] == a1[2]
            assert_matrix_equal("chunks alignment", a1[1], a0[1])
    # loud failure on a residue outside the alphabet, also on the pipelined path
    bad = res.copy()
    bad[len(bad) // 2] = 77
    c = a.Context(0)
    c.set_scoring(M, 12, 1, po.SEMI_LOCAL)
    with pytest.raises(a.AadpError):
        c.fill_batch(bad, off, pq, pt, what, 0.02)
    out = c.fill_batch(res, off, pq, pt, a.W_FWD)   # the context is still usable
    assert_matrix_equal("after error", out["fwd_score"], outs[0][0]["fwd_score"])
    c.close()


def test_enumeration_user_limit_truncation_on_gpu(blosum):
    # ucw.h:72,115-126 / cw.h:76,118-130: once `user_limit` alignments are complete the reference stops branching and
    # completes every pending branch along the optimal predecessors.  The oracle's truncation is pinned to the live
    # reference at its hard-coded limit (tests/test_oracle.py); the GPU walk must give the oracle's set -- same slot
    # order, same fp32 scores -- for small limits, for the constrained variant, and at the reference's own 100000.
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(21)
    L = 26
    q = rng.integers(0, 20, L).astype(np.uint8)
    t = q.copy()
    t[::3] = rng.integers(0, 20, len(t[::3]))
    res, off = a.Context.pack([q, t])
    c = a.Context(0)
    c.set_scoring(M, 3, 1, po.SEMI_LOCAL)
    O = po.Oracle(M, 3, 1, po.SEMI_LOCAL)
    F, fq, ft = O.fill(q, t, po.FWD, True, fast=False)
    sim = O.sim(q, t)
    c.fill_batch(res, off, np.array([0], np.int32), np.array([1], np.int32), a.W_FWD | a.W_SCORES | a.W_TB, 0.5)
    flags = (np.arange(L + 2) // 4) % 2
    for delta, limit, K, constrained in [(0.3, 50, 4000, False), (0.3, 1, 4000, False), (0.35, 700, 20000, False),
                                         (0.4, 300, 20000, True), (0.5, 100000, 120000, False)]:
        thr = O.threshold(float(F[-1, -1]), delta)
        c.set_option("cw_user_limit" if constrained else "ucw_user_limit", limit)
        if constrained:
            st, want = O.cno_enumerate(q, t, F, sim, thr, fq, ft, flags, K, user_limit=limit)
            gst, gthr, alis = c.near_optimal([0], delta, K, subopt_flags=[flags], constrained=True)[0]
        else:
            st, want = O.ucw_enumerate(q, t, F, sim, thr, K, fq, ft, user_limit=limit)
            gst, gthr, alis = c.near_optimal([0], delta, K)[0]
        assert st == 0 and gst == 0 and gthr == thr
        assert len(want) > limit, "the case must cross the limit"
        assert len(alis) == len(want), (delta, limit, len(alis), len(want))
        for (gs, gp), (ws, wp) in zip(alis, want):
            assert gs == ws and np.array_equal(gp, wp)
        # and the limit matters: without it the set is larger
        if limit < 1000:
            c.set_option("cw_user_limit" if constrained else "ucw_user_limit", 0)
            full = c.near_optimal([0], delta, K, **({"subopt_flags": [flags], "constrained": True} if constrained else {}))[0]
            assert len(full[2]) > len(alis) or full[0] == 1
    c.close()


def test_long_pair_wavefront_8000_full_parity(blosum):
    # the multi-CTA wavefront at a size where the stripe hand-off is live for thousands of rows (32 stripes per
    # direction): scores, BOTH traceback matrices and the near-optimal set against the oracle's O(mn) fill, cell by cell
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(1005)
    Lq, Lt = 8000, 8050
    q, t = rand_pair(rng, Lq, Lt)
    t[1000:5000] = q[900:4900]          # a related stretch: a real optimum away from the borders
    t[1500:4800:7] = rng.integers(0, 20, len(t[1500:4800:7]))
    c = a.Context(0)
    try:
        for at in (po.SEMI_LOCAL, po.GLOBAL):
            c.set_scoring(M, 12, 1, at)
            O = po.Oracle(M, 12, 1, at)
            out = c.fill_pair(q, t, a.BOTH, delta_ratio=0.01)
            F, fq, ft = O.fill(q, t, po.FWD, True, fast=True)
            assert_matrix_equal("F", out["score_fwd"], F)
            assert_matrix_equal("fq", out["prevq_fwd"], fq)
            assert_matrix_equal("ft", out["prevt_fwd"], ft)
            del fq, ft
            R, rq, rt = O.fill(q, t, po.REV, True, fast=True)
            assert_matrix_equal("R", out["score_rev"], R)
            assert_matrix_equal("rq", out["prevq_rev"], rq)
            assert_matrix_equal("rt", out["prevt_rev"], rt)
            del rq, rt
            thr = O.threshold(float(F[-1, -1]), 0.01)
            mask, _ = O.nearopt_mask(F, R, O.sim(q, t), thr)
            assert out["threshold"] == thr
            assert_matrix_equal("nearopt", out["nearopt"], mask)
            del out, F, R, mask
    finally:
        c.close()


def test_long_pair_wavefront_30000_properties(blosum):
    # BASELINE.json configs[4] at full size (the oracle would need 11 GB per matrix): size-independent properties --
    # forward optimum == reverse optimum, both optimal alignments are valid paths whose rescoring gives the optimum,
    # and the near-optimal set contains every cell of the optimal alignment
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(1005)
    L = 30000
    seqs = [rng.integers(0, 20, L).astype(np.uint8) for _ in range(2)]
    res, off = a.Context.pack(seqs)
    c = a.Context(0)
    try:
        c.set_scoring(M, 12, 1, po.SEMI_LOCAL)
        out = c.fill_batch(res, off, np.array([0], np.int32), np.array([1], np.int32),
                           a.W_FWD | a.W_REV | a.W_TB | a.W_MASK, 0.01)
        assert out["fwd_score"][0] == out["rev_score"][0]
        opt = float(out["fwd_score"][0])
        for d in (a.FWD, a.REV):
            rc, pairs, sc = c.optimal(0, d, L, L)
            assert rc == 0 and sc == opt
            assert tuple(pairs[0]) == (0, 0) and tuple(pairs[-1]) == (L + 1, L + 1)
            assert np.all(np.diff(pairs[:, 0]) >= 1) and np.all(np.diff(pairs[:, 1]) >= 1)
            assert _rescore(None, seqs[0], seqs[1], [tuple(p) for p in pairs], M, 12.0, 1.0, po.SEMI_LOCAL) == opt
        assert out["nearopt_count"][0] >= len(pairs) - 2
    finally:
        c.close()


def test_fill_batch_submit_wait_equals_fill_batch(blosum):
    # aadp_fill_batch_submit / aadp_fill_batch_wait: the same results as the blocking call, two contexts driven by one
    # thread with batches in flight on both; an invalid residue is reported by wait (packed-only batch) or by submit
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    _, M = blosum
    seqs, pq, pt = synth.pair_workload(91, 40000, 60, 300)   # >= 32768 pairs: the pipelined path
    res, off = a.Context.pack(seqs)
    what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK
    cs = [a.Context(0), a.Context(0)]
    for c in cs:
        c.set_scoring(M, 12, 1, po.SEMI_LOCAL)
    want = cs[0].fill_batch(res, off, pq, pt, what, 0.01)
    outs = [None, None]
    for it in range(4):
        k = it % 2
        if outs[k] is not None:
            got = cs[k].fill_batch_wait()
            for key in want:
                assert_matrix_equal("async %s" % key, got[key], want[key])
        outs[k] = cs[k].fill_batch_submit(res, off, pq, pt, what, 0.01)
    with pytest.raises(a.AadpError):  # a second submit before the wait
        cs[0].fill_batch_submit(res, off, pq, pt, what, 0.01)
    for k in range(2):
        got = cs[k].fill_batch_wait()
        for key in want:
            assert_matrix_equal("async %s" % key, got[key], want[key])
    # the resident products of a waited batch serve the usual follow-up calls
    rc, pairs, sc = cs[1].optimal(5, a.FWD, len(seqs[pq[5]]), len(seqs[pt[5]]))
    assert rc == 0 and sc == want["fwd_score"][5]
    bad = res.copy()
    bad[off[pq[7]]] = 77
    cs[0].fill_batch_submit(bad, off, pq, pt, what, 0.01)
    with pytest.raises(a.AadpError):
        cs[0].fill_batch_wait()
    for c in cs:
        c.close()


def test_float_mode_optimal_alignments_of_a_whole_batch(blosum):
    # aadp_batch_optimal_all[_compact] under the reference's default penalties (exact-float mode: no resident traceback):
    # chunked dense fills with predecessors + one walk per pair; equal to the per-pair call and to the oracle's
    # Optimal::enumerate over the literal fill
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(8)
    seqs = [rng.integers(0, 20, int(L)).astype(np.uint8) for L in rng.integers(1, 160, 60)]
    seqs[3] = seqs[2][:100].copy()
    res, off = a.Context.pack(seqs)
    pq, pt = rng.integers(0, 60, 400).astype(np.int32), rng.integers(0, 60, 400).astype(np.int32)
    pq[0], pt[0] = 2, 3
    for at in (po.SEMI_LOCAL, po.GLOBAL):
        c = a.Context(0)
        c.set_option("general_budget_mcells", 4)   # several chunks
        c.set_scoring(M, 4.73, 0.34, at)
        O = po.Oracle(M, 4.73, 0.34, at)
        out = c.fill_batch(res, off, pq, pt, a.W_FWD)
        aoff, pairs, n, st = c.optimal_all(a.FWD, len(pq))
        coff, cpairs, cn, cst = c.optimal_all_compact(a.FWD, len(pq))
        assert (st == 0).all() and (cst == 0).all() and np.array_equal(n, cn)
        for p in range(len(pq)):
            got = pairs[aoff[p]:aoff[p] + n[p]]
            assert_matrix_equal("compact", cpairs[coff[p]:coff[p + 1]], got)
            if p % 16 == 0:
                q, t = seqs[pq[p]], seqs[pt[p]]
                rc, one, sc = c.optimal(p, a.FWD, len(q), len(t))
                assert rc == 0 and sc == out["fwd_score"][p]
                assert_matrix_equal("per-pair call", got, one)
                F, fq, ft = O.fill(q, t, po.FWD, True, fast=False)
                orc, opairs, osc = O.optimal(F, fq, ft, po.FWD)
                assert orc == 0 and osc == sc
                assert_matrix_equal("oracle", got, opairs)
        with pytest.raises(a.AadpError):
            c.optimal_all(a.REV, len(pq))
        c.close()


def test_enumeration_with_and_without_mask_pruned_scans(blosum):
    # option "enum_mask_prune" (default 1): with the near-optimal set of the same delta resident, the deletion scans of
    # the enumeration kernel only test the cells of the set.  Every alignment, score and slot must be what the unpruned
    # scans give (UCW and the constrained variant, wide and narrow delta, pairs with several thousand near-optimal cells),
    # and a delta that differs from the resident set's must not be pruned with it.
    import alignment_algos_b200 as a
    _, M = blosum
    rng = np.random.default_rng(21)
    seqs, pq, pt = [], [], []
    for k in range(160):
        L = int(rng.integers(40, 420))
        sq = rng.integers(0, 20, L).astype(np.uint8)
        m = sq.copy()
        m[::5] = rng.integers(0, 20, len(m[::5]))
        cut = int(rng.integers(5, L - 5))
        m = np.concatenate([m[:cut], m[cut + int(rng.integers(0, 5)):]])
        seqs += [sq, m]
        pq.append(2 * k)
        pt.append(2 * k + 1)
    pq, pt = np.array(pq, np.int32), np.array(pt, np.int32)
    res, off = a.Context.pack(seqs)
    ids = np.arange(len(pq), dtype=np.int64)
    what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK

    def same(x, y):
        return all(u[0] == v[0] and u[1] == v[1] and len(u[2]) == len(v[2]) and
                   all(s1 == s2 and np.array_equal(p1, p2) for (s1, p1), (s2, p2) in zip(u[2], v[2])) for u, v in zip(x, y))

    for at in (po.SEMI_LOCAL, po.GLOBAL):
        c = a.Context(0)
        c.set_scoring(M, 12, 1, at)
        for delta in (0.01, 0.05):
            c.fill_batch(res, off, pq, pt, what, delta)
            flags = [(rng.random(len(seqs[t]) + 2) < 0.7).astype(np.uint8) for t in pt]
            got = {}
            for prune in (1, 0):
                c.set_option("enum_mask_prune", prune)
                got[prune] = (c.near_optimal(ids, delta, 48), c.near_optimal(ids, delta, 48, subopt_flags=flags, constrained=True),
                              c.near_optimal(ids[:40], delta * 2, 48))   # another delta than the resident set's
            assert sum(len(g[2]) for g in got[1][0]) > 2 * len(ids)
            for k in range(3):
                assert same(got[1][k], got[0][k]), (at, delta, k)
        c.close()
