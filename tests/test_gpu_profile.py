"""Position-specific template profiles on the integer kernels (aadp_set_profile_scoring; run with -m gpu on a B200).

1. Identity profiles (prof[t][j-1, a] = sub[a, t_j]) must reproduce the substitution scoring bit for bit in every
   product -- scores, predecessors, thresholds, near-optimal sets, optimal alignments, cross scores, enumerations -- on
   every kernel path.  The substitution path is pinned to the reference, so this pins every profile lookup.
2. Random position-specific profiles against the oracle's table-driven fill (tests/test_profile_scoring.py checks that
   construction) and against the exact fp32 kernel aadp_fill_pair_general over the same similarity matrix.
3. The limits of the grid rule and the per-template packed bound; 4. validation and refusals.
Every sequence holds both end codes and every matrix is asymmetric, so a query/template swap in a lookup shows."""
import numpy as np
import pytest

from util import po, MODES, MODE_NAMES, assert_matrix_equal
from test_scoring_space import asym_matrix, seq, low_entropy_seq
from test_profile_scoring import identity_profile, profile_sim, affine_tables, profile_fill, random_profile

pytestmark = pytest.mark.gpu

MODE_IDS = [MODE_NAMES[m] for m in MODES]
ALL = 1 | 2 | 4 | 8 | 16  # W_FWD | W_REV | W_TB | W_SCORES | W_MASK
PRUNE_KSORTED, PRUNE_REDUNDANCY = 2, 3  # include/aadp.h


def new_ctx(**options):
    import alignment_algos_b200 as a
    c = a.Context(0)
    for k, v in options.items():
        c.set_option(k, v)
    return c


def kernels(c, fn):
    c.set_profiling(True)
    try:
        out = fn()
        names = [n for n, _, _ in c.profile()]
    finally:
        c.set_profiling(False)
    return out, names


def has(names, prefix, pro):
    return any(n.startswith(prefix) and ("PRO=1" in n) == pro for n in names)


def pairs_of(rng, lens, A, low_entropy=False):
    """Query 2k and template 2k+1 for each (Lq, Lt)."""
    mk = (lambda L: low_entropy_seq(rng, L, A)) if low_entropy else (lambda L: seq(rng, L, A))
    seqs = []
    for Lq, Lt in lens:
        seqs += [mk(Lq), mk(Lt)]
    pq = np.arange(0, len(seqs), 2, dtype=np.int32)
    return seqs, pq, pq + 1


def identity_profiles(sub, seqs, templates):
    return [identity_profile(sub, s) if k in templates else None for k, s in enumerate(seqs)]


def same(tag, x, y):
    if isinstance(x, dict):
        assert x.keys() == y.keys(), tag
        for k in x:
            same(tag + "." + k, x[k], y[k])
    elif isinstance(x, (list, tuple)):
        assert len(x) == len(y), tag
        for i, (u, v) in enumerate(zip(x, y)):
            same("%s[%d]" % (tag, i), u, v)
    elif isinstance(x, np.ndarray) or isinstance(y, np.ndarray):
        assert_matrix_equal(tag, x, y)
    else:
        assert x == y, "%s: %r vs %r" % (tag, x, y)


def products(c, seqs, pq, pt, what, dr, at, enum=True):
    """Everything a resident batch answers, as plain data."""
    import alignment_algos_b200 as a
    res, off = a.Context.pack(seqs)
    out = {"batch": c.fill_batch(res, off, pq, pt, what, dr)}
    for p in range(len(pq)):
        Lq, Lt = len(seqs[pq[p]]), len(seqs[pt[p]])
        out["pair%d" % p] = c.fetch_pair(p, Lq, Lt, fwd=True, rev=True, tb=True, scores=True, mask=bool(what & 16))
    for d, nm in ((a.FWD, "opt_fwd"), (a.REV, "opt_rev")):
        # only the first n[p] rows of slot p are written
        off, pairs, n, st = c.optimal_all(d, len(pq))
        out[nm] = (off, [pairs[off[p]:off[p] + n[p]] for p in range(len(pq))], n, st)
    off, pairs, n, st = c.optimal_all_compact(a.FWD, len(pq))
    out["opt_compact"] = (off, pairs[:off[-1]], n, st)
    out["opt0"] = c.optimal(0, a.FWD, len(seqs[pq[0]]), len(seqs[pt[0]]))
    # the fetched traceback of pair 0, decoded cell by cell (the bits of the int32 kernels' pad columns beyond Lt are
    # never read and may differ)
    Lq0, Lt0 = len(seqs[pq[0]]), len(seqs[pt[0]])
    for d in (a.FWD, a.REV):
        tb, fin = c.fetch_tb(0, d, Lq0, Lt0)
        out["tb0_%d" % d] = (fin, [c.decode_cell(tb, fin, Lq0, Lt0, d, i, j) for i in range(1, Lq0 + 1) for j in range(1, Lt0 + 1)])
    if enum and at != po.LOCAL:
        small = [p for p in range(len(pq)) if len(seqs[pq[p]]) * len(seqs[pt[p]]) <= 400]
        if small:
            out["ucw"] = c.near_optimal(small, 0.02, 500)
            out["cno"] = c.near_optimal(small, 0.02, 500, constrained=True)
            p = small[0]
            for v in (PRUNE_KSORTED, PRUNE_REDUNDANCY):
                out["pruned%d" % v] = c.near_optimal_pruned(p, v, 0.02, len(seqs[pq[p]]), len(seqs[pt[p]]), max_alignments=500)
    return out


# ---- 1. identity profiles: bit-identical to the substitution scoring on every path ----

# name: (align type, options, pair lengths, what, kernel prefixes that must run)
PATHS = {
    "packed": (po.SEMI_LOCAL, {}, [(12, 14), (1, 1), (0, 9), (40, 16), (17, 33), (100, 512), (9, 12)], ALL, ["packed_kernel"]),
    "packed_global": (po.GLOBAL, {}, [(11, 15), (33, 31), (64, 200), (5, 1)], ALL, ["packed_kernel"]),
    "packed_local": (po.LOCAL, {}, [(12, 14), (40, 70), (1, 1), (200, 90)], 1 | 2 | 4 | 8, ["packed_kernel<TB=1,FST=1,MSK=0,LOC=1"]),
    "int32_k8_k16": (po.GLOBAL_LOCAL, {"packed": 0}, [(12, 14), (30, 256), (45, 257), (9, 600)], ALL,
                     ["fill_kernel<K=8", "fill_kernel<K=16", "mask_kernel"]),
    "int32_local": (po.LOCAL, {}, [(12, 14), (30, 700)], ALL, ["fill_kernel<K=16", "mask_kernel"]),
    "wave": (po.LOCAL_GLOBAL, {"wave_min_cells": 1}, [(12, 14), (40, 520), (300, 1100)], ALL, ["wave_kernel", "mask_kernel"]),
}


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("A", [1, 20, 33, 64])
def test_identity_profiles_match_substitution_scoring(A, path):
    import alignment_algos_b200 as a
    at, opts, lens, what, expect = PATHS[path]
    sub = asym_matrix(A, 500 + A)
    gi, ge = 6.0, 2.0
    rng = np.random.default_rng(1000 + 7 * A)
    seqs, pq, pt = pairs_of(rng, lens, A)
    res = {}
    for mode in ("sub", "pro"):
        c = new_ctx(**opts)
        try:
            if mode == "sub":
                c.set_scoring(sub, gi, ge, at)
            else:
                c.set_profile_scoring(identity_profiles(sub, seqs, set(pt.tolist())), gi, ge, at)
            out, names = kernels(c, lambda: products(c, seqs, pq, pt, what, 0.02, at))
            for pre in expect:
                assert has(names, pre, mode == "pro"), (mode, pre, names)
            # cross mode: the packed XM kernel for short templates, the pair-list path for the rest
            rs, off = a.Context.pack(seqs)
            xs, xn = kernels(c, lambda: c.cross_scores(rs, off, pq, pt))
            out["cross"] = xs
            if at != po.LOCAL and opts.get("packed", 1):
                assert has(xn, "packed_kernel<TB=0,FST=0,MSK=0,XM=1", mode == "pro"), xn
            res[mode] = out
        finally:
            c.close()
    same("A%d %s" % (A, path), res["sub"], res["pro"])


@pytest.mark.parametrize("A", [20, 64])
def test_identity_profiles_int32_score_storage(A):
    # |score| bound above 30000 units: the int32 kernels keep int32 scores (int16 otherwise)
    sub = asym_matrix(A, 77 + A, -60, 60)
    rng = np.random.default_rng(A)
    seqs, pq, pt = pairs_of(rng, [(600, 560), (30, 40)], A)
    res = {}
    for mode in ("sub", "pro"):
        c = new_ctx(packed=0)
        try:
            if mode == "sub":
                c.set_scoring(sub, 6.0, 2.0, po.GLOBAL)
            else:
                c.set_profile_scoring(identity_profiles(sub, seqs, set(pt.tolist())), 6.0, 2.0, po.GLOBAL)
            out, names = kernels(c, lambda: products(c, seqs, pq, pt, ALL, 0.02, po.GLOBAL, enum=False))
            assert has(names, "fill_kernel<K=16,TB=1,ST=2", mode == "pro"), names
            res[mode] = out
        finally:
            c.close()
    same("A%d int32 storage" % A, res["sub"], res["pro"])


# ---- 2. position-specific profiles against the oracle and the exact fp32 kernel ----

@pytest.fixture(scope="module", params=["packed", "int32"])
def ctx(request):
    c = new_ctx(packed=1 if request.param == "packed" else 0)
    c.packed = request.param == "packed"
    yield c
    c.close()


@pytest.fixture(scope="module")
def general():
    # aadp_fill_pair_general replaces the resident batch of its context: a context of its own
    c = new_ctx()
    yield c
    c.close()


KINDS = {"int127": (20, 40.0, 3.0), "grid3": (20, 2.5, 0.375), "ties": (4, 1.0, 1.0)}


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("kind", list(KINDS))
def test_position_specific_profiles_against_oracle(ctx, general, kind, at):
    import alignment_algos_b200 as a
    A, gi, ge = KINDS[kind]
    rng = np.random.default_rng(100 * len(kind) + 10 * at + ord(kind[0]))
    lens = [(9, 11), (14, 12), (1, 7), (7, 1), (0, 5), (5, 0), (33, 47), (120, 90)]
    seqs, pq, pt = pairs_of(rng, lens, A, low_entropy=(kind == "ties"))
    profs = [random_profile(rng, len(s), A, kind) if k % 2 else None for k, s in enumerate(seqs)]
    ctx.set_profile_scoring(profs, gi, ge, at)
    what = ALL if at != po.LOCAL else 1 | 2 | 4 | 8
    res, off = a.Context.pack(seqs)
    out, names = kernels(ctx, lambda: ctx.fill_batch(res, off, pq, pt, what, 0.02))
    assert has(names, "packed_kernel" if ctx.packed else "fill_kernel", True), names
    O = po.Oracle(np.zeros((A, A), np.float32), gi, ge, at)
    for p in range(len(pq)):
        q, prof = seqs[pq[p]], profs[pt[p]]
        tag = "%s at%d pair %d (%dx%d)" % (kind, at, p, len(q), prof.shape[0])
        got = ctx.fetch_pair(p, len(q), prof.shape[0], fwd=True, rev=True, tb=True, scores=True, mask=bool(what & 16))
        mats = {}
        for d, nm in ((po.FWD, "fwd"), (po.REV, "rev")):
            s, pqm, ptm, sim = profile_fill(prof, q, gi, ge, at, d)
            assert_matrix_equal(tag + " score_" + nm, got["score_" + nm], s)
            assert_matrix_equal(tag + " prevq_" + nm, got["prevq_" + nm], pqm)
            assert_matrix_equal(tag + " prevt_" + nm, got["prevt_" + nm], ptm)
            mats[nm] = (s, pqm, ptm)
            # the exact fp32 path over the same similarity matrix (pinned to the reference for any similarity)
            gs, gq, gt = general.fill_pair_general(sim, gi, ge, at, d)
            assert_matrix_equal(tag + " general score_" + nm, got["score_" + nm], gs)
            assert_matrix_equal(tag + " general prevq_" + nm, got["prevq_" + nm], gq)
            assert_matrix_equal(tag + " general prevt_" + nm, got["prevt_" + nm], gt)
        assert out["fwd_score"][p] == mats["fwd"][0][-1, -1], tag
        assert out["rev_score"][p] == mats["rev"][0][0, 0], tag
        if what & 16 and len(q) and prof.shape[0]:
            F, R = mats["fwd"][0], mats["rev"][0]
            thr = O.threshold(float(F[-1, -1]), 0.02)
            mask, n = O.nearopt_mask(F, R, sim, thr)
            assert out["threshold"][p] == thr, tag
            assert out["nearopt_count"][p] == n, tag
            assert_matrix_equal(tag + " nearopt", got["nearopt"], mask)
    if at != po.LOCAL:
        small = [p for p in range(len(pq)) if 0 < len(seqs[pq[p]]) * len(seqs[pt[p]]) <= 200]
        ucw = ctx.near_optimal(small, 0.02, 3000)
        cno = ctx.near_optimal(small, 0.02, 3000, constrained=True)
        for k, p in enumerate(small):
            q, prof = seqs[pq[p]], profs[pt[p]]
            F, PQ, PT, sim = profile_fill(prof, q, gi, ge, at, po.FWD)
            thr = O.threshold(float(F[-1, -1]), 0.02)
            for label, gpu, ref in (("ucw", ucw[k], O.ucw_enumerate(q, np.zeros(prof.shape[0], np.uint8), F, sim, thr, 3000, PQ, PT)),
                                    ("cno", cno[k], O.cno_enumerate(q, np.zeros(prof.shape[0], np.uint8), F, sim, thr, PQ, PT,
                                                                    max_alignments=3000))):
                st, gthr, alis = gpu
                assert gthr == thr and st == ref[0], (label, p)
                assert len(alis) == len(ref[1]), (label, p)
                for (s1, p1), (s2, p2) in zip(alis, ref[1]):
                    assert s1 == s2, (label, p)
                    assert_matrix_equal("%s %s pair %d path" % (label, kind, p), p1, p2)


# ---- 3. limits ----

def test_entry_limit_127_units_and_context_survives_refusal():
    import alignment_algos_b200 as a
    A = 20
    rng = np.random.default_rng(9)
    seqs, pq, pt = pairs_of(rng, [(30, 40), (12, 9)], A)
    profs = [random_profile(rng, len(s), A, "int127") if k % 2 else None for k, s in enumerate(seqs)]
    res, off = a.Context.pack(seqs)
    c = new_ctx()
    try:
        c.set_profile_scoring(profs, 5.0, 1.0, po.GLOBAL)
        want = c.fill_batch(res, off, pq, pt, ALL, 0.02)
        bad = [None if p is None else p.copy() for p in profs]
        bad[3][2, 5] = 128.0
        with pytest.raises(a.AadpError, match="sequence 3.*127"):
            c.set_profile_scoring(bad, 5.0, 1.0, po.GLOBAL)
        # on the grid 2^-1: 63.5 is 127 units (accepted), 64 is 128 units (refused)
        half = [None if p is None else np.clip(p, -63, 63) for p in profs]
        half[1][0, 0], half[1][0, 1] = 63.5, 0.5
        c.set_profile_scoring(half, 5.0, 1.0, po.GLOBAL)
        half[1][0, 0] = 64.0
        with pytest.raises(a.AadpError, match="sequence 1.*128 units of 2\\^-1"):
            c.set_profile_scoring(half, 5.0, 1.0, po.GLOBAL)
        nd = [None if p is None else p.copy() for p in profs]
        nd[1][1, 1] = 0.1
        with pytest.raises(a.AadpError, match="aadp_fill_batch_tabulated"):
            c.set_profile_scoring(nd, 5.0, 1.0, po.GLOBAL)
        with pytest.raises(a.AadpError, match="grid"):
            c.set_profile_scoring(profs, 4.73, 0.34, po.GLOBAL)
        # a refusal leaves the context's scoring as it was
        c.set_profile_scoring(profs, 5.0, 1.0, po.GLOBAL)
        same("after refusals", c.fill_batch(res, off, pq, pt, ALL, 0.02), want)
    finally:
        c.close()


def test_packed_bound_uses_each_templates_own_maximum():
    import alignment_algos_b200 as a
    # bound = min(Lq,Lt)*max|entry| + 2gi + ge*(Lq+Lt) in units, gi = 56, ge = 1:
    #   97 x 97 with max 69 -> 6999 (packed), 84 x 84 with max 80 -> 7000 (int32), 30 x 40 with max 9 (packed)
    A, gi, ge = 20, 56.0, 1.0
    rng = np.random.default_rng(21)
    seqs, pq, pt = pairs_of(rng, [(97, 97), (84, 84), (30, 40)], A)

    def prof(L, mx):
        p = rng.integers(-mx + 1, mx, (L, A)).astype(np.float32)
        p[L // 2, 3] = -mx
        return p
    profs = [None, prof(97, 69), None, prof(84, 80), None, prof(40, 9)]
    assert [97 * 69 + 2 * 56 + 194, 84 * 80 + 2 * 56 + 168] == [6999, 7000]
    c = new_ctx()
    try:
        c.set_profile_scoring(profs, gi, ge, po.GLOBAL)
        res, off = a.Context.pack(seqs)
        out, names = kernels(c, lambda: c.fill_batch(res, off, pq, pt, ALL, 0.02))
        assert has(names, "packed_kernel", True) and has(names, "fill_kernel<K=8", True), names
        for p in range(3):
            q, pr = seqs[pq[p]], profs[pt[p]]
            tb, fin = c.fetch_tb(p, a.FWD, len(q), pr.shape[0])
            assert fin[5] == (0 if p == 1 else 1), (p, list(fin))  # layout class: 0 = int32 kernels, 1 = packed
            got = c.fetch_pair(p, len(q), pr.shape[0], fwd=True, rev=True, tb=True, scores=True, mask=True)
            for d, nm in ((po.FWD, "fwd"), (po.REV, "rev")):
                s, pqm, ptm, _ = profile_fill(pr, q, gi, ge, po.GLOBAL, d)
                assert_matrix_equal("p%d score_%s" % (p, nm), got["score_" + nm], s)
                assert_matrix_equal("p%d prevq_%s" % (p, nm), got["prevq_" + nm], pqm)
                assert_matrix_equal("p%d prevt_%s" % (p, nm), got["prevt_" + nm], ptm)
        # under one substitution matrix of max 80 the 97 x 97 pair (bound 8066) leaves the packed kernels too
        c.set_scoring(asym_matrix(A, 3, -80, 80), gi, ge, po.GLOBAL)
        c.fill_batch(res, off, pq, pt, ALL, 0.02)
        assert [c.fetch_tb(p, a.FWD, len(seqs[pq[p]]), len(seqs[pt[p]]))[1][5] for p in range(3)] == [0, 0, 1]
    finally:
        c.close()


# ---- 4. validation ----

def test_validation_refusals_name_the_sequence():
    import alignment_algos_b200 as a
    A = 20
    rng = np.random.default_rng(4)
    seqs, pq, pt = pairs_of(rng, [(10, 12), (8, 9)], A)
    res, off = a.Context.pack(seqs)
    good = [None, random_profile(rng, 12, A, "grid3"), None, random_profile(rng, 9, A, "grid3")]
    c = new_ctx()
    try:
        wrong = list(good)
        wrong[3] = random_profile(rng, 8, A, "grid3")
        c.set_profile_scoring(wrong, 2.0, 0.5, po.GLOBAL)
        with pytest.raises(a.AadpError, match="sequence 3 has 160 entries.*9 residues"):
            c.fill_batch(res, off, pq, pt, ALL, 0.02)
        missing = list(good)
        missing[1] = None
        c.set_profile_scoring(missing, 2.0, 0.5, po.GLOBAL)
        with pytest.raises(a.AadpError, match="sequence 1 is used as a template.*empty"):
            c.fill_batch(res, off, pq, pt, ALL, 0.02)
        with pytest.raises(a.AadpError, match="sequence 1"):
            c.cross_scores(res, off, [0], [1])
        c.set_profile_scoring(good[:3], 2.0, 0.5, po.GLOBAL)
        with pytest.raises(a.AadpError, match="3 profiles for 4 sequences"):
            c.fill_batch(res, off, pq, pt, ALL, 0.02)
        # query-only sequences may have no profile; a template sequence that is also a query is fine
        c.set_profile_scoring(good, 2.0, 0.5, po.GLOBAL)
        out = c.fill_batch(res, off, np.array([0, 2, 1], np.int32), np.array([1, 3, 1], np.int32), ALL, 0.02)
        for p, (qi, ti) in enumerate([(0, 1), (2, 3), (1, 1)]):
            assert out["fwd_score"][p] == profile_fill(good[ti], seqs[qi], 2.0, 0.5, po.GLOBAL, po.FWD)[0][-1, -1]
        # refused in profile mode: no template id, or exact fp32 kernels only
        with pytest.raises(a.AadpError, match="one-pair batch"):
            c.fill_pair(seqs[0], seqs[1], a.BOTH)
        with pytest.raises(a.AadpError, match="aadp_fill_subpair"):
            c.fill_subpair(seqs[0], seqs[1], (0, 0, 11, 13))
        with pytest.raises(a.AadpError, match="aadp_fill_subpair_batch"):
            c.fill_subpair_batch(res, off, [0], [1], [(0, 0, 11, 13)])
    finally:
        c.close()
    c = new_ctx(exact_float=1)
    try:
        with pytest.raises(a.AadpError, match="exact_float"):
            c.set_profile_scoring(good, 2.0, 0.5, po.GLOBAL)
    finally:
        c.close()


@pytest.mark.parametrize("at", [po.SEMI_LOCAL, po.LOCAL])
def test_switching_back_to_substitution_scoring(at):
    import alignment_algos_b200 as a
    A = 20
    sub = asym_matrix(A, 11)
    rng = np.random.default_rng(5 + at)
    seqs, pq, pt = pairs_of(rng, [(10, 12), (80, 300), (40, 600)], A)
    profs = [random_profile(rng, len(s), A, "int127") if k % 2 else None for k, s in enumerate(seqs)]
    what = ALL if at != po.LOCAL else 1 | 2 | 4 | 8
    fresh = new_ctx()
    c = new_ctx()
    try:
        fresh.set_scoring(sub, 6.0, 2.0, at)
        want = products(fresh, seqs, pq, pt, what, 0.02, at)
        c.set_profile_scoring(profs, 6.0, 2.0, at)
        products(c, seqs, pq, pt, what, 0.02, at)
        c.set_scoring(sub, 6.0, 2.0, at)
        with pytest.raises(a.AadpError, match="no valid resident batch"):
            c.run_batch(what)
        got, names = kernels(c, lambda: products(c, seqs, pq, pt, what, 0.02, at))
        assert not any(",PRO=1" in n for n in names), names
        same("switched back", got, want)
    finally:
        c.close()
        fresh.close()
