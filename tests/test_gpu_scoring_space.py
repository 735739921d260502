"""GPU parity outside BLOSUM62 (run with -m gpu on a B200): asymmetric substitution matrices over 1..64-letter alphabets,
a 2^-8 dyadic grid, tie-heavy and zero-gap scoring, and the scoring limits that choose the kernel (packed int16x2 /
int32 / wavefront / exact float) or the score storage (int16 / int32).  Every comparison is bit-exact against the oracle,
which tests/test_scoring_space.py anchors to an independent float64 dynamic program for these same scorings.

A symmetric matrix hides a query/template swap in any substitution lookup; every matrix here is asymmetric where the
alphabet allows and every sequence holds both end codes 0 and A-1, whose two lookups differ."""
import numpy as np
import pytest

from util import po, MODES, MODE_NAMES, assert_matrix_equal
from test_scoring_space import (ALPHABET_SIZES, SWAPPED_MODE, asym_matrix, extreme_matrix, dyadic_matrix, tie_matrix,
                                seq, low_entropy_seq)

pytestmark = pytest.mark.gpu

PACKED_BOUND = 7000      # kPackedBound (aadp_packed.cuh): |score| bound in grid units below which a pair may be packed
FLOOR16 = -13000         # kFloor16: the packed mask clamps its integer threshold to [FLOOR16, PACKED_BOUND]
MODE_IDS = [MODE_NAMES[m] for m in MODES]


@pytest.fixture(scope="module", params=["packed", "int32"])
def ctx(request):
    # like tests/test_gpu_parity.py: each test runs through the packed kernels (where a pair qualifies) and with the
    # int32 kernels forced
    import alignment_algos_b200 as a
    c = a.Context(0)
    c.set_option("packed", 1 if request.param == "packed" else 0)
    c.packed = request.param == "packed"
    yield c
    c.close()


def new_ctx(**options):
    import alignment_algos_b200 as a
    c = a.Context(0)
    for k, v in options.items():
        c.set_option(k, v)
    return c


def bound(Lq, Lt, sub, gi, ge, s=0):
    """The host's |score| bound of a pair in grid units 2^-s: min(Lq,Lt)*max|sub| + 2gi + ge(Lq+Lt)."""
    m = 1 << s
    return min(Lq, Lt) * int(np.abs(sub).max() * m) + 2 * int(gi * m) + int(ge * m) * (Lq + Lt)


def kernels(c, fn):
    """Run fn() with profiling on; returns (fn's result, names of the kernels it launched)."""
    c.set_profiling(True)
    try:
        out = fn()
        names = [n for n, _, _ in c.profile()]
    finally:
        c.set_profiling(False)
    return out, names


def has(names, prefix):
    return any(n.startswith(prefix) for n in names)


def is_float_path(names):
    return has(names, "frec_fill_kernel") or has(names, "general_fill_kernel")


def check_pair(c, O, q, t, tag, mask_dr=None, fast=True):
    """fill_pair against the oracle: scores and both predecessor matrices in both directions; with mask_dr also the
    threshold and the near-optimal cell set.  Returns the names of the kernels the fill launched."""
    import alignment_algos_b200 as a
    out, names = kernels(c, lambda: c.fill_pair(q, t, a.BOTH, delta_ratio=(mask_dr if mask_dr is not None else -1.0)))
    F = R = None
    for d, nm in ((po.FWD, "fwd"), (po.REV, "rev")):
        s, pq, pt = O.fill(q, t, d, True, fast=fast)
        assert_matrix_equal(tag + " score_" + nm, out["score_" + nm], s)
        assert_matrix_equal(tag + " prevq_" + nm, out["prevq_" + nm], pq)
        assert_matrix_equal(tag + " prevt_" + nm, out["prevt_" + nm], pt)
        F, R = (s, R) if d == po.FWD else (F, s)
    if mask_dr is not None:
        thr = O.threshold(float(F[-1, -1]), mask_dr)
        mask, _ = O.nearopt_mask(F, R, O.sim(q, t), thr)
        assert out["threshold"] == thr, tag
        assert_matrix_equal(tag + " nearopt", out["nearopt"], mask)
    return names


def mask_dr_for(at, q, t, dr=0.05):
    return dr if at != po.LOCAL and len(q) and len(t) else None


# ---- 2a. fill_pair, every mode, every alphabet size, lengths at the lane / bucket / stripe edges ----

LENGTHS = [(0, 0), (0, 17), (16, 0), (1, 1), (1, 513), (513, 1), (15, 256), (16, 255), (17, 257), (255, 16), (256, 511),
           (257, 15), (511, 17), (512, 512), (513, 33)]


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("A", ALPHABET_SIZES)
def test_fill_pair_asymmetric_alphabets(ctx, A, at):
    sub = asym_matrix(A, 1000 + A)
    ctx.set_scoring(sub, 7, 2, at)
    O = po.Oracle(sub, 7, 2, at)
    rng = np.random.default_rng(10 * A + at)
    ran_packed = False
    for Lq, Lt in LENGTHS:
        q, t = seq(rng, Lq, A), seq(rng, Lt, A)
        names = check_pair(ctx, O, q, t, "A%d at%d %dx%d" % (A, at, Lq, Lt), mask_dr_for(at, q, t))
        ran_packed |= has(names, "packed_kernel")
    # the 512x512 pair is within the packed bound for every one of these matrices
    assert ran_packed == ctx.packed


SPECIAL = {
    # name: (sub, gi, ge, sequence generator)
    "extreme127": (extreme_matrix(), 40.0, 3.0, seq),
    "dyadic8": (dyadic_matrix(20, 5), 3.0 + 1 / 256.0, 0.5 + 3 / 256.0, seq),
    "ties": (tie_matrix(), 1.0, 1.0, lambda rng, L, A: low_entropy_seq(rng, L, A)),
    "zero_gap": (asym_matrix(4, 77), 0.0, 0.0, seq),
    "zero_gap64": (asym_matrix(64, 78), 0.0, 0.0, seq),
}


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("name", sorted(SPECIAL))
def test_fill_pair_special_scorings(ctx, name, at):
    sub, gi, ge, gen = SPECIAL[name]
    A = sub.shape[0]
    ctx.set_scoring(sub, gi, ge, at)
    O = po.Oracle(sub, gi, ge, at)
    rng = np.random.default_rng(sorted(SPECIAL).index(name) * 10 + at)
    for Lq, Lt in [(1, 1), (2, 3), (9, 8), (17, 16), (30, 41), (64, 33), (120, 90), (255, 257), (40, 513)]:
        q, t = gen(rng, Lq, A), gen(rng, Lt, A)
        check_pair(ctx, O, q, t, "%s at%d %dx%d" % (name, at, Lq, Lt), mask_dr_for(at, q, t))


# ---- 2b. the multi-CTA wavefront, all five modes ----

@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("A", [4, 64])
def test_wavefront_asymmetric(A, at):
    sub = asym_matrix(A, 2000 + A)
    c = new_ctx(wave_min_cells=1)
    try:
        c.set_scoring(sub, 7, 2, at)
        O = po.Oracle(sub, 7, 2, at)
        rng = np.random.default_rng(20 * A + at)
        for Lt in (513, 768, 1025):      # 768 = exactly three 256-column stripes
            for Lq in (1, 40, 700):
                q, t = seq(rng, Lq, A), seq(rng, Lt, A)
                names = check_pair(c, O, q, t, "wave A%d at%d %dx%d" % (A, at, Lq, Lt), mask_dr_for(at, q, t, 0.02))
                assert has(names, "wave_kernel"), names
    finally:
        c.close()


# ---- 2c. one batch with every kernel class under an A = 64 asymmetric matrix ----

@pytest.mark.parametrize("at", [po.SEMI_LOCAL, po.GLOBAL_LOCAL], ids=["semi_local", "global_local"])
def test_mixed_batch_every_class_a64(at):
    import alignment_algos_b200 as a
    A, gi, ge = 64, 7, 2
    sub = asym_matrix(A, 3064, -12, 12)
    rng = np.random.default_rng(64 + at)
    shapes = {"packed": [(int(rng.integers(1, 200)), int(rng.integers(1, 200))) for _ in range(20)] + [(300, 512)],
              "int32_k8": [(2000, 250), (2500, 200)],      # Lt <= 256, bound >= 7000
              "int32_k16": [(700, 500), (900, 400)],       # 256 < Lt <= 512, bound >= 7000
              "wave": [(300, 900), (40, 1025)],
              "empty": [(0, 50), (50, 0), (0, 0)]}
    for cls, lst in shapes.items():
        for Lq, Lt in lst:
            if cls == "packed":
                assert bound(Lq, Lt, sub, gi, ge) < PACKED_BOUND
            elif cls.startswith("int32"):
                assert bound(Lq, Lt, sub, gi, ge) >= PACKED_BOUND
    seqs, pq, pt, cls_of = [], [], [], []
    for cls in ("packed", "int32_k8", "wave", "empty", "int32_k16"):   # classes interleaved in pair order
        for Lq, Lt in shapes[cls]:
            pq.append(len(seqs))
            pt.append(len(seqs) + 1)
            seqs += [seq(rng, Lq, A), seq(rng, Lt, A)]
            cls_of.append(cls)
    perm = rng.permutation(len(pq))
    pq, pt, cls_of = np.array(pq, np.int32)[perm], np.array(pt, np.int32)[perm], [cls_of[i] for i in perm]
    res, off = a.Context.pack(seqs)
    c = new_ctx(wave_min_cells=1)
    try:
        c.set_scoring(sub, gi, ge, at)
        O = po.Oracle(sub, gi, ge, at)
        delta = 0.05
        what = a.W_FWD | a.W_REV | a.W_TB | a.W_SCORES | a.W_MASK
        out, names = kernels(c, lambda: c.fill_batch(res, off, pq, pt, what, delta))
        assert has(names, "packed_kernel") and has(names, "fill_kernel<K=8") and has(names, "fill_kernel<K=16")
        assert has(names, "wave_kernel"), names
        want = {}
        for p in range(len(pq)):
            q, t = seqs[pq[p]], seqs[pt[p]]
            F, fq, ft = O.fill(q, t, po.FWD, True, fast=True)
            R, rq, rt = O.fill(q, t, po.REV, True, fast=True)
            thr = O.threshold(float(F[-1, -1]), delta)
            mask, cnt = O.nearopt_mask(F, R, O.sim(q, t), thr)
            tag = "pair %d (%s %dx%d)" % (p, cls_of[p], len(q), len(t))
            assert out["fwd_score"][p] == F[-1, -1] and out["rev_score"][p] == R[0, 0], tag
            assert out["threshold"][p] == thr and out["nearopt_count"][p] == cnt, tag
            want[p] = (F, fq, ft, R, rq, rt, mask)
        sample = [cls_of.index(k) for k in shapes] + [len(pq) - 1]
        for p in sample:
            q, t = seqs[pq[p]], seqs[pt[p]]
            F, fq, ft, R, rq, rt, mask = want[p]
            got = c.fetch_pair(int(p), len(q), len(t), fwd=True, rev=True, mask=True)
            for k, w in (("score_fwd", F), ("prevq_fwd", fq), ("prevt_fwd", ft), ("score_rev", R), ("prevq_rev", rq),
                         ("prevt_rev", rt), ("nearopt", mask)):
                assert_matrix_equal("%s pair %d (%s)" % (k, p, cls_of[p]), got[k], w)
            for d, od, (S, sq, st) in ((a.FWD, po.FWD, (F, fq, ft)), (a.REV, po.REV, (R, rq, rt))):
                rc, hp, hs = c.optimal(int(p), d, len(q), len(t))
                orc, opairs, osc = O.optimal(S, sq, st, od)
                assert (rc != 0) == (orc != 0), (p, d)
                if rc == 0:
                    assert hs == osc
                    assert_matrix_equal("optimal pair %d dir %d (%s)" % (p, d, cls_of[p]), hp, opairs)
        for d in (a.FWD, a.REV):
            aoff, pairs, n, st = c.optimal_all(d, len(pq))
            for p in range(len(pq)):
                q, t = seqs[pq[p]], seqs[pt[p]]
                rc, hp, _ = c.optimal(int(p), d, len(q), len(t))
                assert st[p] == rc, (p, d, cls_of[p])
                assert_matrix_equal("optimal_all pair %d dir %d (%s)" % (p, d, cls_of[p]), pairs[aoff[p]:aoff[p] + n[p]], hp)
    finally:
        c.close()


# ---- 2d. cross mode ----

@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_cross_scores_asymmetric(ctx, at):
    import alignment_algos_b200 as a
    A = 33
    sub = asym_matrix(A, 4033)
    rng = np.random.default_rng(41 + at)
    lens = list(rng.integers(1, 140, 30)) + [0, 1, 16, 17, 512, 513, 33]
    seqs = [seq(rng, int(L), A) for L in lens]
    res, off = a.Context.pack(seqs)
    q_ids = np.array([3, 0, 31, 30, 7, 36, 12, 5, 34, 9, 3, 20, 21], np.int32)
    t_ids = np.arange(len(seqs), dtype=np.int32)[::-1].copy()
    ctx.set_scoring(sub, 7, 2, at)
    got, names = kernels(ctx, lambda: ctx.cross_scores(res, off, q_ids, t_ids))
    assert has(names, "packed_kernel<TB=0,FST=0,MSK=0,XM=1>") == (ctx.packed and at != po.LOCAL), names
    O = po.Oracle(sub, 7, 2, at)
    want = np.zeros_like(got)
    for i, qs in enumerate(q_ids):
        for j, ts in enumerate(t_ids):
            want[i, j] = O.fill(seqs[qs], seqs[ts], po.FWD, False, fast=True)[0][-1, -1]
    assert_matrix_equal("cross scores", got, want)
    pq = np.repeat(q_ids, len(t_ids)).astype(np.int32)
    pt = np.tile(t_ids, len(q_ids)).astype(np.int32)
    assert_matrix_equal("cross == pair list", got.reshape(-1), ctx.fill_batch(res, off, pq, pt, a.W_FWD)["fwd_score"])


@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
def test_cross_scores_transposition(ctx, at):
    # cross(Q, T, sub, m) == cross(T, Q, sub^T, m')^T: no oracle needed, so the rectangle can be large
    import alignment_algos_b200 as a
    A = 64
    sub = asym_matrix(A, 5064)
    rng = np.random.default_rng(50 + at)
    seqs = [seq(rng, int(L), A) for L in rng.integers(1, 300, 260)]
    res, off = a.Context.pack(seqs)
    Q, T = np.arange(0, 120, dtype=np.int32), np.arange(120, 260, dtype=np.int32)
    ctx.set_scoring(sub, 7, 2, at)
    x = ctx.cross_scores(res, off, Q, T)
    ctx.set_scoring(np.ascontiguousarray(sub.T), 7, 2, SWAPPED_MODE[at])
    y = ctx.cross_scores(res, off, T, Q)
    assert_matrix_equal("transposed cross", x, y.T)
    # and the matrix matters: the untransposed matrix with swapped roles gives other scores
    ctx.set_scoring(sub, 7, 2, SWAPPED_MODE[at])
    z = ctx.cross_scores(res, off, T, Q)
    assert (z.T != x).mean() > 0.5


# ---- 2e. exact float: an asymmetric matrix off every dyadic grid ----

def float_matrix(A, seed):
    rng = np.random.default_rng(seed)
    return (asym_matrix(A, seed) + rng.integers(-50, 51, (A, A)) / 100.0).astype(np.float32)


@pytest.mark.parametrize("records", [1, 0], ids=["records", "scans"])
@pytest.mark.parametrize("A", [4, 64])
def test_exact_float_asymmetric(A, records):
    import alignment_algos_b200 as a
    sub = float_matrix(A, 6000 + A)
    rng = np.random.default_rng(A + records)
    c = new_ctx(general_records=records)
    try:
        for at in MODES:
            c.set_scoring(sub, 4.73, 0.34, at)
            O = po.Oracle(sub, 4.73, 0.34, at)
            for Lq, Lt in [(0, 0), (0, 5), (4, 0), (1, 1), (2, 3), (33, 17), (64, 65), (120, 90), (5, 700)]:
                q, t = seq(rng, Lq, A), seq(rng, Lt, A)
                names = check_pair(c, O, q, t, "float A%d at%d %dx%d" % (A, at, Lq, Lt), mask_dr_for(at, q, t), fast=False)
                if Lq and Lt:
                    assert is_float_path(names), names
            seqs = [seq(rng, int(L), A) for L in rng.integers(1, 160, 40)]
            res, off = a.Context.pack(seqs)
            pq, pt = rng.integers(0, 40, 60).astype(np.int32), rng.integers(0, 40, 60).astype(np.int32)
            what = a.W_FWD | a.W_REV | (0 if at == po.LOCAL else a.W_MASK)
            out = c.fill_batch(res, off, pq, pt, what, 0.02)
            for p in range(len(pq)):
                q, t = seqs[pq[p]], seqs[pt[p]]
                F = O.fill(q, t, po.FWD, True, fast=False)[0]
                R = O.fill(q, t, po.REV, True, fast=False)[0]
                assert out["fwd_score"][p] == F[-1, -1] and out["rev_score"][p] == R[0, 0], (at, p)
                if at != po.LOCAL:
                    thr = O.threshold(float(F[-1, -1]), 0.02)
                    _, cnt = O.nearopt_mask(F, R, O.sim(q, t), thr)
                    assert out["threshold"][p] == thr and out["nearopt_count"][p] == cnt, (at, p)
            if at == po.LOCAL:
                continue
            c.fill_batch(res, off, pq, pt, a.W_FWD)
            aoff, pairs, n, st = c.optimal_all(a.FWD, len(pq))
            for p in range(0, len(pq), 3):
                q, t = seqs[pq[p]], seqs[pt[p]]
                F, fq, ft = O.fill(q, t, po.FWD, True, fast=False)
                orc, opairs, osc = O.optimal(F, fq, ft, po.FWD)
                assert (st[p] != 0) == (orc != 0), (at, p)
                if orc == 0:
                    assert_matrix_equal("float optimal_all pair %d" % p, pairs[aoff[p]:aoff[p] + n[p]], opairs)
    finally:
        c.close()


# ---- 2f. enumeration under asymmetric and tie-heavy scoring ----

@pytest.mark.parametrize("scoring", ["asym4", "ties"])
def test_enumeration_asymmetric_and_ties(ctx, scoring):
    import alignment_algos_b200 as a
    sub, gi, ge = (asym_matrix(4, 7004), 5, 1) if scoring == "asym4" else (tie_matrix(), 1, 1)
    rng = np.random.default_rng(7 if scoring == "ties" else 8)
    seqs = []
    for k in range(14):
        L = int(rng.integers(6, 30))
        s = low_entropy_seq(rng, L) if scoring == "ties" else seq(rng, L, 4)
        m = s.copy()
        m[::5] = rng.integers(0, 4, len(m[::5]))
        seqs += [s, np.concatenate([m[: L // 2], m[L // 2 + int(rng.integers(0, 3)):]])]
    seqs += [seq(rng, L, 4) for L in (0, 1, 2)]
    res, off = a.Context.pack(seqs)
    pq = np.array(list(range(0, 28, 2)) + [28, 29, 30, 3], np.int32)
    pt = np.array(list(range(1, 28, 2)) + [5, 29, 7, 30], np.int32)
    K = 3000
    for at, delta in [(po.SEMI_LOCAL, 0.1), (po.GLOBAL, 0.15), (po.GLOBAL_LOCAL, 0.1), (po.LOCAL_GLOBAL, 0.1)]:
        ctx.set_scoring(sub, gi, ge, at)
        O = po.Oracle(sub, gi, ge, at)
        ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB | a.W_MASK, delta)
        ids = np.arange(len(pq))
        flags = [((np.arange(len(seqs[pt[p]]) + 2) // 3) % 2).astype(np.uint8) for p in ids]
        got = ctx.near_optimal(ids, delta, K)
        con = ctx.near_optimal(ids, delta, K, subopt_flags=flags, constrained=True)
        n_multi = 0
        for k, p in enumerate(ids):
            q, t = seqs[pq[p]], seqs[pt[p]]
            F, fq, ft = O.fill(q, t, po.FWD, True, fast=True)
            sim = O.sim(q, t)
            thr = O.threshold(float(F[-1, -1]), delta)
            for label, g, (st, want) in (("ucw", got[k], O.ucw_enumerate(q, t, F, sim, thr, K)),
                                         ("cno", con[k], O.cno_enumerate(q, t, F, sim, thr, fq, ft, flags[k], K))):
                gst, gthr, alis = g
                assert (gst, gthr, len(alis)) == (st, thr, len(want)), (label, at, p, gst, st, len(alis), len(want))
                for (gs, gp), (ws, wp) in zip(alis, want):
                    assert gs == ws
                    assert_matrix_equal("%s at%d pair %d alignment" % (label, at, p), gp, wp)
            n_multi += len(got[k][2]) > 1
        assert n_multi >= 5


# ---- 2g. local alignments on the packed (LOC = 1) and int32 kernels ----

def test_local_batch_asymmetric(ctx):
    import alignment_algos_b200 as a
    A = 20
    sub = asym_matrix(A, 8020, -9, 6)
    rng = np.random.default_rng(12)
    seqs = [seq(rng, int(L), A) for L in rng.integers(1, 200, 40)]
    for k in range(0, 16, 2):       # related pairs: a shared core in different flanks
        core = seq(rng, int(rng.integers(10, 60)), A)
        seqs[k] = np.concatenate([seq(rng, 7, A), core, seq(rng, 12, A)])
        seqs[k + 1] = np.concatenate([seq(rng, 15, A), core, seq(rng, 3, A)])
    seqs += [np.zeros(0, np.uint8), seq(rng, 400, A)]
    res, off = a.Context.pack(seqs)
    pq = np.concatenate([np.arange(0, 16, 2), rng.integers(0, 42, 30)]).astype(np.int32)
    pt = np.concatenate([np.arange(1, 16, 2), rng.integers(0, 42, 30)]).astype(np.int32)
    ctx.set_scoring(sub, 6, 1, po.LOCAL)
    O = po.Oracle(sub, 6, 1, po.LOCAL)
    out, names = kernels(ctx, lambda: ctx.fill_batch(res, off, pq, pt, a.W_FWD | a.W_REV | a.W_TB | a.W_SCORES))
    assert any("LOC=1" in n for n in names) == ctx.packed, names
    want = {}
    for p in range(len(pq)):
        q, t = seqs[pq[p]], seqs[pt[p]]
        F, fq, ft = O.fill(q, t, po.FWD, True, fast=True)
        R, rq, rt = O.fill(q, t, po.REV, True, fast=True)
        assert out["fwd_score"][p] == F[-1, -1] and out["rev_score"][p] == R[0, 0], p
        want[p] = ((F, fq, ft), (R, rq, rt))
        if p % 3 == 0:
            got = ctx.fetch_pair(int(p), len(q), len(t), fwd=True, rev=True)
            for d, nm in ((0, "fwd"), (1, "rev")):
                for k, w in zip(("score_", "prevq_", "prevt_"), want[p][d]):
                    assert_matrix_equal("local %s%s pair %d" % (k, nm, p), got[k + nm], w)
    for d, od, x in ((a.FWD, po.FWD, 0), (a.REV, po.REV, 1)):
        aoff, pairs, n, st = ctx.optimal_all(d, len(pq))
        for p in range(len(pq)):
            orc, opairs, osc = O.optimal(*want[p][x], od)
            assert st[p] == 0 and orc == 0
            assert_matrix_equal("local optimal pair %d dir %d" % (p, d), pairs[aoff[p]:aoff[p] + n[p]], opairs)


# ---- 3. the limits that choose the kernel or the score storage, each side of each ----

def edge_pair(c, O, q, t, tag, want_prefix, mask_dr=0.05, fast=True):
    names = check_pair(c, O, q, t, tag, mask_dr, fast=fast)
    if want_prefix == "float":
        assert is_float_path(names), (tag, names)
    else:
        assert has(names, want_prefix), (tag, want_prefix, names)
        assert not is_float_path(names), (tag, names)
    return names


@pytest.mark.parametrize("at", [po.GLOBAL, po.SEMI_LOCAL, po.LOCAL_GLOBAL], ids=["global", "semi_local", "local_global"])
def test_packed_bound_edge(at):
    # bd = 300*10 + 2*1699 + 1*(300+Lt): Lt = 301 -> 6999 (packed), Lt = 302 -> 7000 (int32)
    import alignment_algos_b200 as a
    sub = asym_matrix(4, 9004, -10, 10)
    gi, ge = 1699, 1
    rng = np.random.default_rng(at)
    c = new_ctx()
    try:
        c.set_scoring(sub, gi, ge, at)
        O = po.Oracle(sub, gi, ge, at)
        q = seq(rng, 300, 4)
        for Lt, path in ((301, "packed_kernel"), (302, "fill_kernel")):
            assert bound(300, Lt, sub, gi, ge) == PACKED_BOUND - (1 if Lt == 301 else 0)
            t = q[:Lt].copy() if Lt <= 300 else np.concatenate([q, seq(rng, Lt - 300, 4)])
            t[::7] = rng.integers(0, 4, len(t[::7]))
            edge_pair(c, O, q, t, "bd %d" % bound(300, Lt, sub, gi, ge), path)
        # cross mode: the same bound from the query's side (template list of one 300-residue template)
        seqs = [seq(rng, 300, 4), seq(rng, 301, 4), seq(rng, 302, 4)]
        res, off = a.Context.pack(seqs)
        for qi, packed in ((1, True), (2, False)):
            assert (bound(len(seqs[qi]), 300, sub, gi, ge) < PACKED_BOUND) == packed
            got, names = kernels(c, lambda: c.cross_scores(res, off, np.array([qi], np.int32), np.array([0], np.int32)))
            assert has(names, "packed_kernel<TB=0,FST=0,MSK=0,XM=1>") == packed, (qi, names)
            assert got[0, 0] == O.fill(seqs[qi], seqs[0], po.FWD, False, fast=True)[0][-1, -1]
    finally:
        c.close()


def test_packed_gap_limits():
    # gi <= 2048 and ge <= 400 grid units take the packed kernels, 2049 / 401 the int32 kernels; also at s = 1
    sub = asym_matrix(4, 9104)
    half = (asym_matrix(4, 9105) + 0.5).astype(np.float32)   # needs the 2^-1 grid
    rng = np.random.default_rng(3)
    c = new_ctx()
    try:
        for m, gi, ge, L, path in [(sub, 2048, 1, 100, "packed_kernel"), (sub, 2049, 1, 100, "fill_kernel"),
                                   (half, 1024.0, 0.5, 100, "packed_kernel"), (half, 1024.5, 0.5, 100, "fill_kernel"),
                                   (sub, 10, 400, 5, "packed_kernel"), (sub, 10, 401, 5, "fill_kernel"),
                                   (half, 10, 200.0, 4, "packed_kernel"), (half, 10, 200.5, 4, "fill_kernel")]:
            for at in (po.GLOBAL, po.SEMI_LOCAL):
                c.set_scoring(m, gi, ge, at)
                O = po.Oracle(m, gi, ge, at)
                s = 1 if m is half else 0
                assert bound(L, L + 3, m, gi, ge, s) < PACKED_BOUND
                q, t = seq(rng, L, 4), seq(rng, L + 3, 4)
                edge_pair(c, O, q, t, "gi %s ge %s at%d" % (gi, ge, at), path)
    finally:
        c.close()


def test_integer_grid_limits():
    # |sub * 2^s| = 127 and a 2^-8 grid take the integer kernels; 128, or one entry on the 2^-9 grid, exact float
    rng = np.random.default_rng(4)
    m127 = extreme_matrix()
    m128 = m127.copy()
    m128[2, 3] = 128
    d8 = dyadic_matrix(20, 5)
    d9 = d8.copy()
    d9[4, 7] = 3 / 512.0
    h127 = (m127 / 2).astype(np.float32)           # 63.5 = 127 units of 2^-1
    h128 = h127.copy()
    h128[5, 5] = 64.0                               # 128 units of 2^-1
    c = new_ctx()
    try:
        for m, gi, ge, path in [(m127, 40, 3, "int"), (m128, 40, 3, "float"), (d8, 3 + 1 / 256.0, 0.5, "int"),
                                (d9, 3 + 1 / 256.0, 0.5, "float"), (h127, 20.5, 1.5, "int"), (h128, 20.5, 1.5, "float")]:
            for at in (po.GLOBAL, po.SEMI_LOCAL, po.LOCAL):
                c.set_scoring(m, gi, ge, at)
                O = po.Oracle(m, gi, ge, at)
                for Lq, Lt in [(12, 9), (70, 130)]:
                    q, t = seq(rng, Lq, 20), seq(rng, Lt, 20)
                    q[:5], t[:5] = 1, 1                     # the +127 diagonal entry in play
                    tag = "%s at%d %dx%d" % (path, at, Lq, Lt)
                    edge_pair(c, O, q, t, tag, "float" if path == "float" else ("packed_kernel", "fill_kernel"),
                              mask_dr_for(at, q, t), fast=(path == "int"))
    finally:
        c.close()


def _storage_batch(c, O, c_val, wave):
    """A batch whose largest non-packed bound is 600*c_val: two identical 600-residue sequences over A = 1, gi = ge = 0
    (forward optimum = bound), plus packed-sized pairs that do not count towards the bound."""
    import alignment_algos_b200 as a
    rng = np.random.default_rng(c_val)
    seqs = [np.zeros(600, np.uint8), np.zeros(600, np.uint8)] + [np.zeros(int(L), np.uint8) for L in rng.integers(1, 40, 6)]
    res, off = a.Context.pack(seqs)
    pq = np.array([0, 2, 4, 6], np.int32)
    pt = np.array([1, 3, 5, 7], np.int32)
    delta = 0.01
    what = a.W_FWD | a.W_REV | a.W_TB | a.W_SCORES | a.W_MASK
    out, names = kernels(c, lambda: c.fill_batch(res, off, pq, pt, what, delta))
    st = 1 if 600 * c_val < 30000 else 2
    kern = "wave_kernel<K=8,TB=1,ST=%d>" % st if wave else "fill_kernel<K=16,TB=1,ST=%d>" % st
    assert has(names, kern), (kern, names)
    for p in range(len(pq)):
        q, t = seqs[pq[p]], seqs[pt[p]]
        F, fq, ft = O.fill(q, t, po.FWD, True, fast=True)
        R, rq, rt = O.fill(q, t, po.REV, True, fast=True)
        thr = O.threshold(float(F[-1, -1]), delta)
        mask, cnt = O.nearopt_mask(F, R, O.sim(q, t), thr)
        assert out["fwd_score"][p] == F[-1, -1] and out["rev_score"][p] == R[0, 0]
        assert out["threshold"][p] == thr and out["nearopt_count"][p] == cnt
        if p == 0:   # the test must reach the storage range it claims to test
            assert np.abs(F).max() >= 0.9 * 600 * c_val and np.abs(R).max() >= 0.9 * 600 * c_val
        got = c.fetch_pair(p, len(q), len(t), fwd=True, rev=True, mask=True)
        for k, w in (("score_fwd", F), ("prevq_fwd", fq), ("prevt_fwd", ft), ("score_rev", R), ("prevq_rev", rq),
                     ("prevt_rev", rt), ("nearopt", mask)):
            assert_matrix_equal("storage c=%d %s pair %d" % (c_val, k, p), got[k], w)


@pytest.mark.parametrize("wave", [False, True], ids=["int32", "wavefront"])
@pytest.mark.parametrize("c_val", [49, 50])
def test_int16_int32_score_storage_edge(c_val, wave):
    # bound 29400 keeps int16 score storage, 30000 switches to int32
    c = new_ctx(**({"wave_min_cells": 1} if wave else {}))
    try:
        for at in (po.GLOBAL, po.SEMI_LOCAL):
            sub = np.array([[c_val]], np.float32)
            c.set_scoring(sub, 0, 0, at)
            _storage_batch(c, po.Oracle(sub, 0, 0, at), c_val, wave)
    finally:
        c.close()


def test_bound_of_2_24_fails_loudly_and_the_context_recovers():
    import alignment_algos_b200 as a
    sub = asym_matrix(4, 9204)
    gi, ge = 1e6, 1e5                       # the largest gap penalties of the integer path
    rng = np.random.default_rng(5)
    seqs = [seq(rng, 84, 4), seq(rng, 84, 4), seq(rng, 20, 4), seq(rng, 21, 4)]
    assert bound(84, 84, sub, gi, ge) >= 1 << 24 > bound(20, 21, sub, gi, ge)
    res, off = a.Context.pack(seqs)
    c = new_ctx()
    try:
        c.set_scoring(sub, gi, ge, po.GLOBAL)
        with pytest.raises(a.AadpError):
            c.fill_batch(res, off, [0, 2], [1, 3], a.W_FWD | a.W_REV)
        with pytest.raises(a.AadpError):
            c.fill_pair(seqs[0], seqs[1], a.BOTH)
        O = po.Oracle(sub, gi, ge, po.GLOBAL)
        out = c.fill_batch(res, off, [2], [3], a.W_FWD | a.W_REV | a.W_TB | a.W_MASK, 0.05)
        F = O.fill(seqs[2], seqs[3], po.FWD, True, fast=True)[0]
        R = O.fill(seqs[2], seqs[3], po.REV, True, fast=True)[0]
        thr = O.threshold(float(F[-1, -1]), 0.05)
        assert out["fwd_score"][0] == F[-1, -1] and out["rev_score"][0] == R[0, 0] and out["threshold"][0] == thr
        assert out["nearopt_count"][0] == O.nearopt_mask(F, R, O.sim(seqs[2], seqs[3]), thr)[1]
        check_pair(c, O, seqs[2], seqs[3], "after the refusal", 0.05)
        sub2 = asym_matrix(20, 9220)
        c.set_scoring(sub2, 7, 2, po.SEMI_LOCAL)
        O2 = po.Oracle(sub2, 7, 2, po.SEMI_LOCAL)
        q, t = seq(rng, 90, 20), seq(rng, 120, 20)
        check_pair(c, O2, q, t, "normal scoring after the refusal", 0.05)
    finally:
        c.close()


@pytest.mark.parametrize("delta", [0.0, 1.0, 4.0])
def test_mask_threshold_extremes(delta):
    # The packed kernels' fused mask compares with an integer threshold clamped to [kFloor16, kPackedBound]; its mask and
    # count against the int32 kernels' mask_kernel and the oracle, all in global mode:
    #  - gi = 2048 units, bd = 6946 (just under 7000), positive optimum 1710: at delta = 4 the threshold -5130 lies
    #    among the slacks of the off-diagonal cells (down to about -5230), so any clamp above it loses cells;
    #  - gi = 2048 units, a negative optimum;
    #  - gi = 10, positive optimum 4500: at delta = 4 the threshold -13500 is below kFloor16 and the clamp is live.
    sub = asym_matrix(4, 9304, -9, 9)
    np.fill_diagonal(sub, 9)
    rng = np.random.default_rng(int(delta * 10))
    q, q2 = seq(rng, 190, 4), seq(rng, 500, 4)
    cases = [(q, q.copy(), 2048, 3, "positive"), (seq(rng, 250, 4), seq(rng, 60, 4), 2048, 4, "negative"),
             (q2, q2.copy(), 10, 2, "clamped")]
    cp, ci = new_ctx(packed=1), new_ctx(packed=0)
    try:
        for q_, t_, gi, ge, kind in cases:
            assert bound(len(q_), len(t_), sub, gi, ge) < PACKED_BOUND
            O = po.Oracle(sub, gi, ge, po.GLOBAL)
            opt = float(O.fill(q_, t_, po.FWD, True, fast=True)[0][-1, -1])
            assert (opt > 0) == (kind != "negative")
            if delta == 4.0 and kind == "clamped":
                assert np.floor(O.threshold(opt, delta)) < FLOOR16
            for c, path in ((cp, "packed_kernel"), (ci, "mask_kernel")):
                c.set_scoring(sub, gi, ge, po.GLOBAL)
                names = edge_pair(c, O, q_, t_, "delta %s %s %s" % (delta, kind, path), path, mask_dr=delta)
                assert any("MSK=1" in n for n in names) == (c is cp), names
    finally:
        cp.close()
        ci.close()
