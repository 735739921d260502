"""The C++ drop-in boundary: one demo source (tests/cxx/dropin_demo.cpp, shaped like the reference
driver aa_ali.cpp:63-90) is compiled against this repo's include/hmap2 headers (GPU fill) and against
the unmodified reference headers (CPU).  Their DPCell dumps and optimal alignments must be identical.
The reference builds' output is stored in tests/golden/reference_digests.json (tests/util.py, ReferenceResults)."""
import os
import subprocess

import numpy as np
import pytest

from util import ROOT, po, MODES, MODE_NAMES, ReferenceResults

CXX = os.path.join(ROOT, "tests", "cxx")
DEMO = os.path.join(CXX, "dropin_demo")
MATRIX = os.path.join(ROOT, "alignment_algos_b200", "data", "BLOSUM62")
ALPHA = "ARNDCQEGHILKMFPSTWYVBZX*"


def _letters(codes):
    return "".join(ALPHA[c] for c in codes)


def _run(binary, at, gi, ge, q, t):
    out = subprocess.run([binary, MATRIX, str(at), str(gi), str(ge), _letters(q), _letters(t)],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout.splitlines()


def _expected_lines(O, q, t, sub, fast=True):
    """What the demo must print, from the oracle."""
    lines = []
    sim = O.sim(q, t)
    res = {}
    for d, tag in ((po.FWD, "F"), (po.REV, "R")):
        s, pq, pt = O.fill(q, t, d, True, fast=fast)
        res[tag] = (s, pq, pt)
        for i in range(s.shape[0]):
            for j in range(s.shape[1]):
                lines.append("%s %d %d %.6g %d %d %.6g" % (tag, i, j, s[i, j], pq[i, j], pt[i, j], sim[i, j]))
    return lines, res


def test_headers_compile_and_reference_demo_matches_oracle(blosum):
    subprocess.check_call(["make", "-C", CXX, "all"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    assert os.path.exists(DEMO)
    _, M = blosum
    ref = ReferenceResults("test_cxx_dropin.py::test_headers_compile_and_reference_demo_matches_oracle")
    rng = np.random.default_rng(21)
    for at in (po.GLOBAL, po.SEMI_LOCAL, po.LOCAL):
        q = rng.integers(0, 20, 23).astype(np.uint8)
        t = rng.integers(0, 20, 31).astype(np.uint8)
        O = po.Oracle(M, 12, 1, at)
        want, _ = _expected_lines(O, q, t, M)
        ref.check("DPCell lines of the reference demo, mode %d" % at, want)
    ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("at", MODES, ids=[MODE_NAMES[m] for m in MODES])
def test_gpu_dropin_equals_reference_build(blosum, at):
    _, M = blosum
    ref = ReferenceResults("test_cxx_dropin.py::test_gpu_dropin_equals_reference_build[%s]" % MODE_NAMES[at])
    rng = np.random.default_rng(40 + at)
    # the last case is the reference's default scoring (alib.cpp:17-18): not on a dyadic grid -> exact fp32 path
    for (gi, ge, Lq, Lt) in [(12, 1, 37, 52), (3, 1, 64, 20), (10.5, 0.25, 18, 18), (12, 1, 1, 9), (12, 1, 300, 270),
                             (4.73, 0.34, 41, 35)]:
        q = rng.integers(0, 20, Lq).astype(np.uint8)
        t = rng.integers(0, 20, Lt).astype(np.uint8)
        got = _run(DEMO, at, gi, ge, q, t)
        core = [l for l in got if not l.startswith("#") and not l.startswith("@")]
        O = po.Oracle(M, gi, ge, at)
        want, res = _expected_lines(O, q, t, M, fast=(gi != 4.73))
        assert core[:len(want)] == want
        if Lq * Lt < 5000:
            case = "%s %s %dx%d" % (gi, ge, Lq, Lt)
            ref.check("everything the reference build prints, " + case, core)
            # near-optimal alignments (ucw.h) enumerated on the GPU vs. the reference recursion: same set, same scores
            ucw_got = sorted(l for l in got if l.startswith("@"))
            ref.check("UnconstrainedNearOptimal alignments of the reference build, " + case, ucw_got)
            if at != po.LOCAL:
                assert len(ucw_got) >= 2
            if Lq > 7 and Lt > 7:  # the loop list closed in ONE aadp_fill_subpair_batch call vs. one sub-matrix per loop
                assert len([l for l in core if l.startswith("LOOP ")]) == 5
        # optimal alignment line against the oracle traceback
        F, fq, ft = res["F"]
        rc, pairs, sc = O.optimal(F, fq, ft, po.FWD)
        opt = [l for l in core if l.startswith("OPT ")]
        assert len(opt) == 1
        assert opt[0].split(" pairs ")[1].split() == ["%d:%d" % (a, b) for a, b in pairs]
        # extras: reverse traceback and near-optimal cell count
        R, rq, rt = res["R"]
        rrc, rpairs, rsc = O.optimal(R, rq, rt, po.REV)
        rev = [l for l in got if l.startswith("#REV")][0]
        if rrc == 0:
            assert rev.split(" pairs ")[1].split() == ["%d:%d" % (a, b) for a, b in rpairs]
        else:
            assert "Illegal alignment start pair" in rev
        if at != po.LOCAL:
            thr = O.threshold(float(F[-1, -1]), 0.05)
            mask, cnt = O.nearopt_mask(F, R, O.sim(q, t), thr)
            no = [l for l in got if l.startswith("#NEAROPT")][0].split()
            assert int(no[-1]) == cnt and float(no[4]) == pytest.approx(thr, rel=1e-6)
    ref.close()


REFPATCH_GPU = os.path.join(CXX, "refpatch_gpu")
REFPATCH_CPU = os.path.join(CXX, "refpatch_cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("at", MODES, ids=[MODE_NAMES[m] for m in MODES])
def test_unmodified_reference_with_gpu_fill_enumerates_the_same_alignments(at):
    """tests/cxx/refpatch_demo.cpp: the reference's own headers + sources, with DPMatrix::build()/build_subdpm()
    specialised from the outside to call aadp_fill_pair_general.  The reference's own Optimal, UCW and CNO
    enumerators then run over the GPU-filled matrices and must print exactly what the pure reference prints:
    every DPCell, the optimal alignment, and every near-optimal alignment with its score."""
    if not (os.path.exists(REFPATCH_GPU) and os.path.exists(REFPATCH_CPU)):
        pytest.skip("refpatch binaries not built (they need /root/reference at build time)")
    rng = np.random.default_rng(300 + at)
    cases = [(12, 1, 0.2, 18, 22), (4.73, 0.34, 0.1, 25, 21), (3, 1, 0.05, 30, 30), (12, 1, 0.3, 4, 9)]
    n_alignments = 0
    for gi, ge, delta, Lq, Lt in cases:
        # related sequences (a mutated copy) so that the near-optimal set is not trivial
        q = rng.integers(0, 20, Lq).astype(np.uint8)
        t = np.resize(q, Lt).copy()
        mut = rng.random(Lt) < 0.25
        t[mut] = rng.integers(0, 20, int(mut.sum()))
        args = [MATRIX, str(at), str(gi), str(ge), str(delta), _letters(q), _letters(t)]
        got = subprocess.run([REFPATCH_GPU] + args, capture_output=True, text=True, timeout=300)
        want = subprocess.run([REFPATCH_CPU] + args, capture_output=True, text=True, timeout=300)
        assert got.returncode == 0, got.stdout[-400:] + got.stderr[-400:]
        assert want.returncode == 0
        assert got.stdout == want.stdout, "GPU-filled reference and pure reference print different results"
        n_alignments += sum(1 for l in got.stdout.splitlines() if l.startswith(("UCW ", "CNO ")))
    assert at == po.LOCAL or n_alignments > 10


TAB_DEMO = os.path.join(CXX, "tabeval_demo")


@pytest.mark.gpu
@pytest.mark.parametrize("at", MODES, ids=[MODE_NAMES[m] for m in MODES])
def test_user_evaluator_with_positional_gaps_equals_reference_build(at):
    # tests/cxx/tabeval_demo.cpp: a user-defined Evaluator whose gap penalties depend on the template position
    # (hmap_eval.h:63-117 / gn2_eval.h:99-158 shaped).  hmap2::DPMatrix tabulates it and fills on the GPU
    # (aadp_fill_pair_tabulated); the unmodified reference fills on the CPU.  Same source, identical output.
    assert os.path.exists(TAB_DEMO), "tests/cxx/tabeval_demo is built by __graft_entry__.build()"
    ref = ReferenceResults("test_cxx_dropin.py::test_user_evaluator_with_positional_gaps_equals_reference_build[%s]"
                           % MODE_NAMES[at])
    rng = np.random.default_rng(70 + at)
    for style in (1, 2):
        for (gi, ge, Lq, Lt) in [(4.73, 0.34, 33, 47), (7.1, 0.9, 5, 1), (10, 0.5, 80, 75)]:
            q = rng.integers(0, 20, Lq).astype(np.uint8)
            t = rng.integers(0, 20, Lt).astype(np.uint8)
            args = [MATRIX, str(at), str(gi), str(ge), str(style), _letters(q), _letters(t)]
            got = subprocess.run([TAB_DEMO] + args, capture_output=True, text=True, timeout=120)
            assert got.returncode == 0, got.stdout[-300:] + got.stderr[-300:]
            assert len(got.stdout.splitlines()) == 2 * (Lq + 2) * (Lt + 2) + 1
            ref.check("style %d %dx%d: output of the reference build" % (style, Lq, Lt), got.stdout)
    ref.close()


PRUNED_DEMO = os.path.join(CXX, "pruned_demo")


def _run_pruned(binary, at, gi, ge, delta, kl, sl, mo, flags, q, t):
    fl = "-" if flags is None else "".join("1" if f else "0" for f in flags)
    out = subprocess.run([binary, MATRIX, str(at), str(gi), str(ge), str(delta), str(kl), str(sl), str(mo), fl, _letters(q),
                          _letters(t)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout.splitlines()


@pytest.mark.gpu
@pytest.mark.parametrize("at", [po.SEMI_LOCAL, po.GLOBAL, po.GLOBAL_LOCAL], ids=["semi_local", "global", "global_local"])
def test_pruned_enumerators_dropin_equals_reference_build(at):
    # SURVEY.md §8 row f2: include/hmap2/kscw.h + crcw.h (GPU fill + aadp_batch_near_optimal_pruned) against the UNMODIFIED
    # reference headers compiled from the same source: the printed alignment sets (scores and aligned pairs, after the
    # reference's sortSet) must be the same.  Alignments of equal score may be listed in either order.
    assert os.path.exists(PRUNED_DEMO), "tests/cxx/pruned_demo is built by __graft_entry__.build()"
    ref = ReferenceResults("test_cxx_dropin.py::test_pruned_enumerators_dropin_equals_reference_build[%s]"
                           % MODE_NAMES[at])
    rng = np.random.default_rng(60 + at)
    n = 0
    for gi, ge in ((3, 1), (12, 1), (4.73, 0.34)):
        for L, delta in ((24, 0.25), (48, 0.12), (96, 0.06)):
            q = rng.integers(0, 20, L).astype(np.uint8)
            t = q.copy()
            t[::4] = rng.integers(0, 20, len(t[::4]))
            t = np.concatenate([t[: L // 3], t[L // 3 + 2:]])
            for flags in (None, (np.arange(len(t) + 2) // 7) % 2):
                for kl, sl, mo in ((16, 100, 0.3), (4, 10, 0.5)):
                    got = _run_pruned(PRUNED_DEMO, at, gi, ge, delta, kl, sl, mo, flags, q, t)
                    ref.check("%s %s %d %d: output of the reference build" % (gi, ge, L, kl),
                              [l for l in got if " n " in l], sorted(got))
                    # sortSet order: scores must be non-increasing in both
                    for tag in ("KS", "CR"):
                        sc = [float(l.split()[1]) for l in got if l.startswith(tag + " ") and " pairs" in l]
                        assert sc == sorted(sc, reverse=True)
                    n += len(got)
    ref.close()
    assert n > 200
