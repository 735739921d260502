"""SURVEY.md §8 row f2: the pruned near-optimal enumerators (kscw.h k-sorted, crcw.h controlled redundancy).

CPU part (no GPU): the host walk that aadp_batch_near_optimal_pruned runs over a GPU-filled pair
(alignment_algos_b200/csrc/aadp_pruned.h, built into tests/cxx/libpruned_host.so) is driven with the oracle's forward
matrix and compared with the results of the REFERENCE's own KSConstrainedNearOptimal / CRConstrainedNearOptimal (compiled
from the unmodified headers by oracle/ref_harness.cpp), stored in tests/golden/reference_digests.json.  GPU part (-m gpu):
the same comparison through the C ABI over a resident batch.

Bar: identical alignment sets (pairs and fp32 scores).  The reference ranks branch candidates with std::sort /
std::partial_sort on the score alone, so which of several equal-score candidates survive a cut is a property of the
sort implementation; both sides call the same libstdc++ routines on the same key sequence, and the comparison is on
canonically ordered sets."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from util import po, ROOT, ReferenceResults

LIB = os.path.join(ROOT, "tests", "cxx", "libpruned_host.so")


def _host_lib():
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(
            os.path.join(ROOT, "alignment_algos_b200", "csrc", "aadp_pruned.h")):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "cxx"), "libpruned_host.so"])
    return C.CDLL(LIB)


def _p(a, ty):
    return a.ctypes.data_as(C.POINTER(ty))


def host_walk(L, variant, q, t, F, pq, pt, sim, flags, gi, ge, at, delta, k_limit=16, sort_limit=100, max_overlap=0.30,
              user_limit=100000, K=20000):
    Lq, Lt = len(q), len(t)
    delfree = at in (po.LOCAL, po.SEMI_LOCAL, po.LOCAL_GLOBAL)
    insfree = at in (po.LOCAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL)
    cap = K * (Lq + Lt + 4)
    scores = np.zeros(K, np.float32)
    ln = np.zeros(K, np.int32)
    paths = np.zeros((cap, 2), np.int32)
    n = C.c_int(0)
    fl = np.ascontiguousarray(flags, np.uint8) if flags is not None else None
    rc = L.pruned_host_run(variant, Lq, Lt, _p(np.ascontiguousarray(F, np.float32), C.c_float),
                           _p(np.ascontiguousarray(pq, np.int32), C.c_int), _p(np.ascontiguousarray(pt, np.int32), C.c_int),
                           _p(np.ascontiguousarray(sim, np.float32), C.c_float), _p(fl, C.c_uint8) if fl is not None else None,
                           C.c_float(gi), C.c_float(ge), int(delfree), int(insfree), C.c_float(delta), C.c_uint(k_limit),
                           C.c_uint(sort_limit), C.c_float(max_overlap), C.c_uint(user_limit), C.c_long(K), C.byref(n),
                           _p(scores, C.c_float), _p(ln, C.c_int), _p(paths, C.c_int), C.c_long(cap))
    assert rc == 0, rc
    out, o = [], 0
    for k in range(n.value):
        out.append((float(scores[k]), paths[o:o + ln[k]].copy()))
        o += ln[k]
    return out


def canon(alis):
    return sorted((np.float32(s).tobytes(), p.tobytes()) for s, p in alis)


def cases(rng):
    """related pairs (many near-optimal alignments) of several sizes, with several SuboptFlags patterns"""
    for L, delta in ((18, 0.3), (30, 0.2), (45, 0.15), (60, 0.1), (90, 0.06), (120, 0.05)):
        q = rng.integers(0, 20, L).astype(np.uint8)
        t = q.copy()
        t[::4] = rng.integers(0, 20, len(t[::4]))
        cut = int(rng.integers(2, L - 2))
        t = np.concatenate([t[:cut], t[cut + int(rng.integers(0, 3)):]])
        Lt = len(t)
        for flags in (None, (np.arange(Lt + 2) // 6) % 2, 1 - (np.arange(Lt + 2) // 9) % 2, rng.integers(0, 2, Lt + 2)):
            yield q, t, delta, flags


VARIANTS = {2: "kscw", 3: "crcw"}


@pytest.mark.parametrize("variant", [2, 3], ids=["kscw", "crcw"])
def test_host_walk_equals_reference(blosum, variant):
    _, M = blosum
    ref = ReferenceResults("test_pruned.py::test_host_walk_equals_reference[%s]" % VARIANTS[variant])
    L = _host_lib()
    rng = np.random.default_rng(31 + variant)
    total = multi = 0
    for at in (po.SEMI_LOCAL, po.GLOBAL, po.GLOBAL_LOCAL):
        for gi, ge in ((3, 1), (12, 1), (4.73, 0.34)):
            O = po.Oracle(M, gi, ge, at)
            for q, t, delta, flags in cases(rng):
                F, pq, pt = O.fill(q, t, po.FWD, True, fast=False)
                for kl, sl, mo in ((16, 100, 0.30), (4, 100, 0.30), (16, 8, 0.5), (2, 100, 0.1)):
                    got = host_walk(L, variant, q, t, F, pq, pt, O.sim(q, t), flags, gi, ge, at, delta, kl, sl, mo)
                    ref.check("%d %s %dx%d %d %d %s" % (at, gi, len(q), len(t), kl, sl, mo), canon(got))
                    total += len(got)
                    multi += len(got) > 1
    ref.close()
    assert total > 3000 and multi > 100


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [2, 3], ids=["kscw", "crcw"])
def test_gpu_pruned_enumerators_equal_reference(blosum, variant):
    # aadp_batch_near_optimal_pruned over a resident batch (forward fill, traceback and scores produced by the CUDA
    # kernels; integer grid -> packed kernels, 4.73/0.34 -> exact general-gap kernel) against the reference's own
    # KSConstrainedNearOptimal / CRConstrainedNearOptimal
    import alignment_algos_b200 as a
    _, M = blosum
    ref = ReferenceResults("test_pruned.py::test_gpu_pruned_enumerators_equal_reference[%s]" % VARIANTS[variant])
    rng = np.random.default_rng(41 + variant)
    total = 0
    for at, gi, ge in ((po.SEMI_LOCAL, 3, 1), (po.GLOBAL, 12, 1), (po.GLOBAL_LOCAL, 4.73, 0.34)):
        cs = list(cases(rng))
        seqs, pq, pt = [], [], []
        for q, t, delta, flags in cs:
            pq.append(len(seqs)); seqs.append(q)
            pt.append(len(seqs)); seqs.append(t)
        res, off = a.Context.pack(seqs)
        c = a.Context(0)
        c.set_scoring(M, gi, ge, at)
        c.fill_batch(res, off, np.array(pq, np.int32), np.array(pt, np.int32), a.W_FWD | a.W_TB | a.W_SCORES, 0.1)
        for p, (q, t, delta, flags) in enumerate(cs):
            for kl, sl, mo in ((16, 100, 0.30), (4, 8, 0.5)):
                st, thr, got = c.near_optimal_pruned(p, variant, delta, len(q), len(t), flags, kl, sl, mo)
                assert st == 0
                ref.check("%d %s pair %d %d" % (at, gi, p, kl), canon(got))
                total += len(got)
        # a budget smaller than the set: status 1
        st, _, got = c.near_optimal_pruned(1, 2, cs[1][2], len(cs[1][0]), len(cs[1][1]), cs[1][3], max_alignments=1)
        assert st in (0, 1) and len(got) <= 1
        c.close()
    ref.close()
    assert total > 500
