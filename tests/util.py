"""Shared helpers for the parity tests."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import pyoracle as po  # noqa: E402  (tests are allowed to use the oracle)

REFERENCE_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")

MODES = [po.GLOBAL_LOCAL, po.GLOBAL, po.LOCAL_GLOBAL, po.LOCAL, po.SEMI_LOCAL]
MODE_NAMES = {0: "global_local", 1: "global", 2: "local_global", 3: "local", 4: "semi_local"}


def golden_cases(g):
    return [str(n) for n in g["names"]]


def golden_case(g, name):
    gi, ge, at = g[name + ".params"]
    return g[name + ".q"], g[name + ".t"], float(gi), float(ge), int(at)


def rand_pair(rng, Lq, Lt, A=20):
    return rng.integers(0, A, Lq).astype(np.uint8), rng.integers(0, A, Lt).astype(np.uint8)


def digest(*items):
    """BLAKE2b digest of results: arrays by shape and values (integers as int64, floats as float64, so the digest
    does not depend on the container type), numbers exactly, lists and tuples element by element."""
    h = hashlib.blake2b(digest_size=8)

    def feed(x):
        if isinstance(x, np.ndarray):
            x = x.astype(np.float64 if x.dtype.kind == "f" else np.int64)
            h.update(("a%s%s" % (x.dtype.str, x.shape)).encode())
            h.update(np.ascontiguousarray(x).tobytes())
        elif isinstance(x, (list, tuple)):
            h.update(b"(%d" % len(x))
            for y in x:
                feed(y)
            h.update(b")")
        elif isinstance(x, (bool, np.bool_, int, np.integer)):
            h.update(b"i%d" % int(x))
        elif isinstance(x, (float, np.floating)):
            h.update(b"f" + float(x).hex().encode())
        elif isinstance(x, (str, bytes)):
            b = x.encode() if isinstance(x, str) else x
            h.update(b"s%d:" % len(b) + b)
        else:
            raise TypeError("digest: %r" % type(x))
    for x in items:
        feed(x)
    return h.hexdigest()


class ReferenceResults:
    """The results of the reference implementation (the C++ sources this project ports, which are not part of the
    repository) on the seeded inputs of one test, stored as digests in tests/golden/reference_digests.json, one per
    result in the order the test produces them.  A digest keeps the comparison exact while the file stays small.

    These tests used to compare with a reference built from its sources.  The digests were recorded from this project's
    side of each comparison (the oracle, the host walk or the GPU) with the code of commit 5fbca29, at which every one
    of these tests ran against the live reference on exactly these inputs and passed: they are the reference's results.

    With AADP_RECORD_REFERENCE_DIGESTS=<file> set, the digests of what the test computes are written to <file> instead
    of compared; that is only a record of the reference where the same results were compared with it."""

    def __init__(self, test):
        self.test = test
        self.record = os.environ.get("AADP_RECORD_REFERENCE_DIGESTS")
        self.got = []
        self.want = None
        if not self.record:
            with open(REFERENCE_DIGESTS) as f:
                self.want = json.load(f).get(test)
            assert self.want, "no reference results stored for " + test

    def check(self, label, *items):
        d = digest(*items)
        i = len(self.got)
        self.got.append(d)
        if self.record:
            return
        assert i < len(self.want), "%s: more results than the reference has (%s)" % (self.test, label)
        assert d == self.want[i], "%s: result %d (%s) differs from the reference's" % (self.test, i, label)

    def close(self):
        if self.record:
            data = {}
            if os.path.exists(self.record):
                with open(self.record) as f:
                    data = json.load(f)
            data[self.test] = self.got
            with open(self.record, "w") as f:
                json.dump(data, f, indent=0, sort_keys=True)
                f.write("\n")
        else:
            assert len(self.got) == len(self.want), "%s: %d results, the reference has %d" % (
                self.test, len(self.got), len(self.want))


def assert_matrix_equal(name, got, want):
    got = np.asarray(got)
    want = np.asarray(want)
    assert got.shape == want.shape, "%s: shape %s vs %s" % (name, got.shape, want.shape)
    bad = np.argwhere(got != want)
    assert len(bad) == 0, "%s: %d mismatching cells, first at %s: got %s want %s" % (
        name, len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])


def subali_walk(S, PQ, PT, rect):
    """Optimal_Subali::enumerate (optimal_subali.h:59-83) over reference-shaped dense matrices: (status, aligned pairs
    from (q1_end, t1_end) to (q2_beg, t2_beg), score of the final cell)."""
    q1, t1, q2, t2 = [int(x) for x in rect]
    i, j = q2, t2
    path = [(i, j)]
    while i > q1:
        i, j = int(PQ[i, j]), int(PT[i, j])
        path.insert(0, (i, j))
    return (0 if (i, j) == (q1, t1) else 3), np.array(path, np.int32).reshape(-1, 2), S[q2, t2]
