"""Thin Python view of the C ABI (include/aadp.h), used by the tests and by bench.py.

The product's host side is C++ (include/hmap2/*.h mirrors the reference's template API);
this module only marshals numpy / torch buffers into the same C entry points.
"""
import ctypes as C

import numpy as np

from ._lib import lib

GLOBAL_LOCAL, GLOBAL, LOCAL_GLOBAL, LOCAL, SEMI_LOCAL = 0, 1, 2, 3, 4  # alib.h:20-26
FWD, REV, BOTH = 1, 2, 3                                               # dpmatrix.h:23-26
REPRO_REV_BUG = 1
W_FWD, W_REV, W_TB, W_SCORES, W_MASK = 1, 2, 4, 8, 16


class AadpError(RuntimeError):
    pass


def _ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """One device + stream.  Mirrors the life of a reference DPMatrix/Evaluator pair."""

    def __init__(self, device=0):
        self.L = lib()
        self.h = self.L.aadp_create(device)
        if not self.h:
            raise AadpError(self.L.aadp_last_error().decode())
        self.align_type = None
        self.flags = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.aadp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise AadpError(self.L.aadp_last_error().decode())

    def set_stream(self, cuda_stream_ptr):
        self._ck(self.L.aadp_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))

    def set_option(self, key, value):
        self._ck(self.L.aadp_set_option(self.h, key.encode(), int(value)))

    def synchronize(self):
        self._ck(self.L.aadp_synchronize(self.h))

    def set_scoring(self, sub, gi, ge, align_type, flags=REPRO_REV_BUG):
        sub = np.ascontiguousarray(sub, dtype=np.float32)
        assert sub.ndim == 2 and sub.shape[0] == sub.shape[1]
        self._ck(self.L.aadp_set_scoring(self.h, _ptr(sub), sub.shape[0], gi, ge, align_type, flags))
        self.align_type, self.flags = align_type, flags

    @staticmethod
    def pack_profiles(profiles):
        """Position-specific template profiles, indexed by sequence id: an (L, A) array per sequence (row j-1 = the scores
        of query codes 0..A-1 against template position j) or None for a sequence that is only ever a query.
        Returns (prof float32[total], prof_off int64[n+1], A) as aadp_set_profile_scoring takes them."""
        arrs = [None if p is None else np.asarray(p, np.float32) for p in profiles]
        widths = {a.shape[1] for a in arrs if a is not None and a.ndim == 2}
        if any(a is not None and a.ndim != 2 for a in arrs) or len(widths) != 1:
            raise ValueError("profiles: (L, A) arrays with one A for every sequence (None for query-only sequences)")
        A = widths.pop()
        off = np.zeros(len(arrs) + 1, np.int64)
        off[1:] = np.cumsum([0 if a is None else a.size for a in arrs])
        data = [a.ravel() for a in arrs if a is not None and a.size]
        prof = np.ascontiguousarray(np.concatenate(data) if data else np.zeros(0, np.float32), np.float32)
        return prof, off, A

    def set_profile_scoring(self, profiles, gi, ge, align_type, flags=REPRO_REV_BUG):
        """aadp_set_profile_scoring: a pair with template sequence t scores sim(i, j) = profiles[t][j-1, q_i]."""
        prof, off, A = self.pack_profiles(profiles)
        self._ck(self.L.aadp_set_profile_scoring(self.h, _ptr(prof), _ptr(off), len(off) - 1, A, gi, ge, align_type, flags))
        self.align_type, self.flags = align_type, flags

    # ---- single pair (DPMatrix constructor replacement) ----
    def fill_pair(self, q, t, direction=FWD, delta_ratio=-1.0, want_tb=True, want_scores=True):
        q = np.ascontiguousarray(q, dtype=np.uint8)
        t = np.ascontiguousarray(t, dtype=np.uint8)
        sz = (len(q) + 2, len(t) + 2)
        out = {}

        def mk(name, dt, cond):
            out[name] = np.zeros(sz, dt) if cond else None
            return _ptr(out[name])

        f, r = bool(direction & 1), bool(direction & 2)
        args = [mk("score_fwd", np.float32, f and want_scores), mk("prevq_fwd", np.int32, f and want_tb),
                mk("prevt_fwd", np.int32, f and want_tb), mk("score_rev", np.float32, r and want_scores),
                mk("prevq_rev", np.int32, r and want_tb), mk("prevt_rev", np.int32, r and want_tb)]
        want_mask = delta_ratio >= 0 and direction == BOTH
        args.append(mk("nearopt", np.uint8, want_mask))
        thr = C.c_float(0)
        self._ck(self.L.aadp_fill_pair(self.h, _ptr(q), len(q), _ptr(t), len(t), direction, delta_ratio,
                                       *args, C.cast(C.byref(thr), C.c_void_p) if want_mask else None))
        out["threshold"] = thr.value if want_mask else None
        return out

    def fill_subpair(self, q, t, rect, direction=FWD):
        """build_subdpm (dpmatrix.h:319-353): rect = (q1_end, t1_end, q2_beg, t2_beg), matrix indices."""
        q = np.ascontiguousarray(q, dtype=np.uint8)
        t = np.ascontiguousarray(t, dtype=np.uint8)
        sz = (len(q) + 2, len(t) + 2)
        s, pq, pt = np.zeros(sz, np.float32), np.zeros(sz, np.int32), np.zeros(sz, np.int32)
        self._ck(self.L.aadp_fill_subpair(self.h, _ptr(q), len(q), _ptr(t), len(t), int(rect[0]), int(rect[1]),
                                          int(rect[2]), int(rect[3]), direction, _ptr(s), _ptr(pq), _ptr(pt)))
        return s, pq, pt

    def fill_subpair_batch(self, residues, seq_off, item_q, item_t, rects, direction=FWD, want_alignments=True):
        """Many build_subdpm fills + Optimal_Subali tracebacks in one call (ssss.h:621-633 loop closure).
        rects: (n, 4) = (q1_end, t1_end, q2_beg, t2_beg) per item.  Returns (score[n], ali_off[n+1], pairs[(total,2)],
        n_out[n], status[n]); the last three are None when want_alignments is False (or direction is REV)."""
        item_q = np.ascontiguousarray(item_q, np.int32)
        item_t = np.ascontiguousarray(item_t, np.int32)
        rects = np.ascontiguousarray(rects, np.int32).reshape(-1, 4)
        n = len(item_q)
        assert len(item_t) == n and len(rects) == n
        off = np.zeros(n + 1, np.int64)
        self._ck(self.L.aadp_fill_subpair_batch(self.h, _ptr(residues), _ptr(seq_off), len(seq_off) - 1, _ptr(item_q),
                                                _ptr(item_t), _ptr(rects), n, direction, None, _ptr(off), None, 0, None,
                                                None))
        score = np.zeros(n, np.float32)
        ali = want_alignments and direction == FWD
        pairs = np.zeros((max(int(off[-1]), 1), 2), np.int32) if ali else None
        n_out = np.zeros(n, np.int32) if ali else None
        st = np.zeros(n, np.int32) if ali else None
        self._ck(self.L.aadp_fill_subpair_batch(self.h, _ptr(residues), _ptr(seq_off), len(seq_off) - 1, _ptr(item_q),
                                                _ptr(item_t), _ptr(rects), n, direction, _ptr(score), _ptr(off),
                                                _ptr(pairs), int(off[-1]), _ptr(n_out), _ptr(st)))
        return score, off, pairs, n_out, st

    def fill_pair_general(self, sim, gi, ge, align_type, direction=FWD, rect=None, flags=REPRO_REV_BUG):
        """Any evaluator with uniform affine gaps: sim is the (Lq+2, Lt+2) similarity matrix of simmatrix.h."""
        sim = np.ascontiguousarray(sim, dtype=np.float32)
        sz = sim.shape
        s, pq, pt = np.zeros(sz, np.float32), np.zeros(sz, np.int32), np.zeros(sz, np.int32)
        r = np.ascontiguousarray(rect, np.int32) if rect is not None else None
        self._ck(self.L.aadp_fill_pair_general(self.h, _ptr(sim), sz[0] - 2, sz[1] - 2, gi, ge, align_type, flags,
                                               direction, _ptr(r), _ptr(s), _ptr(pq), _ptr(pt)))
        return s, pq, pt

    def fill_pair_tabulated(self, sim, del_tab, ins_tab, is_local=False, direction=FWD, flags=REPRO_REV_BUG):
        """Any evaluator, position-dependent gaps included: sim (Lq+2, Lt+2), del_tab (Lt+2, Lt+2), ins_tab (Lq+1, Lt+2)
        as described in include/aadp.h (aadp_fill_pair_tabulated)."""
        sim = np.ascontiguousarray(sim, dtype=np.float32)
        del_tab = np.ascontiguousarray(del_tab, dtype=np.float32)
        ins_tab = np.ascontiguousarray(ins_tab, dtype=np.float32)
        sz = sim.shape
        assert del_tab.shape == (sz[1], sz[1]) and ins_tab.shape == (sz[0] - 1, sz[1])
        s, pq, pt = np.zeros(sz, np.float32), np.zeros(sz, np.int32), np.zeros(sz, np.int32)
        self._ck(self.L.aadp_fill_pair_tabulated(self.h, _ptr(sim), sz[0] - 2, sz[1] - 2, _ptr(del_tab), _ptr(ins_tab),
                                                 int(bool(is_local)), flags, direction, _ptr(s), _ptr(pq), _ptr(pt)))
        return s, pq, pt

    def fill_batch_tabulated(self, sims, dels, inss, is_local=False, direction=BOTH, want_alignments=True, flags=REPRO_REV_BUG):
        """Many tabulated pairs in one call (aadp_fill_batch_tabulated): lists of per-item sim / del_tab / ins_tab arrays.
        Returns (fwd_score, rev_score, ali_off, pairs, n_out, status)."""
        n = len(sims)
        Lq = np.array([s.shape[0] - 2 for s in sims], np.int32)
        Lt = np.array([s.shape[1] - 2 for s in sims], np.int32)

        def blob(arrs):
            off = np.zeros(n + 1, np.int64)
            off[1:] = np.cumsum([a.size for a in arrs])
            data = np.concatenate([np.ascontiguousarray(a, np.float32).ravel() for a in arrs]) if n else np.zeros(0, np.float32)
            return np.ascontiguousarray(data, np.float32), off

        (sb, so), (db, do), (ib, io) = blob(sims), blob(dels), blob(inss)
        fs = np.zeros(n, np.float32) if direction & 1 else None
        rs = np.zeros(n, np.float32) if direction & 2 else None
        aoff = np.zeros(n + 1, np.int64)
        ali = want_alignments and not is_local and (direction & 1)
        args = [self.h, n, _ptr(Lq), _ptr(Lt), _ptr(sb), _ptr(so), _ptr(db), _ptr(do), _ptr(ib), _ptr(io), int(bool(is_local)),
                flags, direction]
        self._ck(self.L.aadp_fill_batch_tabulated(*args, None, None, _ptr(aoff), None, 0, None, None))
        pairs = np.zeros((max(int(aoff[-1]), 1), 2), np.int32) if ali else None
        n_out = np.zeros(n, np.int32) if ali else None
        st = np.zeros(n, np.int32) if ali else None
        self._ck(self.L.aadp_fill_batch_tabulated(*args, _ptr(fs), _ptr(rs), _ptr(aoff), _ptr(pairs), int(aoff[-1]), _ptr(n_out),
                                                  _ptr(st)))
        return fs, rs, aoff, pairs, n_out, st

    # ---- batches ----
    @staticmethod
    def pack(seqs):
        lens = np.array([len(s) for s in seqs], np.int64)
        off = np.zeros(len(seqs) + 1, np.int64)
        off[1:] = np.cumsum(lens)
        res = np.concatenate([np.asarray(s, np.uint8) for s in seqs]) if len(seqs) else np.zeros(0, np.uint8)
        return np.ascontiguousarray(res, np.uint8), off

    def fill_batch(self, residues, seq_off, pair_q, pair_t, what, delta_ratio=0.01):
        pair_q = np.ascontiguousarray(pair_q, np.int32)
        pair_t = np.ascontiguousarray(pair_t, np.int32)
        n = len(pair_q)
        fs = np.zeros(n, np.float32) if what & W_FWD else None
        rs = np.zeros(n, np.float32) if what & W_REV else None
        th = np.zeros(n, np.float32) if what & W_MASK else None
        cn = np.zeros(n, np.int64) if what & W_MASK else None
        self._ck(self.L.aadp_fill_batch(self.h, _ptr(residues), _ptr(seq_off), len(seq_off) - 1, _ptr(pair_q),
                                        _ptr(pair_t), n, what, delta_ratio, _ptr(fs), _ptr(rs), _ptr(th), _ptr(cn)))
        return {"fwd_score": fs, "rev_score": rs, "threshold": th, "nearopt_count": cn}

    def fill_batch_submit(self, residues, seq_off, pair_q, pair_t, what, delta_ratio=0.01, out=None):
        """aadp_fill_batch_submit: host scheduling + everything enqueued, no final wait.  `out` may hold preallocated
        result arrays ("fwd_score", "rev_score", "threshold", "nearopt_count"; PINNED memory keeps the device-to-host
        copies asynchronous); inputs and outputs must stay alive and untouched until fill_batch_wait()."""
        pair_q = np.ascontiguousarray(pair_q, np.int32)
        pair_t = np.ascontiguousarray(pair_t, np.int32)
        n = len(pair_q)
        out = dict(out) if out else {}
        want = {"fwd_score": (what & W_FWD, np.float32), "rev_score": (what & W_REV, np.float32),
                "threshold": (what & W_MASK, np.float32), "nearopt_count": (what & W_MASK, np.int64)}
        for k, (on, ty) in want.items():
            if not on:
                out[k] = None
            elif out.get(k) is None:
                out[k] = np.zeros(n, ty)
        self._ck(self.L.aadp_fill_batch_submit(self.h, _ptr(residues), _ptr(seq_off), len(seq_off) - 1, _ptr(pair_q),
                                               _ptr(pair_t), n, what, delta_ratio, _ptr(out["fwd_score"]), _ptr(out["rev_score"]),
                                               _ptr(out["threshold"]), _ptr(out["nearopt_count"])))
        self._pending = (residues, seq_off, pair_q, pair_t, out)  # keep the buffers alive (a refused submit leaves the old ones)
        return out

    def fill_batch_wait(self):
        """aadp_fill_batch_wait: returns when the results of the submitted batch are in the output arrays."""
        self._ck(self.L.aadp_fill_batch_wait(self.h))
        out = getattr(self, "_pending", (None,) * 5)[4]
        self._pending = None
        return out

    def upload_batch(self, residues, seq_off, pair_q, pair_t, what):
        pair_q = np.ascontiguousarray(pair_q, np.int32)
        pair_t = np.ascontiguousarray(pair_t, np.int32)
        self._ck(self.L.aadp_upload_batch(self.h, _ptr(residues), _ptr(seq_off), len(seq_off) - 1, _ptr(pair_q),
                                          _ptr(pair_t), len(pair_q), what))

    def run_batch(self, what, delta_ratio=0.01, d_fwd=None, d_rev=None, d_thr=None, d_cnt=None):
        """d_* are raw device pointers (ints) or None."""
        self._ck(self.L.aadp_run_batch(self.h, what, delta_ratio, d_fwd, d_rev, d_thr, d_cnt))

    # ---- all queries x all templates, forward score only ----
    def upload_sequences(self, residues, seq_off):
        self._ck(self.L.aadp_upload_sequences(self.h, _ptr(residues), _ptr(seq_off), len(seq_off) - 1))

    def cross_run(self, q_ids, t_ids, d_scores):
        """d_scores: raw device pointer (int) to len(q_ids)*len(t_ids) floats."""
        q_ids = np.ascontiguousarray(q_ids, np.int32)
        t_ids = np.ascontiguousarray(t_ids, np.int32)
        self._ck(self.L.aadp_cross_run(self.h, _ptr(q_ids), len(q_ids), _ptr(t_ids), len(t_ids), d_scores))

    def cross_scores(self, residues, seq_off, q_ids, t_ids):
        q_ids = np.ascontiguousarray(q_ids, np.int32)
        t_ids = np.ascontiguousarray(t_ids, np.int32)
        out = np.zeros((len(q_ids), len(t_ids)), np.float32)
        self._ck(self.L.aadp_cross_scores(self.h, _ptr(residues), _ptr(seq_off), len(seq_off) - 1, _ptr(q_ids),
                                          len(q_ids), _ptr(t_ids), len(t_ids), _ptr(out)))
        return out

    def last_cross_cell_updates(self):
        return self.L.aadp_last_cross_cell_updates(self.h)

    def resident_bytes(self, which):
        return self.L.aadp_batch_resident_bytes(self.h, which)

    def last_launch_count(self):
        return self.L.aadp_last_launch_count(self.h)

    def last_transfer_bytes(self):
        return self.L.aadp_last_h2d_bytes(self.h), self.L.aadp_last_d2h_bytes(self.h)

    def last_cell_updates(self):
        return self.L.aadp_last_cell_updates(self.h)

    def set_profiling(self, on):
        self._ck(self.L.aadp_set_profiling(self.h, int(bool(on))))

    def profile(self):
        """[(kernel name, ms, cell updates)] of the last run (needs set_profiling(True))."""
        out = []
        buf = C.create_string_buffer(96)
        for i in range(self.L.aadp_profile_count(self.h)):
            ms, cells = C.c_float(0), C.c_double(0)
            self._ck(self.L.aadp_profile_get(self.h, i, C.cast(buf, C.c_void_p), 96,
                                             C.cast(C.byref(ms), C.c_void_p), C.cast(C.byref(cells), C.c_void_p)))
            out.append((buf.value.decode(), ms.value, cells.value))
        return out

    def fetch_pair(self, p, Lq, Lt, fwd=True, rev=False, tb=True, scores=True, mask=False):
        sz = (Lq + 2, Lt + 2)
        out = {}

        def mk(name, dt, cond):
            out[name] = np.zeros(sz, dt) if cond else None
            return _ptr(out[name])

        args = [mk("score_fwd", np.float32, fwd and scores), mk("prevq_fwd", np.int32, fwd and tb),
                mk("prevt_fwd", np.int32, fwd and tb), mk("score_rev", np.float32, rev and scores),
                mk("prevq_rev", np.int32, rev and tb), mk("prevt_rev", np.int32, rev and tb),
                mk("nearopt", np.uint8, mask)]
        self._ck(self.L.aadp_batch_fetch_pair(self.h, p, *args))
        return out

    def optimal(self, p, direction, Lq, Lt):
        cap = Lq + Lt + 8
        pairs = np.zeros((cap, 2), np.int32)
        n = C.c_int32(0)
        s = C.c_float(0)
        rc = self.L.aadp_batch_optimal(self.h, p, direction, _ptr(pairs), cap, C.cast(C.byref(n), C.c_void_p),
                                       C.cast(C.byref(s), C.c_void_p))
        if rc not in (0, 3):
            raise AadpError(self.L.aadp_last_error().decode())
        return rc, pairs[: min(n.value, cap)].copy(), s.value

    def optimal_all(self, direction, npairs, bufs=None):
        """Optimal alignments of every pair of the resident batch (GPU traceback).
        Returns (ali_off, pairs[(total,2)], n[npairs], status[npairs]).  bufs = (off, pairs, n, status): caller-owned
        (e.g. pinned) arrays reused across calls; pairs must hold ali_off[-1] rows."""
        off = np.zeros(npairs + 1, np.int64) if bufs is None else bufs[0]
        self._ck(self.L.aadp_batch_optimal_all(self.h, direction, _ptr(off), None, 0, None, None))
        if bufs is None:
            pairs = np.zeros((max(int(off[-1]), 1), 2), np.int32)
            n = np.zeros(npairs, np.int32)
            st = np.zeros(npairs, np.int32)
        else:
            _, pairs, n, st = bufs
            if len(pairs) < int(off[-1]):
                raise AadpError("optimal_all: pairs buffer too small (%d rows needed)" % int(off[-1]))
        self._ck(self.L.aadp_batch_optimal_all(self.h, direction, _ptr(off), _ptr(pairs), int(off[-1]), _ptr(n), _ptr(st)))
        return off, pairs, n, st

    def optimal_all_compact(self, direction, npairs, pairs=None, pairs_cap=None):
        """Optimal alignments of every pair, packed: (ali_off[npairs+1], pairs[(cap,2)], n[npairs], status[npairs]).
        pairs: caller-owned (e.g. pinned) (cap,2) int32 array; by default sized by the capacity bound."""
        off = np.zeros(npairs + 1, np.int64)
        if pairs is None:
            capo = np.zeros(npairs + 1, np.int64)
            self._ck(self.L.aadp_batch_optimal_all(self.h, direction, _ptr(capo), None, 0, None, None))
            pairs = np.zeros((max(int(capo[-1]), 1), 2), np.int32)
        n = np.zeros(npairs, np.int32)
        st = np.zeros(npairs, np.int32)
        self._ck(self.L.aadp_batch_optimal_all_compact(self.h, direction, _ptr(off), _ptr(pairs), len(pairs), _ptr(n), _ptr(st)))
        return off, pairs, n, st

    def near_optimal(self, pair_ids, delta_ratio, max_alignments, subopt_flags=None, constrained=False):
        """UnconstrainedNearOptimal::enumerate (ucw.h:63-191, before sortSet) of the listed pairs on the GPU -- or, with
        constrained=True, ConstrainedNearOptimal::enumerate (cw.h:60-284) with subopt_flags = one array of Lt+2 flags per
        listed pair (None = all true).
        Returns a list (one entry per listed pair) of (status, threshold, [(score, pairs[(len,2)]) in depth-first order])."""
        ids = np.ascontiguousarray(pair_ids, np.int64)
        n, K = len(ids), int(max_alignments)
        off = np.zeros(n + 1, np.int64)
        if constrained:
            fl, fo = None, None
            if subopt_flags is not None:
                fo = np.zeros(n + 1, np.int64)
                fo[1:] = np.cumsum([len(f) for f in subopt_flags])
                fl = np.ascontiguousarray(np.concatenate([np.asarray(f, np.uint8) for f in subopt_flags]), np.uint8)

            def call(*a):
                return self.L.aadp_batch_near_optimal_constrained(self.h, _ptr(ids), n, _ptr(fl), _ptr(fo), delta_ratio, K, *a)
        else:
            def call(*a):
                return self.L.aadp_batch_near_optimal(self.h, _ptr(ids), n, delta_ratio, K, *a)
        self._ck(call(None, None, None, None, _ptr(off), None, 0, None))
        n_ali, st = np.zeros(n, np.int32), np.zeros(n, np.int32)
        scores, ln = np.zeros((n, K), np.float32), np.zeros((n, K), np.int32)
        paths = np.zeros((max(int(off[-1]), 1), 2), np.int32)
        thr = np.zeros(n, np.float32)
        self._ck(call(_ptr(n_ali), _ptr(st), _ptr(scores), _ptr(ln), _ptr(off), _ptr(paths), int(off[-1]), _ptr(thr)))
        out = []
        for k in range(n):
            slot = (off[k + 1] - off[k]) // K
            alis = [(float(scores[k, a]), paths[off[k] + a * slot: off[k] + a * slot + ln[k, a]].copy())
                    for a in range(n_ali[k])]
            out.append((int(st[k]), float(thr[k]), alis))
        return out

    def near_optimal_pruned(self, p, variant, delta_ratio, Lq, Lt, flags=None, k_limit=16, sort_limit=100, max_overlap=0.30,
                            user_limit=100000, max_alignments=20000):
        """KSConstrainedNearOptimal (variant=PRUNE_KSORTED, kscw.h) / CRConstrainedNearOptimal (PRUNE_REDUNDANCY, crcw.h) of
        pair p of the resident batch: (status, threshold, [(score, pairs[(len,2)])]) in the reference's slot order."""
        K = int(max_alignments)
        cap = K * (Lq + Lt + 4)
        scores = np.zeros(K, np.float32)
        ln = np.zeros(K, np.int32)
        paths = np.zeros((cap, 2), np.int32)
        n, st, thr = C.c_int32(0), C.c_int32(0), C.c_float(0)
        fl = np.ascontiguousarray(flags, np.uint8) if flags is not None else None
        self._ck(self.L.aadp_batch_near_optimal_pruned(
            self.h, int(p), int(variant), _ptr(fl) if fl is not None else None, delta_ratio, k_limit, sort_limit, max_overlap,
            user_limit, K, C.cast(C.byref(n), C.c_void_p), C.cast(C.byref(st), C.c_void_p), _ptr(scores), _ptr(ln), _ptr(paths),
            cap, C.cast(C.byref(thr), C.c_void_p)))
        out, o = [], 0
        for k in range(min(n.value, K)):
            out.append((float(scores[k]), paths[o:o + ln[k]].copy()))
            o += ln[k]
        return st.value, thr.value, out

    def fetch_tb(self, p, direction, Lq, Lt):
        nbytes = max(int(self.L.aadp_batch_tb_bytes(self.h, p)), 1)
        tb = np.zeros(nbytes, np.uint8)
        fin = np.zeros(6, np.int32)
        self._ck(self.L.aadp_batch_fetch_tb(self.h, p, direction, _ptr(tb), nbytes, _ptr(fin)))
        return tb, fin

    def decode_cell(self, tb, fin, Lq, Lt, direction, i, j):
        pq, pt = C.c_int32(0), C.c_int32(0)
        self._ck(self.L.aadp_decode_cell(_ptr(tb), Lq, Lt, direction, self.align_type, self.flags, _ptr(fin), i, j,
                                         C.cast(C.byref(pq), C.c_void_p), C.cast(C.byref(pt), C.c_void_p)))
        return pq.value, pt.value
