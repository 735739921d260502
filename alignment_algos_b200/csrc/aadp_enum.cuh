// aadp_enum.cuh -- near-optimal ENUMERATION on the GPU for sm_100a (SURVEY.md §8 row f1).
//
// UnconstrainedNearOptimal::enumerate / branch (ucw.h:63-191): a depth-first walk from the final cell towards the
// anchor that follows every predecessor satisfying Waterman's condition  F[pred] + r - g > threshold, where r is the
// score accumulated from the end of the alignment and g the gap penalty of the step.  Each root-to-leaf path of the
// walk is one near-optimal alignment; the reference numbers them in depth-first order (slot k of the AlignmentSet)
// and sorts them by score afterwards (sortSet, alignment.h:922-932).
//
// Mapping.  The walk of ONE pair is sequential, but the two candidate scans of a node (ucw.h:154-180: a whole row and
// a whole column of the forward matrix) are not: one WARP owns a pair, its 32 lanes test 32 candidates at a time and a
// ballot picks the first one in the reference's order (match, deletions t0-2..1, insertions q0-2..1).  The
// recursion is an explicit stack of frames in HBM (one frame per alignment position, <= Lq+1 deep).  The forward
// scores are read straight from the RESIDENT batch products (packed int16 diagonal-major blob of the packed kernels or
// the row-major blob of the int32 kernels) -- no dense matrix is expanded.  Batch-level parallelism: one warp per
// listed pair, thousands of pairs per launch.
//
// ConstrainedNearOptimal (cw.h:60-284, template CNO=1) is the same walk with branching restricted by per-template-
// position SuboptFlags: after every accepted branch the optimal predecessors (DPCell::prev_*, here the packed traceback
// decoded on the fly) are followed until the flag changes state (cw.h:247-272, rule #1), and only there the candidates
// are scanned again.  Both variants share one kernel: the current partial alignment lives in a per-warp path buffer,
// a frame remembers its length.
//
// Arithmetic is the reference's fp32 in the reference's order: r = curr + sim; (f + r) - g > thr; score = r - g;
// leaf: score += D[q0][t0].score.  On the dyadic grid the integer kernels require, every value is exact, so the
// alignments, their order and their scores are bit-identical.  The opt_path fallback (ucw.h:182-236) is reachable
// through rounding (a cell that passed always has a passing predecessor in exact arithmetic) and through the
// reference's alignment limit (ucw.h:72: 100000, cw.h:76: 1000000), reproduced here as `user_limit`: beyond it every
// further branch() completes its alignment along the optimal predecessors (needs the traceback).  A pair that exceeds
// its OUTPUT budget is flagged (status 1); a walk that needs predecessors the batch did not keep is flagged status 2.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "aadp_kernels.cuh"

namespace aadp {

struct UcwParams {
  int A;
  const float* subf;          // A*A substitution scores
  float gi, ge;               // gap(len) = gi + ge*(len-1) (aasubalib.h:37-38)
  int delfree, insfree;       // free end gaps (aasubalib.h:39-42, 65-68)
  float inv_scale;            // score units -> float
  const uint8_t* residues;
  const int64_t* seq_off;
  const int32_t* pair_q;
  const int32_t* pair_t;
  const uint8_t* fmt;         // per pair: layout class (1 = packed)
  const void* sc_blob;        // forward score blob
  const int64_t* sc_off;      // per pair
  int st_mode_v1;             // storage of the non-packed pairs: 1 = int16, 2 = int32
  int bias16;                 // bias of the packed int16 domain
  const int32_t* fin_score;   // per pair: D[last][last].score in score units
  const uint32_t* mask;       // near-optimal cell set of the batch (same delta_ratio), or null: prunes the deletion scans
  const int64_t* mask_off;    // per pair (32-bit words)
  const uint8_t* tb;          // packed forward traceback blob (the optimal walks of cw.h), or null
  const int64_t* tb_off;
  // exact-float mode (one listed pair per launch): the dense fp32 forward matrix of the general-gap kernel and its
  // predecessors instead of the resident integer products; null otherwise
  const float* denseF;
  const int32_t* densePQ;
  const int32_t* densePT;
  const int64_t* dense_off;   // per listed pair of the launch: offset of its dense matrices
  const int64_t* ids;         // listed pairs
  int n;
  float delta_ratio;
  int max_ali;                // output budget per pair
  int user_limit;             // ucw.h:72 / cw.h:76: once this many alignments are complete, every further branch() forces
                              // the optimal path to the beginning (ucw.h:115-126, cw.h:118-130) instead of branching
  const uint8_t* subopt;      // CNO: SuboptFlags per template position (Lt+2 bytes per listed pair), null = all true
  const int64_t* subopt_off;  // per listed pair
  const int64_t* path_off;    // per listed pair: first slot; alignment a of pair k lives at path_off[k] + a*(Lq+2)
  int2* paths;                // aligned pairs front to back, (0,0) first
  int32_t* ali_len;           // [k*max_ali + a]
  float* scores;              // [k*max_ali + a]
  int32_t* n_ali;             // per listed pair
  int32_t* status;            // per listed pair: 0, 1 = more than max_ali alignments (output truncated), 2 = see above
  float* threshold;           // per listed pair, or null
  const int64_t* stack_off;   // per listed pair: first entry of its frame stack / path buffer (Lq+2 entries each)
  int4* stack;                // frames: (q0, t0, __float_as_int(curr), next candidate | any<<30)
  int32_t* frame_plen;        // per frame: length of the path buffer when the frame was entered
  int2* pathbuf;              // the partial alignment from the final cell down to the current node
};

// PRO = 1: sim() reads the fp32 position-specific template profile (ProfDev, aadp_set_profile_scoring); exact on the grid.
template <int CNO, int PRO = 0>
__global__ void __launch_bounds__(128, 8) ucw_enum_kernel(const UcwParams P, const ProfDev pd) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= P.n) return;
  const int64_t pair = P.ids[warp];
  const int qs = P.pair_q[pair], ts = P.pair_t[pair];
  const int64_t qo = P.seq_off[qs], to = P.seq_off[ts];
  const int Lq = (int)(P.seq_off[qs + 1] - qo), Lt = (int)(P.seq_off[ts + 1] - to);
  const uint8_t* qseq = P.residues + qo;
  const uint8_t* tseq = P.residues + to;
  const int fmt = P.denseF ? 0 : P.fmt[pair];  // exact-float batches have no layout tables
  const Layout L = make_layout(Lq, Lt, fmt, 0);
  const int st_mode = fmt == 1 ? 1 : P.st_mode_v1;
  const int bias = fmt == 1 ? P.bias16 : 0;
  const int64_t sco = P.denseF ? 0 : P.sc_off[pair];
  const uint8_t* tb = (P.denseF || !P.tb) ? nullptr : P.tb + P.tb_off[pair];
  const float inv = P.inv_scale;
  const int sz2 = Lt + 2;
  const int64_t dbase = P.denseF ? P.dense_off[warp] : 0;
  const float* denseF = P.denseF ? P.denseF + dbase : nullptr;
  const int32_t* densePQ = P.densePQ ? P.densePQ + dbase : nullptr;
  const int32_t* densePT = P.densePT ? P.densePT + dbase : nullptr;
  // DPCell::score of the forward matrix (interior cells and the final cell)
  auto F = [&](int i, int j) -> float {
    if (denseF) return denseF[(int64_t)i * sz2 + j];
    if (i == Lq + 1 && j == Lt + 1) return (float)P.fin_score[pair] * inv;
    int si;
    if (st_mode == 1) si = (int)((const int16_t*)P.sc_blob)[sco + layout_sc_index(L, i, j)] - bias;
    else si = ((const int32_t*)((const int16_t*)P.sc_blob + sco))[layout_sc_index(L, i, j)];
    return (float)si * inv;
  };
  auto sim = [&](int i, int j) -> float {  // aasubalib.h:17-25
    if (i < 1 || i > Lq || j < 1 || j > Lt) return 0.f;
    if constexpr (PRO) return pd.pf[pd.offf[ts] + (int64_t)(j - 1) * P.A + (int)qseq[i - 1]];
    return P.subf[(int)qseq[i - 1] * P.A + (int)tseq[j - 1]];
  };
  auto pen = [&](int len) { return __fadd_rn(P.gi, __fmul_rn(P.ge, (float)(len - 1))); };
  // DPCell::prev_* of an interior cell; false when this batch cannot answer (no traceback kept / the final cell)
  auto prev = [&](int a, int b, int* pa, int* pb) -> bool {
    if (densePQ) { *pa = densePQ[(int64_t)a * sz2 + b]; *pb = densePT[(int64_t)a * sz2 + b]; return true; }
    if (!tb || a > Lq || b > Lt) return false;
    decode_prev(tb, L, a, b, pa, pb);
    return true;
  };
  // gap penalty of the step (pa,pb) -> (a,b) as opt_path evaluates it (ucw.h:222-226, cw.h:262-266)
  auto step_gap = [&](int pa, int pb, int a, int b) -> float {
    if (a - pa == 1) {  // deletion(pq,q0,pt,t0), aasubalib.h:27-51
      const int len = b - pb - 1;
      return (len >= 1 && !(P.delfree && (pb == 0 || b == Lt + 1))) ? pen(len) : 0.f;
    }
    const int len = a - pa - 1;  // insertion(pq,q0,pt,t0), aasubalib.h:53-77
    return (len >= 1 && !(P.insfree && (pa == 0 || a == Lq + 1))) ? pen(len) : 0.f;
  };
  const uint8_t* so_flags = (CNO && P.subopt) ? P.subopt + P.subopt_off[warp] : nullptr;
  auto subopt = [&](int t) -> bool { return so_flags ? so_flags[t] != 0 : true; };

  const float opt = F(Lq + 1, Lt + 1);
  const float thr = fminf(__fmul_rn(1.f - P.delta_ratio, opt), __fsub_rn(opt, 0.1f));  // ucw.h:81-83, cw.h:86-88
  if (lane == 0 && P.threshold) P.threshold[warp] = thr;

  // near-optimal set of this pair as 16-bit slot words (packed layout only: reverse-flow coordinates, diagonal-major)
  const uint16_t* mkrow = (P.mask && !P.denseF && fmt == 1) ? reinterpret_cast<const uint16_t*>(P.mask + P.mask_off[pair]) : nullptr;
  const int cap = Lq + 2;  // every step lowers the query index: at most Lq+2 aligned pairs
  int2* paths = P.paths + P.path_off[warp];
  int4* stack = P.stack + P.stack_off[warp];
  int32_t* frame_plen = P.frame_plen + P.stack_off[warp];
  int2* pathbuf = P.pathbuf + P.stack_off[warp];
  int32_t* ali_len = P.ali_len + (int64_t)warp * P.max_ali;
  float* scores = P.scores + (int64_t)warp * P.max_ali;
  int count = 0, status = 0, plen = 0, depth = 0;

  // base case (ucw.h:94-101, cw.h:102-110): the alignment is (0,0), the leaf, then the partial alignment back to front.
  // CNO keeps all of it in the path buffer (frames and optimal walks interleaved); UCW has one node per frame, so the
  // frame stack IS the path and the buffer only holds the nodes of a forced optimal walk below the deepest frame.
  auto emit = [&](int lq, int lt, float s) -> bool {
    if (count >= P.max_ali) { status = 1; return false; }
    __syncwarp();
    int2* out = paths + (int64_t)count * cap;
    const int len = (CNO ? 0 : depth) + plen + 2;
    for (int k = lane; k < len; k += 32) {
      int2 v;
      if (k == 0) v = make_int2(0, 0);
      else if (k == 1) v = make_int2(lq, lt);
      else if (k < plen + 2) v = pathbuf[plen + 1 - k];
      else { const int4 f = stack[depth - 1 - (k - plen - 2)]; v = make_int2(f.x, f.y); }
      out[k] = v;
    }
    if (lane == 0) { ali_len[count] = len; scores[count] = s; }
    ++count;
    return true;
  };
  // opt_path (ucw.h:194-236, cw.h:213-281): follow the stored predecessors from (a,b), extending the alignment and its
  // score; forced = to the base case, otherwise (cw.h rule #1) until the SuboptFlag of the template position changes.
  auto walk = [&](int& a, int& b, float& s, bool forced) -> bool {
    const bool flag = !subopt(b);
    while (b > 1 && a > 1) {
      if (!forced && subopt(b) == flag) break;
      if (lane == 0) pathbuf[plen] = make_int2(a, b);
      ++plen;
      s = __fadd_rn(s, sim(a, b));
      int pa, pb;
      if (!prev(a, b, &pa, &pb)) { status = 2; return false; }
      s = __fsub_rn(s, step_gap(pa, pb, a, b));
      a = pa; b = pb;
    }
    return true;
  };

  // frame in registers (uniform across the warp); stack[d] holds the frames below it
  int q0 = Lq + 1, t0 = Lt + 1, next = 0, any = 0;
  float curr = 0.f;
  for (;;) {
    if (q0 == 1 || t0 == 1) {
      if (!emit(q0, t0, __fadd_rn(curr, F(q0, t0)))) break;
    } else if (next == 0 && count >= P.user_limit) {
      // as.size() > user_limit at the ENTRY of a branch() call (as.size() = completed alignments + the one in progress):
      // the reference stops branching and completes this alignment along the optimal predecessors.  A frame that is
      // re-entered (next > 0) is a branch() that started before the limit was reached: its candidate loops continue.
      int a = q0, b = t0;
      float s = curr;
      if (!walk(a, b, s, true)) break;
      if (!emit(a, b, __fadd_rn(s, F(a, b)))) break;
    } else {
      const float r = __fadd_rn(curr, sim(q0, t0));  // ucw.h:141
      const int ndel = t0 - 2, total = 1 + ndel + (q0 - 2);
      int found = -1, cq = 0, ct = 0;
      float cg = 0.f;
      int scan_from = next;
      if (mkrow && next <= ndel) {
        // PRUNED deletion scan (packed pairs with a resident near-optimal set of the same delta): a predecessor can
        // only pass  F[pred] + r - g > thr  if it lies in the set  F + R - sim > thr  (r - g is the score of ONE way to
        // continue from it, R - sim of the best one; exact on the integer grid).  The set's bits of matrix row q0-1 sit
        // in one 16-bit word per 16-column slot: lane s fetches slot s, then only the non-empty slots are tested, 16
        // candidates at a time, in the reference's order (match first, then template positions t0-2 .. 1).
        const int iq = q0 - 1;
        const int a_rev = Lq + 1 - iq;                 // reverse-flow row of matrix row iq
        const int shift = Lt + 2 - t0;                 // candidate index of reverse-flow column bb: idx = bb - shift
        unsigned m16 = 0;
        if (lane < L.n) {
          const unsigned v = mkrow[((int64_t)(a_rev - 1 + lane) * L.n + lane)];  // byte (cc & 1), bit 7 - (cc >> 1)
#pragma unroll
          for (int cc = 0; cc < 16; ++cc) {
            const int idx = 16 * lane + cc + 1 - shift;
            if (idx >= max(next, 1) && idx <= ndel && ((v >> (8 * (cc & 1) + 7 - (cc >> 1))) & 1u)) m16 |= 1u << cc;
          }
        }
        bool first = true;
        for (;;) {
          const unsigned nonempty = __ballot_sync(0xffffffffu, m16 != 0);
          const bool with_match = first && next == 0;
          if (!nonempty && !with_match) break;
          const int sl = nonempty ? __ffs(nonempty) - 1 : 0;
          const unsigned ms = nonempty ? __shfl_sync(0xffffffffu, m16, sl) : 0u;
          bool pass = false;
          int it = 0, idx = 0;
          float g = 0.f;
          if (lane < 16) {
            if ((ms >> lane) & 1u) {
              idx = 16 * sl + lane + 1 - shift;
              it = t0 - 1 - idx;
              g = (P.delfree && t0 == Lt + 1) ? 0.f : pen(t0 - it - 1);
              pass = __fsub_rn(__fadd_rn(F(iq, it), r), g) > thr;
            }
          } else if (lane == 31 && with_match) {  // the match candidate (idx 0) rides along in the first round
            it = t0 - 1;
            pass = __fadd_rn(F(iq, it), r) > thr;
          }
          first = false;
          const unsigned pm = __ballot_sync(0xffffffffu, pass);
          if (pm) {
            const int src = (pm >> 31) ? 31 : __ffs(pm) - 1;  // the match precedes every deletion
            found = __shfl_sync(0xffffffffu, idx, src);
            cq = iq;
            ct = __shfl_sync(0xffffffffu, it, src);
            cg = __shfl_sync(0xffffffffu, g, src);
            break;
          }
          if (nonempty && lane == sl) m16 = 0;
        }
        scan_from = ndel + 1;  // the insertion candidates follow unpruned
      }
      for (int base = max(next, scan_from); base < total && found < 0; base += 32) {
        const int idx = base + lane;
        bool pass = false;
        int iq = 0, it = 0;
        float g = 0.f;
        if (idx < total) {
          if (idx == 0) {  // match (ucw.h:142-150)
            iq = q0 - 1; it = t0 - 1;
            pass = __fadd_rn(F(iq, it), r) > thr;
          } else if (idx <= ndel) {  // deletions, i = t0-2 .. 1 (ucw.h:154-165)
            iq = q0 - 1; it = t0 - 1 - idx;
            const int len = t0 - it - 1;
            g = (P.delfree && t0 == Lt + 1) ? 0.f : pen(len);  // aasubalib.h:39-42 (it >= 1: never the Head)
            pass = __fsub_rn(__fadd_rn(F(iq, it), r), g) > thr;
          } else {  // insertions, j = q0-2 .. 1 (ucw.h:169-180)
            iq = q0 - 1 - (idx - ndel); it = t0 - 1;
            const int len = q0 - iq - 1;
            g = (P.insfree && q0 == Lq + 1) ? 0.f : pen(len);  // aasubalib.h:65-68
            pass = __fsub_rn(__fadd_rn(F(iq, it), r), g) > thr;
          }
        }
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (m) {
          const int src = __ffs(m) - 1;
          found = base + src;
          cq = __shfl_sync(0xffffffffu, iq, src);
          ct = __shfl_sync(0xffffffffu, it, src);
          cg = __shfl_sync(0xffffffffu, g, src);
        }
      }
      if (found >= 0) {
        // descend: the child continues slot k (first passing branch) or a copy of `curr` (later ones), ucw.h:145-149
        if (lane == 0) {
          stack[depth] = make_int4(q0, t0, __float_as_int(curr), (found + 1) | (1 << 30));
          if (CNO) {
            frame_plen[depth] = plen;
            pathbuf[plen] = make_int2(q0, t0);
          }
        }
        if (CNO) ++plen;
        ++depth;
        curr = found == 0 ? r : __fsub_rn(r, cg);
        q0 = cq; t0 = ct; next = 0; any = 0;
        // cw.h:150,163,177: the constrained variant continues with opt_path -- no branching until the flag changes
        if (CNO && q0 > 1 && t0 > 1 && !walk(q0, t0, curr, false)) break;
        continue;
      }
      if (!any) {
        // The score fell below the threshold after extending the branch (ucw.h:182-189, cw.h:195-201): only rounding can
        // do that; the reference then forces the optimal path to the beginning.
        int a = q0, b = t0;
        float s = curr;
        if (!walk(a, b, s, true)) break;
        if (!emit(a, b, __fadd_rn(s, F(a, b)))) break;
      }
    }
    // return to the parent frame
    if (depth == 0) break;
    --depth;
    __syncwarp();
    const int4 f = stack[depth];
    q0 = f.x; t0 = f.y; curr = __int_as_float(f.z); next = f.w & 0x3fffffff; any = (f.w >> 30) & 1;
    plen = CNO ? frame_plen[depth] : 0;
  }
  if (lane == 0) { P.n_ali[warp] = count; P.status[warp] = status; }
}

}  // namespace aadp
