// aadp_general.cuh -- exact GENERAL-GAP fill in fp32 for sm_100a (SURVEY.md §8 row f3).
//
// The reference fill is not an affine three-state recurrence: every interior cell (i,j) scans the whole
// previous row and the whole previous column (dpmatrix.h:459-480) and evaluates, per candidate,
//     s = D[pred].score;  s -= gap penalty;  s += sim[i][j];  if (s > opt_s) take it
// in fp32.  For scores/penalties that are not on a common dyadic grid (the reference defaults 4.73 / 0.34,
// alib.cpp:17-18) the O(mn) recurrence of aadp_kernels.cuh cannot reproduce those roundings, so this kernel
// performs the SAME scan with the SAME fp32 operations in the SAME order -- results are bit-identical to
// the reference (scores, every DPCell predecessor, the near-optimal cell set), 0 ulp.
//
// Parallel mapping.  Row a of the flow depends on rows < a only (the column scan of cell (a,b) reads
// D[k][b-1] for k < a-1, the row scan reads D[a-1][k]): one CTA owns one (pair, direction), its threads own
// the columns, rows are processed in order with the previous row and the penalty table in shared memory.
// The column scan reads the score matrix itself (coalesced across the threads, L1/L2 resident).
// Cost O(Lq*Lt*(Lq+Lt)) like the reference; many pairs run concurrently (grid = pairs x directions).
//
// Gap penalties: pen(len) = gi + ge*(float)(len-1) (aasubalib.h:37-38, two roundings: the multiply and the
// add, no fused multiply-add) tabulated once per CTA; free end gaps per aasubalib.h:39-42,65-68.
// Flow coordinates as everywhere in this library: the reverse fill is the forward fill of the mirrored
// problem (dpmatrix.h:691-877 scans k descending in matrix coordinates = ascending in flow coordinates).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace aadp {

struct GeneralParams {
  int A;
  const float* subf;         // A*A substitution scores (SubstitutionMatrix::score, submatrix.h:36-38)
  float gi, ge;
  int delfree, insfree, local, repro_rev_bug;
  const uint8_t* residues;
  const int64_t* seq_off;
  const int32_t* pair_q;
  const int32_t* pair_t;
  const int32_t* items;      // pair ids of this launch (blockIdx.x indexes it); null = identity + item0
  int item0;
  int dirs[2];               // blockIdx.y -> 0 forward, 1 reverse
  const int64_t* dense_off;  // per item: offset (in cells) of its (Lq+2)*(Lt+2) matrices; null = 0
  const float* simov;        // similarity override: dense (Lq+2)*(Lt+2) matrices per item (same offsets as the
                             // outputs), as SimilarityMatrix (simmatrix.h:40-73) built them from ANY Evaluator; null =
                             // substitution table lookup
  const int4* rects;         // per item: anchors (q1_end, t1_end, q2_beg, t2_beg) of build_subdpm (dpmatrix.h:319-353),
                             // matrix indices; null = the whole matrix (0, 0, Lq+1, Lt+1)
  // Tabulated gap model (TAB=1, single pair, whole matrix): the two gap functions of ANY Evaluator over every
  // argument combination the fill can pass (dpmatrix.h:356-1030), so evaluators with position-dependent penalties
  // (hmap_eval.h:63-117, gn2_eval.h:99-158) run the same scan.  sz2 = Lt+2:
  const float* del_tab;      //   [t_pos1*sz2 + t_pos2] = deletion(., ., t_pos1, t_pos2), t_pos1 < t_pos2
  const float* del_tabT;     //   its transpose (the reverse fill scans it by column)
  const float* ins_tab;      //   [(q_pos2-q_pos1-1)*sz2 + t_pos2] = insertion(q_pos1, q_pos2, t_pos2-1, t_pos2)
  const int64_t* del_off;    //   per item: offset of its deletion table (batches of tabulated pairs), or null
  const int64_t* ins_off;    //   per item: offset of its insertion table, or null
  int compact;               // 1: an item stores only its rectangle, (q2_beg-q1_end+1) x (t2_beg-t1_end+1) cells with the
                             // first anchor at offset 0 (batched loop-closure fills: many small rectangles of large
                             // matrices); predecessors stay matrix indices
  int fin_by_item;           // 1: fin[] is indexed by item0 + item instead of by pair
  int max_nt;                // launch-wide shared-memory layout (general_fill_kernel): the most interior columns of an
  int max_len;               // item and the longest gap an item can take, max(nq, nt) -- for sub-rectangles those of the
                             // rectangles, not of the sequences (a loop in a 30 000-residue pair needs a few hundred floats)
  float* score[2];          // per direction: dense score matrices (always)
  int32_t* prevq[2];         // per direction: dense predecessor rows/cols, or null
  int32_t* prevt[2];
  float* fin[2];             // per direction, per PAIR: score of the final cell, or null
  float* pmcol[2];           // per direction: dense matrices of column prefix maxima (same offsets as score), or null.
                             // With them the scans are PRUNED without changing any result: max(D[1..k]) - pen(len) + sim is
                             // monotone in k (fp32 rounding preserves order, pen grows with len) and bounds every candidate
                             // up to k, so a binary search finds the first candidate that can still beat the current optimum;
                             // every earlier one fails the reference's strict '>' anyway.  Not for tabulated penalties.
};

__device__ __forceinline__ float gg_pen(float gi, float ge, int len) {  // aasubalib.h:37-38
  return __fadd_rn(gi, __fmul_rn(ge, (float)(len - 1)));
}

// First k in [lo, hi) for which the MONOTONE predicate viable(k) holds (false ... false true ... true), hi if none.
// Plain binary search: an 8-ary variant (seven independent probes per round) was measured 48 % slower -- the kernel is
// bound by executed instructions, not by the latency of the probes.
template <class Pred>
__device__ __forceinline__ int first_viable(int lo, int hi, Pred viable) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (viable(mid)) hi = mid; else lo = mid + 1;
  }
  return lo;
}

template <int TBM, int TAB = 0>
__global__ void __launch_bounds__(512) general_fill_kernel(const GeneralParams P) {
  extern __shared__ __align__(16) float gg_smem[];
  const int item = blockIdx.x;
  const int pair = P.items ? P.items[item] : P.item0 + item;
  const int dsel = blockIdx.y;
  const int rev = P.dirs[dsel];
  const int qs = P.pair_q[pair], ts = P.pair_t[pair];
  const int64_t qo = P.seq_off[qs], to = P.seq_off[ts];
  const int Lq = (int)(P.seq_off[qs + 1] - qo), Lt = (int)(P.seq_off[ts + 1] - to);
  // anchors of the filled rectangle: (q0,t0) and (mq1,mt1) in matrix indices.  q1/t1 = FLOW index of the final
  // cell, nq/nt = interior rows/columns of the rectangle.  A whole matrix is (0,0)-(Lq+1,Lt+1).
  int q0 = 0, t0 = 0, mq1 = Lq + 1, mt1 = Lt + 1;
  if (P.rects) { const int4 r = P.rects[blockIdx.x]; q0 = r.x; t0 = r.y; mq1 = r.z; mt1 = r.w; }
  const int sz2 = Lt + 2, q1 = mq1 - q0, t1 = mt1 - t0, nq = q1 - 1, nt = t1 - 1;
  // storage of the outputs: the whole matrix, or (compact) the rectangle alone
  const int ld = P.compact ? t1 + 1 : sz2, nrows = P.compact ? q1 + 1 : Lq + 2;
  const int r0 = P.compact ? q0 : 0, c0 = P.compact ? t0 : 0;
  const int fin_idx = P.fin_by_item ? P.item0 + item : pair;
  const int64_t base = P.dense_off ? P.dense_off[item] : 0;
  float* D = P.score[dsel] + base;
  int32_t* PQ = TBM ? P.prevq[dsel] + base : nullptr;
  int32_t* PT = TBM ? P.prevt[dsel] + base : nullptr;
  const uint8_t* qseq = P.residues + qo;
  const uint8_t* tseq = P.residues + to;
  const int tid = threadIdx.x, nth = blockDim.x;
  const float gi = P.gi, ge = P.ge;
  const bool local = P.local != 0;

  // indexed by flow column (prow, pm) and by gap length (pen): sized by the launch (nt <= max_nt, max(nq, nt) <= max_len)
  float* prow = gg_smem;                // D[a-1][0..nt]
  float* pen = gg_smem + (P.max_nt + 2);  // pen[len], len >= 1
  float* pm = pen + (P.max_len + 2);    // pm[k] = max(prow[1..k])  (pruned scans)
  float* wmax = pm + (P.max_nt + 2);    // 32 warp maxima of the block-wide prefix scan
  const bool PRUNE = !TAB && P.pmcol[dsel] != nullptr;
  float* PMC = PRUNE ? P.pmcol[dsel] + base : nullptr;
  const float* del_tab = TAB ? P.del_tab + (P.del_off ? P.del_off[item] : 0) : nullptr;
  const float* del_tabT = (TAB && P.del_tabT) ? P.del_tabT + (P.del_off ? P.del_off[item] : 0) : nullptr;
  const float* ins_tab = TAB ? P.ins_tab + (P.ins_off ? P.ins_off[item] : 0) : nullptr;
  const int maxlen = max(nq, nt);
  if (!TAB)
    for (int l = 1 + tid; l <= maxlen; l += nth) pen[l] = gg_pen(gi, ge, l);

  // matrix index of flow cell (a,b); matrix row / column of a flow row / column
  auto rowof = [&](int a) { return rev ? mq1 - a : q0 + a; };
  auto colof = [&](int b) { return rev ? mt1 - b : t0 + b; };
  auto at = [&](int a, int b) -> int64_t { return (int64_t)(rowof(a) - r0) * ld + (colof(b) - c0); };
  auto clampl = [&](float s) { return (local && s < 0.f) ? 0.f : s; };
  const float* simov = P.simov ? P.simov + base : nullptr;
  auto sim = [&](int a, int b) -> float {  // flow cell -> similarity (interior cells only)
    const int i = rowof(a), j = colof(b);
    if (simov) return simov[(int64_t)i * sz2 + j];
    return P.subf[(int)qseq[i - 1] * P.A + (int)tseq[j - 1]];
  };
  // gap between flow columns b0 < b1 / flow rows a0 < a1, with the free end gaps of aasubalib.h:39-42,65-68:
  // free when the lower matrix position is the Head or the upper one is the Tail (anchors of a sub-rectangle
  // are ordinary residues unless they are the Head / the Tail)
  // template position pair of an insertion taken by a cell of flow column b: (j-1, j) forward (dpmatrix.h:473),
  // (j, j+1) reverse (dpmatrix.h:812); the table is indexed by the upper one
  auto t2of = [&](int b) { return rev ? colof(b) + 1 : colof(b); };
  auto gdel = [&](int b0, int b1) -> float {
    const int len = b1 - b0 - 1;
    if (len < 1) return 0.f;
    const int x = colof(b0), y = colof(b1);
    if (TAB) return del_tab[(int64_t)min(x, y) * sz2 + max(x, y)];
    if (P.delfree && (min(x, y) == 0 || max(x, y) == Lt + 1)) return 0.f;
    return pen[len];
  };
  auto gins = [&](int a0, int a1, int b) -> float {
    const int len = a1 - a0 - 1;
    if (len < 1) return 0.f;
    if (TAB) return ins_tab[(int64_t)len * sz2 + t2of(b)];
    const int x = rowof(a0), y = rowof(a1);
    if (P.insfree && (min(x, y) == 0 || max(x, y) == Lq + 1)) return 0.f;
    return pen[len];
  };
  // similarity of the final cell: 0 at the Head / Tail (aasubalib.h:19-21), a real score at an interior anchor
  float simf = 0.f;
  {
    const int i = rowof(q1), j = colof(t1);
    if (simov) simf = simov[(int64_t)i * sz2 + j];
    else if (i >= 1 && i <= Lq && j >= 1 && j <= Lt) simf = P.subf[(int)qseq[i - 1] * P.A + (int)tseq[j - 1]];
  }

  // DPCell::DPCell (dpmatrix.cpp:17-25): score 0, predecessors null
  for (int64_t o = tid; o < (int64_t)nrows * ld; o += nth) {
    D[o] = 0.f;
    if (TBM) { PQ[o] = -1; PT[o] = -1; }
  }
  __syncthreads();

  auto set_tb = [&](int a, int b, int pa, int pb, float s) {  // dpmatrix.cpp:27-32
    const int64_t o = at(a, b);
    D[o] = s;
    if (TBM) { PQ[o] = rowof(pa); PT[o] = colof(pb); }
  };

  // Special cases #1/#2 (dpmatrix.h:374-390, 712-728): an empty sequence forces one gap; not clamped
  if (nq == 0 || nt == 0) {
    if (tid == 0) {
      float s = 0.f;
      s = __fsub_rn(s, nq == 0 ? gdel(0, t1) : gins(0, q1, t1));
      s = __fadd_rn(s, simf);
      set_tb(q1, t1, 0, 0, s);
      if (P.fin[dsel]) P.fin[dsel][fin_idx] = s;
    }
    return;
  }

  // boundary row and column of the flow (dpmatrix.h:408-426, 746-764, 579-599, 920-940)
  for (int b = 1 + tid; b <= nt; b += nth) {
    float s = 0.f;
    if (b >= 2) s = __fsub_rn(s, gdel(0, b));
    s = clampl(__fadd_rn(s, sim(1, b)));
    set_tb(1, b, 0, 0, s);
    prow[b] = s;
  }
  for (int a = 2 + tid; a <= nq; a += nth) {
    float s = 0.f;
    s = __fsub_rn(s, gins(0, a, 1));
    s = clampl(__fadd_rn(s, sim(a, 1)));
    set_tb(a, 1, 0, 0, s);
  }
  __syncthreads();

  // Row hand-over: prow[1..nt] <- row a of D (own cells and the boundary column), the column prefix maxima of that row,
  // and pm[1..nt] = inclusive prefix maximum of prow (block-wide: warp shuffles + one hop through shared memory).
  // load_row = false: prow is already in place (the boundary row).  Two barriers per chunk of blockDim columns.
  auto hand_over = [&](int a, bool load_row) {
    float carry = -3.0e38f;
    const int lane = tid & 31, wid = tid >> 5, nw = (nth + 31) >> 5;
    for (int c0 = 1; c0 <= nt; c0 += nth) {
      const int b = c0 + tid;
      float v = -3.0e38f;
      if (b <= nt) {
        if (load_row) { v = D[at(a, b)]; prow[b] = v; } else v = prow[b];
        if (PRUNE) PMC[at(a, b)] = a > 1 ? fmaxf(PMC[at(a - 1, b)], v) : v;
      }
      if (PRUNE) {
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float u = __shfl_up_sync(0xffffffffu, v, o);
          if (lane >= o) v = fmaxf(v, u);
        }
        if (lane == 31) wmax[wid] = v;
      }
      __syncthreads();
      if (PRUNE) {
        float pre = carry, tot = carry;
        for (int w = 0; w < nw; ++w) {
          const float x = wmax[w];
          if (w < wid) pre = fmaxf(pre, x);
          tot = fmaxf(tot, x);
        }
        if (b <= nt) pm[b] = fmaxf(v, pre);
        carry = tot;
        __syncthreads();
      }
    }
  };
  if (PRUNE) hand_over(1, false);

  // interior rows (dpmatrix.h:446-497): match, deletions k ascending, insertions k ascending, strict '>'
  for (int a = 2; a <= nq; ++a) {
    const float* subrow = simov ? simov + (int64_t)rowof(a) * sz2 : P.subf + (int)qseq[rowof(a) - 1] * P.A;
    for (int b = 2 + tid; b <= nt; b += nth) {
      const float simc = simov ? subrow[colof(b)] : subrow[(int)tseq[colof(b) - 1]];
      int oa = a - 1, ob = b - 1;
      float os = clampl(__fadd_rn(prow[b - 1], simc));
      // tabulated penalties of this cell: deletion column (rows = the other template position), insertion column
      // (reverse fill without a transposed table: the row of the table is scanned instead of its column)
      const bool dT = TAB && rev && !del_tabT;
      const float* dcol = TAB ? (dT ? del_tab + (int64_t)colof(b) * sz2 : (rev ? del_tabT : del_tab) + colof(b)) : nullptr;
      const int64_t dstr = dT ? 1 : sz2;
      const float* icol = TAB ? ins_tab + t2of(b) : nullptr;
      const float* colp = D + at(1, b - 1);
      const int64_t cstride = rev ? -(int64_t)ld : (int64_t)ld;
      // Pruned scans: bound(k) = rn(rn(max(D[1..k]) - pen(len)) + sim) is monotone in k and bounds candidate k, so every
      // candidate before the first k with bound(k) > os fails the reference's strict '>' and is skipped (binary search).
      // A variant scanning down from the nearest candidate with a running bound was also exact but 60 % slower.
      int kr = 1, kc = 1;
      if (PRUNE) {
        kr = first_viable(1, b - 1, [&](int k) { return clampl(__fadd_rn(__fsub_rn(pm[k], pen[b - k - 1]), simc)) > os; });
      }
      if (PRUNE && TBM) {
        for (int k = kr; k < b - 1; ++k) {  // dpmatrix.h:459-468
          const float s = clampl(__fadd_rn(__fsub_rn(prow[k], pen[b - k - 1]), simc));
          if (s > os) { ob = k; os = s; }
        }
        const float* pmp = PMC + at(1, b - 1);
        kc = first_viable(1, a - 1, [&](int k) { return clampl(__fadd_rn(__fsub_rn(pmp[(int64_t)(k - 1) * cstride], pen[a - k - 1]), simc)) > os; });
        bool col = false;
        int ka = 0;
        for (int k = kc; k < a - 1; ++k) {  // dpmatrix.h:471-480
          const float s = clampl(__fadd_rn(__fsub_rn(colp[(int64_t)(k - 1) * cstride], pen[a - k - 1]), simc));
          if (s > os) { col = true; ka = k; os = s; }
        }
        if (col) { oa = ka; ob = b - 1; }
      } else if (PRUNE) {
#pragma unroll 4
        for (int k = kr; k < b - 1; ++k) os = fmaxf(os, __fadd_rn(__fsub_rn(prow[k], pen[b - k - 1]), simc));
        const float* pmp = PMC + at(1, b - 1);
        kc = first_viable(1, a - 1, [&](int k) { return __fadd_rn(__fsub_rn(pmp[(int64_t)(k - 1) * cstride], pen[a - k - 1]), simc) > os; });
#pragma unroll 4
        for (int k = kc; k < a - 1; ++k) os = fmaxf(os, __fadd_rn(__fsub_rn(colp[(int64_t)(k - 1) * cstride], pen[a - k - 1]), simc));
        os = clampl(os);
      } else if (TBM) {
        for (int k = 1; k < b - 1; ++k) {  // dpmatrix.h:459-468
          float s = __fsub_rn(prow[k], TAB ? dcol[(int64_t)colof(k) * dstr] : pen[b - k - 1]);
          s = clampl(__fadd_rn(s, simc));
          if (s > os) { ob = k; os = s; }
        }
        bool col = false;
        int ka = 0;
        for (int k = 1; k < a - 1; ++k) {  // dpmatrix.h:471-480
          float s = __fsub_rn(colp[(int64_t)(k - 1) * cstride], TAB ? icol[(int64_t)(a - k - 1) * sz2] : pen[a - k - 1]);
          s = clampl(__fadd_rn(s, simc));
          if (s > os) { col = true; ka = k; os = s; }
        }
        if (col) { oa = ka; ob = b - 1; }
      } else {
        // score only: the strict-'>' scan and a running maximum give the same value; the clamp commutes with max
#pragma unroll 4
        for (int k = 1; k < b - 1; ++k)
          os = fmaxf(os, __fadd_rn(__fsub_rn(prow[k], TAB ? dcol[(int64_t)colof(k) * dstr] : pen[b - k - 1]), simc));
#pragma unroll 4
        for (int k = 1; k < a - 1; ++k)
          os = fmaxf(os, __fadd_rn(__fsub_rn(colp[(int64_t)(k - 1) * cstride], TAB ? icol[(int64_t)(a - k - 1) * sz2] : pen[a - k - 1]), simc));
        os = clampl(os);
      }
      set_tb(a, b, oa, ob, os);
    }
    __syncthreads();  // every thread is done reading the previous row
    hand_over(a, true);
  }

  // final cell (dpmatrix.h:504-534, 844-874, 654-687, 995-1028): match, bottom row, right column.
  // Its similarity is 0 at the Tail / Head, a real score at an interior anchor.  Serial: nq + nt candidates.
  if (tid == 0) {
    int oa = nq, ob = nt;
    bool from_col = false;
    float os = clampl(__fadd_rn(D[at(nq, nt)], simf));
    for (int k = 1; k < t1; ++k) {
      float s = __fsub_rn(D[at(nq, k)], gdel(k, t1));
      s = clampl(__fadd_rn(s, simf));
      if (s > os) { oa = nq; ob = k; os = s; }
    }
    for (int k = 1; k < q1; ++k) {
      float s = __fsub_rn(D[at(k, nt)], gins(k, q1, t1));
      s = clampl(__fadd_rn(s, simf));
      if (s > os) { oa = k; ob = nt; os = s; from_col = true; }
    }
    set_tb(q1, t1, oa, ob, os);
    // dpmatrix.h:868: the global reverse fill records opt_j = t1_m1 (a matrix column) for left-column candidates
    if (TBM && rev && !local && P.repro_rev_bug && from_col) PT[at(q1, t1)] = mt1 - 1;
    if (P.fin[dsel]) P.fin[dsel][fin_idx] = os;
  }
}

// Near-optimal cell set on dense matrices, the reference arithmetic: v = F + R; v -= sim; v > thr
// (ucw.h:141-180 with the threshold of cw.h:86-88).  One CTA per item.
struct GeneralMaskParams {
  int A;
  const float* subf;
  const uint8_t* residues;
  const int64_t* seq_off;
  const int32_t* pair_q;
  const int32_t* pair_t;
  const int32_t* items;
  int item0;
  const int64_t* dense_off;
  const float* F;
  const float* R;
  const float* fin_fwd;      // per pair
  float delta_ratio;
  uint8_t* mask;             // dense bytes per item (same offsets), or null
  float* threshold;          // per pair, or null
  long long* count;          // per pair, or null
};

__global__ void __launch_bounds__(256) general_mask_kernel(const GeneralMaskParams P) {
  const int item = blockIdx.x;
  const int pair = P.items ? P.items[item] : P.item0 + item;
  const int qs = P.pair_q[pair], ts = P.pair_t[pair];
  const int64_t qo = P.seq_off[qs], to = P.seq_off[ts];
  const int Lq = (int)(P.seq_off[qs + 1] - qo), Lt = (int)(P.seq_off[ts + 1] - to);
  const int sz2 = Lt + 2;
  const int64_t base = P.dense_off ? P.dense_off[item] : 0;
  const float opt = P.fin_fwd[pair];
  const float thr = fminf(__fmul_rn(1.f - P.delta_ratio, opt), __fsub_rn(opt, 0.1f));  // cw.h:86-88
  long long cnt = 0;
  // row by row (no 64-bit division per cell); the border cells of a dense mask stay 0
  if (P.mask) {
    for (int j = threadIdx.x; j < sz2; j += blockDim.x) { P.mask[base + j] = 0; P.mask[base + (int64_t)(Lq + 1) * sz2 + j] = 0; }
    for (int i = 1 + threadIdx.x; i <= Lq; i += blockDim.x) { P.mask[base + (int64_t)i * sz2] = 0; P.mask[base + (int64_t)i * sz2 + Lt + 1] = 0; }
  }
  for (int i = 1; i <= Lq; ++i) {
    const float* subrow = P.subf + (int)P.residues[qo + i - 1] * P.A;
    const int64_t ro = base + (int64_t)i * sz2;
    for (int j = 1 + threadIdx.x; j <= Lt; j += blockDim.x) {
      float v = __fadd_rn(P.F[ro + j], P.R[ro + j]);
      v = __fsub_rn(v, subrow[(int)P.residues[to + j - 1]]);
      const int m = v > thr ? 1 : 0;
      if (P.mask) P.mask[ro + j] = (uint8_t)m;
      cnt += m;
    }
  }
  __shared__ long long s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  for (int o = 16; o >= 1; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd((unsigned long long*)&s_cnt, (unsigned long long)cnt);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (P.count) P.count[pair] = s_cnt;
    if (P.threshold) P.threshold[pair] = thr;
  }
}

// Optimal sub-alignment of every rectangle of a compact batch: Optimal_Subali::enumerate (optimal_subali.h:59-83).
// One thread per item follows DPCell::prev_* from (q2_beg, t2_beg) while q_last > q1_end, then requires the walk to
// have ended on (q1_end, t1_end) (status 3 = "Illegal alignment start pair", optimal_subali.h:80).  Every step lowers
// the query index, so a slot of q2_beg - q1_end + 1 aligned pairs always suffices.
struct SubTraceParams {
  const int32_t* PQ;
  const int32_t* PT;
  const float* D;
  const int64_t* dense_off;  // per item of this launch
  const int4* rects;         // per item of this launch
  const int64_t* cap_off;    // per item of the whole batch (index item0 + item)
  int item0, n;
  int2* out;                 // slots, front to back
  int32_t* out_n;
  int32_t* out_status;
  float* out_score;          // D[q2_beg][t2_beg].score (optimal_subali.h:68), or null
};

__global__ void __launch_bounds__(128) subali_trace_kernel(const SubTraceParams P) {
  const int item = blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= P.n) return;
  const int4 r = P.rects[item];
  const int ld = r.w - r.y + 1;
  const int64_t base = P.dense_off[item];
  auto idx = [&](int i, int j) -> int64_t { return base + (int64_t)(i - r.x) * ld + (j - r.y); };
  const int cap = r.z - r.x + 1;
  int len = 1, i = r.z, j = r.w;
  while (i > r.x && len <= cap) {
    const int64_t o = idx(i, j);
    i = P.PQ[o];
    j = P.PT[o];
    ++len;
  }
  const bool ok = (i == r.x && j == r.y);
  const int64_t slot = P.cap_off[P.item0 + item];
  len = min(len, cap);
  i = r.z;
  j = r.w;
  for (int k = len - 1; k >= 0; --k) {  // prepend order: the slot reads front to back
    P.out[slot + k] = make_int2(i, j);
    if (k) {
      const int64_t o = idx(i, j);
      i = P.PQ[o];
      j = P.PT[o];
    }
  }
  P.out_n[P.item0 + item] = len;
  P.out_status[P.item0 + item] = ok ? 0 : 3;
  if (P.out_score) P.out_score[P.item0 + item] = P.D[idx(r.z, r.w)];
}

}  // namespace aadp
