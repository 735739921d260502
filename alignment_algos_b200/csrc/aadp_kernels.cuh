// aadp_kernels.cuh -- hand-written sm_100a kernels for the affine-gap DP fill of
// christang/alignment-algos (dpmatrix.h:356-1030 driven by AASubstitutionEval, aasubalib.h:8-87).
//
// Recurrence.  The reference scans, for every interior cell (i,j), the whole previous row and the
// whole previous column (dpmatrix.h:459-480).  For the affine gap cost gi+ge*(len-1) that is the
// three-state recurrence (SURVEY.md App. A.2), written here in FLOW coordinates (flow = matrix
// coordinates for the forward fill, mirrored coordinates for the reverse fill):
//     M(i,j) = sim(i,j) + X(i-1,j-1)                       X = max3(M,E,F), ties M > E > F
//     E(i,j) = max(E(i,j-1) - ge, M(i,j-1) - gi)           ties keep the extension (smaller k)
//     F(i,j) = max(F(i-1,j) - ge, M(i-1,j) - gi)           ties keep the extension (smaller k)
// which reproduces the reference's strict-'>' scan order match -> deletions(k asc) -> insertions
// (k asc) (dpmatrix.h:463,475) exactly when all scores are integers in the chosen units.
// M is the reference's DPCell::score.  E and F never chain into each other (a predecessor moves
// one index by exactly 1, dpmatrix.h:453-480).
//
// Mapping (one warp per pair, "striped + skewed"): lane l owns K consecutive template columns and
// processes row i = step - l + 1, so the E chain crosses lanes with three __shfl_up_sync per step
// and everything else stays in registers.  Substitution scores come from a per-pair int8
// template profile staged in shared memory (prof[a][column] = sub[a][t_column]); the row's query
// residue selects the profile row, one 8/16-byte conflict-free LDS per lane per step.
//
// Packed traceback (4 bit/cell, "planes"): for flow cell (i,j)
//     plane0 selE  = [E > M]          plane1 selF  = [F > max(M,E)]
//     plane2 eopen = [M(i,j-1)-gi > E(i,j-1)-ge]     plane3 fopen = [M(i-1,j)-gi > F(i-1,j)-ge]
// stored per row as 32-bit words covering 8 columns: byte p = plane p, bit (7-c) = column 8g+c+1.
// The absolute predecessor the reference stores in DPCell (dpmatrix.h:28-37) is recovered by
// walking eopen / fopen bits (see decode_prev below).
#pragma once
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>

namespace aadp {

constexpr int kNeg32 = -(1 << 30);    // "-infinity" for E/F seeds (int32 path)
constexpr int kFloor32 = -(1 << 29);  // clamp floor of M (never reached by real scores)
constexpr int kWarpsPerCta = 4;
constexpr int kQRing = 1024;           // per-warp query staging ring (bytes)
// multi-CTA wavefront (long pairs): columns per lane / per stripe (one warp per stripe).  Every stripe has to
// walk all Lq rows, so the run time is (Lq + pipeline skew) x (time of one row step); measured on B200
// (30k x 30k, fwd+rev): K = 4 -> 13.9 ms (705 cycles/step), K = 8 -> 12.3 ms (703), K = 16 -> 13.5 ms (824):
// the step time is set by serialized latencies (shuffle -> E chain -> publish), not by the cells per lane.
constexpr int kWaveK = 8;
constexpr int kWaveCols = 32 * kWaveK;

__host__ __device__ inline int64_t round_up64(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
// packed-traceback row stride in bytes: one 32-bit word per 8 columns, rows padded to 16 B
__host__ __device__ inline int64_t tb_row_bytes(int Lt) { return round_up64(4 * (int64_t)((Lt + 7) / 8), 16); }
// score-matrix row stride in elements (rows hold columns 1..Lt, padded to 16 elements)
__host__ __device__ inline int64_t sc_row_elems(int Lt) { return round_up64(Lt, 16); }

struct Scoring {
  int A;        // alphabet size
  int gi, ge;   // gap penalties in integer units (scaled by 2^scale_log2)
  int delfree;  // aasubalib.h:39-42: free end gaps in the template (local, semi_local, local_global)
  int insfree;  // aasubalib.h:65-68: free end gaps in the query (local, semi_local, global_local)
  int local;    // align_type == local (dpmatrix.h:155): clamp at 0
  int scale_log2;
};

struct FillParams {
  Scoring sc;
  const int8_t* sub8;        // A*A scaled substitution scores
  const uint8_t* residues;   // sequence arena
  const int64_t* seq_off;    // nseq+1
  const int32_t* pair_q;     // npairs
  const int32_t* pair_t;
  const int32_t* order;      // work list (pair ids) for this launch
  int n_items;
  int rev;                   // 0 = forward flow, 1 = reverse flow
  unsigned int* counter;     // dynamic work counter (zeroed before launch)
  uint8_t* tb;               // packed traceback blob of this direction (or null)
  const int64_t* tb_off;     // per pair byte offset
  void* sc_blob;             // score blob of this direction (int16 or int32 elements)
  const int64_t* sc_off;     // per pair offset in int16 units (int32 pairs use two units per element)
  int32_t* fin_score;        // per pair: final-cell score (integer units)
  int32_t* fin_kind;         // 0 = diagonal, 1 = row (deletion), 2 = column (insertion)
  int32_t* fin_k;            // kind 1: flow column k of the predecessor; kind 2: -1 (resolved by decode)
  int4* bbuf;                // stripe boundary buffer: [warp slot][bb_rows]
  int bb_rows;
  double cells_hint;         // host-side bookkeeping only (cell updates of this launch)
  // ---- multi-CTA wavefront mode (one long pair, one CTA per 32*K-column stripe)
  int wave_pair;             // pair id
  int wave_nstripes;
  unsigned long long* wave_ll;  // [stripe][bb_rows][3] boundary (X, E, M-gi) of the stripe's last column per row, each
                             // value published as ONE 8-byte word {value, tag}: data and flag travel together, so
                             // neither side needs a fence or a separate progress counter (cf. NCCL's LL protocol)
  unsigned int wave_tag;     // tag of this launch (the buffer is zeroed when allocated, tags never repeat)
  int* wave_ready;           // [stripe] Lq+1 once the stripe is completely done (final-cell partials chain)
  int4* wave_part;           // [stripe] final-row partials (rb_val, rb_k, diag, col)
  long long* wave_dbg;       // optional [stripe][2]: cycles spent waiting for the left neighbour, total cycles
};

// Position-specific template profiles (aadp_set_profile_scoring): sim(i,j) = profile of the template at position j,
// query code q_i.  The int8 copy (grid units) is laid out per sequence and FLOW: sequence s owns 2*A*16n bytes at
// p8 + off8[s] (n = ceil(L/16)), the forward flow first, then the reverse flow.  Row a of a flow holds 16n bytes; byte k
// is the score of query code a at flow column j = k + 1 - sig, -128 where that column does not exist.  Forward: sig =
// 16n - L (right-aligned like the packed forward pass); reverse: sig = 0 and flow column j is template position L+1-j.
// A packed lane therefore loads its 16 columns of a row with one aligned 16-byte load.  pf / offf: the profiles as
// given (fp32, [offf[s] + (j-1)*A + a]) for the enumeration kernel.
struct ProfDev {
  const int8_t* p8;
  const int64_t* off8;
  const float* pf;
  const int64_t* offf;
};
__host__ __device__ inline int prof_row_bytes(int L) { return 16 * ((L + 15) >> 4); }
// row 0 of the flow `rev` of sequence s (template length L)
__device__ __forceinline__ const int8_t* prof_flow(const ProfDev& pd, int s, int L, int A, int rev) {
  return pd.p8 + pd.off8[s] + (rev ? (int64_t)A * prof_row_bytes(L) : 0);
}

__device__ __forceinline__ int ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
// 8-byte {value, tag} words: single-copy atomic, L1-bypassing, no fence
__device__ __forceinline__ void st_ll(unsigned long long* p, int v, unsigned int tag) {
  const unsigned long long w = (unsigned long long)(unsigned int)v | ((unsigned long long)tag << 32);
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(w) : "memory");
}
__device__ __forceinline__ unsigned long long ld_ll(const unsigned long long* p) {
  unsigned long long w;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
  return w;
}

// gap(len) in integer units; 0 for len < 1 (aasubalib.h:33-38)
__host__ __device__ inline int gap_w(int gi, int ge, int len) { return len < 1 ? 0 : gi + ge * (len - 1); }

// prmt.b32 with the full 4-bit selector nibbles (bit 3 = replicate the sign of the selected byte).
// __byte_perm() masks the selector to 3 bits, so the PTX instruction is issued directly.
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

__device__ __forceinline__ int sext8(uint32_t w, int c) {
  // byte c of w -> int32: byte 0 = the byte, bytes 1..3 = its sign
  const uint32_t sel = (uint32_t)c | ((uint32_t)(c | 8) << 4) | ((uint32_t)(c | 8) << 8) | ((uint32_t)(c | 8) << 12);
  return (int)prmt(w, 0u, sel);
}

// ------------------------------------------------------------------------------------------------
// One warp fills one pair in one direction.  K = columns per lane (8 or 16).
// TBM: write packed traceback.  STM: 0 = no score matrix, 1 = int16, 2 = int32.
// ------------------------------------------------------------------------------------------------
// WAVE = 1: this warp (one CTA) fills ONLY stripe `wave_st` of the pair; stripe st consumes the boundary
// column of stripe st-1 from global memory 32 rows at a time, gated by release/acquire progress flags --
// the CTAs of one launch form an anti-diagonal wavefront over the column stripes of one long pair.
// PRO = 1: the stripe profile is copied from the template's position-specific profile (ProfDev) instead of being
// built from the substitution table; nothing else changes.
template <int K, int TBM, int STM, int WAVE, int PRO = 0>
__device__ __forceinline__ void fill_pair_warp(const FillParams& P, int pair, int8_t* prof, uint8_t* qring,
                                               const int8_t* s_sub, int4* bb, int lane, int wave_st = 0,
                                               const ProfDev& pd = ProfDev{}) {
  constexpr int W = 32 * K;
  const Scoring& S = P.sc;
  const int gi = S.gi, ge = S.ge;
  const int floorM = S.local ? 0 : kFloor32;

  const int qs = P.pair_q[pair], ts = P.pair_t[pair];
  const int64_t qo = P.seq_off[qs], to = P.seq_off[ts];
  const int Lq = (int)(P.seq_off[qs + 1] - qo), Lt = (int)(P.seq_off[ts + 1] - to);
  const uint8_t* qseq = P.residues + qo;
  const uint8_t* tseq = P.residues + to;
  const int rev = P.rev;

  // Special cases #1/#2 (dpmatrix.h:374-390, 712-728): an empty sequence forces one gap.
  if (Lq == 0 || Lt == 0) {
    if (lane == 0) {
      int s;
      if (Lq == 0) s = -(S.delfree ? 0 : gap_w(gi, ge, Lt));
      else s = -(S.insfree ? 0 : gap_w(gi, ge, Lq));
      P.fin_score[pair] = s;
      P.fin_kind[pair] = 0;
      P.fin_k[pair] = 0;
    }
    return;
  }

  const int64_t tbs = tb_row_bytes(Lt);
  const int64_t scs = sc_row_elems(Lt);
  uint8_t* const tbp = TBM ? P.tb + P.tb_off[pair] : nullptr;
  const int64_t sco = STM ? P.sc_off[pair] : 0;  // hoisted: a per-step global load here stalls every row

  const int nstripes = (Lt + W - 1) / W;
  // running row-part of the final cell: best M(Lq,k) - pen(Lt-k) over k < Lt, smallest k on ties
  int rb_val = kNeg32, rb_k = 0;
  int diag_val = kNeg32, col_val = kNeg32;

  const int st_lo = WAVE ? wave_st : 0, st_hi = WAVE ? wave_st + 1 : nstripes;
  for (int st = st_lo; st < st_hi; ++st) {
    // WAVE: this stripe's published boundary column, and the one it consumes (the stripe to its left)
    unsigned long long* ll_out = WAVE ? P.wave_ll + (int64_t)st * P.bb_rows * 3 : nullptr;
    const unsigned long long* ll_in = WAVE ? P.wave_ll + (int64_t)(st - 1) * P.bb_rows * 3 : nullptr;
    int4* wblk = reinterpret_cast<int4*>(qring + kQRing);  // WAVE: 32 staged rows of the input boundary (512 B)
    const int jbase = st * W + lane * K;  // flow column of register c is jbase + c + 1
    const int cols_here = min(W, Lt - st * W);
    const int n_act = (cols_here + K - 1) / K;

    // ---- template profile for this stripe: prof[a*W + lane*K + c] = sub8[a][t_(jbase+c+1)]
    if (PRO) {
      // flow column j of the stripe sits at byte j-1+sig of the row; columns beyond Lt are never read back
      const int nb = prof_row_bytes(Lt), sig = rev ? 0 : nb - Lt;
      const int8_t* src = prof_flow(pd, ts, Lt, S.A, rev) + sig - 1;
      __syncwarp();  // previous users of prof are done
      for (int a = 0; a < S.A; ++a) {
        uint32_t* dst = reinterpret_cast<uint32_t*>(prof + a * W + lane * K);
#pragma unroll
        for (int w = 0; w < K / 4; ++w) {
          uint32_t o = 0;
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const int j = jbase + w * 4 + b + 1;
            if (j <= Lt) o |= (uint32_t)(uint8_t)src[a * nb + j] << (8 * b);
          }
          dst[w] = o;
        }
      }
      __syncwarp();
    } else {
      uint32_t tc[K / 4];
#pragma unroll
      for (int w = 0; w < K / 4; ++w) {
        uint32_t x = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          int j = jbase + w * 4 + b + 1;
          uint32_t code = 0;
          if (j <= Lt) code = rev ? tseq[Lt - j] : tseq[j - 1];
          x |= code << (8 * b);
        }
        tc[w] = x;
      }
      __syncwarp();  // previous users of prof are done
      for (int a = 0; a < S.A; ++a) {
        const int8_t* row = s_sub + a * S.A;
        uint32_t* dst = reinterpret_cast<uint32_t*>(prof + a * W + lane * K);
#pragma unroll
        for (int w = 0; w < K / 4; ++w) {
          uint32_t x = tc[w], o = 0;
#pragma unroll
          for (int b = 0; b < 4; ++b) o |= (uint32_t)(uint8_t)row[(x >> (8 * b)) & 0xff] << (8 * b);
          dst[w] = o;
        }
      }
      __syncwarp();
    }

    // ---- state for virtual row 0
    int Xp[K], Fs[K], Mg[K], nge[K];
#pragma unroll
    for (int c = 0; c < K; ++c) {
      int j = jbase + c + 1;
      Xp[c] = -(S.delfree ? 0 : gap_w(gi, ge, j));  // X(0,j): dpmatrix.h:412-418
      Fs[c] = kNeg32;
      Mg[c] = kNeg32;
      nge[c] = (S.insfree && j == Lt) ? 0 : -ge;  // zero-penalty F chain in the last column
    }
    int xl_hold;  // X(i-1, jbase): diagonal input of the lane's first column
    {
      int jl = jbase;  // column to the left of the lane's first column
      xl_hold = (jl == 0) ? 0 : -(S.delfree ? 0 : gap_w(gi, ge, jl));
    }
    int x_pub = 0, e_pub = kNeg32, mg_pub = kNeg32;
    // Query residues are staged in a kQRing-byte shared-memory ring, kQRing/2 rows at a time:
    // lanes are skewed by one row, so at step s rows s-30..s+2 are live; block b (rows
    // b*H+1..b*H+H, H = kQRing/2) is loaded at step (b-1)*H+32, after lane 31 has left block b-2.
    constexpr int H = kQRing / 2;
    __syncwarp();
#pragma unroll
    for (int u = 0; u < kQRing / 32; ++u) {
      int r = u * 32 + lane;  // 0-based flow row
      if (r < Lq && r < kQRing) qring[r] = rev ? qseq[Lq - 1 - r] : qseq[r];
    }
    __syncwarp();
    int a_nxt = 0;
    if (lane == 0) a_nxt = qring[0];

    const int nsteps = Lq + n_act - 1;
    long long dbg_wait = 0;
    const long long dbg_t0 = (WAVE && P.wave_dbg) ? clock64() : 0;
    for (int s = 0; s < nsteps; ++s) {
      if (s >= H + 32 && ((s - 32) & (H - 1)) == 0) {  // refill: block b = (s-32)/H + 1
        const int r0 = ((s - 32) / H + 1) * H;
        __syncwarp();
#pragma unroll
        for (int u = 0; u < H / 32; ++u) {
          int r = r0 + u * 32 + lane;
          if (r < Lq) qring[r & (kQRing - 1)] = rev ? qseq[Lq - 1 - r] : qseq[r];
        }
        __syncwarp();
      }
      int xn = __shfl_up_sync(0xffffffffu, x_pub, 1);
      int e_in = __shfl_up_sync(0xffffffffu, e_pub, 1);
      int mg_in = __shfl_up_sync(0xffffffffu, mg_pub, 1);
      const int i = s - lane + 1;
      const int a_cur = a_nxt;
      {
        int inx = i + 1;
        if (inx >= 1 && inx <= Lq) a_nxt = qring[(inx - 1) & (kQRing - 1)];
      }
      if (WAVE && st > 0) {
        const int i0 = s + 1;  // row lane 0 works on in this step
        if (i0 <= Lq && ((i0 - 1) & 31) == 0) {
          // a new 32-row block of the left neighbour's boundary: lane l fetches row i0+l and spins until all three
          // words carry this launch's tag (they are published row by row, in order), then stages it
          const int r = i0 + lane;
          unsigned long long w0 = 0, w1 = 0, w2 = 0;
          const long long t_w0 = P.wave_dbg ? clock64() : 0;
          for (;;) {
            bool ok = true;
            if (r <= Lq) {
              const unsigned long long* src = ll_in + (int64_t)r * 3;
              w0 = ld_ll(src); w1 = ld_ll(src + 1); w2 = ld_ll(src + 2);
              ok = (unsigned int)(w0 >> 32) == P.wave_tag && (unsigned int)(w1 >> 32) == P.wave_tag &&
                   (unsigned int)(w2 >> 32) == P.wave_tag;
            }
            if (__all_sync(0xffffffffu, ok)) break;
            __nanosleep(32);
          }
          if (P.wave_dbg) dbg_wait += clock64() - t_w0;
          wblk[lane] = make_int4((int)(unsigned int)w0, (int)(unsigned int)w1, (int)(unsigned int)w2, 0);
          __syncwarp();
        }
        if (i0 <= Lq) {
          const int4 bv = wblk[(i0 - 1) & 31];  // same address for every lane: one broadcast LDS.128
          if (lane == 0) { xn = bv.x; e_in = bv.y; mg_in = bv.z; }
        }
      }
      if (lane == 0) {
        if (st == 0) {
          xn = -(S.insfree ? 0 : gap_w(gi, ge, i));  // X(i,0): dpmatrix.h:420-426
          e_in = kNeg32;
          mg_in = kNeg32;
        } else if (!WAVE && i <= Lq) {
          int4 b = bb[i];
          xn = b.x;
          e_in = b.y;
          mg_in = b.z;
        }
      }
      const bool active = (i >= 1) && (i <= Lq) && (lane < n_act);
      if (active) {
        uint32_t pw[K / 4];
        if (K == 16) {
          uint4 v = *reinterpret_cast<const uint4*>(prof + a_cur * W + lane * K);
          pw[0] = v.x; pw[1] = v.y; pw[K / 4 - 2] = v.z; pw[K / 4 - 1] = v.w;
        } else if (K == 8) {
          uint2 v = *reinterpret_cast<const uint2*>(prof + a_cur * W + lane * K);
          pw[0] = v.x; pw[K / 4 - 1] = v.y;
        } else {
          pw[0] = *reinterpret_cast<const uint32_t*>(prof + a_cur * W + lane * K);
        }
        int Xd = xl_hold, E = e_in, Mgl = mg_in;
        uint32_t acc0 = 0, acc1 = 0, acc2 = 0, acc3 = 0;
        uint32_t tbw[(K + 7) / 8];
        int mrow[K];
#pragma unroll
        for (int c = 0; c < K; ++c) {
          const int sim = sext8(pw[c >> 2], c & 3);
          const int M = __viaddmax_s32(sim, Xd, floorM);
          Xd = Xp[c];
          int F, X;
          if (TBM) {
            const int Eext = E - ge;
            const int Fext = Fs[c] + nge[c];
            const int dE = Eext - Mgl;  // < 0  <=> the open candidate wins strictly
            E = max(Eext, Mgl);
            const int dF = Fext - Mg[c];
            F = max(Fext, Mg[c]);
            const int dS1 = M - E;  // < 0 <=> E > M
            const int t = max(M, E);
            const int dS2 = t - F;  // < 0 <=> F > max(M,E)
            X = max(t, F);
            acc0 = __funnelshift_l((uint32_t)dS1, acc0, 1);
            acc1 = __funnelshift_l((uint32_t)dS2, acc1, 1);
            acc2 = __funnelshift_l((uint32_t)dE, acc2, 1);
            acc3 = __funnelshift_l((uint32_t)dF, acc3, 1);
            if (K >= 8 && (c & 7) == 7)
              tbw[c >> 3] = __byte_perm(__byte_perm(acc0, acc1, 0x0040), __byte_perm(acc2, acc3, 0x0040), 0x5410);
            if (K == 4 && c == 3)  // nibble layout: byte 0 = planes 0|1, byte 1 = planes 2|3
              tbw[0] = ((acc0 << 4) | acc1) | (((acc2 << 4) | acc3) << 8);
          } else {
            E = __viaddmax_s32(E, -ge, Mgl);
            F = __viaddmax_s32(Fs[c], nge[c], Mg[c]);
            X = __vimax3_s32(M, E, F);
          }
          Mgl = M - gi;
          Xp[c] = X;
          Fs[c] = F;
          Mg[c] = Mgl;
          if (STM) mrow[c] = M;
        }
        xl_hold = xn;
        x_pub = Xp[K - 1];
        e_pub = E;
        mg_pub = Mgl;
        if (TBM) {
          uint8_t* dst = tbp + (int64_t)(i - 1) * tbs + (int64_t)(st * W + lane * K) / 2;
          if (K == 16) *reinterpret_cast<uint2*>(dst) = make_uint2(tbw[0], tbw[(K + 7) / 8 - 1]);
          else if (K == 8) *reinterpret_cast<uint32_t*>(dst) = tbw[0];
          else *reinterpret_cast<uint16_t*>(dst) = (uint16_t)tbw[0];
        }
        if (STM == 1) {
          int16_t* dst = reinterpret_cast<int16_t*>(P.sc_blob) + sco + (int64_t)(i - 1) * scs + st * W + lane * K;
          uint32_t pk[K / 2];
#pragma unroll
          for (int c = 0; c < K / 2; ++c) pk[c] = __byte_perm((uint32_t)mrow[2 * c], (uint32_t)mrow[2 * c + 1], 0x5410);
          if (K == 4) *reinterpret_cast<uint2*>(dst) = make_uint2(pk[0], pk[K / 2 - 1]);
#pragma unroll
          for (int c = 0; c < K / 8; ++c)
            reinterpret_cast<uint4*>(dst)[c] = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
        } else if (STM == 2) {
          int32_t* dst = reinterpret_cast<int32_t*>(reinterpret_cast<int16_t*>(P.sc_blob) + sco) + (int64_t)(i - 1) * scs + st * W + lane * K;
#pragma unroll
          for (int c = 0; c < K / 4; ++c)
            reinterpret_cast<int4*>(dst)[c] = make_int4(mrow[4 * c], mrow[4 * c + 1], mrow[4 * c + 2], mrow[4 * c + 3]);
        }
        if (st + 1 < nstripes && lane == 31) {
          if (WAVE) {  // publish this row of the boundary column: three self-validating 8-byte words
            unsigned long long* o = ll_out + (int64_t)i * 3;
            st_ll(o, x_pub, P.wave_tag);
            st_ll(o + 1, e_pub, P.wave_tag);
            st_ll(o + 2, mg_pub, P.wave_tag);
          } else {
            bb[i] = make_int4(x_pub, e_pub, mg_pub, 0);
          }
        }
      }
    }

    if (WAVE && P.wave_dbg && lane == 0) {
      P.wave_dbg[2 * st] = dbg_wait;
      P.wave_dbg[2 * st + 1] = clock64() - dbg_t0;
    }
    // ---- after the last row: contributions of this stripe's columns to the final cell
    // (dpmatrix.h:504-534).  Mg[c] + gi = M(Lq, j).
#pragma unroll
    for (int c = 0; c < K; ++c) {
      int j = jbase + c + 1;
      int m = Mg[c] + gi;
      if (j < Lt) {
        int v = m - (S.delfree ? 0 : gap_w(gi, ge, Lt - j));
        if (v > rb_val) { rb_val = v; rb_k = j; }
      } else if (j == Lt) {
        diag_val = m;
        col_val = (Lq >= 2) ? Fs[c] + (S.insfree ? gi : 0) : kNeg32;
      }
    }
    __syncwarp();
  }

  // ---- final cell: match, then bottom-row candidates (k ascending), then right-column
  // candidates, strict '>' (dpmatrix.h:504-534 / 844-874)
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    int v2 = __shfl_xor_sync(0xffffffffu, rb_val, o);
    int k2 = __shfl_xor_sync(0xffffffffu, rb_k, o);
    if (v2 > rb_val || (v2 == rb_val && k2 < rb_k)) { rb_val = v2; rb_k = k2; }
    diag_val = max(diag_val, __shfl_xor_sync(0xffffffffu, diag_val, o));
    col_val = max(col_val, __shfl_xor_sync(0xffffffffu, col_val, o));
  }
  if (WAVE) {
    // stripe partial -> global; completion is chained stripe by stripe so that the last stripe sees them all
    if (lane == 0) {
      P.wave_part[wave_st] = make_int4(rb_val, rb_k, diag_val, col_val);
      if (wave_st > 0) while (ld_acquire(P.wave_ready + wave_st - 1) < Lq + 1) __nanosleep(64);
      __threadfence();
      st_release(P.wave_ready + wave_st, Lq + 1);
    }
    __syncwarp();
    if (wave_st != nstripes - 1) return;
    rb_val = kNeg32; rb_k = 0; diag_val = kNeg32; col_val = kNeg32;
    for (int t = lane; t < nstripes; t += 32) {  // ascending stripes per lane: '>' keeps the smallest k
      const int4 v = P.wave_part[t];
      if (v.x > rb_val) { rb_val = v.x; rb_k = v.y; }
      diag_val = max(diag_val, v.z);
      col_val = max(col_val, v.w);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      int v2 = __shfl_xor_sync(0xffffffffu, rb_val, o);
      int k2 = __shfl_xor_sync(0xffffffffu, rb_k, o);
      if (v2 > rb_val || (v2 == rb_val && k2 < rb_k)) { rb_val = v2; rb_k = k2; }
      diag_val = max(diag_val, __shfl_xor_sync(0xffffffffu, diag_val, o));
      col_val = max(col_val, __shfl_xor_sync(0xffffffffu, col_val, o));
    }
  }
  if (lane == 0) {
    int best = diag_val, kind = 0, k = Lt;
    if (S.local) best = max(best, 0);
    if (Lt >= 2 && rb_val > best) { best = rb_val; kind = 1; k = rb_k; }
    if (col_val > best) { best = col_val; kind = 2; k = -1; }
    P.fin_score[pair] = best;
    P.fin_kind[pair] = kind;
    P.fin_k[pair] = k;
  }
}

// PRO = 1: position-specific template profiles (aadp_set_profile_scoring, read from pd); PRO = 0 ignores pd
template <int K, int TBM, int STM, int PRO>
__global__ void __launch_bounds__(kWarpsPerCta * 32) fill_kernel(const FillParams P, const ProfDev pd) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int W = 32 * K;
  const int A = P.sc.A;
  int8_t* s_sub = reinterpret_cast<int8_t*>(smem);
  const int sub_bytes = (A * A + 15) / 16 * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* qring = smem + sub_bytes + warp * kQRing;
  int8_t* prof = reinterpret_cast<int8_t*>(smem + sub_bytes + kWarpsPerCta * kQRing + warp * A * W);
  if (!PRO)
    for (int x = threadIdx.x; x < A * A; x += blockDim.x) s_sub[x] = P.sub8[x];
  __syncthreads();
  const int slot = blockIdx.x * kWarpsPerCta + warp;
  int4* bb = P.bbuf ? P.bbuf + (int64_t)slot * P.bb_rows : nullptr;
  for (;;) {
    unsigned int item = 0;
    if (lane == 0) item = atomicAdd(P.counter, 1u);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= (unsigned int)P.n_items) break;
    fill_pair_warp<K, TBM, STM, 0, PRO>(P, P.order[item], prof, qring, s_sub, bb, lane, 0, pd);
  }
}

// One long pair, both directions in one launch: CTA b (one warp) fills stripe b % nstripes of direction
// b / nstripes.  All CTAs must be co-resident (they wait on each other): launched cooperatively.
template <int K, int TBM, int STM, int PRO>
__global__ void __launch_bounds__(32) wave_kernel(const FillParams Pf, const FillParams Pr, int ndirs, const ProfDev pd) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int W = 32 * K;
  const int nst = Pf.wave_nstripes;
  const int d = blockIdx.x / nst, st = blockIdx.x % nst;
  if (d >= ndirs) return;
  const FillParams& P = d ? Pr : Pf;
  const int A = P.sc.A;
  int8_t* s_sub = reinterpret_cast<int8_t*>(smem);
  const int sub_bytes = (A * A + 15) / 16 * 16;
  const int lane = threadIdx.x;
  uint8_t* qring = smem + sub_bytes;  // followed by the 512-byte staging block of the input boundary
  int8_t* prof = reinterpret_cast<int8_t*>(smem + sub_bytes + kQRing + 512);
  if (!PRO)
    for (int x = threadIdx.x; x < A * A; x += blockDim.x) s_sub[x] = P.sub8[x];
  __syncwarp();
  fill_pair_warp<K, TBM, STM, 1, PRO>(P, P.wave_pair, prof, qring, s_sub, nullptr, lane, st, pd);
}


// ------------------------------------------------------------------------------------------------
// Packed-traceback decode (shared by host and device).
// tb: packed traceback of one pair in FLOW coordinates. Returns the flow predecessor of flow
// cell (a,b), 1 <= a <= Lq, 1 <= b <= Lt.
// ------------------------------------------------------------------------------------------------
// Storage layout of one pair's products in one direction.
//   sig  = number of leading pad columns (0 for the int32 kernels and the packed reverse pass,
//          16*ceil(Lt/16)-Lt for the right-aligned packed forward pass);
//   skew = 0: row-major (int32 kernels).  1: diagonal-major (packed kernels): the 16-column chunk
//          k of flow row a lives in "skew row" (a-1)+k, so everything a warp produces in one step
//          is contiguous in memory (the lanes of a segment are skewed by one row per lane).
//   nib  = 1: row-major like skew = 0, but the traceback is grouped by FOUR columns (the multi-CTA wavefront
//          kernel owns 4 columns per lane): 2 bytes per group, byte 0 = planes 0|1, byte 1 = planes 2|3 as
//          high|low nibbles, bit 3-(c&3) of a nibble = column c of the group.
struct Layout {
  int Lq, Lt, n;  // n = ceil(Lt/16) chunks
  int sig, skew, nib;
};
// fmt: 0 = int32 kernels, 1 = packed kernels, 2 = wavefront kernel (the per-pair class of the host scheduler)
__host__ __device__ inline Layout make_layout(int Lq, int Lt, int fmt, int rev) {
  Layout L;
  L.Lq = Lq; L.Lt = Lt; L.n = (Lt + 15) >> 4;
  L.skew = fmt == 1 ? 1 : 0;
  L.nib = (fmt == 2 && kWaveK == 4) ? 1 : 0;
  L.sig = (fmt == 1 && !rev) ? 16 * L.n - Lt : 0;
  return L;
}
// bytes of packed traceback / int16 units of scores / 32-bit words of mask one pair occupies
__host__ __device__ inline int64_t layout_tb_bytes(const Layout& L) {
  return L.skew ? (int64_t)(L.Lq + L.n - 1) * L.n * 8 : (int64_t)L.Lq * tb_row_bytes(L.Lt);
}
__host__ __device__ inline int64_t layout_sc_elems(const Layout& L) {
  return L.skew ? (int64_t)(L.Lq + L.n - 1) * L.n * 16 : (int64_t)L.Lq * sc_row_elems(L.Lt);
}
__host__ __device__ inline int64_t layout_mask_words(const Layout& L) {
  return L.skew ? ((int64_t)(L.Lq + L.n - 1) * L.n * 2 + 3) / 4 : (int64_t)L.Lq * ((L.Lt + 31) / 32);
}
// byte offset of the traceback byte holding plane `plane` of flow cell (a,b); *bit = bit index in it
__host__ __device__ inline int64_t layout_tb_byte(const Layout& L, int a, int b, int plane, int* bit) {
  const int pos = b - 1 + L.sig;
  if (L.nib) {
    *bit = ((plane & 1) ? 0 : 4) + 3 - (pos & 3);
    return (int64_t)(a - 1) * tb_row_bytes(L.Lt) + 2 * (pos >> 2) + (plane >> 1);
  }
  *bit = 7 - (pos & 7);
  if (L.skew) {
    const int k = pos >> 4;
    return ((int64_t)(a - 1 + k) * L.n + k) * 8 + 4 * ((pos >> 3) & 1) + plane;
  }
  return (int64_t)(a - 1) * tb_row_bytes(L.Lt) + 4 * (pos >> 3) + plane;
}
// element index (int16 or int32 units) of the score of flow cell (a,b)
__host__ __device__ inline int64_t layout_sc_index(const Layout& L, int a, int b) {
  const int pos = b - 1 + L.sig;
  if (L.skew) {
    const int k = pos >> 4, e = pos & 15;
    return (((int64_t)(a - 1 + k) * 2 + (e >> 3)) * L.n + k) * 8 + (e & 7);
  }
  return (int64_t)(a - 1) * sc_row_elems(L.Lt) + pos;
}
__host__ __device__ inline int tb_plane(const uint8_t* tb, const Layout& L, int a, int b, int plane) {
  int bit;
  const uint8_t byte = tb[layout_tb_byte(L, a, b, plane, &bit)];
  return (byte >> bit) & 1;
}

__host__ __device__ inline void decode_prev(const uint8_t* tb, const Layout& L, int a, int b, int* pa, int* pb) {
  if (a == 1 || b == 1) { *pa = 0; *pb = 0; return; }  // dpmatrix.h:408-426: boundary cells point at the anchor
  const int r = a - 1, c = b - 1;
  if (tb_plane(tb, L, r, c, 1)) {  // F won: walk up column c while the gap was extended
    int rr = r;
    while (rr > 1 && !tb_plane(tb, L, rr, c, 3)) --rr;
    *pa = rr - 1; *pb = c;
  } else if (tb_plane(tb, L, r, c, 0)) {  // E won: walk left along row r
    int cc = c;
    while (cc > 1 && !tb_plane(tb, L, r, cc, 2)) --cc;
    *pa = r; *pb = cc - 1;
  } else {
    *pa = r; *pb = c;
  }
}

// Predecessor of the final flow cell (Lq+1, Lt+1) from the per-pair record.
__host__ __device__ inline void decode_final(const uint8_t* tb, const Layout& L, int kind, int k, int* pa, int* pb) {
  const int Lq = L.Lq, Lt = L.Lt;
  if (Lq == 0 || Lt == 0) { *pa = 0; *pb = 0; return; }
  if (kind == 0) { *pa = Lq; *pb = Lt; }
  else if (kind == 1) { *pa = Lq; *pb = k; }
  else {
    int rr = Lq;
    while (rr > 1 && !tb_plane(tb, L, rr, Lt, 3)) --rr;
    *pa = rr - 1; *pb = Lt;
  }
}

// ------------------------------------------------------------------------------------------------
// Near-optimal cell set (SURVEY.md §0.9; consumed by ucw.h:141-180): one block per pair.
// mask bit (j-1) of row (i-1) is set iff F(i,j) + R(i,j) - sim(i,j) > thr, thr = cw.h:86-88.
// ------------------------------------------------------------------------------------------------
struct MaskParams {
  Scoring sc;
  const int8_t* sub8;
  const uint8_t* residues;
  const int64_t* seq_off;
  const int32_t* pair_q;
  const int32_t* pair_t;
  int n_pairs;
  int st_mode;               // 1 = int16 scores, 2 = int32
  const void* scF; const void* scR;
  const int64_t* sc_off;
  const int32_t* fin_fwd;    // forward final score (integer units)
  float delta_ratio;
  uint32_t* mask;            // bit blob
  const int64_t* mask_off;   // per pair word offset
  float* threshold;          // per pair (may be null)
  long long* count;          // per pair (may be null)
  const uint8_t* fmt;        // per pair: 0 = int32 kernels, 1 = packed kernels, 2 = wavefront (long pair)
  int want_fmt;              // which class this launch handles
  int only_pair;             // >= 0: this launch covers one pair, rows split over blockIdx.y
};

__host__ __device__ inline int64_t mask_row_words(int Lt) { return (Lt + 31) / 32; }

__device__ __forceinline__ float nearopt_threshold(float opt, float delta_ratio) {
  float thr = __fmul_rn(1.f - delta_ratio, opt);  // (1.f - delta_ratio) * opt, cw.h:86-87
  float alt = __fsub_rn(opt, 0.1f);               // cw.h:88
  return fminf(thr, alt);
}

#ifndef AADP_MASK_U
#define AADP_MASK_U 4
#endif
constexpr int kMaskU = AADP_MASK_U;  // 32-column groups a warp loads before it uses any (bytes in flight per thread)
template <int PRO>
__global__ void __launch_bounds__(256) mask_kernel(const MaskParams P, const ProfDev pd) {
  const int pair = P.only_pair >= 0 ? P.only_pair : blockIdx.x;
  if (P.fmt[pair] != P.want_fmt) return;
  const int qs = P.pair_q[pair], ts = P.pair_t[pair];
  const int64_t qo = P.seq_off[qs], to = P.seq_off[ts];
  const int Lq = (int)(P.seq_off[qs + 1] - qo), Lt = (int)(P.seq_off[ts + 1] - to);
  const float inv = 1.f / (float)(1 << P.sc.scale_log2);
  const float opt = (float)P.fin_fwd[pair] * inv;
  const float thr = nearopt_threshold(opt, P.delta_ratio);
  if (threadIdx.x == 0 && blockIdx.y == 0 && P.threshold) P.threshold[pair] = thr;
  if (Lq == 0 || Lt == 0) { if (threadIdx.x == 0 && blockIdx.y == 0 && P.count) P.count[pair] = 0; return; }
  const int64_t scs = sc_row_elems(Lt), mws = mask_row_words(Lt);
  const int64_t so = P.sc_off[pair];
  uint32_t* mk = P.mask + P.mask_off[pair];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int A = P.sc.A;
  long long cnt = 0;
  // a block owns a contiguous band of rows and walks it row by row, its warps side by side along the row:
  // few concurrent DRAM streams (two per block), each fully sequential
  const int rows_per_blk = (Lq + gridDim.y - 1) / gridDim.y;
  const int i_lo = 1 + rows_per_blk * blockIdx.y, i_hi = min(Lq, i_lo + rows_per_blk - 1);
  // Integer form of  (F + R) - sim > thr  (ucw.h:141-180): on the dyadic grid every term is an exact fp32 number, so the
  // reference's float comparison equals  slack > floor(thr * 2^s)  on the integers (the packed kernels use the same form).
  const int thr_i = (int)fminf(fmaxf(floorf(thr * (float)(1 << P.sc.scale_log2)), -2.0e9f), 2.0e9f);
  const uint8_t* tres = P.residues + to;
  // PRO: the forward-flow profile row of the query code, shifted so that column jm+1 is subrow[jm]
  const int8_t* prof0 = PRO ? prof_flow(pd, ts, Lt, A, 0) + (prof_row_bytes(Lt) - Lt) : nullptr;
  for (int i = i_lo; i <= i_hi; ++i) {
    const int qa = P.residues[qo + i - 1];
    const int8_t* subrow = PRO ? prof0 + qa * prof_row_bytes(Lt) : P.sub8 + qa * A;
    // row pointers: forward row i ascending, reverse row Lq-i descending (the reverse matrix is stored in flow coordinates)
    const int16_t* f16 = (const int16_t*)P.scF + so + (int64_t)(i - 1) * scs;
    const int16_t* r16 = (const int16_t*)P.scR + so + (int64_t)(Lq - i) * scs + (Lt - 1);
    const int32_t* f32 = (const int32_t*)((const int16_t*)P.scF + so) + (int64_t)(i - 1) * scs;
    const int32_t* r32 = (const int32_t*)((const int16_t*)P.scR + so) + (int64_t)(Lq - i) * scs + (Lt - 1);
    uint32_t* mrow = mk + (int64_t)(i - 1) * mws;
    // kMaskU*32 columns per iteration: the loads of kMaskU 32-column groups are issued before any of them is used
    for (int j0 = 32 * kMaskU * warp; j0 < Lt; j0 += 32 * kMaskU * nw) {
      bool on[kMaskU];
#pragma unroll
      for (int u = 0; u < kMaskU; ++u) {
        const int jm = j0 + 32 * u + lane;  // column index - 1
        on[u] = false;
        if (jm < Lt) {
          int f, r;
          if (P.st_mode == 1) { f = f16[jm]; r = r16[-jm]; }
          else { f = f32[jm]; r = r32[-jm]; }
          on[u] = f + r - (int)subrow[PRO ? jm : tres[jm]] > thr_i;
        }
      }
      uint32_t mine = 0;
#pragma unroll
      for (int u = 0; u < kMaskU; ++u) {
        const uint32_t bits = __ballot_sync(0xffffffffu, on[u]);
        if (lane == u) mine = bits;
      }
      if (lane < kMaskU && j0 + 32 * lane < Lt) { mrow[(j0 >> 5) + lane] = mine; cnt += __popc(mine); }
    }
  }
  if (P.count) {
    __shared__ long long s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    if (cnt) atomicAdd((unsigned long long*)&s_cnt, (unsigned long long)cnt);
    __syncthreads();
    if (threadIdx.x == 0) {
      if (gridDim.y == 1) P.count[pair] = s_cnt;
      else atomicAdd((unsigned long long*)&P.count[pair], (unsigned long long)s_cnt);  // zeroed by the host
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Dense, reference-shaped expansion of one pair (DPCell::score / prev_*; dpmatrix.h:28-37).
// ------------------------------------------------------------------------------------------------
struct DenseParams {
  Scoring sc;
  int Lq, Lt, rev, repro_rev_bug;
  Layout lay;
  int bias;  // packed kernels store biased scores
  int st_mode;
  const void* sc_blob; int64_t sc_off;
  const uint8_t* tb;  // packed traceback of this pair/direction (or null)
  int fin_score, fin_kind, fin_k;
  float* score;       // (Lq+2)*(Lt+2) or null
  int32_t* prev_q;    // or null
  int32_t* prev_t;
};

__global__ void dense_kernel(const DenseParams P) {
  const int sz1 = P.Lq + 2, sz2 = P.Lt + 2;
  const int64_t n = (int64_t)sz1 * sz2;
  const float inv = 1.f / (float)(1 << P.sc.scale_log2);
  for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < n; o += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(o / sz2), j = (int)(o % sz2);
    // flow coordinates
    const int a = P.rev ? P.Lq + 1 - i : i, b = P.rev ? P.Lt + 1 - j : j;
    float s = 0.f;
    int pa = -1, pb = -1;  // flow predecessor; -1 = DPCell::null
    const bool interior = a >= 1 && a <= P.Lq && b >= 1 && b <= P.Lt;
    int si = 0;
    if (interior) {
      if (P.st_mode == 1) si = ((const int16_t*)P.sc_blob)[P.sc_off + layout_sc_index(P.lay, a, b)] - P.bias;
      else if (P.st_mode == 2) si = ((const int32_t*)((const int16_t*)P.sc_blob + P.sc_off))[layout_sc_index(P.lay, a, b)];
      s = (float)si * inv;
      if (P.tb) {
        decode_prev(P.tb, P.lay, a, b, &pa, &pb);
        // local fills: a cell clamped to 0 keeps the match predecessor (dpmatrix.h:616-646)
        if (P.sc.local && si == 0 && a > 1 && b > 1) { pa = a - 1; pb = b - 1; }
      }
    } else if (a == P.Lq + 1 && b == P.Lt + 1) {
      s = (float)P.fin_score * inv;
      if (P.Lq == 0 || P.Lt == 0) { pa = 0; pb = 0; }
      else if (P.tb) decode_final(P.tb, P.lay, P.fin_kind, P.fin_k, &pa, &pb);
      else if (P.fin_kind == 0) { pa = P.Lq; pb = P.Lt; }
      else if (P.fin_kind == 1) { pa = P.Lq; pb = P.fin_k; }
    }
    if (P.score) P.score[o] = s;
    if (P.prev_q) {
      int pi = -1, pj = -1;
      if (pa >= 0) {
        pi = P.rev ? P.Lq + 1 - pa : pa;
        pj = P.rev ? P.Lt + 1 - pb : pb;
        // dpmatrix.h:868: the global reverse fill stores opt_j = t1_m1 for left-column candidates
        if (P.rev && !P.sc.local && P.repro_rev_bug && !interior && P.fin_kind == 2 && P.Lq > 0 && P.Lt > 0) pj = P.Lt;
      }
      P.prev_q[o] = pi;
      P.prev_t[o] = pj;
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Optimal alignments of a whole batch on the GPU (SURVEY.md §8 row f1): one thread per pair follows the
// packed traceback in HBM from the final cell to the anchor -- Optimal::enumerate (optimal.h:47-75) for the
// forward matrices, Optimal_Rev::enumerate (optimal_rev.h:47-78) for the reverse ones.  The walk is a chain
// of dependent byte loads (latency bound), so the parallelism is across the pairs of the batch.
// Output slot of pair p: cap_off[p] .. cap_off[p+1] (capacity Lq+Lt+2 aligned pairs), filled front to back
// with (query_idx, template_idx) in matrix coordinates, including (0,0) and (last,last).
// ------------------------------------------------------------------------------------------------
struct TraceParams {
  const uint8_t* tb;         // packed traceback blob of the direction
  const int64_t* tb_off;
  const uint8_t* fmt;        // per pair: layout class (see make_layout)
  const int64_t* seq_off;
  const int32_t* pair_q;
  const int32_t* pair_t;
  const int32_t* fin_kind;
  const int32_t* fin_k;
  int n_pairs;
  int rev;                   // 0: forward matrices, 1: reverse matrices
  int repro_rev_bug;
  const int64_t* cap_off;    // per pair: first slot (in aligned pairs); slot p has Lq+Lt+2 entries
  int2* out;                 // aligned pairs
  int32_t* out_n;            // per pair: number of aligned pairs written
  int32_t* out_status;       // per pair: 0, or 3 = "Illegal alignment start pair" (optimal.h:74)
};

__global__ void __launch_bounds__(128) traceback_kernel(const TraceParams P) {
  const int pair = blockIdx.x * blockDim.x + threadIdx.x;
  if (pair >= P.n_pairs) return;
  const int qs = P.pair_q[pair], ts = P.pair_t[pair];
  const int Lq = (int)(P.seq_off[qs + 1] - P.seq_off[qs]), Lt = (int)(P.seq_off[ts + 1] - P.seq_off[ts]);
  const uint8_t* tb = P.tb + P.tb_off[pair];
  const Layout L = make_layout(Lq, Lt, P.fmt[pair], P.rev);
  const int kind = P.fin_kind[pair], fk = P.fin_k[pair];
  int2* out = P.out + P.cap_off[pair];
  const int cap = Lq + Lt + 2;
  // flow coordinates: (a,b) runs from the final flow cell (Lq+1,Lt+1) down to the anchor (0,0)
  int a = Lq + 1, b = Lt + 1, n = 0;
  bool first = true, ok = true;
  for (;;) {
    // matrix coordinates of the current cell; forward alignments are built with prepend(): fill from the back
    const int i = P.rev ? Lq + 1 - a : a, j = P.rev ? Lt + 1 - b : b;
    if (n < cap) out[P.rev ? n : cap - 1 - n] = make_int2(i, j);
    ++n;
    if (a <= 0 || n > cap) break;  // optimal.h:61 loops while the query index is positive (rev: below last)
    int pa = -1, pb = -1;
    if (first) {
      decode_final(tb, L, kind, fk, &pa, &pb);
      // dpmatrix.h:868: the global reverse fill stores opt_j = t1_m1 (a MATRIX column) for left-column
      // candidates; followed literally the walk leaves the legal path and the reference throws
      if (P.rev && P.repro_rev_bug && kind == 2 && Lq > 0 && Lt > 0) pb = Lt + 1 - Lt;  // matrix column Lt -> flow column 1
      first = false;
    } else if (a >= 1 && a <= Lq && b >= 1 && b <= Lt) {
      decode_prev(tb, L, a, b, &pa, &pb);
    }
    if (pa < 0 || pb < 0) {  // DPCell::null reached: recorded like the reference would read it, then stop
      if (n < cap) out[P.rev ? n : cap - 1 - n] = make_int2(-1, -1);
      ++n;
      ok = false;
      break;
    }
    a = pa;
    b = pb;
  }
  if (ok && (a != 0 || b != 0)) ok = false;  // "Illegal alignment start pair"
  if (n > cap) { n = cap; ok = false; }
  if (!P.rev && n < cap)  // move the tail-filled forward alignment to the front of its slot
    for (int k = 0; k < n; ++k) out[k] = out[cap - n + k];
  P.out_n[pair] = n;
  P.out_status[pair] = ok ? 0 : 3;
}

// ------------------------------------------------------------------------------------------------
// LOCAL optimal alignments of a whole batch: Optimal::enumerate_local + find_max (optimal.h:76-124) for the forward
// matrices, Optimal_Rev::enumerate_local + find_max (optimal_rev.h:79-131) for the reverse ones.  One warp per pair:
// the 32 lanes search the stored score matrix for its first maximum in the reference's scan order (strict '<' over
// ascending flow coordinates; the starting candidate is D[sz1-2][sz2-2] forward but D[0][0] -- the final cell of the
// reverse fill -- in reverse, an asymmetry of the reference that is kept), then lane 0 follows the packed traceback
// until a predecessor with score <= 0.  Scores are compared in integer units (exact).
// Output slot as in traceback_kernel; (last,last) forward / (0,0) reverse frames the alignment as the reference does.
// ------------------------------------------------------------------------------------------------
struct LocalTraceParams {
  TraceParams t;
  const void* sc_blob;       // score blob of the direction
  const int64_t* sc_off;
  int st_mode_v1;            // storage of the non-packed pairs: 1 = int16, 2 = int32
  int bias16;
  const int32_t* fin_score;  // per pair: score of the final flow cell
  float inv_scale;
  float* out_score;          // per pair: AlignedPairList::score, or null
};

__global__ void __launch_bounds__(128) local_traceback_kernel(const LocalTraceParams Q) {
  const TraceParams& P = Q.t;
  const int pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (pair >= P.n_pairs) return;
  const int qs = P.pair_q[pair], ts = P.pair_t[pair];
  const int Lq = (int)(P.seq_off[qs + 1] - P.seq_off[qs]), Lt = (int)(P.seq_off[ts + 1] - P.seq_off[ts]);
  const uint8_t* tb = P.tb + P.tb_off[pair];
  const int fmt = P.fmt[pair];
  const Layout L = make_layout(Lq, Lt, fmt, P.rev);
  const int st_mode = fmt == 1 ? 1 : Q.st_mode_v1, bias = fmt == 1 ? Q.bias16 : 0;
  const int64_t sco = Q.sc_off[pair];
  const int fin = Q.fin_score[pair];
  auto score = [&](int a, int b) -> int {  // flow cell -> DPCell::score in integer units
    if (a >= 1 && a <= Lq && b >= 1 && b <= Lt) {
      if (st_mode == 1) return (int)((const int16_t*)Q.sc_blob)[sco + layout_sc_index(L, a, b)] - bias;
      return ((const int32_t*)((const int16_t*)Q.sc_blob + sco))[layout_sc_index(L, a, b)];
    }
    return (a == Lq + 1 && b == Lt + 1) ? fin : 0;
  };
  // find_max: first interior maximum in ascending flow order (cells of flow row/column 0 hold 0 and never win '<')
  int best = INT_MIN;
  int64_t bidx = 0;
  const int64_t ncell = (int64_t)Lq * Lt;
  if (fmt == 1) {
    // packed pairs: the blob is walked in STORAGE order (diagonal-major, 16-byte chunks of 8 columns: coalesced) instead of
    // matrix order; "first maximum in ascending flow order" then needs the index in the comparison
    const int nchunk = (Lq + L.n - 1) * 2 * L.n;
    const int16_t* sc = (const int16_t*)Q.sc_blob + sco;
    for (int c = lane; c < nchunk; c += 32) {
      const int k = c % L.n, rh = c / L.n, h = rh & 1, r = rh >> 1;
      const int a = r - k + 1;
      if (a < 1 || a > Lq) continue;
      const uint4 w = *reinterpret_cast<const uint4*>(sc + (int64_t)c * 8);
      const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
      const int b0 = 16 * k + 8 * h - L.sig + 1;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int b = b0 + e;
        if (b < 1 || b > Lt) continue;
        const int v = (int)(short)((ww[e >> 1] >> (16 * (e & 1))) & 0xffffu) - bias;
        const int64_t idx = (int64_t)(a - 1) * Lt + (b - 1);
        if (v > best || (v == best && idx < bidx)) { best = v; bidx = idx; }
      }
    }
  } else {
    for (int a = 1; a <= Lq; ++a)  // (row by row: a lane meets its cells in ascending order without a 64-bit division per cell)
      for (int b = 1 + lane; b <= Lt; b += 32) {
        const int v = score(a, b);
        if (v > best) { best = v; bidx = (int64_t)(a - 1) * Lt + (b - 1); }
      }
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const int ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int64_t oi = __shfl_xor_sync(0xffffffffu, bidx, o);
    if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
  }
  if (lane != 0) return;
  // the starting candidate of the reference's scan (optimal.h:111-113 / optimal_rev.h:118-120)
  int a = P.rev ? Lq + 1 : Lq, b = P.rev ? Lt + 1 : Lt;
  int s = score(a, b);
  if (ncell > 0 && best > s) { a = (int)(bidx / Lt) + 1; b = (int)(bidx % Lt) + 1; s = best; }
  auto prev = [&](int ca, int cb, int* pa, int* pb) {
    *pa = -1; *pb = -1;
    if (ca == Lq + 1 && cb == Lt + 1) { decode_final(tb, L, P.fin_kind[pair], P.fin_k[pair], pa, pb); return; }
    if (ca < 1 || ca > Lq || cb < 1 || cb > Lt) return;
    decode_prev(tb, L, ca, cb, pa, pb);
    if (score(ca, cb) == 0 && ca > 1 && cb > 1) { *pa = ca - 1; *pb = cb - 1; }  // clamped cell: dpmatrix.h:616-646
  };
  // two passes over the same walk: count, then write front to back in matrix order
  const int cap = Lq + Lt + 2;
  int2* out = P.out + P.cap_off[pair];
  int n_walk = 1, ea = a, eb = b;  // cells from the maximum down the traceback (the maximum included)
  {
    int ca = a, cb = b;
    while (ca > 0) {
      int pa, pb;
      prev(ca, cb, &pa, &pb);
      ca = pa; cb = pb;
      ea = ca; eb = cb;
      if (ca < 0 || score(ca, cb) <= 0) break;
      ++n_walk;
    }
  }
  const bool frame0 = (ea != 0 && eb != 0);  // optimal.h:105: prepend (0,0) unless the walk ended on row or column 0
  const int total = n_walk + 1 + (frame0 ? 1 : 0);
  auto put = [&](int k, int fa, int fb) {  // k-th pair counted from the frame (last,last) [fwd] / (0,0) [rev]
    const int i = P.rev ? Lq + 1 - fa : fa, j = P.rev ? Lt + 1 - fb : fb;
    const int pos = P.rev ? k : total - 1 - k;
    if (pos >= 0 && pos < cap) out[pos] = make_int2(i, j);
  };
  put(0, Lq + 1, Lt + 1);
  {
    int ca = a, cb = b;
    for (int k = 0; k < n_walk; ++k) {
      put(1 + k, ca, cb);
      int pa, pb;
      prev(ca, cb, &pa, &pb);
      ca = pa; cb = pb;
    }
  }
  if (frame0) put(1 + n_walk, 0, 0);
  P.out_n[pair] = min(total, cap);
  P.out_status[pair] = 0;
  if (Q.out_score) Q.out_score[pair] = (float)s * Q.inv_scale;
}

}  // namespace aadp
