// aadp_packed.cuh -- the fast path: packed int16x2 ("two pairs per register") segmented systolic
// fill kernel for sm_100a, built on the DPX instructions VIADDMNMX.S16x2 / VIMNMX.S16x2 /
// VIADD.16x2 and on PRMT sign-replication for the traceback bit gather.
//
// Same recurrence and tie rules as aadp_kernels.cuh (dpmatrix.h:356-1030; SURVEY.md App. A.2).
// What changes is the mapping:
//   * every 32-bit register holds the same DP quantity of TWO independent pairs (a "couple":
//     pair A in the low half, pair B in the high half), so one instruction updates two cells;
//   * a warp is split into contiguous lane SEGMENTS; a segment of n = ceil(Lt/16) lanes owns one
//     couple, lane `off` of a segment owns 16 consecutive template columns and runs `off` rows
//     behind lane 0 (skewed systolic array).  Short templates therefore use few lanes and several
//     couples share a warp ("task"); the host bin-packs couples of similar query length into tasks;
//   * the forward pass is RIGHT-aligned (the last template column is always register 15 of the
//     segment's last lane, pad columns come first and reproduce the boundary column through the F
//     recurrence), the reverse pass is LEFT-aligned in its own flow.  Both therefore cut the
//     template into the SAME 16-column chunks, so the reverse pass reads the forward scores with
//     aligned 16-byte loads and emits the near-optimal cell set F+R-sim > thr (ucw.h:141-180,
//     cw.h:86-88) on the fly -- the forward+reverse fusion of BASELINE.json's north_star.
//
// Layouts (struct Layout in aadp_kernels.cuh; `sig` = number of leading pad columns): DIAGONAL-MAJOR.
// Lane `off` of a segment works on flow row a = step-off+1, so chunk k of row a is produced at step
// r = (a-1)+k.  Everything is stored by "skew row" r, which makes every store of a step contiguous
// across the lanes of a segment (fully coalesced), and -- because the reverse pass is skewed the
// opposite way -- makes the reverse pass read ONE contiguous skew row of forward scores per step:
//   traceback  [r][slot k] 8 bytes: two 32-bit words (8 columns each), byte p = plane p,
//              bit 7-(c&7) = register c; register c of slot k is flow column 16k+c+1-sig
//   scores     int16 [r][c>>3][slot k][c&7]   (two 16-byte halves per slot, each half contiguous over k)
//   mask       reverse-flow coordinates [r][slot k] 2 bytes: byte (c&1), bit 7-(c>>1)
#pragma once
#include "aadp_kernels.cuh"
#include <cuda_fp16.h>

namespace aadp {

// BIASED DOMAIN.  Every DP value v is held as v + kBias16 in an unsigned 16-bit half with
//   1024 <= v + kBias16 < 0x7C00.
// Two things follow.  (1) The halves are positive, normal fp16 bit patterns whose fp16 order equals
// their integer order, so HSET2.GT (one instruction on the fp16 pipe, no predicates) yields a
// 0xFFFF/0 mask per half for the traceback decisions.  (2) Adding a packed non-positive constant is
// a plain 32-bit add (the low half always carries into the high half, which the constant
// pre-compensates), so those adds can issue on the FMA pipe (IMAD.IADD) instead of the ALU pipe.
// kBias16 is chosen so that (a) single-biased values v + B stay inside [1024, 0x7C00) for v in [kNeg16 - drift, bound)
// and (b) DOUBLY biased sums F + X (the near-optimal slack, v in [-2*bound, bound)) stay inside (0x8000, 0xFC00):
// there they are negative, finite fp16 patterns whose fp16 order is the REVERSE of their integer order, so the same
// one-instruction sign test decides slack > thr without removing a bias first (see the MSK pass).
constexpr int kBias16 = 24000;
constexpr int kNeg16 = -20000;    // "-infinity" seed of E/F chains (only ever extended once)
constexpr int kFloor16 = -13000;  // clamp floor of M / slack
constexpr int kPackedBound = 7000;  // |score| bound (integer units) a pair must satisfy to use this kernel
// Build-time toggles of the variant measurements (profiles/r02_packed_variants.md); the defaults are the shipped kernel.
#ifndef AADP_GAT_IMAD
#define AADP_GAT_IMAD 1   // traceback / mask bit gather: 1 = multiply-add on the FMA pipe, 0 = LOP3 on the ALU pipe
#endif
#ifndef AADP_PROF_AHEAD
#define AADP_PROF_AHEAD 1  // profile words of the next row loaded during the current step (software pipelining)
#endif
#ifndef AADP_SLACK_IMAD
#define AADP_SLACK_IMAD 1  // near-optimal slack: 1 = one FMA-pipe add + double-biased compare, 0 = three-input ALU add
#endif
constexpr int kFwdAhead = 8;      // rows of L2 prefetch distance for the forward scores the reverse+mask pass reads
constexpr int kPackedWarps = 1;   // warps per CTA (one: finest shared-memory granularity -> most warps per SM)
// per-warp cp.async staging: query rings (1 KB: 2 halves x 2 blocks of 8 rows per lane) + forward-score chunks
// (6 KB, reverse+mask pass only).  Shared memory is what bounds the warps per SM, so nothing else gets a region of
// its own: the padded substitution table is only needed while a profile is being built and ALIASES the staging
// area (copied in per task, before the first cp.async of the task is issued), and the 512-byte reduction scratch
// of the final cells aliases the profile (dead by then) -- except in cross mode, where the profile outlives the
// query couples of an item and the scratch has its own 512 bytes.
// Per CTA: forward 21.5 KB -> 10 warps/SM, reverse+mask 27 KB -> 8 warps/SM (was 23.5 / 29.6 KB: 9 and 7).
// bytes of the padded substitution table: A rows of A+1 entries (entry A = pad = -128), rounded up to 16
__host__ __device__ inline int packed_sub_bytes(int A) { return (A * (A + 1) + 15) / 16 * 16; }
__host__ __device__ inline int packed_stage_bytes(int A, int msk) {
  const int st = msk ? 1024 + 6144 : 1024;
  return st > packed_sub_bytes(A) ? st : packed_sub_bytes(A);  // alphabets above 31 letters need more than 1 KB
}
// xm (cross mode): both halves of a couple align against the SAME template, so one profile serves both
__host__ __device__ inline size_t packed_smem_bytes(int A, int msk, int xm = 0) {
  return (size_t)kPackedWarps * ((xm ? 32 * sizeof(int4) : 0) + packed_stage_bytes(A, msk) + (xm ? 1 : 2) * A * 512);
}

struct PackedParams {
  Scoring sc;
  const int8_t* sub8;        // A*A scaled substitution scores
  const int8_t* sub8p;       // the same, padded: A rows of A+1 entries (entry A = -128), packed_sub_bytes(A) bytes
  const uint8_t* arena;      // 4-byte aligned sequence arena in the FLOW order of this direction
  const int32_t* aoff;       // per sequence: byte offset into arena
  const int64_t* seq_off;    // nseq+1 (lengths)
  const int32_t* pair_q;
  const int32_t* pair_t;
  const int32_t* tasks;      // n_tasks * 64: pair id (or -1) of lane l, half h at [task*64 + h*32 + l]
  int n_tasks;
  int rev;
  unsigned int* counter;
  uint8_t* tb;               // packed traceback blob of this direction
  const int64_t* tb_off;
  int16_t* sc_out;           // score blob of this direction (written when FST)
  const int16_t* scF;        // forward score blob (read when MSK)
  const int64_t* sc_off;
  uint32_t* mask;            // near-optimal bit blob (written when MSK)
  const int64_t* mask_off;
  const int32_t* fin_fwd;    // forward final scores, integer units (MSK)
  float delta_ratio;
  float* threshold;          // per pair, may be null (MSK)
  long long* count;          // per pair, may be null (MSK)
  int32_t* fin_score;
  int32_t* fin_kind;
  int32_t* fin_k;
  double cells_hint;
  // ---- cross mode (XM = 1): every query of a list against every template of a list, forward score only.
  // Work item = (layout, group of x_group query couples); a layout assigns 32 lanes to whole templates.
  const int32_t* x_layout;   // n_layouts * 32: template LIST index of lane l, or -1
  const int32_t* x_qc;       // n_qcouples * 2: query LIST indices of the two halves (both always valid)
  const int32_t* x_qid;      // query list index -> sequence id
  const int32_t* x_tid;      // template list index -> sequence id
  int x_nlayouts, x_nqc, x_group;
  long long x_nt;            // row stride of x_scores
  float* x_scores;           // [query list index][template list index] = D[last][last].score
  ProfDev prof;              // position-specific template profiles (read by the PRO = 1 kernels only)
};

__device__ __forceinline__ uint32_t pk2(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }
// biased pack
__device__ __forceinline__ uint32_t pkb(int lo, int hi) { return pk2(lo + kBias16, hi + kBias16); }
// 32-bit addend that subtracts dlo from the low half and dhi from the high half (dlo,dhi >= 0) of a
// biased pair: the low half borrows nothing (values >= 1024 > d), i.e. adding 65536-dlo always carries
// into the high half, so the high constant is reduced by that carry.
__device__ __forceinline__ uint32_t pkdec(int dlo, int dhi) {
  const uint32_t lo = (uint32_t)(-dlo) & 0xffffu;
  const uint32_t carry = dlo != 0 ? 1u : 0u;
  return lo | (((uint32_t)(-dhi) - carry) << 16);
}
// packed add of a pkdec() constant: a single 32-bit integer add, written as a multiply-add so that it
// issues on the FMA pipe (IMAD) and leaves the ALU pipe to the DPX min/max instructions
__device__ __forceinline__ uint32_t addc(uint32_t x, uint32_t c) {
  uint32_t d;
  asm("mad.lo.u32 %0, %1, 1, %2;" : "=r"(d) : "r"(x), "r"(c));
  return d;
}
// fp16x2 difference a - b of two biased pairs (HADD2 with a negated operand, on the fp16/FMA-lite pipe):
// only its SIGN bits (bit 15 / bit 31) are used -- set exactly where a < b, because the biased halves
// are positive fp16 bit patterns ordered like the integers and an fp16 difference never rounds across 0.
// Measured on B200 (profiles/microbench/pipes.cu): HSET2, PRMT and VIADDMNMX are half-rate on the ALU
// pipe the VIMNMX chain lives on, HADD2 / VIADD.16x2 run on a different pipe.
__device__ __forceinline__ uint32_t lt_sign(uint32_t a, uint32_t b) {
  const __half2 d = __hsub2(*reinterpret_cast<const __half2*>(&a), *reinterpret_cast<const __half2*>(&b));
  return *reinterpret_cast<const uint32_t*>(&d);
}
__device__ __forceinline__ int lo16(uint32_t v) { return (int)(short)(v & 0xffffu); }
__device__ __forceinline__ int hi16(uint32_t v) { return ((int)v) >> 16; }
__device__ __forceinline__ int half16(uint32_t v, int h) { return h ? hi16(v) : lo16(v); }
__device__ __forceinline__ int unb16(uint32_t v, int h) { return (int)((v >> (16 * h)) & 0xffffu) - kBias16; }
// Asynchronous global->shared staging (LDGSTS): the prefetched bytes never occupy a register, so no
// instruction waits on them until cp_async_wait() one or more rows later.
// 32-bit shared-window address of a generic pointer into shared memory, computed ONCE (asm volatile: the compiler
// may not rematerialise it).  Left to itself it rebuilds the window base (S2R SR_CgaCtaId + LEA) in every row step
// for every shared-memory access made through a generic pointer.
__device__ __forceinline__ unsigned smem_u32(const void* p) {
  unsigned r;
  asm volatile("{ .reg .u64 t; cvta.to.shared.u64 t, %1; cvt.u32.u64 %0, t; }" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ uint4 lds128(unsigned sa) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(sa));
  return v;
}
__device__ __forceinline__ int lds_u8(unsigned sa) {
  unsigned v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(sa));
  return (int)v;
}
// A location in shared memory, held both as a generic pointer and as a pinned 32-bit shared-window address.  SA picks
// which one an access uses: the score-only kernels (few registers, short rows) gain 7 % from the pinned addresses,
// the traceback kernels lose 0.6 % to the extra live registers and keep the generic pointers.
struct SPtr {
  uint8_t* p;
  unsigned sa;
  __device__ __forceinline__ SPtr operator+(int o) const { return SPtr{p + o, sa + (unsigned)o}; }
};
template <bool SA> __device__ __forceinline__ SPtr sptr(void* p) { return SPtr{reinterpret_cast<uint8_t*>(p), SA ? smem_u32(p) : 0u}; }
template <bool SA> __device__ __forceinline__ uint4 ld16(const SPtr& x) { return SA ? lds128(x.sa) : *reinterpret_cast<const uint4*>(x.p); }
template <bool SA> __device__ __forceinline__ int ld1(const SPtr& x) { return SA ? lds_u8(x.sa) : (int)*x.p; }
__device__ __forceinline__ void cp_async16(unsigned sa, const void* gsrc, int cond) {
  asm volatile("{ .reg .pred q; setp.ne.s32 q, %2, 0; @q cp.async.ca.shared.global [%0], [%1], 16; }"
               :: "r"(sa), "l"(gsrc), "r"(cond) : "memory");
}
__device__ __forceinline__ void cp_async8(unsigned sa, const void* gsrc, int cond) {
  asm volatile("{ .reg .pred q; setp.ne.s32 q, %2, 0; @q cp.async.ca.shared.global [%0], [%1], 8; }"
               :: "r"(sa), "l"(gsrc), "r"(cond) : "memory");
}
// L2 prefetch of one sector (no destination, no scoreboard): the DRAM latency of a later cp.async is paid early
template <bool SA> __device__ __forceinline__ void cpa16(const SPtr& d, const void* g, int cond) {
  cp_async16(SA ? d.sa : (unsigned)__cvta_generic_to_shared(d.p), g, cond);
}
template <bool SA> __device__ __forceinline__ void cpa8(const SPtr& d, const void* g, int cond) {
  cp_async8(SA ? d.sa : (unsigned)__cvta_generic_to_shared(d.p), g, cond);
}
__device__ __forceinline__ void prefetch_l2(const void* gsrc, int cond) {
  asm volatile("{ .reg .pred q; setp.ne.s32 q, %1, 0; @q prefetch.global.L2 [%0]; }" :: "l"(gsrc), "r"(cond) : "memory");
}
// Predicated global stores: the per-half store blocks of a row step become straight-line code (no BSSY/BRA)
__device__ __forceinline__ void stg16_if(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d, bool cond) {
  asm volatile("{ .reg .pred q; setp.ne.s32 q, %5, 0; @q st.global.v4.u32 [%0], {%1,%2,%3,%4}; }"
               :: "l"(p), "r"(a), "r"(b), "r"(c), "r"(d), "r"((int)cond) : "memory");
}
__device__ __forceinline__ void stg8_if(void* p, uint32_t a, uint32_t b, bool cond) {
  asm volatile("{ .reg .pred q; setp.ne.s32 q, %3, 0; @q st.global.v2.u32 [%0], {%1,%2}; }"
               :: "l"(p), "r"(a), "r"(b), "r"((int)cond) : "memory");
}
__device__ __forceinline__ void stg2_if(void* p, uint32_t a, bool cond) {
  asm volatile("{ .reg .pred q; setp.ne.s32 q, %2, 0; @q st.global.u16 [%0], %1; }"
               :: "l"(p), "h"((unsigned short)a), "r"((int)cond) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
// Bit gather on the FMA pipe.  t holds four bytes that are 0xFF or 0x00 (PRMT sign replication); bit k of byte j of
// the result must be set where byte j of t is 0xFF.  Instead of  acc |= t & (0x01010101 << k)  (LOP3, ALU pipe -- the
// pipe the VIMNMX/PRMT recurrence saturates), accumulate  acc -= t << k  with ONE multiply-add (IMAD, FMA pipe):
// 0xFF << (8j+k) = 2^(8j+8+k) - 2^(8j+k), so the sum over the eight cells of a group telescopes to B - (B << 8),
// B being the wanted word, and B = acc * (1 + 2^8 + 2^16 + 2^24) mod 2^32 -- one more IMAD per group (gat_fin).
__device__ __forceinline__ uint32_t gat(uint32_t acc, uint32_t t, int k) {
#if AADP_GAT_IMAD
  uint32_t d;
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(t), "r"(0u - (1u << k)), "r"(acc));
  return d;
#else
  return acc | (t & (0x01010101u << k));
#endif
}
__device__ __forceinline__ uint32_t gat_fin(uint32_t acc) {
#if AADP_GAT_IMAD
  uint32_t d;
  asm("mul.lo.u32 %0, %1, 0x01010101;" : "=r"(d) : "r"(acc));
  return d;
#else
  return acc;
#endif
}

// Per-lane, per-half final-row summary (what the final cell needs from this lane's 16 columns).
struct RowSum {
  int rb_val, rb_k;  // best bottom-row candidate M(Lq,k) - pen(Lt-k), k < Lt (smallest k on ties)
  int diag, col;     // M(Lq,Lt) and the right-column candidate (lane owning column Lt only)
};

// LOC = 1: local alignments (dpmatrix.h:538-689, 879-1030): every candidate is clamped at 0 before it is compared
// (s = max(0.f, s), :580 etc.), i.e. M = max(0, sim + X); the gap states stay unclamped (they only ever lose against
// M >= 0 where the clamp would have mattered), a cell clamped to 0 keeps its match predecessor (decoded from the
// stored score, dense_kernel / local_traceback_kernel).  One more VIMNMX per packed cell.
// PRO = 1: position-specific template profiles (ProfDev, aadp_set_profile_scoring): the profile rows are copied from the
// template's int8 profile of this flow instead of being built from the substitution table; the row loop is unchanged.
// RB = 1 (forward pass with score spill, FST = 1): the final-row summary reads M(Lq, .) back from the score blob instead
// of parking the row state in local memory inside the row loop (see the capture below).
template <int TBM, int FST, int MSK, int XM, int LOC = 0, int PRO = 0, int RB = 0>
__device__ __forceinline__ void packed_task(const PackedParams& P, int task, int8_t* prof, int4* red,
                                            uint8_t* stage, int lane) {
  const Scoring& S = P.sc;
  const int gi = S.gi, ge = S.ge, A = S.A;
  const int W = 512;  // profile row stride: 32 lanes * 16 columns
  int8_t* profA = prof;
  int8_t* profB = XM ? prof : prof + A * W;

  // cross mode: this item's layout (which template each lane works on) and its group of query couples
  int x_tl = -1, x_qc0 = 0, nrep = 1;
  if (XM) {
    const int layout = task % P.x_nlayouts, qg = task / P.x_nlayouts;
    x_tl = P.x_layout[layout * 32 + lane];
    x_qc0 = qg * P.x_group;
    nrep = min(P.x_group, P.x_nqc - x_qc0);
  }
  for (int rep = 0; rep < nrep; ++rep) {
  // ---- who am I: pair ids of both halves (cross mode: the template list index), segment geometry
  int x_ql[2] = {0, 0};
  if (XM) { x_ql[0] = P.x_qc[(x_qc0 + rep) * 2]; x_ql[1] = P.x_qc[(x_qc0 + rep) * 2 + 1]; }
  const int pid[2] = {XM ? x_tl : P.tasks[task * 64 + lane], XM ? x_tl : P.tasks[task * 64 + 32 + lane]};
  const int prev_pid = __shfl_up_sync(0xffffffffu, pid[0], 1);
  const bool seg_start = (lane == 0) || (prev_pid != pid[0]);
  const unsigned starts = __ballot_sync(0xffffffffu, seg_start);
  const int seg_lane0 = 31 - __clz(starts & (0xffffffffu >> (31 - lane)));
  const int off = lane - seg_lane0;

  int Lq[2] = {0, 0}, Lt[2] = {0, 0}, sig[2] = {0, 0};
  const uint8_t* qp[2] = {P.arena, P.arena};
  const uint8_t* tp[2] = {P.arena, P.arena};
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (pid[h] >= 0) {
      const int qs = XM ? P.x_qid[x_ql[h]] : P.pair_q[pid[h]], ts = XM ? P.x_tid[pid[h]] : P.pair_t[pid[h]];
      Lq[h] = (int)(P.seq_off[qs + 1] - P.seq_off[qs]);
      Lt[h] = (int)(P.seq_off[ts + 1] - P.seq_off[ts]);
      qp[h] = P.arena + P.aoff[qs];
      tp[h] = P.arena + P.aoff[ts];
      const int n = (Lt[h] + 15) >> 4;
      sig[h] = P.rev ? 0 : 16 * n - Lt[h];  // forward pass is right-aligned
    }
  }
  const int nl = (Lt[0] + 15) >> 4;  // lanes of this segment (both halves have the same n)
  const int Lqmax = max(Lq[0], Lq[1]);
  int nsteps = (pid[0] >= 0 || pid[1] >= 0) ? Lqmax + nl - 1 : 0;
  nsteps = __reduce_max_sync(0xffffffffu, nsteps);

  // ---- template profiles: prof[a*512 + lane*16 + c] = sub8[a][t_(column of register c)], pads = -128
  // (cross mode: one profile for both halves, built once per item and reused by every query couple)
  if constexpr (PRO) {
    if (!XM || rep == 0) {
      // lane `off` of a segment owns bytes 16*off .. 16*off+15 of every profile row of the flow: one aligned 16-byte load
      // per row; the -128 pad columns are already in place.  A half without a pair gets pad columns only.
      __syncwarp();
#pragma unroll
      for (int h = 0; h < (XM ? 1 : 2); ++h) {
        const int ts = pid[h] < 0 ? -1 : (XM ? P.x_tid[pid[h]] : P.pair_t[pid[h]]);
        const int nb = prof_row_bytes(Lt[h]);
        const int8_t* src = ts < 0 ? nullptr : prof_flow(P.prof, ts, Lt[h], A, P.rev) + off * 16;
        int8_t* dst = (h ? profB : profA) + lane * 16;
        for (int a = 0; a < A; ++a)
          *reinterpret_cast<uint4*>(dst + a * W) = ts < 0 ? make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u)
                                                          : *reinterpret_cast<const uint4*>(src + a * nb);
      }
      __syncwarp();
    }
  } else if (!XM || rep == 0) {
    // padded substitution table (A rows of A+1 entries, entry A = pad = -128) into the staging area: no cp.async
    // of this task has been issued yet and the previous task drained its own
    int8_t* s_sub = reinterpret_cast<int8_t*>(stage);
    __syncwarp();
    for (int x = lane; x < packed_sub_bytes(A) / 16; x += 32)
      reinterpret_cast<uint4*>(s_sub)[x] = reinterpret_cast<const uint4*>(P.sub8p)[x];
    uint32_t tc[2][4];
#pragma unroll
    for (int h = 0; h < (XM ? 1 : 2); ++h)
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        uint32_t x = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int j = off * 16 + w * 4 + b + 1 - sig[h];
          uint32_t code = (uint32_t)A;  // pad column -> extra table column holding -128
          if (pid[h] >= 0 && j >= 1 && j <= Lt[h]) code = tp[h][j - 1];
          x |= code << (8 * b);
        }
        tc[h][w] = x;
      }
    __syncwarp();
    for (int a = 0; a < A; ++a) {
      const int8_t* row = s_sub + a * (A + 1);
#pragma unroll
      for (int h = 0; h < (XM ? 1 : 2); ++h) {
        uint4 o;
        uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const uint32_t x = tc[h][w];
          uint32_t v = 0;
#pragma unroll
          for (int b = 0; b < 4; ++b) v |= (uint32_t)(uint8_t)row[(x >> (8 * b)) & 0xff] << (8 * b);
          ow[w] = v;
        }
        *reinterpret_cast<uint4*>((h ? profB : profA) + a * W + lane * 16) = o;
      }
    }
    __syncwarp();
  }

  // ---- state for virtual row 0 (packed: A low, B high).  Fn[c] is the F of the row ABOUT to be processed: it is
  // updated as soon as M of the current row is known (F(i+1,c) = max(F(i,c) - ge, M(i,c) - gi)), so no copy of
  // M - gi has to live across a row; its open/extend decision bit belongs to the next row's traceback word and is
  // carried there in fprev[].
  uint32_t Xp[16], Fn[16], nge[16];
  uint32_t xl_hold;
  uint32_t fprev[2] = {0u, 0u};  // fopen plane of the next row: byte 1 = pair A, byte 3 = pair B (8 columns per word)
  {
    int xh[2];
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      int x[2], f[2], m[2], g[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = off * 16 + c + 1 - sig[h];
        if (j < 0) { x[h] = kFloor16; f[h] = kNeg16; m[h] = kNeg16; g[h] = -ge; }
        else if (j == 0) {  // the boundary column lives in a pad register: X(i,0) comes from its F chain
          x[h] = 0;
          f[h] = S.insfree ? 0 : kNeg16;
          m[h] = S.insfree ? kNeg16 : -gi;
          g[h] = S.insfree ? 0 : -ge;
        } else {
          x[h] = -(S.delfree ? 0 : gap_w(gi, ge, j));  // X(0,j): dpmatrix.h:412-418
          f[h] = kNeg16;
          m[h] = kNeg16;
          g[h] = (S.insfree && j == Lt[h]) ? 0 : -ge;  // zero-penalty F chain in the last column
        }
        // F of row 1 and its decision bit ("the open candidate wins strictly")
        if (TBM && f[h] + g[h] < m[h]) fprev[c >> 3] |= 1u << (8 * (2 * h + 1) + 7 - (c & 7));
        f[h] = max(f[h] + g[h], m[h]);
      }
      Xp[c] = pkb(x[0], x[1]);
      Fn[c] = pkb(f[0], f[1]);
      nge[c] = pkdec(-g[0], -g[1]);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int jl = off * 16 - sig[h];  // column left of register 0
      xh[h] = jl < 0 ? kFloor16 : (jl == 0 ? 0 : -(S.delfree ? 0 : gap_w(gi, ge, jl)));
    }
    xl_hold = pkb(xh[0], xh[1]);
  }
  // injection at the segment's first lane: X(i,0) when register 0 is column 1, "-inf" when it is a pad.
  // xn = (shuffled & inj_keep) | (binj & inj_b_mask) | inj_floor;  binj = X(s+1,0) of the segment's first lane,
  // advanced by one gap extension per step (dpmatrix.h:420-426)
  const uint32_t inj_b_mask = (seg_start ? ((sig[0] == 0 ? 0x0000ffffu : 0u) | (sig[1] == 0 ? 0xffff0000u : 0u)) : 0u);
  const uint32_t inj_keep = seg_start ? 0u : 0xffffffffu;
  const uint32_t NEG2 = pkb(kNeg16, kNeg16);
  const uint32_t FLOOR2 = pkb(kFloor16, kFloor16);
  const uint32_t inj_floor = seg_start ? (FLOOR2 & ~inj_b_mask) : 0u;
  const uint32_t inj_neg = seg_start ? NEG2 : 0u;
  const uint32_t NGE2 = pkdec(ge, ge);
  const uint32_t ZERO2 = pkb(0, 0);
  const uint32_t NGI2 = pkdec(gi, gi);
  uint32_t binj = S.insfree ? pkb(0, 0) : pkb(-gi, -gi);
  const uint32_t binj_step = S.insfree ? 0u : NGE2;
  // ---- per-half output bases (diagonal-major: the address of a step is base + step * stride)
  uint8_t* tbp[2] = {nullptr, nullptr};
  int16_t* scp[2] = {nullptr, nullptr};
  const int16_t* fp[2] = {nullptr, nullptr};
  uint8_t* mkp[2] = {nullptr, nullptr};
  uint32_t THR2 = 0, THR1 = 0;
  const uint32_t NBIAS1 = pkdec(kBias16, kBias16);
  float thr_f[2] = {0.f, 0.f};
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (pid[h] < 0) continue;
    if (TBM) tbp[h] = P.tb + P.tb_off[pid[h]] + off * 8;                 // + step * nl*8
    if (FST) scp[h] = P.sc_out + P.sc_off[pid[h]] + off * 8;             // + step * nl*16 (+ nl*8 for the upper half)
    if (MSK) {
      // forward chunk (nl-1-off) of forward row Lq+1-a sits in forward skew row Lq+nl-2-step: the same
      // skew row for every lane of the segment
      fp[h] = P.scF + P.sc_off[pid[h]] + (int64_t)(Lq[h] + nl - 2) * nl * 16 + (nl - 1 - off) * 8;  // - step * nl*16
      mkp[h] = reinterpret_cast<uint8_t*>(P.mask + P.mask_off[pid[h]]) + off * 2;  // + step * nl*2
      const float inv = 1.f / (float)(1 << S.scale_log2);
      const float opt = (float)P.fin_fwd[pid[h]] * inv;
      thr_f[h] = nearopt_threshold(opt, P.delta_ratio);
    }
  }
  if (MSK) {
    int ti[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float t = floorf(thr_f[h] * (float)(1 << S.scale_log2));  // slack (integer) > thr  <=>  slack > floor(thr)
      ti[h] = (int)fminf(fmaxf(t, (float)kFloor16), (float)kPackedBound);
    }
    THR2 = pk2(ti[0] + 2 * kBias16, ti[1] + 2 * kBias16);  // compared with the doubly biased sum F + X
    THR1 = pkb(ti[0], ti[1]);
  }

  // ---- query residues: each lane stages its own rows in a private 16-byte ring per half
  // (two 8-row blocks), refilled with cp.async one block (8 rows) ahead of use.
  constexpr bool SA = (TBM == 0);
  const SPtr stage_s = sptr<SA>(stage), profA_s = sptr<SA>(profA) + lane * 16, profB_s = XM ? profA_s : sptr<SA>(profB) + lane * 16;
  // Per-lane staging: a 16-byte query ring per half and (MSK) a private triple buffer of forward-score chunks
  // (3 x 32 bytes per half), requested two rows ahead.  These strides make the ring byte loads 8-way and the chunk
  // loads / cp.async writes 4-way bank conflicted (ncu: L1/shared data pipe of the reverse+mask kernel at 72 %), but the
  // conflict-free layouts ([buffer][quarter][lane] chunks, word-interleaved rings) were MEASURED SLOWER on every
  // workload (profiles/r02_packed_variants.md #14: C3 -1.3 %, C2 -9 %, C4 -11 % against this layout): their extra address
  // arithmetic per step costs more than the wavefronts they save.
  const SPtr qst[2] = {stage_s + lane * 32, stage_s + (lane * 32 + 16)};
  const SPtr fst[2] = {stage_s + (1024 + lane * 192), stage_s + (1024 + lane * 192 + 96)};
  constexpr int kFBuf = 32;  // bytes per chunk buffer of a lane and half
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    cpa8<SA>(qst[h], qp[h], 1);
    cpa8<SA>(qst[h] + 8, qp[h] + 8, 1);
  }

  uint32_t x_pub = FLOOR2, e_pub = NEG2, mg_pub = NEG2;
  if (MSK) {
    // rows 1 and 2 of this lane (steps off and off+1) -> buffers 1 and 2
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
      for (int r = 1; r <= 2; ++r) {
        const int ok = pid[h] >= 0 && Lq[h] >= r;
        const int16_t* src = fp[h] - (int64_t)(off + r - 1) * nl * 16;
        cpa16<SA>(fst[h] + kFBuf * (r % 3), src, ok);
        cpa16<SA>(fst[h] + (kFBuf * (r % 3) + 16), src + nl * 8, ok);
      }
    }
  }
  cp_async_commit();
  // Row 1 of every lane: its residues and profile words are read here, before the loop, instead of behind an i == 1
  // test in every step.  Waiting for the first group costs nothing extra: lane 0 of the warp waits for it in step 0.
  cp_async_wait_all();
  int qa_n0 = ld1<SA>(qst[0]), qa_n1 = ld1<SA>(qst[1]);  // query residues of the NEXT row (read one row ahead)
  uint4 pnA = make_uint4(0, 0, 0, 0), pnB = make_uint4(0, 0, 0, 0);  // profile words of the next row
#if AADP_PROF_AHEAD
  pnA = ld16<SA>(profA_s + qa_n0 * W);
  pnB = ld16<SA>(profB_s + qa_n1 * W);
#endif
  // valid (non-pad) registers in the layout of accM: A bytes 0/1 (even/odd c), B bytes 2/3
  uint32_t VM = 0;
  if (MSK) {
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const int j = off * 16 + c + 1 - sig[h];
        if (pid[h] >= 0 && j >= 1 && j <= Lt[h]) VM |= 1u << (8 * (2 * h + (c & 1)) + 7 - (c >> 1));
      }
  }
  // triple-buffer offsets of the forward-score chunks: row i lives in buffer i % 3, row i+2 in buffer (i+2) % 3 =
  // (i-1) % 3; rotated once per row instead of dividing by 3 (a lane's active rows are consecutive, from 1)
  int fcur_off = kFBuf, fnxt_off = 0;
  uint32_t cnt[2] = {0u, 0u};  // near-optimal cells of this lane: at most 16 * Lq
  RowSum fin[2] = {{kNeg32, 0, kNeg32, kNeg32}, {kNeg32, 0, kNeg32, kNeg32}};

  // What the final cell needs from this lane's 16 columns (RowSum) is M(Lq,.) and F(Lq,Lt).  The loop-carried state
  // holds exactly the inputs of that row -- X(Lq-1,.) and F(Lq,.) -- at the END of the step of row Lq-1 (before the
  // loop when Lq = 1), and the two halves of a couple get there at different steps.  A rare branch at that point
  // only parks the raw registers in local memory (volatile: the compiler otherwise promotes the arrays to 66 more
  // registers); the summary itself is computed after the loop.  Computing it inside the loop cost ~50 registers.
  // RB: the lane has stored M(Lq, .) of its 16 columns itself (skew row Lq - 1 + off of the score blob, LOC clamp
  // included), and F(Lq, Lt) is always register 15 of the segment's last lane in the right-aligned forward pass: one
  // branch-free select per step keeps it (fcol), and nothing is parked.
  volatile uint32_t capX[2][17], capF[2][16];
  int capQ[2] = {0, 0};
  uint32_t fcol = 0;
  auto capture = [&](int h, int qa) {
#pragma unroll
    for (int c = 0; c < 16; ++c) { capX[h][c + 1] = Xp[c]; capF[h][c] = Fn[c]; }
    capX[h][0] = xl_hold;
    capQ[h] = qa;
  };
  if (!RB)
    for (int h = 0; h < 2; ++h)
      if (pid[h] >= 0 && Lq[h] == 1) capture(h, (int)qp[h][0]);

  for (int s = 0; s < nsteps; ++s) {
    uint32_t xn = __shfl_up_sync(0xffffffffu, x_pub, 1);
    uint32_t e_in = __shfl_up_sync(0xffffffffu, e_pub, 1);
    uint32_t mg_in = __shfl_up_sync(0xffffffffu, mg_pub, 1);
    const int r0 = s - off;  // row - 1 of this lane
    const int i = r0 + 1;
    xn = (xn & inj_keep) | ((binj & inj_b_mask) | inj_floor);
    e_in = (e_in & inj_keep) | inj_neg;
    mg_in = (mg_in & inj_keep) | inj_neg;
    binj = addc(binj, binj_step);
    const bool act0 = (unsigned)r0 < (unsigned)Lq[0];  // Lq is 0 for an empty half
    const bool act1 = (unsigned)r0 < (unsigned)Lq[1];
    if (act0 || act1) {
      // One cp.async group is committed per row.  Query blocks are requested 8 rows ahead and forward
      // scores 2 rows ahead, so only the most recent group(s) may still be in flight.
      if (MSK) cp_async_wait_group<1>();
      else cp_async_wait_group<4>();
#if AADP_PROF_AHEAD
      // The profile words of THIS row were loaded during the previous step (the first row: before the loop): the
      // step starts with register operands only.  The residue of the next row comes out of the ring now and its
      // profile row follows as soon as the residue is there -- both loads have a whole step to complete.
      const uint32_t pwA[4] = {pnA.x, pnA.y, pnA.z, pnA.w};
      const uint32_t pwB[4] = {pnB.x, pnB.y, pnB.z, pnB.w};
      qa_n0 = ld1<SA>(qst[0] + (i & 15));
      qa_n1 = ld1<SA>(qst[1] + (i & 15));
      pnA = ld16<SA>(profA_s + qa_n0 * W);
      pnB = ld16<SA>(profB_s + qa_n1 * W);
#else
      const int qa0 = qa_n0, qa1 = qa_n1;
      const uint4 pa = ld16<SA>(profA_s + qa0 * W);
      const uint4 pb = ld16<SA>(profB_s + qa1 * W);
      qa_n0 = ld1<SA>(qst[0] + (i & 15));
      qa_n1 = ld1<SA>(qst[1] + (i & 15));
      const uint32_t pwA[4] = {pa.x, pa.y, pa.z, pa.w};
      const uint32_t pwB[4] = {pb.x, pb.y, pb.z, pb.w};
#endif
      uint32_t fcur[2][8];
      if (MSK) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint4 a = ld16<SA>(fst[h] + fcur_off), b = ld16<SA>(fst[h] + (fcur_off + 16));
          fcur[h][0] = a.x; fcur[h][1] = a.y; fcur[h][2] = a.z; fcur[h][3] = a.w;
          fcur[h][4] = b.x; fcur[h][5] = b.y; fcur[h][6] = b.z; fcur[h][7] = b.w;
        }
      }
      {
        // stage ahead: the next 8-row query block (once per 8 rows) and the forward scores of row i+2
        const int blk = (r0 >> 3) + 2;  // blocks 0 and 1 were requested up front
        const int newblk = ((r0 & 7) == 0) && r0 > 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          cpa8<SA>(qst[h] + 8 * ((blk - 1) & 1), qp[h] + 8 * (blk - 1), newblk);
          if (MSK) {
            const int more = pid[h] >= 0 && (i + 2) <= Lq[h];
            const int16_t* src = fp[h] - (size_t)((uint32_t)(s + 2) * (uint32_t)nl * 16u);
            cpa16<SA>(fst[h] + fnxt_off, src, more);
            cpa16<SA>(fst[h] + (fnxt_off + 16), src + nl * 8, more);
            // two rows (~700 cycles) do not cover a DRAM round trip under load: pull the chunk of row
            // i+kFwdAhead into L2 now, so that the cp.async issued for it later is an L2 hit
            const int far = pid[h] >= 0 && (i + kFwdAhead) <= Lq[h];
            const int16_t* psrc = fp[h] - (size_t)((uint32_t)(s + kFwdAhead) * (uint32_t)nl * 16u);
            prefetch_l2(psrc, far);
            prefetch_l2(psrc + nl * 8, far);
          }
        }
        cp_async_commit();
      }

      uint32_t E = e_in, Mgl = mg_in;
      uint32_t accM = 0, acc01 = 0, acc23 = 0;
      uint32_t tbA[2], tbB[2], oA[8], oB[8];
      // ---- phase 1: every M of the row (independent adds), and the near-optimal test of the reverse pass.
      // Doing this first frees the previous row's X registers, so phase 2 updates the state in place.
      uint32_t Mv[16];
      {
        uint32_t Xd = xl_hold, d5prev = 0;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const int k = c & 3;
          const uint32_t ssel = (uint32_t)k | ((uint32_t)(k | 8) << 4) | ((uint32_t)(4 + k) << 8) | ((uint32_t)((4 + k) | 8) << 12);
          const uint32_t simp = prmt(pwA[c >> 2], pwB[c >> 2], ssel);
          // plain packed add (VIADD.16x2, off the ALU pipe): no clamp is needed -- real cells stay far above the
          // floor and pad columns only drift down by ge per row (bounded by the host-side score bound)
          Mv[c] = LOC ? __vmaxs2(__vadd2(simp, Xd), ZERO2) : __vadd2(simp, Xd);
          if (MSK) {
            // slack = F(i,j) + R(i,j) - sim(i,j) = F(i,j) + X_rev(i+1,j+1) (<= optimum, so it stays in range);
            // element 15-c of the forward chunk.
            const int e = 15 - c;
            const uint32_t fv = prmt(fcur[0][e >> 1], fcur[1][e >> 1], (e & 1) ? 0x7632u : 0x5410u);
            // both halves are positive 16-bit numbers whose sum stays below 65536: a plain 32-bit add (IMAD, FMA
            // pipe) without a carry between the halves.  The sum carries the bias TWICE and is a negative fp16
            // pattern, like THR2: among negative patterns the larger integer is the smaller fp16 number, so the
            // sign of (slack - thr) as fp16 numbers is set exactly where slack > thr as integers.
#if AADP_SLACK_IMAD
            const uint32_t slack = addc(fv, Xd);
            const uint32_t d5 = lt_sign(slack, THR2);
#else
            const uint32_t slack = fv + Xd + NBIAS1;  // one bias removed on the ALU pipe (IADD3), singly biased compare
            const uint32_t d5 = lt_sign(THR1, slack);
#endif
            // gather the sign bits of two cells at once: bytes [A(c-1), A(c), B(c-1), B(c)] = 0xFF / 0x00
            if (c & 1) accM = gat(accM, prmt(d5prev, d5, 0xFBD9u), 7 - (c >> 1));
            else d5prev = d5;
          }
          Xd = Xp[c];
        }
      }
      // ---- phase 2: E chain, X, next row's F, traceback bits
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const uint32_t M = Mv[c];
        const uint32_t F = Fn[c];
        uint32_t X;
        if (TBM) {
          const uint32_t Eext = addc(E, NGE2);
          const uint32_t dE = lt_sign(Eext, Mgl);   // the open candidate wins strictly
          E = __vmaxs2(Eext, Mgl);
          const uint32_t dS1 = lt_sign(M, E);       // E > M
          const uint32_t t = __vmaxs2(M, E);
          const uint32_t dS2 = lt_sign(t, F);       // F > max(M,E)
          X = __vmaxs2(t, F);
          Mgl = addc(M, NGI2);
          const uint32_t Fext = addc(F, nge[c]);
          const uint32_t dF = lt_sign(Fext, Mgl);   // decision of the NEXT row's F
          Fn[c] = __vmaxs2(Fext, Mgl);
          // PRMT with sign replication turns four sign bits into four 0xFF/0x00 bytes [A.x, A.y, B.x, B.y]
          acc01 = gat(acc01, prmt(dS1, dS2, 0xFBD9u), 7 - (c & 7));
          acc23 = gat(acc23, prmt(dE, dF, 0xFBD9u), 7 - (c & 7));
          if ((c & 7) == 7) {
            const uint32_t b01 = gat_fin(acc01), b23 = gat_fin(acc23);
            // eopen of this row, fopen computed one row earlier
            const uint32_t m23 = (b23 & 0x00ff00ffu) | (fprev[c >> 3] & 0xff00ff00u);
            fprev[c >> 3] = b23;
            tbA[c >> 3] = prmt(b01, m23, 0x5410u);  // planes selE, selF, eopen, fopen of pair A
            tbB[c >> 3] = prmt(b01, m23, 0x7632u);
            acc01 = 0;
            acc23 = 0;
          }
        } else {
          E = __viaddmax_s16x2(E, pk2(-ge, -ge), Mgl);
          X = __vimax3_s16x2(M, E, F);
          Mgl = addc(M, NGI2);
          Fn[c] = __vmaxs2(addc(F, nge[c]), Mgl);
        }
        Xp[c] = X;
        if (FST && (c & 1)) {
          oA[c >> 1] = prmt(Mv[c - 1], M, 0x5410u);
          oB[c >> 1] = prmt(Mv[c - 1], M, 0x7632u);
        }
      }
      if (MSK) {
        accM = gat_fin(accM) & VM;
        fnxt_off = fcur_off;
        fcur_off = fcur_off == 2 * kFBuf ? 0 : fcur_off + kFBuf;
      }
      xl_hold = xn;
      x_pub = Xp[15];
      e_pub = E;
      mg_pub = Mgl;
      // byte offsets of this step inside a pair's products fit 32 bits (Lt <= 512, bounded Lq): one 32-bit
      // multiply shared by both halves, then base + offset per store
      const uint32_t snl = (uint32_t)s * (uint32_t)nl;
      // every word and address of the step first, then the stores of both halves, predicated in one place
      uint8_t* const tba = tbp[0] + (size_t)(snl * 8u);
      uint8_t* const tbb = tbp[1] + (size_t)(snl * 8u);
      uint8_t* const sca = reinterpret_cast<uint8_t*>(scp[0]) + (size_t)(snl * 32u);
      uint8_t* const scb = reinterpret_cast<uint8_t*>(scp[1]) + (size_t)(snl * 32u);
      const size_t sch = (size_t)((uint32_t)nl * 16u);
      uint8_t* const mka = mkp[0] + (size_t)(snl * 2u);
      uint8_t* const mkb = mkp[1] + (size_t)(snl * 2u);
      if (TBM) {
        stg8_if(tba, tbA[0], tbA[1], act0);
        stg8_if(tbb, tbB[0], tbB[1], act1);
      }
      if (FST) {
        stg16_if(sca, oA[0], oA[1], oA[2], oA[3], act0);
        stg16_if(sca + sch, oA[4], oA[5], oA[6], oA[7], act0);
        stg16_if(scb, oB[0], oB[1], oB[2], oB[3], act1);
        stg16_if(scb + sch, oB[4], oB[5], oB[6], oB[7], act1);
      }
      if (MSK) {
        stg2_if(mka, accM, act0);
        stg2_if(mkb, accM >> 16, act1);
        cnt[0] += act0 ? __popc(accM & 0xffffu) : 0;
        cnt[1] += act1 ? __popc(accM >> 16) : 0;
      }
      if constexpr (RB) {
        const uint32_t sel = (i + 1 == Lq[0] ? 0x0000ffffu : 0u) | (i + 1 == Lq[1] ? 0xffff0000u : 0u);
        fcol = (Fn[15] & sel) | (fcol & ~sel);
      } else {
#ifndef AADP_EXP_NOCAP  // (timing experiment only: without the capture the final scores are wrong)
        if (i + 1 == Lq[0] || i + 1 == Lq[1]) {
          for (int h = 0; h < 2; ++h)
            if (i + 1 == Lq[h]) capture(h, h ? qa_n1 : qa_n0);
        }
#endif
      }
    }
  }

  // ---- final-row summaries: M(Lq,j) = sim(Lq,j) + X(Lq-1,j-1) from the parked state, or read back (RB)
  for (int h = 0; h < 2; ++h) {
    if (pid[h] < 0) continue;
    const int8_t* prow = (h ? profB : profA) + capQ[h] * W + lane * 16;
    uint32_t mrow[8];  // RB: the stored words of this half, biased M of columns 2w (low) and 2w+1 (high)
    if (RB) {
      const int16_t* row = scp[h] + (size_t)(Lq[h] - 1 + off) * (size_t)(nl * 16);
      const uint4 a = *reinterpret_cast<const uint4*>(row), b = *reinterpret_cast<const uint4*>(row + nl * 8);
      mrow[0] = a.x; mrow[1] = a.y; mrow[2] = a.z; mrow[3] = a.w;
      mrow[4] = b.x; mrow[5] = b.y; mrow[6] = b.z; mrow[7] = b.w;
    }
    RowSum r = {kNeg32, 0, kNeg32, kNeg32};
    for (int c = 0; c < 16; ++c) {
      const int j = off * 16 + c + 1 - sig[h];
      int m = RB ? unb16(mrow[c >> 1], c & 1) : unb16(capX[h][c], h) + (int)prow[c];  // M(Lq, j)
      if (LOC) m = max(m, 0);
      if (j >= 1 && j < Lt[h]) {
        const int v = m - (S.delfree ? 0 : gap_w(gi, ge, Lt[h] - j));
        if (v > r.rb_val) { r.rb_val = v; r.rb_k = j; }
      } else if (j == Lt[h]) {
        r.diag = m;
        r.col = (Lq[h] >= 2) ? unb16(RB ? fcol : capF[h][c], h) + (S.insfree ? gi : 0) : kNeg32;
      }
    }
    fin[h] = r;
  }
  // ---- final cells (dpmatrix.h:504-534 / 844-874): match, bottom row (k ascending), right column
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const RowSum r = fin[h];
    __syncwarp();
    red[lane] = make_int4(r.rb_val, r.rb_k, r.diag, r.col);
    __syncwarp();
    if (seg_start && pid[h] >= 0) {
      int rb = kNeg32, rk = 0, dg = kNeg32, cl = kNeg32;
      for (int l = 0; l < nl; ++l) {
        const int4 v = red[lane + l];
        if (v.x > rb) { rb = v.x; rk = v.y; }  // lanes ascend in column order: '>' keeps the smallest k
        dg = max(dg, v.z);
        cl = max(cl, v.w);
      }
      int best = dg, kind = 0, k = Lt[h];
      if (LOC) best = max(best, 0);
      if (Lt[h] >= 2 && rb > best) { best = rb; kind = 1; k = rk; }
      if (cl > best) { best = cl; kind = 2; k = -1; }
      if (XM) {
        P.x_scores[(long long)x_ql[h] * P.x_nt + pid[h]] = (float)best * (1.f / (float)(1 << S.scale_log2));
      } else {
        P.fin_score[pid[h]] = best;
        P.fin_kind[pid[h]] = kind;
        P.fin_k[pid[h]] = k;
      }
      if (MSK && P.threshold) P.threshold[pid[h]] = thr_f[h];
    }
    if (MSK && P.count) {
      __syncwarp();
      reinterpret_cast<long long*>(red)[lane] = (long long)cnt[h];
      __syncwarp();
      if (seg_start && pid[h] >= 0) {
        long long t = 0;
        for (int l = 0; l < nl; ++l) t += reinterpret_cast<long long*>(red)[lane + l];
        P.count[pid[h]] = t;
      }
    }
  }
  cp_async_wait_all();  // the staging area is recycled by the next couple / task
  __syncwarp();
  }  // rep
}

template <int TBM, int FST, int MSK, int XM, int LOC = 0, int PRO = 0, int RB = 0>
__global__ void __launch_bounds__(kPackedWarps * 32) __maxnreg__(XM ? 168 : (MSK ? 255 : (TBM ? 224 : 200))) packed_kernel(const PackedParams P) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int A = P.sc.A;
  const int warp = threadIdx.x >> 5;
  int lane;
  // read once and pinned in a register: the compiler otherwise re-reads SR_TID.X (S2R, ~25 cycles) in every
  // step of the row loop to rebuild the per-lane shared-memory addresses
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
  const int kStage = packed_stage_bytes(A, MSK);
  const int per_warp = (XM ? 512 : 0) + kStage + (XM ? 1 : 2) * A * 512;
  unsigned char* mine = smem + warp * per_warp;
  uint8_t* stage = mine + (XM ? 512 : 0);
  int8_t* prof = reinterpret_cast<int8_t*>(stage + kStage);
  int4* red = XM ? reinterpret_cast<int4*>(mine) : reinterpret_cast<int4*>(prof);
  for (;;) {
    unsigned int item = 0;
    if (lane == 0) item = atomicAdd(P.counter, 1u);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= (unsigned int)P.n_tasks) break;
    packed_task<TBM, FST, MSK, XM, LOC, PRO, RB>(P, (int)item, prof, red, stage, lane);
  }
}

}  // namespace aadp
