// aadp_api.cu -- C ABI (include/aadp.h) + host orchestration of the sm_100a fill kernels.
// The product path: there is no CPU fallback anywhere in this file; every compute entry point
// fails with an error message when no CUDA device / kernel image is available.
#include "../../include/aadp.h"
#include "aadp_kernels.cuh"
#include "aadp_packed.cuh"
#include "aadp_general.cuh"
#include "aadp_frec.cuh"
#include "aadp_enum.cuh"
#include "aadp_pruned.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <numeric>
#include <string>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

using namespace aadp;

namespace {

thread_local std::string g_err;


int fail(const std::string& m) {
  g_err = m;
  return 1;
}

#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      g_err = std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #call;        \
      return 1;                                                                           \
    }                                                                                     \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      e = cudaMalloc(&p, bytes);
      want = bytes;
    }
    if (e != cudaSuccess) {
      g_err = std::string("cudaMalloc failed for ") + std::to_string(bytes) + " bytes: " + cudaGetErrorString(e);
      p = nullptr;
      return 1;
    }
    cap = want;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct Batch {
  int64_t nseq = 0, npairs = 0;
  bool have_seqs = false;
  std::vector<int64_t> seq_off;
  std::vector<int32_t> pair_q, pair_t;
  std::vector<int64_t> tb_off, sc_off, mask_off;  // per pair, +1 total at the end
  std::vector<int32_t> order[2];                  // bucket 0: K=8, bucket 1: K=16
  double bucket_cells[2] = {0, 0};
  int max_Lq = 0, max_Lt = 0;
  int st_mode = 1;  // 1 = int16 score storage possible, 2 = int32
  // packed (int16x2) path
  std::vector<uint8_t> fmt;       // per pair: 0 = int32 kernels, 1 = packed kernels, 2 = multi-CTA wavefront (long pair)
  std::vector<int32_t> wave_pairs;
  std::vector<int32_t> aoff;      // per sequence byte offset into the aligned arenas
  double packed_cells = 0;
  int64_t n_tasks = 0;
  // the packed task list may be built (and launched) in several chunks of consecutive pair ids, so that the
  // kernels of chunk k run while the host schedules chunk k+1 (aadp_fill_batch)
  std::vector<int64_t> chunk_first, chunk_ntasks;
  std::vector<double> chunk_cells;
  std::vector<int64_t> chunk_max_seq;  // largest sequence id a chunk references
  std::vector<int64_t> piece_end;      // residue pieces of a pipelined upload: first sequence id after piece j
  size_t piece_waited = 0;             // pieces the compute stream already waits for
  double cells = 0;
  uint32_t uploaded_what = 0;
  uint32_t ran_what = 0;
  // The schedule (pair classes, product offsets, task lists, score-storage mode) and the residue validation were
  // derived from the scoring in force at upload time.  sched_ok is cleared by aadp_set_scoring and by every entry
  // point that reuses the batch storage for its own items; aadp_run_batch refuses to run a stale schedule.
  bool sched_ok = false;
  int seq_A = 0;  // alphabet size the resident residues were validated against
};

struct HostPool {
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv, done;
  std::function<void(int)>* fn = nullptr;
  uint64_t gen = 0;
  int active = 0, pending = 0;
  bool stop = false;
  void start(int n);
  void run(int T, std::function<void(int)> f);
  ~HostPool();
};

// per-host-thread scratch of the scheduler, kept between batches (fresh allocations page-fault, and page
// faults of concurrent threads serialise on the process' address-space lock)
struct SchedItem { int32_t p; int n; int Lq; };
struct SchedCouple { int32_t a, b; int n; int Lq; };
struct SchedScratch {
  std::vector<SchedItem> items, items2;
  std::vector<SchedCouple> couples, couples2;
  std::vector<int32_t> cnt, tasks, order[2], wave;
};

}  // namespace

struct aadp_ctx {
  int device = 0;
  int num_sms = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  bool have_scoring = false;
  Scoring sc{};
  int align_type = AADP_GLOBAL;
  uint32_t flags = 0;
  std::vector<int8_t> sub8_h;
  std::vector<float> subf_h;  // the substitution table as given (host copy: similarity matrix of the pruned enumerators)
  int max_abs_sub = 0;
  DevBuf sub8p;
  // position-specific template profiles (aadp_set_profile_scoring): replace sub8 / sub8p / subf while prof_mode is set
  bool prof_mode = false;
  int64_t prof_nseq = 0;              // profiles given (one per sequence id)
  std::vector<int64_t> prof_len;      // per sequence: entries (L*A), 0 = no profile
  std::vector<int> prof_max;          // per sequence: max |entry| in grid units (the per-template score bound)
  std::vector<float> proff_h;         // the profiles as given (host copy: similarity matrix of the pruned enumerators)
  std::vector<int64_t> proff_off_h;
  DevBuf prof8, prof8_off, proff, proff_off;
  ProfDev prof_dev() const { return ProfDev{prof8.as<int8_t>(), prof8_off.as<int64_t>(), proff.as<float>(), proff_off.as<int64_t>()}; }
  DevBuf sub8, residues, seq_off, pair_q, pair_t, order[2], tb_off, sc_off, mask_off;
  DevBuf tb[2], scb[2], mask, fin_score[2], fin_kind[2], fin_k[2], counter, bbuf, thr, count, fscore[2];
  DevBuf scratch_a, scratch_b, scratch_c, scratch_d;
  DevBuf fmt, tasks, aoff, arena_f, arena_r, badflag;
  bool allow_packed = true;
  bool allow_wave = true;
  int host_threads = 0;  // 0 = min(hardware threads, 8)
  int pipeline_chunks = 2;  // aadp_fill_batch: task-list chunks whose scheduling overlaps the previous chunk's kernel
  HostPool pool;
  std::vector<SchedScratch> sched;
  std::vector<int32_t> Lq32, Lt32;
  int64_t wave_min_cells = 4000000;  // pairs at least this large use the multi-CTA wavefront
  DevBuf wave_bb, wave_ready, wave_part, wave_dbg;
  unsigned int wave_tag = 0;
  DevBuf x_layout, x_qc, x_qid, x_tid, x_scores;
  // exact general-gap fp32 path (aadp_general.cuh): scoring that is not on a dyadic grid, or forced
  bool float_mode = false, force_float = false;
  float gi_f = 0.f, ge_f = 0.f;
  float last_delta = -1.f;
  int64_t gg_budget_cells = 1000000000;  // dense cells per direction and chunk of a batch (8-16 B per cell and direction)
  DevBuf ali_cap, ali_out, ali_n, ali_status, gg_rect;
  DevBuf ucw_ids, ucw_path_off, ucw_stack_off, ucw_stack, ucw_paths, ucw_len, ucw_scores, ucw_n, ucw_status, ucw_thr, ucw_plen, ucw_pathbuf, ucw_flags, ucw_flag_off;
  DevBuf subf, gg_score[2], gg_pq[2], gg_pt[2], gg_mask, gg_off, gg_fin[2], gg_pm[2], gg_items, tb_del, tb_ins, tb_del_off, tb_ins_off;
  int gg_threads_cap = 256;  // CTA size limit of the exact general-gap kernel (option "general_threads"): 512 -> 256 measured +12 %
  int ucw_user_limit = 100000, cw_user_limit = 1000000;  // ucw.h:72, cw.h:76
  int gg_prune = 1;  // pruned scans of the exact general-gap kernel (results identical either way)
  int enum_mask_prune = 1;  // enumeration kernel: prune the deletion scans with the resident near-optimal set
  int gg_records = 1;  // record-list kernel (aadp_frec.cuh) for affine gaps in exact-float mode (results identical either way)
  double x_cells = 0;  // cell updates of the last aadp_cross_run
  // pinned host staging for metadata uploads (bump-allocated per upload)
  uint8_t* pin = nullptr;
  size_t pin_cap = 0, pin_used = 0;
  int* pin_flag = nullptr;
  bool pending = false;        // aadp_fill_batch_submit without its aadp_fill_batch_wait
  bool flag_deferred = false;  // ... whose residue validation flag has not been looked at yet
  cudaEvent_t ev_flag = nullptr;  // recorded after the residue validation flag has been copied back
  cudaStream_t copy_stream = nullptr;  // pipelined uploads (aadp_fill_batch)
  cudaEvent_t ev_piece[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}, ev_start = nullptr;
  Batch b;
  int64_t launches = 0;
  int64_t h2d_bytes = 0, d2h_bytes = 0;  // of the last upload / fill call
  int bb_rows = 0;
  // optional per-launch timing
  bool profiling = false;
  struct Prof { std::string name; cudaEvent_t e0, e1; double cells; };
  std::vector<Prof> prof;       // launches of the last run
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  cudaEvent_t next_event() {
    if (ev_used == ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); ev_pool.push_back(e); }
    return ev_pool[ev_used++];
  }
  void prof_begin(const char* name, double cells) {
    if (!profiling) return;
    Prof p{name, next_event(), next_event(), cells};
    cudaEventRecord(p.e0, stream);
    prof.push_back(p);
  }
  void prof_end() {
    if (!profiling) return;
    cudaEventRecord(prof.back().e1, stream);
  }
};

// cudaFuncSetAttribute and the occupancy query are made ONCE per (device, kernel, size) and cached.  Measured on B200
// (AADP_TIMING marks, two contexts on two host threads): cudaFuncSetAttribute on a kernel that is RUNNING -- launched by
// another context of the process -- blocks the calling host thread until that kernel has finished, 10-13 ms per C3 step,
// which serialised the host scheduling of one context behind the GPU work of the other.
#include <map>
#include <tuple>
static std::mutex g_attr_mu;
static std::map<std::pair<int, const void*>, size_t> g_attr_smem;
static std::map<std::tuple<int, const void*, int, size_t>, int> g_attr_occ;
static cudaError_t cached_max_smem(const void* f, size_t smem) {
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(g_attr_mu);
  auto it = g_attr_smem.find({dev, f});
  if (it != g_attr_smem.end() && it->second >= smem) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) g_attr_smem[{dev, f}] = smem;
  return e;
}
static cudaError_t cached_occupancy(int* occ, const void* f, int threads, size_t smem) {
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(g_attr_mu);
  const auto key = std::make_tuple(dev, f, threads, smem);
  auto it = g_attr_occ.find(key);
  if (it != g_attr_occ.end()) { *occ = it->second; return cudaSuccess; }
  const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, f, threads, smem);
  if (e == cudaSuccess) g_attr_occ[key] = *occ;
  return e;
}

namespace {

// AADP_TIMING=1: host-side time marks of one aadp_fill_batch call (diagnostics of the end-to-end pipeline)
struct TimeMarks {
  bool on = false;
  std::chrono::steady_clock::time_point t0;
  std::string log;
  void start() { on = getenv("AADP_TIMING") != nullptr; t0 = std::chrono::steady_clock::now(); log.clear(); }
  void mark(const char* what) {
    if (!on) return;
    char b[96];
    snprintf(b, sizeof b, " %s %.2f", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    log += b;
  }
};
thread_local TimeMarks g_marks;

template <int K, int TBM, int STM, int PRO>
int launch_fill_t(aadp_ctx* c, FillParams& P) {
  auto kern = fill_kernel<K, TBM, STM, PRO>;
  const int A = P.sc.A;
  const size_t smem = (size_t)((A * A + 15) / 16 * 16) + (size_t)kWarpsPerCta * (kQRing + A * 32 * K);
  CK(cached_max_smem((const void*)kern, (size_t)(smem)));
  int occ = 0;
  CK(cached_occupancy(&occ, (const void*)kern, kWarpsPerCta * 32, smem));
  if (occ < 1) return fail("fill kernel does not fit on an SM");
  int grid = c->num_sms * occ;
  const int need = (P.n_items + kWarpsPerCta - 1) / kWarpsPerCta;
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  // multi-stripe pairs need a boundary buffer slot per resident warp
  if (c->b.max_Lt > 32 * K) {
    c->bb_rows = c->b.max_Lq + 2;
    if (c->bbuf.reserve((size_t)c->num_sms * occ * kWarpsPerCta * c->bb_rows * sizeof(int4))) return 1;
    P.bbuf = c->bbuf.as<int4>();
    P.bb_rows = c->bb_rows;
  }
  char nm[64];
  snprintf(nm, sizeof nm, "fill_kernel<K=%d,TB=%d,ST=%d%s>%s", K, TBM, STM, PRO ? ",PRO=1" : "", P.rev ? "rev" : "fwd");
  c->prof_begin(nm, P.cells_hint);
  kern<<<grid, kWarpsPerCta * 32, smem, c->stream>>>(P, c->prof_dev());
  c->prof_end();
  CK(cudaGetLastError());
  c->launches++;
  return 0;
}

template <int K, int PRO>
int launch_fill_kp(aadp_ctx* c, FillParams& P, int tbm, int stm) {
  if (tbm == 0) {
    if (stm == 0) return launch_fill_t<K, 0, 0, PRO>(c, P);
    if (stm == 1) return launch_fill_t<K, 0, 1, PRO>(c, P);
    return launch_fill_t<K, 0, 2, PRO>(c, P);
  }
  if (stm == 0) return launch_fill_t<K, 1, 0, PRO>(c, P);
  if (stm == 1) return launch_fill_t<K, 1, 1, PRO>(c, P);
  return launch_fill_t<K, 1, 2, PRO>(c, P);
}
template <int K>
int launch_fill_k(aadp_ctx* c, FillParams& P, int tbm, int stm) {
  return c->prof_mode ? launch_fill_kp<K, 1>(c, P, tbm, stm) : launch_fill_kp<K, 0>(c, P, tbm, stm);
}

// Builds the 16-byte aligned forward and reversed sequence arenas on the device and validates the
// residue codes (submatrix.h:36-38 is undefined behaviour for letters outside the matrix).
__global__ void arena_kernel(const uint8_t* __restrict__ res, const int64_t* __restrict__ seq_off,
                             const int32_t* __restrict__ aoff, int64_t s_begin, int64_t nseq, int A,
                             uint8_t* __restrict__ af, uint8_t* __restrict__ ar, int* __restrict__ bad) {
  for (int64_t sq = s_begin + blockIdx.x; sq < nseq; sq += gridDim.x) {
    const int64_t o = seq_off[sq];
    const int L = (int)(seq_off[sq + 1] - o);
    const int64_t d = aoff[sq];
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
      uint8_t v = res[o + i];
      if (v >= A) { *bad = 1; v = 0; }  // reported as an error by the host; kernels already in flight stay in bounds
      af[d + i] = v;
      ar[d + L - 1 - i] = v;
    }
  }
}

template <int TBM, int FST, int MSK, int LOC = 0, int PRO = 0>
int launch_packed_t(aadp_ctx* c, PackedParams& P) {
  // the forward pass with score spill reads its final row back (RB); a reverse pass with scores keeps the capture, its
  // column Lt sits in a register picked at run time
  auto kern = (FST && !MSK && !P.rev) ? packed_kernel<TBM, FST, MSK, 0, LOC, PRO, FST && !MSK> : packed_kernel<TBM, FST, MSK, 0, LOC, PRO>;
  const int A = P.sc.A;
  size_t smem = packed_smem_bytes(A, MSK);
  // measurement aid: AADP_PACKED_SMEM_PAD="fwd,rev" extra bytes per CTA lower the resident warps per SM
  if (const char* e = getenv("AADP_PACKED_SMEM_PAD")) {
    int pf = 0, pr = 0;
    if (sscanf(e, "%d,%d", &pf, &pr) >= 1) smem += (size_t)(P.rev ? pr : pf);
  }
  CK(cached_max_smem((const void*)kern, (size_t)(smem)));
  int occ = 0;
  CK(cached_occupancy(&occ, (const void*)kern, kPackedWarps * 32, smem));
  if (occ < 1) return fail("packed kernel does not fit on an SM");
  int grid = c->num_sms * occ;
  const int need = (P.n_tasks + kPackedWarps - 1) / kPackedWarps;
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  char nm[64];
  snprintf(nm, sizeof nm, "packed_kernel<TB=%d,FST=%d,MSK=%d%s%s>%s", TBM, FST, MSK, LOC ? ",LOC=1" : "", PRO ? ",PRO=1" : "",
           P.rev ? "rev" : "fwd");
  c->prof_begin(nm, P.cells_hint);
  P.prof = c->prof_dev();
  kern<<<grid, kPackedWarps * 32, smem, c->stream>>>(P);
  c->prof_end();
  CK(cudaGetLastError());
  c->launches++;
  return 0;
}

template <int PRO>
int launch_packed_p(aadp_ctx* c, PackedParams& P, int tbm, int fst, int msk) {
  const int key = tbm * 4 + fst * 2 + msk;
  if (P.sc.local) {  // local alignments: the clamped variants (never with the fused near-optimal pass)
    if (msk) return fail("internal: local alignments have no fused near-optimal pass");
    switch (key) {
      case 0: return launch_packed_t<0, 0, 0, 1, PRO>(c, P);
      case 2: return launch_packed_t<0, 1, 0, 1, PRO>(c, P);
      case 4: return launch_packed_t<1, 0, 0, 1, PRO>(c, P);
      default: return launch_packed_t<1, 1, 0, 1, PRO>(c, P);
    }
  }
  switch (key) {
    case 0: return launch_packed_t<0, 0, 0, 0, PRO>(c, P);
    case 1: return launch_packed_t<0, 0, 1, 0, PRO>(c, P);
    case 2: return launch_packed_t<0, 1, 0, 0, PRO>(c, P);
    case 3: return launch_packed_t<0, 1, 1, 0, PRO>(c, P);
    case 4: return launch_packed_t<1, 0, 0, 0, PRO>(c, P);
    case 5: return launch_packed_t<1, 0, 1, 0, PRO>(c, P);
    case 6: return launch_packed_t<1, 1, 0, 0, PRO>(c, P);
    default: return launch_packed_t<1, 1, 1, 0, PRO>(c, P);
  }
}
int launch_packed(aadp_ctx* c, PackedParams& P, int tbm, int fst, int msk) {
  return c->prof_mode ? launch_packed_p<1>(c, P, tbm, fst, msk) : launch_packed_p<0>(c, P, tbm, fst, msk);
}

// shared memory of a wavefront CTA (one warp = one stripe): substitution table, query ring + staging block, profile
static size_t wave_smem_bytes(int A) {
  return (size_t)((A * A + 15) / 16 * 16) + kQRing + 512 + (size_t)A * 32 * kWaveK;
}
// CTAs of the wavefront kernel that can be resident at once (all stripes of a pair wait on each other)
static int wave_resident_ctas(aadp_ctx* c, int A) {
  // the largest variant
  const void* kern = c->prof_mode ? (const void*)wave_kernel<kWaveK, 1, 2, 1> : (const void*)wave_kernel<kWaveK, 1, 2, 0>;
  const size_t smem = wave_smem_bytes(A);
  if (cached_max_smem((const void*)kern, smem) != cudaSuccess) return 0;
  int occ = 0;
  if (cached_occupancy(&occ, (const void*)kern, 32, smem) != cudaSuccess) return 0;
  return occ * c->num_sms;
}

template <int TBM, int STM>
int launch_wave_t(aadp_ctx* c, FillParams& Pf, FillParams& Pr, int ndirs, int nst) {
  const bool pro = c->prof_mode;
  const void* kern = pro ? (const void*)wave_kernel<kWaveK, TBM, STM, 1> : (const void*)wave_kernel<kWaveK, TBM, STM, 0>;
  const int A = Pf.sc.A;
  const size_t smem = wave_smem_bytes(A);
  CK(cached_max_smem((const void*)kern, (size_t)(smem)));
  int occ = 0;
  CK(cached_occupancy(&occ, (const void*)kern, 32, smem));
  const int grid = ndirs * nst;
  if (occ < 1 || grid > occ * c->num_sms) return fail("wavefront kernel: stripes of this pair cannot all be resident");
  char nm[64];
  snprintf(nm, sizeof nm, "wave_kernel<K=%d,TB=%d,ST=%d%s>x%d", kWaveK, TBM, STM, pro ? ",PRO=1" : "", ndirs);
  c->prof_begin(nm, Pf.cells_hint * ndirs);
  int nd = ndirs;
  ProfDev pd = c->prof_dev();
  void* args[] = {(void*)&Pf, (void*)&Pr, (void*)&nd, (void*)&pd};
  CK(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(32), args, smem, c->stream));
  c->prof_end();
  c->launches++;
  return 0;
}

int launch_wave(aadp_ctx* c, FillParams& Pf, FillParams& Pr, int ndirs, int nst, int tbm, int stm) {
  if (tbm == 0) {
    if (stm == 0) return launch_wave_t<0, 0>(c, Pf, Pr, ndirs, nst);
    if (stm == 1) return launch_wave_t<0, 1>(c, Pf, Pr, ndirs, nst);
    return launch_wave_t<0, 2>(c, Pf, Pr, ndirs, nst);
  }
  if (stm == 0) return launch_wave_t<1, 0>(c, Pf, Pr, ndirs, nst);
  if (stm == 1) return launch_wave_t<1, 1>(c, Pf, Pr, ndirs, nst);
  return launch_wave_t<1, 2>(c, Pf, Pr, ndirs, nst);
}

__global__ void scores_to_float_kernel(const int32_t* fin, float* out, int64_t n, int scale_log2) {
  const float inv = 1.f / (float)(1 << scale_log2);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (float)fin[i] * inv;
}

int check_ctx(aadp_ctx* c, bool need_scoring) {
  if (!c) return fail("null context");
  // between aadp_fill_batch_submit and aadp_fill_batch_wait the context belongs to the batch in flight
  if (c->pending) return fail("a submitted batch is pending on this context: call aadp_fill_batch_wait first");
  if (need_scoring && !c->have_scoring) return fail("aadp_set_scoring has not been called");
  cudaError_t e = cudaSetDevice(c->device);
  if (e != cudaSuccess) return fail(std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  return 0;
}

// Persistent host worker pool (the schedule of a batch is built on several host threads; spawning
// threads per call costs more than the work itself).  run(T, f) executes f(t) for t in [0,T): the
// caller is thread 0, workers take 1..T-1.
void HostPool::start(int n) {
  while ((int)workers.size() < n) {
    const int id = (int)workers.size() + 1;
    workers.emplace_back([this, id]() {
      uint64_t seen = 0;
      for (;;) {
        std::function<void(int)>* f = nullptr;
        {
          std::unique_lock<std::mutex> lk(mu);
          cv.wait(lk, [&]() { return stop || gen != seen; });
          if (stop) return;
          seen = gen;
          if (id < active) f = fn;
        }
        if (f) {
          (*f)(id);
          std::unique_lock<std::mutex> lk(mu);
          if (--pending == 0) done.notify_one();
        }
      }
    });
  }
}
void HostPool::run(int T, std::function<void(int)> f) {
  if (T <= 1) { f(0); return; }
  start(T - 1);
  {
    std::unique_lock<std::mutex> lk(mu);
    fn = &f;
    active = T;
    pending = T - 1;
    ++gen;
  }
  cv.notify_all();
  f(0);
  std::unique_lock<std::mutex> lk(mu);
  done.wait(lk, [&]() { return pending == 0; });
  fn = nullptr;
}
HostPool::~HostPool() {
  {
    std::unique_lock<std::mutex> lk(mu);
    stop = true;
  }
  cv.notify_all();
  for (std::thread& t : workers) t.join();
}

// Couple pairs of equal lane width and similar query length (they share a segment, one per register
// half), then bin-pack the couples into 32-lane tasks of similar duration.  Works on the packed pairs of
// the id range [lo,hi) only, so that several host threads can schedule disjoint ranges independently;
// S.tasks receives 64 pair ids per task, longest tasks first.
void build_tasks_range(const Batch& b, const int32_t* Lq32, const int32_t* Lt32, int64_t lo, int64_t hi, SchedScratch& S) {
  typedef SchedItem Item;
  typedef SchedCouple Couple;
  std::vector<int32_t>& out = S.tasks;
  out.clear();
  std::vector<Item>& items = S.items;
  items.clear();
  for (int64_t p = lo; p < hi; ++p) {
    if (b.fmt[p] != 1) continue;
    items.push_back({(int32_t)p, (Lt32[p] + 15) / 16, Lq32[p]});
  }
  if (items.empty()) return;
  // order by (lane width desc, query length desc, pair id): a counting sort when the key space is small
  // (the usual case: Lq up to a few thousand), std::sort otherwise
  int maxLq = 0;
  for (const Item& it : items) maxLq = std::max(maxLq, it.Lq);
  auto cmp = [](const Item& x, const Item& y) {
    if (x.n != y.n) return x.n > y.n;
    if (x.Lq != y.Lq) return x.Lq > y.Lq;
    return x.p < y.p;
  };
  std::vector<int32_t>& cnt = S.cnt;
  if ((int64_t)33 * (maxLq + 1) <= (int64_t)4 * (int64_t)items.size() + 65536) {
    const int64_t nb = (int64_t)33 * (maxLq + 1);
    cnt.assign((size_t)nb + 1, 0);
    auto key = [&](const Item& it) { return (int64_t)(32 - it.n) * (maxLq + 1) + (maxLq - it.Lq); };
    for (const Item& it : items) cnt[(size_t)key(it) + 1]++;
    for (int64_t k = 0; k < nb; ++k) cnt[(size_t)k + 1] += cnt[(size_t)k];
    std::vector<Item>& sorted = S.items2;
    sorted.resize(items.size());
    for (const Item& it : items) sorted[(size_t)cnt[(size_t)key(it)]++] = it;  // stable: pair ids stay ascending
    items.swap(sorted);
  } else {
    std::sort(items.begin(), items.end(), cmp);
  }
  std::vector<Couple>& couples = S.couples;
  couples.clear();
  for (size_t i = 0; i < items.size();) {
    if (i + 1 < items.size() && items[i + 1].n == items[i].n) {
      couples.push_back({items[i].p, items[i + 1].p, items[i].n, items[i].Lq});  // a has the longer query
      i += 2;
    } else {
      couples.push_back({items[i].p, -1, items[i].n, items[i].Lq});
      i += 1;
    }
  }
  // stable order by query length, longest first (longest tasks are scheduled first)
  if ((int64_t)maxLq + 1 <= (int64_t)4 * (int64_t)couples.size() + 65536) {
    cnt.assign((size_t)maxLq + 2, 0);
    for (const Couple& cp : couples) cnt[(size_t)(maxLq - cp.Lq) + 1]++;
    for (int k = 0; k <= maxLq; ++k) cnt[(size_t)k + 1] += cnt[(size_t)k];
    std::vector<Couple>& sorted = S.couples2;
    sorted.resize(couples.size());
    for (const Couple& cp : couples) sorted[(size_t)cnt[(size_t)(maxLq - cp.Lq)]++] = cp;
    couples.swap(sorted);
  } else {
    std::stable_sort(couples.begin(), couples.end(), [](const Couple& x, const Couple& y) { return x.Lq > y.Lq; });
  }
  struct Open { int64_t task; int used; };
  Open open[49];
  int n_open = 0;
  int64_t n_tasks = 0;
  for (const Couple& cp : couples) {
    int best = -1;
    for (int k = 0; k < n_open; ++k)
      if (32 - open[k].used >= cp.n && (best < 0 || open[k].used > open[best].used)) best = k;
    if (best < 0) {
      if (n_open >= 48) {  // drop the oldest open task: its query lengths are the least similar
        for (int k = 1; k < n_open; ++k) open[k - 1] = open[k];
        --n_open;
      }
      out.resize(out.size() + 64, -1);
      open[n_open] = {n_tasks++, 0};
      best = n_open++;
    }
    Open& o = open[best];
    int32_t* dst = &out[(size_t)o.task * 64 + o.used];
    for (int l = 0; l < cp.n; ++l) {
      dst[l] = cp.a;
      dst[32 + l] = cp.b;
    }
    o.used += cp.n;
    if (o.used == 32) {
      for (int k = best + 1; k < n_open; ++k) open[k - 1] = open[k];
      --n_open;
    }
  }
}

// Profile scoring: one profile per sequence id of the batch, and a template's profile must hold L_t*A entries.
int profile_count_refusal(aadp_ctx* c, int64_t nseq) {
  if (c->prof_nseq >= nseq) return 0;
  return fail("profile scoring: " + std::to_string(c->prof_nseq) + " profiles for " + std::to_string(nseq) +
              " sequences; aadp_set_profile_scoring needs one profile (possibly empty) per sequence id");
}
int profile_refusal(aadp_ctx* c, int64_t ts, int64_t Lt) {
  const int64_t n = c->prof_len[(size_t)ts];
  if (n == 0)
    return fail("profile scoring: sequence " + std::to_string(ts) + " is used as a template (" + std::to_string(Lt) +
                " residues) but its profile is empty");
  return fail("profile scoring: the profile of sequence " + std::to_string(ts) + " has " + std::to_string(n) +
              " entries, but the template has " + std::to_string(Lt) + " residues: L*A = " + std::to_string(Lt * c->sc.A) +
              " entries are needed");
}

// Classifies every pair (packed / int32 / wavefront), sizes its resident products and builds the packed
// task list.  All O(npairs) passes run on `host_threads` threads over disjoint pair ranges; the per-range
// task lists (each longest first) are interleaved round-robin so the global order stays longest first.
// (build_task_chunk builds the packed task list, per chunk of consecutive pair ids.)
int build_batch_meta(aadp_ctx* c, uint32_t what) {
  Batch& b = c->b;
  const int64_t np = b.npairs;
  b.tb_off.resize(np + 1);
  b.sc_off.resize(np + 1);
  b.mask_off.resize(np + 1);
  b.tb_off[0] = b.sc_off[0] = b.mask_off[0] = 0;
  b.order[0].clear();
  b.order[1].clear();
  b.max_Lq = b.max_Lt = 0;
  b.cells = 0;
  b.bucket_cells[0] = b.bucket_cells[1] = 0;
  b.fmt.resize(np);
  b.wave_pairs.clear();
  b.packed_cells = 0;
  b.n_tasks = 0;
  b.chunk_first.clear();
  b.chunk_ntasks.clear();
  b.chunk_cells.clear();
  b.chunk_max_seq.clear();
  int T = c->host_threads;
  if (T <= 0) T = (int)std::min<unsigned>(std::max<unsigned>(std::thread::hardware_concurrency(), 1u), 8u);
  T = (int)std::max<int64_t>(1, std::min<int64_t>(T, np / 4096));
  if ((int)c->sched.size() < T) c->sched.resize((size_t)T);
  c->Lq32.resize((size_t)np);
  c->Lt32.resize((size_t)np);
  int32_t* const Lq32 = c->Lq32.data();
  int32_t* const Lt32 = c->Lt32.data();
  if (c->prof_mode && profile_count_refusal(c, b.nseq)) return 1;
  struct Part {
    int err = 0, max_Lq = 0, max_Lt = 0;
    int64_t bad_seq = 0;
    int64_t bound = 0, sum[3] = {0, 0, 0};
    double cells = 0, packed_cells = 0, bucket_cells[2] = {0, 0};
  };
  std::vector<Part> part((size_t)T);
  const int wave_budget = c->allow_wave ? wave_resident_ctas(c, c->sc.A) : 0;
  auto range = [&](int t, int64_t* lo, int64_t* hi) { *lo = np * t / T; *hi = np * (t + 1) / T; };
  // ---- pass 1: lengths, class, score bound
  c->pool.run(T, [&](int t) {
    Part P;
    SchedScratch& S = c->sched[(size_t)t];
    S.order[0].clear();
    S.order[1].clear();
    S.wave.clear();
    int64_t lo, hi;
    range(t, &lo, &hi);
    for (int64_t p = lo; p < hi; ++p) {
      const int qs = b.pair_q[p], ts = b.pair_t[p];
      if (qs < 0 || qs >= b.nseq || ts < 0 || ts >= b.nseq) { P.err = 1; break; }
      const int64_t Lq = b.seq_off[qs + 1] - b.seq_off[qs], Lt = b.seq_off[ts + 1] - b.seq_off[ts];
      if (Lq < 0 || Lt < 0 || Lq > (1 << 24) || Lt > (1 << 24)) { P.err = 2; break; }
      Lq32[p] = (int32_t)Lq;
      Lt32[p] = (int32_t)Lt;
      P.max_Lq = std::max<int>(P.max_Lq, (int)Lq);
      P.max_Lt = std::max<int>(P.max_Lt, (int)Lt);
      const int64_t cl = Lq * Lt;
      P.cells += (double)cl;
      // |similarity| bound: the substitution table's, or (profile scoring) the template's own
      int64_t mx = c->max_abs_sub;
      if (c->prof_mode) {
        if (c->prof_len[(size_t)ts] != Lt * c->sc.A) { P.err = 3; P.bad_seq = ts; break; }
        mx = c->prof_max[(size_t)ts];
      }
      // |score| bound in integer units: matches + one end gap on each side
      const int64_t bd = std::min(Lq, Lt) * mx + 2 * (int64_t)c->sc.gi + (int64_t)c->sc.ge * (Lq + Lt);
      // (local alignments: the packed kernel has no fused near-optimal pass for them -- F + R - sim needs both clamped
      // matrices -- so a local run that asks for the cell set keeps the int32 kernels + mask_kernel)
      const bool packed_ok = c->allow_packed && (!c->sc.local || !(what & AADP_W_MASK)) && Lq >= 1 && Lt >= 1 && Lt <= 512 && bd < kPackedBound &&
                             c->sc.ge <= 400 && c->sc.gi <= 2048;
      // long pairs: one CTA per kWaveCols-column stripe, all stripes of both directions co-resident
      // (both directions in one cooperative launch: every CTA of both must be resident; the budget is the kernel's real
      // occupancy, queried once per batch -- a pair that does not fit takes the int32 kernel instead of failing later)
      const bool wave_ok = !packed_ok && c->allow_wave && Lq >= 1 && Lt > 512 && cl >= (int64_t)c->wave_min_cells &&
                           2 * ((Lt + kWaveCols - 1) / kWaveCols) <= (int64_t)wave_budget;
      b.fmt[(size_t)p] = packed_ok ? 1 : (wave_ok ? 2 : 0);
      if (packed_ok) {
        P.packed_cells += (double)cl;
      } else if (wave_ok) {
        S.wave.push_back((int32_t)p);
        P.bound = std::max(P.bound, bd);
      } else {
        S.order[Lt <= 256 ? 0 : 1].push_back((int32_t)p);
        P.bucket_cells[Lt <= 256 ? 0 : 1] += (double)cl;
        P.bound = std::max(P.bound, bd);
      }
    }
    part[(size_t)t] = P;
  });
  int64_t bound = 0;
  for (int t = 0; t < T; ++t) {
    const Part& P = part[(size_t)t];
    const SchedScratch& S = c->sched[(size_t)t];
    if (P.err == 1) return fail("pair index out of range");
    if (P.err == 2) return fail("bad sequence length");
    if (P.err == 3) return profile_refusal(c, P.bad_seq, b.seq_off[(size_t)P.bad_seq + 1] - b.seq_off[(size_t)P.bad_seq]);
    b.max_Lq = std::max(b.max_Lq, P.max_Lq);
    b.max_Lt = std::max(b.max_Lt, P.max_Lt);
    b.cells += P.cells;
    b.packed_cells += P.packed_cells;
    bound = std::max(bound, P.bound);
    for (int k = 0; k < 2; ++k) {
      b.bucket_cells[k] += P.bucket_cells[k];
      b.order[k].insert(b.order[k].end(), S.order[k].begin(), S.order[k].end());
    }
    b.wave_pairs.insert(b.wave_pairs.end(), S.wave.begin(), S.wave.end());
  }
  b.st_mode = bound < 30000 ? 1 : 2;
  if (bound >= (1 << 24)) return fail("scores exceed the exactly-representable float range (2^24 units)");
  // ---- pass 2: product sizes (scores in int16 units; 16-byte aligned per pair) and the packed tasks
  const bool want_tb = (what & AADP_W_TB) != 0, want_sc = (what & (AADP_W_SCORES | AADP_W_MASK)) != 0,
             want_mk = (what & AADP_W_MASK) != 0;
  c->pool.run(T, [&](int t) {
    int64_t lo, hi, s0 = 0, s1 = 0, s2 = 0;
    range(t, &lo, &hi);
    for (int64_t p = lo; p < hi; ++p) {
      const Layout L = make_layout(Lq32[p], Lt32[p], b.fmt[(size_t)p], 0);
      const int64_t units = (b.fmt[(size_t)p] == 1 || b.st_mode == 1) ? 1 : 2;
      const int64_t z0 = want_tb ? round_up64(layout_tb_bytes(L), 16) : 0;
      const int64_t z1 = want_sc ? round_up64(layout_sc_elems(L) * units, 8) : 0;
      const int64_t z2 = want_mk ? round_up64(layout_mask_words(L), 4) : 0;
      s0 += z0; s1 += z1; s2 += z2;
      b.tb_off[(size_t)p + 1] = s0;  // range-local inclusive sums; the range base is added below
      b.sc_off[(size_t)p + 1] = s1;
      b.mask_off[(size_t)p + 1] = s2;
    }
    part[(size_t)t].sum[0] = s0; part[(size_t)t].sum[1] = s1; part[(size_t)t].sum[2] = s2;
  });
  // ---- range bases, added to the range-local sums
  std::vector<int64_t> base((size_t)T * 3 + 3, 0);
  for (int t = 0; t < T; ++t)
    for (int k = 0; k < 3; ++k) base[(size_t)(t + 1) * 3 + k] = base[(size_t)t * 3 + k] + part[(size_t)t].sum[k];
  c->pool.run(T, [&](int t) {
    int64_t lo, hi;
    range(t, &lo, &hi);
    const int64_t b0 = base[(size_t)t * 3], b1 = base[(size_t)t * 3 + 1], b2 = base[(size_t)t * 3 + 2];
    if (t > 0)
      for (int64_t p = lo; p < hi; ++p) {
        b.tb_off[(size_t)p + 1] += b0;
        b.sc_off[(size_t)p + 1] += b1;
        b.mask_off[(size_t)p + 1] += b2;
      }
  });
  for (int k = 0; k < 2; ++k)
    std::stable_sort(b.order[k].begin(), b.order[k].end(), [&](int32_t x, int32_t y) {
      return (int64_t)Lq32[x] * Lt32[x] > (int64_t)Lq32[y] * Lt32[y];
    });
  return 0;
}

// Packed task list of the pairs [lo,hi): scheduled on the host threads over sub-ranges, the per-range lists (each
// longest first) interleaved round-robin (task i of range t right after task i of range t-1) directly into the
// pinned staging pool.  Appends one chunk to the batch; *tasks_pinned / *ntasks describe it.
int build_task_chunk(aadp_ctx* c, int64_t lo, int64_t hi, int32_t** tasks_pinned, int64_t* ntasks) {
  Batch& b = c->b;
  int T = c->host_threads;
  if (T <= 0) T = (int)std::min<unsigned>(std::max<unsigned>(std::thread::hardware_concurrency(), 1u), 8u);
  T = (int)std::max<int64_t>(1, std::min<int64_t>(T, (hi - lo) / 4096));
  if ((int)c->sched.size() < T) c->sched.resize((size_t)T);
  const int32_t* Lq32 = c->Lq32.data();
  const int32_t* Lt32 = c->Lt32.data();
  c->pool.run(T, [&](int t) {
    const int64_t l2 = lo + (hi - lo) * t / T, h2 = lo + (hi - lo) * (t + 1) / T;
    build_tasks_range(b, Lq32, Lt32, l2, h2, c->sched[(size_t)t]);
  });
  std::vector<int64_t> nt((size_t)T);
  int64_t total = 0;
  for (int t = 0; t < T; ++t) {
    nt[(size_t)t] = (int64_t)c->sched[(size_t)t].tasks.size() / 64;
    total += nt[(size_t)t];
  }
  const size_t at = (c->pin_used + 63) / 64 * 64, bytes = (size_t)total * 64 * sizeof(int32_t);
  if (at + bytes > c->pin_cap) return fail("internal: pinned staging pool too small");
  int32_t* const tdst = reinterpret_cast<int32_t*>(c->pin + at);
  c->pin_used = at + bytes;
  c->pool.run(T, [&](int t) {
    const std::vector<int32_t>& src = c->sched[(size_t)t].tasks;
    for (int64_t i = 0; i < nt[(size_t)t]; ++i) {
      int64_t pos = 0;
      for (int u = 0; u < T; ++u) pos += std::min(nt[(size_t)u], i) + ((u < t && nt[(size_t)u] > i) ? 1 : 0);
      memcpy(tdst + pos * 64, &src[(size_t)i * 64], 64 * sizeof(int32_t));
    }
  });
  double cells = 0;
  int64_t max_seq = 0;
  for (int64_t p = lo; p < hi; ++p) {
    if (b.fmt[(size_t)p] == 1) cells += (double)Lq32[p] * (double)Lt32[p];
    max_seq = std::max<int64_t>(max_seq, std::max(b.pair_q[(size_t)p], b.pair_t[(size_t)p]));
  }
  b.chunk_max_seq.push_back(max_seq);
  b.chunk_first.push_back(b.n_tasks);
  b.chunk_ntasks.push_back(total);
  b.chunk_cells.push_back(cells);
  b.n_tasks += total;
  *tasks_pinned = tdst;
  *ntasks = total;
  return 0;
}

int pin_reserve(aadp_ctx* c, size_t bytes) {
  c->pin_used = 0;
  if (bytes <= c->pin_cap) return 0;
  if (c->pin) cudaFreeHost(c->pin);
  c->pin = nullptr;
  c->pin_cap = 0;
  const size_t want = bytes + bytes / 4 + 4096;
  if (cudaHostAlloc((void**)&c->pin, want, cudaHostAllocDefault) != cudaSuccess) return fail("cudaHostAlloc failed");
  c->pin_cap = want;
  return 0;
}

// copy a host vector into the pinned pool and start its (truly asynchronous) upload
template <class T>
int upload_vec(aadp_ctx* c, DevBuf& d, const std::vector<T>& v, cudaStream_t stream = nullptr, bool use_stream = false) {
  const size_t bytes = v.size() * sizeof(T);
  if (d.reserve(std::max<size_t>(bytes, 16))) return 1;
  if (!bytes) return 0;
  const size_t at = (c->pin_used + 63) / 64 * 64;
  if (at + bytes > c->pin_cap) return fail("internal: pinned staging pool too small");
  memcpy(c->pin + at, v.data(), bytes);
  c->pin_used = at + bytes;
  c->h2d_bytes += (int64_t)bytes;
  CK(cudaMemcpyAsync(d.p, c->pin + at, bytes, cudaMemcpyHostToDevice, use_stream ? stream : c->stream));
  return 0;
}

// Device buffers of one direction (sizes are known once build_batch_meta has run).
int reserve_direction(aadp_ctx* c, int dir, uint32_t what) {
  Batch& b = c->b;
  const int tbm = (what & AADP_W_TB) ? 1 : 0;
  const int64_t np = b.npairs;
  const bool have_v1 = !b.order[0].empty() || !b.order[1].empty() || !b.wave_pairs.empty();
  // the packed reverse pass fuses the mask and needs no reverse score matrix of its own
  const bool need_blob = (what & AADP_W_SCORES) || ((what & AADP_W_MASK) && (dir == 0 || have_v1));
  if (c->fin_score[dir].reserve(std::max<size_t>(np * 4, 16))) return 1;
  if (c->fin_kind[dir].reserve(std::max<size_t>(np * 4, 16))) return 1;
  if (c->fin_k[dir].reserve(std::max<size_t>(np * 4, 16))) return 1;
  if (tbm && c->tb[dir].reserve(std::max<size_t>((size_t)b.tb_off[np], 16))) return 1;
  if (need_blob && c->scb[dir].reserve(std::max<size_t>((size_t)b.sc_off[np] * 2, 16))) return 1;
  return 0;
}

constexpr size_t kAllChunks = (size_t)-1;
// Packed kernel of one direction over the tasks of one chunk.
int launch_packed_chunk(aadp_ctx* c, int dir, uint32_t what, float delta_ratio, float* d_threshold, int64_t* d_count,
                        size_t chunk) {
  Batch& b = c->b;
  const int tbm = (what & AADP_W_TB) ? 1 : 0;
  // chunk == kAllChunks: ONE launch over the task lists of all chunks (they are contiguous on the device) -- every
  // launch that is not needed for the host/GPU pipelining of aadp_fill_batch only adds a kernel tail
  const bool all = chunk == kAllChunks;
  if (all) {
    if (b.chunk_ntasks.empty() || b.n_tasks == 0) return 0;
    chunk = 7;  // its own work counter
  } else {
    if (chunk >= b.chunk_ntasks.size() || b.chunk_ntasks[chunk] == 0) return 0;
    if (chunk >= 7) return fail("internal: too many task chunks");
  }
  {
    PackedParams Q{};
    Q.sc = c->sc;
    Q.sub8 = c->sub8.as<int8_t>();
    Q.sub8p = c->sub8p.as<int8_t>();
    Q.arena = dir ? c->arena_r.as<uint8_t>() : c->arena_f.as<uint8_t>();
    Q.aoff = c->aoff.as<int32_t>();
    Q.seq_off = c->seq_off.as<int64_t>();
    Q.pair_q = c->pair_q.as<int32_t>();
    Q.pair_t = c->pair_t.as<int32_t>();
    Q.tasks = c->tasks.as<int32_t>() + (all ? b.chunk_first[0] : b.chunk_first[chunk]) * 64;
    Q.n_tasks = (int)(all ? b.n_tasks : b.chunk_ntasks[chunk]);
    Q.rev = dir;
    Q.counter = c->counter.as<unsigned int>() + (16 + 8 * dir + (int)chunk);
    Q.tb = tbm ? c->tb[dir].as<uint8_t>() : nullptr;
    Q.tb_off = c->tb_off.as<int64_t>();
    const int msk = (dir == 1 && (what & AADP_W_MASK)) ? 1 : 0;
    const int fst = (dir == 0) ? ((what & (AADP_W_SCORES | AADP_W_MASK)) ? 1 : 0) : ((what & AADP_W_SCORES) ? 1 : 0);
    Q.sc_out = fst ? c->scb[dir].as<int16_t>() : nullptr;
    Q.scF = msk ? c->scb[0].as<int16_t>() : nullptr;
    Q.sc_off = c->sc_off.as<int64_t>();
    Q.mask = msk ? c->mask.as<uint32_t>() : nullptr;
    Q.mask_off = c->mask_off.as<int64_t>();
    Q.fin_fwd = c->fin_score[0].as<int32_t>();
    Q.delta_ratio = delta_ratio;
    Q.threshold = msk ? d_threshold : nullptr;
    Q.count = msk ? reinterpret_cast<long long*>(d_count) : nullptr;
    Q.fin_score = c->fin_score[dir].as<int32_t>();
    Q.fin_kind = c->fin_kind[dir].as<int32_t>();
    Q.fin_k = c->fin_k[dir].as<int32_t>();
    Q.cells_hint = all ? b.packed_cells : b.chunk_cells[chunk];
    if (launch_packed(c, Q, tbm, fst, msk)) return 1;
  }
  return 0;
}

// The int32 kernels of one direction (pairs that do not qualify for the packed path).
int run_direction_int32(aadp_ctx* c, int dir /*0 fwd,1 rev*/, uint32_t what) {
  Batch& b = c->b;
  const int tbm = (what & AADP_W_TB) ? 1 : 0;
  const int stm = (what & (AADP_W_SCORES | AADP_W_MASK)) ? b.st_mode : 0;
  for (int k = 0; k < 2; ++k) {
    if (b.order[k].empty()) continue;
    FillParams P{};
    P.sc = c->sc;
    P.sub8 = c->sub8.as<int8_t>();
    P.residues = c->residues.as<uint8_t>();
    P.seq_off = c->seq_off.as<int64_t>();
    P.pair_q = c->pair_q.as<int32_t>();
    P.pair_t = c->pair_t.as<int32_t>();
    P.order = c->order[k].as<int32_t>();
    P.n_items = (int)b.order[k].size();
    P.rev = dir;
    P.counter = c->counter.as<unsigned int>() + (dir * 2 + k);
    P.tb = tbm ? c->tb[dir].as<uint8_t>() : nullptr;
    P.tb_off = c->tb_off.as<int64_t>();
    P.sc_blob = stm ? c->scb[dir].p : nullptr;
    P.sc_off = c->sc_off.as<int64_t>();
    P.fin_score = c->fin_score[dir].as<int32_t>();
    P.fin_kind = c->fin_kind[dir].as<int32_t>();
    P.fin_k = c->fin_k[dir].as<int32_t>();
    P.bbuf = nullptr;
    P.bb_rows = 0;
    P.cells_hint = b.bucket_cells[k];
    int rc = (k == 0) ? launch_fill_k<8>(c, P, tbm, stm) : launch_fill_k<16>(c, P, tbm, stm);
    if (rc) return rc;
  }
  return 0;
}

// Long pairs: one cooperative launch per pair, covering both directions when both are requested.
int run_wave_pairs(aadp_ctx* c, uint32_t what) {
  Batch& b = c->b;
  if (b.wave_pairs.empty()) return 0;
  const int tbm = (what & AADP_W_TB) ? 1 : 0;
  const int stm = (what & (AADP_W_SCORES | AADP_W_MASK)) ? b.st_mode : 0;
  for (int32_t p : b.wave_pairs) {
    const int qs = b.pair_q[p], ts = b.pair_t[p];
    const int Lq = (int)(b.seq_off[qs + 1] - b.seq_off[qs]), Lt = (int)(b.seq_off[ts + 1] - b.seq_off[ts]);
    const int nst = (Lt + kWaveCols - 1) / kWaveCols;
    const int bb_rows = Lq + 2;
    int dirs[2], nd = 0;
    if (what & AADP_W_FWD) dirs[nd++] = 0;
    if (what & AADP_W_REV) dirs[nd++] = 1;
    {
      // boundary words carry the tag of their launch; the buffer is zeroed whenever it is (re)allocated and
      // tags never repeat within an allocation, so stale words are never mistaken for published ones
      const void* old = c->wave_bb.p;
      if (c->wave_bb.reserve((size_t)nd * nst * bb_rows * 3 * sizeof(unsigned long long))) return 1;
      if (c->wave_bb.p != old || c->wave_tag == 0xffffffffu) {
        CK(cudaMemsetAsync(c->wave_bb.p, 0, c->wave_bb.cap, c->stream));
        c->wave_tag = 0;
      }
      ++c->wave_tag;
    }
    if (c->wave_ready.reserve((size_t)nd * nst * sizeof(int) + 16)) return 1;
    if (c->wave_part.reserve((size_t)nd * nst * sizeof(int4))) return 1;
    CK(cudaMemsetAsync(c->wave_ready.p, 0, (size_t)nd * nst * sizeof(int), c->stream));
    FillParams P[2];
    for (int k = 0; k < nd; ++k) {
      const int dir = dirs[k];
      FillParams& Q = P[k];
      Q = FillParams{};
      Q.sc = c->sc;
      Q.sub8 = c->sub8.as<int8_t>();
      Q.residues = c->residues.as<uint8_t>();
      Q.seq_off = c->seq_off.as<int64_t>();
      Q.pair_q = c->pair_q.as<int32_t>();
      Q.pair_t = c->pair_t.as<int32_t>();
      Q.rev = dir;
      Q.tb = tbm ? c->tb[dir].as<uint8_t>() : nullptr;
      Q.tb_off = c->tb_off.as<int64_t>();
      Q.sc_blob = stm ? c->scb[dir].p : nullptr;
      Q.sc_off = c->sc_off.as<int64_t>();
      Q.fin_score = c->fin_score[dir].as<int32_t>();
      Q.fin_kind = c->fin_kind[dir].as<int32_t>();
      Q.fin_k = c->fin_k[dir].as<int32_t>();
      Q.bb_rows = bb_rows;
      Q.cells_hint = (double)Lq * Lt;
      Q.wave_pair = p;
      Q.wave_nstripes = nst;
      Q.wave_ll = c->wave_bb.as<unsigned long long>() + (size_t)k * nst * bb_rows * 3;
      Q.wave_tag = c->wave_tag;
      Q.wave_dbg = nullptr;
      if (getenv("AADP_WAVE_DEBUG")) {
        if (c->wave_dbg.reserve((size_t)2 * nst * 2 * sizeof(long long))) return 1;
        Q.wave_dbg = c->wave_dbg.as<long long>() + (size_t)k * nst * 2;
      }
      Q.wave_ready = c->wave_ready.as<int>() + (size_t)k * nst;
      Q.wave_part = c->wave_part.as<int4>() + (size_t)k * nst;
    }
    if (nd == 1) P[1] = P[0];
    if (launch_wave(c, P[0], P[1], nd, nst, tbm, stm)) return 1;
    if (getenv("AADP_WAVE_DEBUG")) {  // per-stripe wait / total cycles of the launch (diagnostics)
      std::vector<long long> h((size_t)nd * nst * 2);
      CK(cudaStreamSynchronize(c->stream));
      CK(cudaMemcpy(h.data(), c->wave_dbg.p, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
      for (int k = 0; k < nd; ++k) {
        fprintf(stderr, "[aadp] wave dir %d: stripe wait%%/total:", dirs[k]);
        for (int st = 0; st < nst; st += std::max(1, nst / 24)) {
          const long long* e = &h[((size_t)k * nst + st) * 2];
          fprintf(stderr, " %d:%.0f/%.2fms", st, 100.0 * (double)e[0] / (double)std::max<long long>(1, e[1]), (double)e[1] / 1.965e6);
        }
        fprintf(stderr, "\n");
      }
    }
  }
  return 0;
}

int dense_pair(aadp_ctx* c, int64_t p, int dir, float* h_score, int32_t* h_pq, int32_t* h_pt) {
  if (!h_score && !h_pq && !h_pt) return 0;
  Batch& b = c->b;
  const int qs = b.pair_q[p], ts = b.pair_t[p];
  const int Lq = (int)(b.seq_off[qs + 1] - b.seq_off[qs]), Lt = (int)(b.seq_off[ts + 1] - b.seq_off[ts]);
  const int64_t n = (int64_t)(Lq + 2) * (Lt + 2);
  const bool have_tb = (b.ran_what & AADP_W_TB) != 0;
  const bool have_sc = (b.ran_what & (AADP_W_SCORES | AADP_W_MASK)) != 0;
  if (h_score && !have_sc) return fail("score matrices were not kept (run with AADP_W_SCORES)");
  if ((h_pq || h_pt) && !have_tb) return fail("traceback was not kept (run with AADP_W_TB)");
  if ((h_pq || h_pt) && c->sc.local && !have_sc) return fail("local tracebacks need AADP_W_SCORES");
  int32_t fin[3];
  CK(cudaMemcpyAsync(&fin[0], c->fin_score[dir].as<int32_t>() + p, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&fin[1], c->fin_kind[dir].as<int32_t>() + p, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&fin[2], c->fin_k[dir].as<int32_t>() + p, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  DenseParams D{};
  D.sc = c->sc;
  D.Lq = Lq;
  D.Lt = Lt;
  D.rev = dir;
  D.repro_rev_bug = (c->flags & AADP_REPRO_REV_BUG) ? 1 : 0;
  const bool packed = b.fmt[p] == 1;
  D.lay = make_layout(Lq, Lt, b.fmt[p], dir);
  D.bias = packed ? kBias16 : 0;
  // the packed reverse pass fuses the near-optimal mask and writes no score matrix of its own unless AADP_W_SCORES asks
  // for it: there is nothing to read then (reading it anyway was an out-of-bounds access when only the traceback of such
  // a pair was fetched)
  const bool sc_here = have_sc && !(packed && dir == 1 && !(b.ran_what & AADP_W_SCORES));
  if (h_score && !sc_here) return fail("reverse score matrices were not kept (run with AADP_W_SCORES)");
  D.st_mode = sc_here ? (packed ? 1 : b.st_mode) : 0;
  D.sc_blob = sc_here ? c->scb[dir].p : nullptr;
  D.sc_off = b.sc_off[p];
  D.tb = have_tb ? c->tb[dir].as<uint8_t>() + b.tb_off[p] : nullptr;
  D.fin_score = fin[0];
  D.fin_kind = fin[1];
  D.fin_k = fin[2];
  if (h_score) { if (c->scratch_a.reserve(n * 4)) return 1; D.score = c->scratch_a.as<float>(); }
  if (h_pq || h_pt) {
    if (c->scratch_b.reserve(n * 4) || c->scratch_c.reserve(n * 4)) return 1;
    D.prev_q = c->scratch_b.as<int32_t>();
    D.prev_t = c->scratch_c.as<int32_t>();
  }
  const int threads = 256;
  const int grid = (int)std::min<int64_t>((n + threads - 1) / threads, 148 * 8);
  dense_kernel<<<grid, threads, 0, c->stream>>>(D);
  CK(cudaGetLastError());
  c->launches++;
  if (h_score) CK(cudaMemcpyAsync(h_score, D.score, n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (h_pq) CK(cudaMemcpyAsync(h_pq, D.prev_q, n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (h_pt) CK(cudaMemcpyAsync(h_pt, D.prev_t, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int dense_mask(aadp_ctx* c, int64_t p, uint8_t* h_mask) {
  if (!h_mask) return 0;
  Batch& b = c->b;
  if (!(b.ran_what & AADP_W_MASK)) return fail("near-optimal mask was not computed (run with AADP_W_MASK)");
  const int qs = b.pair_q[p], ts = b.pair_t[p];
  const int Lq = (int)(b.seq_off[qs + 1] - b.seq_off[qs]), Lt = (int)(b.seq_off[ts + 1] - b.seq_off[ts]);
  const int sz2 = Lt + 2;
  const int64_t mws = mask_row_words(Lt);
  const Layout L = make_layout(Lq, Lt, b.fmt[p], 1);
  const int64_t nwords = layout_mask_words(L);
  std::vector<uint32_t> bits((size_t)std::max<int64_t>(nwords, 1));
  if (nwords > 0) {
    CK(cudaMemcpyAsync(bits.data(), c->mask.as<uint32_t>() + b.mask_off[p], (size_t)nwords * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  memset(h_mask, 0, (size_t)(Lq + 2) * sz2);
  if (b.fmt[p] != 1) {
    for (int i = 1; i <= Lq; ++i)
      for (int j = 1; j <= Lt; ++j)
        h_mask[(size_t)i * sz2 + j] = (bits[(size_t)(i - 1) * mws + ((j - 1) >> 5)] >> ((j - 1) & 31)) & 1u;
  } else {
    // packed reverse pass: reverse-flow coordinates, diagonal-major, 2 bytes per 16-column slot:
    // byte (c&1), bit 7-(c>>1)
    const uint8_t* by = reinterpret_cast<const uint8_t*>(bits.data());
    for (int i = 1; i <= Lq; ++i)
      for (int j = 1; j <= Lt; ++j) {
        const int a = Lq + 1 - i, bb = Lt + 1 - j;
        const int slot = (bb - 1) >> 4, cc = (bb - 1) & 15;
        const uint8_t v = by[((size_t)(a - 1 + slot) * L.n + slot) * 2 + (cc & 1)];
        h_mask[(size_t)i * sz2 + j] = (v >> (7 - (cc >> 1))) & 1u;
      }
  }
  return 0;
}

}  // namespace

extern "C" {

const char* aadp_last_error(void) { return g_err.c_str(); }
const char* aadp_version(void) { return "aadp 0.1 (sm_100a)"; }

aadp_ctx* aadp_create(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    g_err = std::string("no CUDA device available (") + (e != cudaSuccess ? cudaGetErrorString(e) : "count 0") +
            "); this library has no CPU fallback";
    return nullptr;
  }
  if (device < 0 || device >= n) { g_err = "device index out of range"; return nullptr; }
  if (cudaSetDevice(device) != cudaSuccess) { g_err = "cudaSetDevice failed"; return nullptr; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { g_err = "cudaGetDeviceProperties failed"; return nullptr; }
  if (prop.major != 10) {
    g_err = "this build contains sm_100a kernels only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor);
    return nullptr;
  }
  aadp_ctx* c = new aadp_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_err = "cudaStreamCreate failed";
    delete c;
    return nullptr;
  }
  c->stream = c->own_stream;
  if (const char* e = getenv("AADP_HOST_THREADS")) c->host_threads = atoi(e);
  else if (const char* lw = getenv("LOCAL_WORLD_SIZE")) {
    // one process per GPU (torchrun): the ranks of a box share its cores, so each scheduler takes its share
    const int ranks = std::max(1, atoi(lw));
    const int hw = (int)std::max<unsigned>(std::thread::hardware_concurrency(), 1u);
    c->host_threads = std::max(2, std::min(8, hw / ranks));
  }
  if (const char* e = getenv("AADP_PIPELINE_CHUNKS")) c->pipeline_chunks = std::max(1, std::min(atoi(e), 7));
  return c;
}

void aadp_destroy(aadp_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  DevBuf* all[] = {&c->sub8, &c->residues, &c->seq_off, &c->pair_q, &c->pair_t, &c->order[0], &c->order[1], &c->tb_off,
                   &c->sc_off, &c->mask_off, &c->tb[0], &c->tb[1], &c->scb[0], &c->scb[1], &c->mask, &c->fin_score[0],
                   &c->fin_score[1], &c->fin_kind[0], &c->fin_kind[1], &c->fin_k[0], &c->fin_k[1], &c->counter, &c->bbuf,
                   &c->thr, &c->count, &c->fscore[0], &c->fscore[1], &c->scratch_a, &c->scratch_b, &c->scratch_c, &c->scratch_d,
                   &c->fmt, &c->tasks, &c->aoff, &c->arena_f, &c->arena_r, &c->badflag, &c->wave_bb, &c->wave_ready, &c->wave_part,
                   &c->x_layout, &c->x_qc, &c->x_qid, &c->x_tid, &c->x_scores,
                   &c->subf, &c->gg_score[0], &c->gg_score[1], &c->gg_pq[0], &c->gg_pq[1], &c->gg_pt[0], &c->gg_pt[1],
                   &c->gg_mask, &c->gg_off, &c->gg_fin[0], &c->gg_fin[1], &c->gg_pm[0], &c->gg_pm[1], &c->gg_items, &c->tb_del, &c->tb_ins, &c->tb_del_off, &c->tb_ins_off, &c->ali_cap, &c->ali_out, &c->ali_n, &c->ali_status, &c->gg_rect, &c->sub8p,
                   &c->ucw_ids, &c->ucw_path_off, &c->ucw_stack_off, &c->ucw_stack, &c->ucw_paths, &c->ucw_len, &c->ucw_scores, &c->ucw_n, &c->ucw_status, &c->ucw_thr, &c->ucw_plen, &c->ucw_pathbuf, &c->ucw_flags, &c->ucw_flag_off,
                   &c->prof8, &c->prof8_off, &c->proff, &c->proff_off};
  for (DevBuf* d : all) d->release();
  if (c->pin) cudaFreeHost(c->pin);
  if (c->pin_flag) cudaFreeHost(c->pin_flag);
  if (c->ev_flag) cudaEventDestroy(c->ev_flag);
  if (c->ev_start) cudaEventDestroy(c->ev_start);
  for (int j = 0; j < 8; ++j) if (c->ev_piece[j]) cudaEventDestroy(c->ev_piece[j]);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

int aadp_set_stream(aadp_ctx* c, void* s) {
  if (!c) return fail("null context");
  // NULL is a valid handle: the legacy default stream (what torch.cuda.current_stream() is
  // unless the caller switched streams).  aadp_create() starts on a private non-blocking stream.
  c->stream = reinterpret_cast<cudaStream_t>(s);
  return 0;
}

int aadp_set_option(aadp_ctx* c, const char* key, int value) {
  if (!c || !key) return fail("null argument");
  if (!strcmp(key, "packed")) { c->allow_packed = value != 0; return 0; }
  if (!strcmp(key, "wave")) { c->allow_wave = value != 0; return 0; }
  if (!strcmp(key, "wave_min_cells")) { c->wave_min_cells = value; return 0; }
  if (!strcmp(key, "host_threads")) { c->host_threads = value; return 0; }
  if (!strcmp(key, "pipeline_chunks")) { c->pipeline_chunks = std::max(1, std::min(value, 8)); return 0; }
  // exact_float = 1: route everything through the exact general-gap fp32 kernel (takes effect at the next
  // aadp_set_scoring); scoring that is not on a dyadic grid always uses it
  if (!strcmp(key, "exact_float")) { c->force_float = value != 0; return 0; }
  if (!strcmp(key, "general_threads")) { c->gg_threads_cap = std::max(32, std::min(512, value / 32 * 32)); return 0; }
  if (!strcmp(key, "general_prune")) { c->gg_prune = value ? 1 : 0; return 0; }
  if (!strcmp(key, "general_records")) { c->gg_records = value ? 1 : 0; return 0; }
  if (!strcmp(key, "enum_mask_prune")) { c->enum_mask_prune = value ? 1 : 0; return 0; }
  // alignment limits of the enumerators (ucw.h:72 hard-codes 100000, cw.h:76 1000000): beyond them the reference
  // forces optimal paths instead of branching; <= 0 restores the reference's value
  if (!strcmp(key, "ucw_user_limit")) { c->ucw_user_limit = value > 0 ? value : 100000; return 0; }
  if (!strcmp(key, "cw_user_limit")) { c->cw_user_limit = value > 0 ? value : 1000000; return 0; }
  if (!strcmp(key, "general_budget_mcells")) { c->gg_budget_cells = (int64_t)std::max(value, 1) * 1000000; return 0; }
  return fail(std::string("unknown option ") + key);
}

int aadp_synchronize(aadp_ctx* c) {
  if (check_ctx(c, false)) return 1;
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int aadp_set_scoring(aadp_ctx* c, const float* sub, int A, float gi, float ge, int align_type, uint32_t flags) {
  if (check_ctx(c, false)) return 1;
  if (!sub || A < 1 || A > 64) return fail("alphabet size must be 1..64");
  if (align_type < 0 || align_type > 4) return fail("Illegal gap style");  // aasubalib.h:49
  if (!(gi >= 0.f) || !(ge >= 0.f)) return fail("gap penalties must be non-negative");
  // find the dyadic grid: smallest s with everything integral in units of 2^-s
  int s = -1;
  for (int t = 0; t <= 8 && s < 0; ++t) {
    const float m = (float)(1 << t);
    bool ok = (gi * m == rintf(gi * m)) && (ge * m == rintf(ge * m));
    for (int i = 0; i < A * A && ok; ++i) ok = (sub[i] * m == rintf(sub[i] * m));
    if (ok) s = t;
  }
  c->prof_mode = false;
  c->sc.A = A;
  c->sc.delfree = (align_type == AADP_LOCAL || align_type == AADP_SEMI_LOCAL || align_type == AADP_LOCAL_GLOBAL);
  c->sc.insfree = (align_type == AADP_LOCAL || align_type == AADP_SEMI_LOCAL || align_type == AADP_GLOBAL_LOCAL);
  c->sc.local = (align_type == AADP_LOCAL);
  c->align_type = align_type;
  c->flags = flags;
  c->gi_f = gi;
  c->ge_f = ge;
  c->subf_h.assign(sub, sub + (size_t)A * A);
  if (c->subf.reserve((size_t)A * A * 4)) return 1;
  CK(cudaMemcpyAsync(c->subf.p, sub, (size_t)A * A * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->b.ran_what = 0;
  c->b.sched_ok = false;  // classification, score bounds and storage modes depend on the scoring
  if (c->b.seq_A != A) c->b.have_seqs = false;  // the residues were validated against another alphabet
  // the integer kernels also need the scaled substitution scores inside the int8 profile range and moderate gap
  // penalties; anything else (e.g. an integer matrix scaled by 10 whose entries exceed 127) is still a legal
  // reference input and takes the exact general-gap path instead of being refused
  bool fits = s >= 0;
  if (fits) {
    const float m = (float)(1 << s);
    for (int i = 0; i < A * A && fits; ++i) fits = fabsf(sub[i] * m) <= 127.f;
    fits = fits && gi * m <= 1e6f && ge * m <= 1e5f;
  }
  if (!fits || c->force_float) {
    // not representable on an integer grid (e.g. the reference defaults 4.73 / 0.34, alib.cpp:17-18): the exact
    // general-gap fp32 kernel reproduces the reference's own scan and roundings (aadp_general.cuh)
    c->float_mode = true;
    c->sc.gi = c->sc.ge = 0;
    c->sc.scale_log2 = 0;
    c->max_abs_sub = 0;
    c->have_scoring = true;
    return 0;
  }
  c->float_mode = false;
  const float m = (float)(1 << s);
  c->sub8_h.resize((size_t)A * A);
  int mx = 0;
  for (int i = 0; i < A * A; ++i) {
    const float v = sub[i] * m;
    c->sub8_h[i] = (int8_t)(int)v;
    mx = std::max(mx, std::abs((int)v));
  }
  c->max_abs_sub = mx;
  c->sc.A = A;
  c->sc.gi = (int)(gi * m);
  c->sc.ge = (int)(ge * m);
  c->sc.delfree = (align_type == AADP_LOCAL || align_type == AADP_SEMI_LOCAL || align_type == AADP_LOCAL_GLOBAL);
  c->sc.insfree = (align_type == AADP_LOCAL || align_type == AADP_SEMI_LOCAL || align_type == AADP_GLOBAL_LOCAL);
  c->sc.local = (align_type == AADP_LOCAL);
  c->sc.scale_log2 = s;
  c->align_type = align_type;
  c->flags = flags;
  if (c->sub8.reserve((size_t)A * A)) return 1;
  CK(cudaMemcpyAsync(c->sub8.p, c->sub8_h.data(), (size_t)A * A, cudaMemcpyHostToDevice, c->stream));
  {  // padded copy for the packed kernels' profile build: A rows of A+1 entries, entry A = pad column (-128)
    std::vector<int8_t> pad((size_t)packed_sub_bytes(A), (int8_t)-128);
    for (int a = 0; a < A; ++a)
      for (int b2 = 0; b2 < A; ++b2) pad[(size_t)a * (A + 1) + b2] = c->sub8_h[(size_t)a * A + b2];
    if (c->sub8p.reserve(pad.size())) return 1;
    CK(cudaMemcpy(c->sub8p.p, pad.data(), pad.size(), cudaMemcpyHostToDevice));
  }
  CK(cudaStreamSynchronize(c->stream));
  c->have_scoring = true;
  return 0;
}

int aadp_set_profile_scoring(aadp_ctx* c, const float* prof, const int64_t* prof_off, int64_t nprof, int A, float gi,
                             float ge, int align_type, uint32_t flags) {
  if (check_ctx(c, false)) return 1;
  if (A < 1 || A > 64) return fail("alphabet size must be 1..64");
  if (align_type < 0 || align_type > 4) return fail("Illegal gap style");  // aasubalib.h:49
  if (!(gi >= 0.f) || !(ge >= 0.f)) return fail("gap penalties must be non-negative");
  if (nprof < 0 || nprof > 0x7fffffff || !prof_off) return fail("null input");
  if (prof_off[nprof] > prof_off[0] && !prof) return fail("null input");
  const char* other = "; position-specific similarities off that grid run on the exact fp32 kernels of aadp_fill_batch_tabulated / "
                      "aadp_fill_pair_general";
  if (c->force_float)
    return fail(std::string("aadp_set_profile_scoring: profile scoring runs on the integer kernels only and the option exact_float "
                            "is set") + other);
  for (int64_t s2 = 0; s2 < nprof; ++s2) {
    const int64_t n = prof_off[s2 + 1] - prof_off[s2];
    if (n < 0) return fail("aadp_set_profile_scoring: profile offsets must be non-decreasing");
    if (n % A) return fail("aadp_set_profile_scoring: the profile of sequence " + std::to_string(s2) + " has " + std::to_string(n) +
                           " entries, not a multiple of A = " + std::to_string(A));
  }
  const float* p0 = prof ? prof + prof_off[0] : nullptr;
  const int64_t ntot = prof_off[nprof] - prof_off[0];
  // the dyadic grid of aadp_set_scoring: smallest s <= 8 with every entry, gi and ge integral in units of 2^-s
  int s = -1;
  for (int t = 0; t <= 8 && s < 0; ++t) {
    const float m = (float)(1 << t);
    bool ok = (gi * m == rintf(gi * m)) && (ge * m == rintf(ge * m));
    for (int64_t i = 0; i < ntot && ok; ++i) ok = (p0[i] * m == rintf(p0[i] * m));
    if (ok) s = t;
  }
  if (s < 0) return fail(std::string("aadp_set_profile_scoring: the profile entries, gi and ge are not on one dyadic grid 2^-s, s <= 8") + other);
  const float m = (float)(1 << s);
  if (gi * m > 1e6f || ge * m > 1e5f) return fail(std::string("aadp_set_profile_scoring: gap penalties too large for the integer kernels") + other);
  std::vector<int> pmax((size_t)nprof, 0);
  for (int64_t s2 = 0; s2 < nprof; ++s2)
    for (int64_t i = prof_off[s2]; i < prof_off[s2 + 1]; ++i) {
      const float v = fabsf(prof[i] * m);
      if (v > 127.f) {
        char e[256];
        snprintf(e, sizeof e, "aadp_set_profile_scoring: the profile of sequence %lld has an entry of %g = %g units of 2^-%d, above 127 units",
                 (long long)s2, (double)prof[i], (double)v, s);
        return fail(e + std::string(other));
      }
      pmax[(size_t)s2] = std::max(pmax[(size_t)s2], (int)v);
    }
  // int8 layout (ProfDev, aadp_kernels.cuh): per sequence, forward flow then reverse flow, A rows of prof_row_bytes(L)
  std::vector<int64_t> off8((size_t)nprof + 1, 0), offf((size_t)nprof + 1, 0);
  for (int64_t s2 = 0; s2 < nprof; ++s2) {
    const int L = (int)((prof_off[s2 + 1] - prof_off[s2]) / A);
    off8[(size_t)s2 + 1] = off8[(size_t)s2] + 2 * (int64_t)A * prof_row_bytes(L);
    offf[(size_t)s2 + 1] = prof_off[s2 + 1] - prof_off[0];
  }
  std::vector<int8_t> p8((size_t)std::max<int64_t>(off8[(size_t)nprof], 16), (int8_t)-128);
  for (int64_t s2 = 0; s2 < nprof; ++s2) {
    const float* ps = prof + prof_off[s2];
    const int L = (int)((prof_off[s2 + 1] - prof_off[s2]) / A), nb = prof_row_bytes(L), sig = nb - L;
    int8_t* fwd = p8.data() + off8[(size_t)s2];
    int8_t* rev = fwd + (int64_t)A * nb;
    for (int j = 1; j <= L; ++j)
      for (int a = 0; a < A; ++a) {
        const int8_t v = (int8_t)(int)(ps[(int64_t)(j - 1) * A + a] * m);
        fwd[(int64_t)a * nb + j - 1 + sig] = v;  // forward flow column j
        rev[(int64_t)a * nb + L - j] = v;        // reverse flow column L+1-j
      }
  }
  // everything checked: the profiles replace the context's scoring
  CK(cudaStreamSynchronize(c->stream));
  if (c->prof8.reserve(p8.size()) || c->prof8_off.reserve(off8.size() * 8) || c->proff.reserve(std::max<size_t>((size_t)ntot * 4, 16)) ||
      c->proff_off.reserve(offf.size() * 8))
    return 1;
  CK(cudaMemcpy(c->prof8.p, p8.data(), p8.size(), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c->prof8_off.p, off8.data(), off8.size() * 8, cudaMemcpyHostToDevice));
  if (ntot) CK(cudaMemcpy(c->proff.p, p0, (size_t)ntot * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(c->proff_off.p, offf.data(), offf.size() * 8, cudaMemcpyHostToDevice));
  c->proff_h.assign(p0, p0 + ntot);
  c->proff_off_h = offf;
  c->prof_len.resize((size_t)nprof);
  for (int64_t s2 = 0; s2 < nprof; ++s2) c->prof_len[(size_t)s2] = prof_off[s2 + 1] - prof_off[s2];
  c->prof_max = pmax;
  c->prof_nseq = nprof;
  c->prof_mode = true;
  c->float_mode = false;
  c->max_abs_sub = 0;
  c->sc.A = A;
  c->sc.gi = (int)(gi * m);
  c->sc.ge = (int)(ge * m);
  c->sc.delfree = (align_type == AADP_LOCAL || align_type == AADP_SEMI_LOCAL || align_type == AADP_LOCAL_GLOBAL);
  c->sc.insfree = (align_type == AADP_LOCAL || align_type == AADP_SEMI_LOCAL || align_type == AADP_GLOBAL_LOCAL);
  c->sc.local = (align_type == AADP_LOCAL);
  c->sc.scale_log2 = s;
  c->align_type = align_type;
  c->flags = flags;
  c->gi_f = gi;
  c->ge_f = ge;
  c->b.ran_what = 0;
  c->b.sched_ok = false;  // as aadp_set_scoring: classification, bounds and storage modes depend on the scoring
  if (c->b.seq_A != A) c->b.have_seqs = false;
  c->have_scoring = true;
  return 0;
}

// ---- the two halves of an upload.  Both only ENQUEUE work on the context stream (the pinned pool must
// have been reserved by the caller) and leave the synchronisation to the caller.
// npieces > 1 (aadp_fill_batch): the residues travel in pieces of consecutive sequences on a separate copy stream,
// each followed by its part of the arena build and an event; the compute stream only waits for the piece a
// chunk of pairs actually references, so the first kernels run while the rest of the residues are still in flight.
static int upload_sequences_impl(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq, int npieces = 1) {
  Batch& b = c->b;
  b.nseq = nseq;
  b.seq_off.assign(seq_off, seq_off + nseq + 1);
  const int64_t nres = seq_off[nseq];
  // aligned arena offsets (16-byte aligned sequences, zero padding absorbs read-ahead)
  b.aoff.assign(nseq + 1, 0);
  int64_t cur = 0, maxL = 0;
  for (int64_t s2 = 0; s2 < nseq; ++s2) {
    const int64_t L = seq_off[s2 + 1] - seq_off[s2];
    if (L < 0) return fail("sequence offsets must be non-decreasing");
    if (cur > 0x7fff0000LL) return fail("sequence arena too large");
    b.aoff[s2] = (int32_t)cur;
    maxL = std::max(maxL, L);
    cur += (L + 15) / 16 * 16;
  }
  const size_t arena_bytes = (size_t)(cur + maxL + 128);
  if (!c->pin_flag && cudaHostAlloc((void**)&c->pin_flag, 64, cudaHostAllocDefault) != cudaSuccess) return fail("cudaHostAlloc failed");
  if (c->residues.reserve(std::max<size_t>(nres, 16))) return 1;
  if (c->arena_f.reserve(arena_bytes) || c->arena_r.reserve(arena_bytes) || c->badflag.reserve(16)) return 1;
  c->h2d_bytes += nres;
  c->d2h_bytes += 4;
  if (!c->ev_flag) CK(cudaEventCreateWithFlags(&c->ev_flag, cudaEventDisableTiming));
  npieces = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(npieces, 8), nres >> 22));  // >= 4 MB per piece
  b.piece_end.clear();
  cudaStream_t cs = c->stream;
  if (npieces > 1) {
    if (!c->copy_stream) CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int j = 0; j < npieces; ++j)
      if (!c->ev_piece[j]) CK(cudaEventCreateWithFlags(&c->ev_piece[j], cudaEventDisableTiming));
    if (!c->ev_start) CK(cudaEventCreateWithFlags(&c->ev_start, cudaEventDisableTiming));
    // the copy stream may not touch the buffers before earlier work of the compute stream is done with them
    CK(cudaEventRecord(c->ev_start, c->stream));
    cs = c->copy_stream;
    CK(cudaStreamWaitEvent(cs, c->ev_start, 0));
  }
  if (upload_vec(c, c->seq_off, b.seq_off, cs, true)) return 1;
  if (upload_vec(c, c->aoff, b.aoff, cs, true)) return 1;
  CK(cudaMemsetAsync(c->arena_f.p, 0, arena_bytes, cs));
  CK(cudaMemsetAsync(c->arena_r.p, 0, arena_bytes, cs));
  CK(cudaMemsetAsync(c->badflag.p, 0, 16, cs));
  int64_t s_begin = 0;
  for (int j = 0; j < npieces; ++j) {
    // piece j: sequences [s_begin, s_end) holding about 1/npieces of the residues
    int64_t s_end = nseq;
    if (j + 1 < npieces) {
      const int64_t target = nres * (j + 1) / npieces;
      s_end = std::upper_bound(seq_off, seq_off + nseq + 1, target) - seq_off - 1;
      s_end = std::max(s_begin, std::min(s_end, nseq));
    }
    const int64_t r0 = seq_off[s_begin], r1 = seq_off[s_end];
    if (r1 > r0) CK(cudaMemcpyAsync(c->residues.as<uint8_t>() + r0, residues + r0, (size_t)(r1 - r0), cudaMemcpyHostToDevice, cs));
    if (s_end > s_begin) {
      const int grid = (int)std::min<int64_t>(s_end - s_begin, 148 * 32);
      arena_kernel<<<grid, 128, 0, cs>>>(c->residues.as<uint8_t>(), c->seq_off.as<int64_t>(), c->aoff.as<int32_t>(), s_begin, s_end,
                                         c->sc.A, c->arena_f.as<uint8_t>(), c->arena_r.as<uint8_t>(), c->badflag.as<int>());
      CK(cudaGetLastError());
    }
    if (npieces > 1) CK(cudaEventRecord(c->ev_piece[j], cs));
    b.piece_end.push_back(s_end);
    s_begin = s_end;
  }
  CK(cudaMemcpyAsync(c->pin_flag, c->badflag.p, 4, cudaMemcpyDeviceToHost, cs));
  CK(cudaEventRecord(c->ev_flag, cs));
  b.have_seqs = true;
  b.seq_A = c->sc.A;
  return 0;
}

// Makes the compute stream wait for the residue pieces that hold every sequence up to `max_seq` (no-op when the
// sequences were uploaded on the compute stream itself).
static int wait_for_sequences(aadp_ctx* c, int64_t max_seq) {
  Batch& b = c->b;
  if (b.piece_end.size() <= 1) return 0;
  size_t j = 0;
  while (j + 1 < b.piece_end.size() && b.piece_end[j] <= max_seq) ++j;
  for (size_t k = b.piece_waited; k <= j; ++k) CK(cudaStreamWaitEvent(c->stream, c->ev_piece[k], 0));
  b.piece_waited = std::max(b.piece_waited, j + 1);
  return 0;
}

static size_t pairs_pin_bytes(int64_t npairs) { return (size_t)npairs * (8 + 1 + 4 + 24 + 64 * 4 / 2 + 64) + 65536; }

// pair list -> classification, product sizes, packed task list, and their uploads.  With nsplit > 1 the task
// list is built in chunks of consecutive pair ids and on_chunk(k) runs right after chunk k is enqueued for
// upload -- aadp_fill_batch launches the forward kernel of chunk k there, so the GPU works on it while the host
// schedules chunk k+1.
static int set_pairs_impl(aadp_ctx* c, const int32_t* pair_q, const int32_t* pair_t, int64_t npairs, uint32_t what,
                          int nsplit = 1, const std::function<int(size_t)>* on_chunk = nullptr) {
  Batch& b = c->b;
  b.sched_ok = false;
  b.npairs = npairs;
  b.pair_q.assign(pair_q, pair_q + npairs);
  b.pair_t.assign(pair_t, pair_t + npairs);
  if (c->float_mode) {  // exact general-gap path: no packed schedule, no resident products
    b.cells = 0;
    b.n_tasks = 0;
    b.tb_off.clear();
    for (int64_t p = 0; p < npairs; ++p) {
      const int qs = b.pair_q[p], ts = b.pair_t[p];
      if (qs < 0 || qs >= b.nseq || ts < 0 || ts >= b.nseq) return fail("pair index out of range");
      b.cells += (double)(b.seq_off[qs + 1] - b.seq_off[qs]) * (double)(b.seq_off[ts + 1] - b.seq_off[ts]);
    }
    b.uploaded_what = what;
    b.ran_what = 0;
    if (upload_vec(c, c->pair_q, b.pair_q)) return 1;
    if (upload_vec(c, c->pair_t, b.pair_t)) return 1;
    b.sched_ok = true;
    return 0;
  }
  b.sched_ok = false;
  if (build_batch_meta(c, what)) return 1;
  g_marks.mark("meta");
  b.uploaded_what = what;
  b.ran_what = 0;
  if (upload_vec(c, c->fmt, b.fmt)) return 1;
  if (upload_vec(c, c->pair_q, b.pair_q)) return 1;
  if (upload_vec(c, c->pair_t, b.pair_t)) return 1;
  if (upload_vec(c, c->order[0], b.order[0])) return 1;
  if (upload_vec(c, c->order[1], b.order[1])) return 1;
  if (upload_vec(c, c->tb_off, b.tb_off)) return 1;
  if (upload_vec(c, c->sc_off, b.sc_off)) return 1;
  if (upload_vec(c, c->mask_off, b.mask_off)) return 1;
  // packed task list: at most one task per couple, one unpaired couple per lane width, host range and chunk
  nsplit = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(nsplit, 7), npairs / 16384));
  if (c->tasks.reserve(((size_t)npairs / 2 + (size_t)33 * 8 * nsplit + 64) * 64 * sizeof(int32_t))) return 1;
  for (int k = 0; k < nsplit; ++k) {
    // the first chunk is the smallest: its kernel should start as early as possible
    const int64_t lo = k == 0 ? 0 : npairs * (2 * k - 1) / (2 * nsplit - 1), hi = npairs * (2 * k + 1) / (2 * nsplit - 1);
    int32_t* tasks_pinned = nullptr;
    int64_t nt = 0;
    if (build_task_chunk(c, lo, std::min(hi, npairs), &tasks_pinned, &nt)) return 1;
    g_marks.mark("tasks");
    const size_t bytes = (size_t)nt * 64 * sizeof(int32_t);
    if (bytes)
      CK(cudaMemcpyAsync(c->tasks.as<int32_t>() + b.chunk_first[(size_t)k] * 64, tasks_pinned, bytes, cudaMemcpyHostToDevice, c->stream));
    c->h2d_bytes += (int64_t)bytes;
    if (k == 0) b.sched_ok = true;  // on_chunk launches from this schedule
    if (on_chunk && (*on_chunk)((size_t)k)) return 1;
  }
  b.sched_ok = true;
  return 0;
}

int aadp_upload_batch(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq, const int32_t* pair_q,
                      const int32_t* pair_t, int64_t npairs, uint32_t what) {
  if (check_ctx(c, true)) return 1;
  if (nseq < 0 || npairs < 0 || npairs > 0x7fffffff) return fail("bad batch size");
  if (!seq_off || (npairs && (!pair_q || !pair_t))) return fail("null input");
  if (seq_off[0] < 0) return fail("sequence offsets must start at a non-negative offset");
  if (nseq && !residues && seq_off[nseq] > seq_off[0]) return fail("null input");
  if ((what & AADP_W_MASK) && (what & (AADP_W_FWD | AADP_W_REV)) != (AADP_W_FWD | AADP_W_REV))
    return fail("AADP_W_MASK needs both AADP_W_FWD and AADP_W_REV");
  const auto t_begin = std::chrono::steady_clock::now();
  Batch& b = c->b;
  if (pin_reserve(c, (size_t)(nseq + 1) * 12 + pairs_pin_bytes(npairs))) return 1;
  c->h2d_bytes = 0;
  c->d2h_bytes = 0;
  // 1. start the big transfer and the device-side arena build / validation first ...
  if (upload_sequences_impl(c, residues, seq_off, nseq)) return 1;
  // 2. ... and build the schedule on the host while they run
  const auto t_meta0 = std::chrono::steady_clock::now();
  if (set_pairs_impl(c, pair_q, pair_t, npairs, what)) return 1;
  const auto t_up = std::chrono::steady_clock::now();
  CK(cudaStreamSynchronize(c->stream));  // the caller may reuse its buffers; the validation flag is back
  if (getenv("AADP_TIMING")) {
    const auto t_end = std::chrono::steady_clock::now();
    auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
      return std::chrono::duration<double, std::milli>(b - a).count();
    };
    fprintf(stderr, "[aadp] upload: sequences %.2f ms, schedule+stage %.2f ms, drain %.2f ms (tasks %lld)\n",
            ms(t_begin, t_meta0), ms(t_meta0, t_up), ms(t_up, t_end), (long long)b.n_tasks);
  }
  if (*c->pin_flag) { b.have_seqs = false; return fail("residue code outside the substitution alphabet"); }
  return 0;
}

int aadp_upload_sequences(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq) {
  return aadp_upload_batch(c, residues, seq_off, nseq, nullptr, nullptr, 0, 0);
}

// ---- cross mode: every query of a list against every template of a list, forward score only ----------
__global__ void scatter_scores_kernel(const float* __restrict__ src, const int32_t* __restrict__ qi,
                                      const int32_t* __restrict__ ti, int64_t n, int64_t nt, float* __restrict__ dst) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[(int64_t)qi[i] * nt + ti[i]] = src[i];
}

int aadp_cross_run(aadp_ctx* c, const int32_t* q_ids, int64_t nq, const int32_t* t_ids, int64_t nt, float* d_scores) {
  if (check_ctx(c, true)) return 1;
  Batch& b = c->b;
  if (!b.have_seqs) return fail("aadp_cross_run: no resident sequences (call aadp_upload_sequences first)");
  if (nq < 0 || nt < 0 || nq > 0x7fffffff || nt > 0x7fffffff) return fail("bad list size");
  if ((nq && !q_ids) || (nt && !t_ids) || (nq && nt && !d_scores)) return fail("null argument");
  c->launches = 0;
  c->x_cells = 0;
  if (nq == 0 || nt == 0) return 0;
  auto len = [&](int32_t s2) { return b.seq_off[(size_t)s2 + 1] - b.seq_off[(size_t)s2]; };
  for (int64_t i = 0; i < nq; ++i) if (q_ids[i] < 0 || q_ids[i] >= b.nseq) return fail("query id out of range");
  for (int64_t i = 0; i < nt; ++i) if (t_ids[i] < 0 || t_ids[i] >= b.nseq) return fail("template id out of range");
  if (c->prof_mode) {
    if (profile_count_refusal(c, b.nseq)) return 1;
    for (int64_t i = 0; i < nt; ++i)
      if (c->prof_len[(size_t)t_ids[i]] != len(t_ids[i]) * c->sc.A) return profile_refusal(c, t_ids[i], len(t_ids[i]));
  }
  // ---- which templates / queries qualify for the packed int16x2 kernel (same rules as build_batch_meta)
  const bool packed_mode = c->allow_packed && !c->float_mode && !c->sc.local && c->sc.ge <= 400 && c->sc.gi <= 2048;
  std::vector<int32_t> te, qe, tbad, qbad;  // LIST indices
  int64_t maxLt = 0;
  int64_t mx = c->max_abs_sub;  // |similarity| bound; profile scoring: the largest of the packed templates of this call
  for (int64_t i = 0; i < nt; ++i) {
    const int64_t L = len(t_ids[i]);
    if (packed_mode && L >= 1 && L <= 512) {
      te.push_back((int32_t)i);
      maxLt = std::max(maxLt, L);
      if (c->prof_mode) mx = std::max<int64_t>(mx, c->prof_max[(size_t)t_ids[i]]);
    }
    else tbad.push_back((int32_t)i);
  }
  for (int64_t i = 0; i < nq; ++i) {
    const int64_t L = len(q_ids[i]);
    const int64_t bd = std::min(L, maxLt) * mx + 2 * (int64_t)c->sc.gi + (int64_t)c->sc.ge * (L + maxLt);
    if (!te.empty() && L >= 1 && bd < kPackedBound) qe.push_back((int32_t)i);
    else qbad.push_back((int32_t)i);
  }
  CK(cudaStreamSynchronize(c->stream));  // the pinned staging pool may still feed an earlier upload
  if (pin_reserve(c, (size_t)(nq + nt) * 16 + (size_t)nt * 32 * 4 + 65536)) return 1;
  if (!qe.empty()) {
    // templates: best-fit decreasing by lane width into 32-lane layouts
    std::vector<int32_t> layouts;
    {
      std::vector<std::vector<int32_t>> byn(33);
      for (int32_t i : te) byn[(size_t)((len(t_ids[i]) + 15) / 16)].push_back(i);
      std::vector<std::vector<int32_t>> open(33);  // open[u] = layouts with u lanes in use
      int64_t nlay = 0;
      for (int n = 32; n >= 1; --n)
        for (int32_t i : byn[(size_t)n]) {
          int u = 32 - n;
          while (u > 0 && open[(size_t)u].empty()) --u;
          int64_t lay;
          if (u > 0) { lay = open[(size_t)u].back(); open[(size_t)u].pop_back(); }
          else { lay = nlay++; layouts.resize(layouts.size() + 32, -1); }
          for (int l = 0; l < n; ++l) layouts[(size_t)lay * 32 + u + l] = i;
          if (u + n < 32) open[(size_t)(u + n)].push_back((int32_t)lay);
        }
    }
    const int64_t nlay = (int64_t)layouts.size() / 32;
    // queries: longest first, adjacent ones share a register (couple); an odd one out is paired with itself
    std::stable_sort(qe.begin(), qe.end(), [&](int32_t x, int32_t y) { return len(q_ids[x]) > len(q_ids[y]); });
    std::vector<int32_t> qc;
    for (size_t i = 0; i < qe.size(); i += 2) { qc.push_back(qe[i]); qc.push_back(i + 1 < qe.size() ? qe[i + 1] : qe[i]); }
    const int64_t nqc = (int64_t)qc.size() / 2;
    std::vector<int32_t> qid(q_ids, q_ids + nq), tid(t_ids, t_ids + nt);
    if (upload_vec(c, c->x_layout, layouts) || upload_vec(c, c->x_qc, qc) || upload_vec(c, c->x_qid, qid) ||
        upload_vec(c, c->x_tid, tid)) return 1;
    const bool pro = c->prof_mode;
    const void* kern = pro ? (const void*)packed_kernel<0, 0, 0, 1, 0, 1> : (const void*)packed_kernel<0, 0, 0, 1, 0, 0>;
    const int A = c->sc.A;
    const size_t smem = packed_smem_bytes(A, 0, 1);
    CK(cached_max_smem((const void*)kern, (size_t)(smem)));
    int occ = 0;
    CK(cached_occupancy(&occ, (const void*)kern, kPackedWarps * 32, smem));
    if (occ < 1) return fail("packed kernel does not fit on an SM");
    const int64_t resident = (int64_t)c->num_sms * occ;
    // query couples per item: reuse the template profile as often as possible while keeping >= 8 items per warp
    int64_t group = std::max<int64_t>(1, std::min<int64_t>(8, nlay * nqc / (8 * resident)));
    const int64_t ngroups = (nqc + group - 1) / group;
    if (nlay * ngroups > 0x7fffffffLL) return fail("aadp_cross_run: too many work items; split the lists into blocks");
    PackedParams Q{};
    Q.sc = c->sc;
    Q.sub8 = c->sub8.as<int8_t>();
    Q.sub8p = c->sub8p.as<int8_t>();
    Q.arena = c->arena_f.as<uint8_t>();
    Q.aoff = c->aoff.as<int32_t>();
    Q.seq_off = c->seq_off.as<int64_t>();
    Q.n_tasks = (int)(nlay * ngroups);
    Q.rev = 0;
    if (c->counter.reserve(64)) return 1;
    CK(cudaMemsetAsync(c->counter.p, 0, 64, c->stream));
    Q.counter = c->counter.as<unsigned int>() + 8;
    Q.x_layout = c->x_layout.as<int32_t>();
    Q.x_qc = c->x_qc.as<int32_t>();
    Q.x_qid = c->x_qid.as<int32_t>();
    Q.x_tid = c->x_tid.as<int32_t>();
    Q.x_nlayouts = (int)nlay;
    Q.x_nqc = (int)nqc;
    Q.x_group = (int)group;
    Q.x_nt = nt;
    Q.x_scores = d_scores;
    double sq = 0, st = 0;
    for (int32_t i : qe) sq += (double)len(q_ids[i]);
    for (int32_t i : te) st += (double)len(t_ids[i]);
    Q.cells_hint = sq * st;
    c->x_cells += sq * st;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(resident, Q.n_tasks));
    c->prof_begin(pro ? "packed_kernel<TB=0,FST=0,MSK=0,XM=1,PRO=1>fwd" : "packed_kernel<TB=0,FST=0,MSK=0,XM=1>fwd", Q.cells_hint);
    Q.prof = c->prof_dev();
    if (pro) packed_kernel<0, 0, 0, 1, 0, 1><<<grid, kPackedWarps * 32, smem, c->stream>>>(Q);
    else packed_kernel<0, 0, 0, 1, 0, 0><<<grid, kPackedWarps * 32, smem, c->stream>>>(Q);
    c->prof_end();
    CK(cudaGetLastError());
    c->launches++;
  }
  // ---- everything else (long / empty sequences, local mode, scores beyond the int16 bound): explicit pair
  // lists through the general batch path, scattered into the matrix.  This replaces the resident pair batch.
  if (!qbad.empty() || !tbad.empty()) {
    std::vector<int32_t> pq, pt, lq, lt;
    const int64_t chunk = 1 << 20;
    auto flush = [&]() -> int {
      if (pq.empty()) return 0;
      const int64_t n = (int64_t)pq.size();
      CK(cudaStreamSynchronize(c->stream));
      if (pin_reserve(c, pairs_pin_bytes(n) + (size_t)n * 8)) return 1;
      const int64_t launches = c->launches;
      if (set_pairs_impl(c, pq.data(), pt.data(), n, AADP_W_FWD)) return 1;
      if (c->fscore[0].reserve((size_t)n * 4)) return 1;
      if (aadp_run_batch(c, AADP_W_FWD, 0.f, c->fscore[0].as<float>(), nullptr, nullptr, nullptr)) return 1;
      if (upload_vec(c, c->x_qc, lq) || upload_vec(c, c->x_layout, lt)) return 1;
      scatter_scores_kernel<<<(int)std::min<int64_t>((n + 255) / 256, 148 * 8), 256, 0, c->stream>>>(
          c->fscore[0].as<float>(), c->x_qc.as<int32_t>(), c->x_layout.as<int32_t>(), n, nt, d_scores);
      CK(cudaGetLastError());
      c->launches += launches + 1;
      c->x_cells += b.cells;
      pq.clear(); pt.clear(); lq.clear(); lt.clear();
      return 0;
    };
    auto add = [&](int32_t qi, int32_t ti) -> int {
      pq.push_back(q_ids[qi]); pt.push_back(t_ids[ti]); lq.push_back(qi); lt.push_back(ti);
      return (int64_t)pq.size() >= chunk ? flush() : 0;
    };
    for (int32_t qi : qbad) for (int64_t ti = 0; ti < nt; ++ti) if (add(qi, (int32_t)ti)) return 1;
    for (int32_t qi : qe) for (int32_t ti : tbad) if (add(qi, ti)) return 1;
    if (flush()) return 1;
  }
  return 0;
}

int aadp_cross_scores(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq, const int32_t* q_ids,
                      int64_t nq, const int32_t* t_ids, int64_t nt, float* scores) {
  if (aadp_upload_sequences(c, residues, seq_off, nseq)) return 1;
  const int64_t h2d = c->h2d_bytes;
  if (nq <= 0 || nt <= 0) return (nq < 0 || nt < 0) ? fail("bad list size") : 0;
  if (!scores) return fail("null argument");
  if (c->x_scores.reserve((size_t)nq * nt * 4)) return 1;
  if (aadp_cross_run(c, q_ids, nq, t_ids, nt, c->x_scores.as<float>())) return 1;
  CK(cudaMemcpyAsync(scores, c->x_scores.p, (size_t)nq * nt * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->h2d_bytes += h2d;
  c->d2h_bytes += nq * nt * 4;
  return 0;
}

// ---- exact general-gap fp32 path (aadp_general.cuh) ------------------------------------------------
// Fills the n consecutive pairs [p0, p0+n) of the batch in the directions of `dirmask` (bit 0 forward,
// bit 1 reverse) into the dense scratch matrices of the context.  off = n+1 cell offsets of the pairs.
// Scoring override of one general-gap launch (aadp_fill_pair_general): a dense similarity matrix from any
// Evaluator plus the uniform affine gap model, instead of the context's substitution table.
struct GeneralOverride {
  float gi, ge;
  int align_type;
  uint32_t flags;
  const float* d_sim;
  // tabulated gap model (aadp_fill_pair_tabulated); null = the affine model above
  const float* d_del;
  const float* d_delT;
  const float* d_ins;
  int tab_local;
  const int64_t* d_del_off;  // batches of tabulated pairs: per-item table offsets (device), or null
  const int64_t* d_ins_off;
};

static int gg_fill(aadp_ctx* c, int64_t p0, int64_t n, int dirmask, bool tb, const std::vector<int64_t>& off,
                   float* d_fin_fwd, float* d_fin_rev, const int* rect = nullptr, const GeneralOverride* ov = nullptr,
                   bool compact = false, const int64_t* ids = nullptr) {
  // ids != nullptr: the n items are the listed pairs ids[0..n) instead of the consecutive pairs p0..p0+n
  Batch& b = c->b;
  const int64_t cells = off[(size_t)n];
  // What the kernels keep per item in shared memory is indexed by flow column (at most nt, the interior columns) and by
  // gap length (at most max(nq, nt)): for a whole matrix nt = Lt and nq = Lq, for a sub-rectangle only the rectangle
  // counts, however long its sequences are.  The widest item picks the kernel, its variant and the shared memory.
  int maxNt = 0, maxLen = 0;
  for (int64_t k = 0; k < n; ++k) {
    int nq, nt;
    if (rect) {
      nq = rect[4 * k + 2] - rect[4 * k] - 1;
      nt = rect[4 * k + 3] - rect[4 * k + 1] - 1;
    } else {
      const int64_t p = ids ? ids[k] : p0 + k;
      const int qs = b.pair_q[p], ts = b.pair_t[p];
      nq = (int)(b.seq_off[qs + 1] - b.seq_off[qs]);
      nt = (int)(b.seq_off[ts + 1] - b.seq_off[ts]);
    }
    maxNt = std::max(maxNt, nt);
    maxLen = std::max(maxLen, std::max(nq, nt));
  }
  const size_t smem = (size_t)(2 * (maxNt + 2) + maxLen + 2 + 32) * sizeof(float);
  if (smem > 220 * 1024) return fail("exact general-gap path: sequences too long for the shared-memory row and penalty tables");
  // the pruned scans (prefix maxima + binary searches) only pay off when the scans are long
  int longest = maxLen;
  if (rect) {
    longest = 1;
    for (int64_t k = 0; k < n; ++k)
      longest = std::max(longest, std::max(rect[4 * k + 2] - rect[4 * k], rect[4 * k + 3] - rect[4 * k + 1]));
  }
  const bool prune_pays = longest >= 96;
  // record-list kernel (aadp_frec.cuh): affine gaps only; one warp per (pair, direction), rows and column leaders in
  // shared memory, 16-bit flow row/column indices, at most 64 key columns per lane
  const int rec_cap = frec_cap(maxNt);
  const bool use_rec = c->gg_records && !(ov && ov->d_del) && maxLen < 32000 && maxNt <= 2048 && frec_smem_bytes(rec_cap) <= 200 * 1024;
  GeneralParams G{};
  G.max_nt = maxNt;
  G.max_len = maxLen;
  G.A = c->sc.A;
  G.subf = c->subf.as<float>();
  G.gi = c->gi_f;
  G.ge = c->ge_f;
  G.delfree = c->sc.delfree;
  G.insfree = c->sc.insfree;
  G.local = c->sc.local;
  G.repro_rev_bug = (c->flags & AADP_REPRO_REV_BUG) ? 1 : 0;
  if (ov) {
    G.gi = ov->gi;
    G.ge = ov->ge;
    G.delfree = (ov->align_type == AADP_LOCAL || ov->align_type == AADP_SEMI_LOCAL || ov->align_type == AADP_LOCAL_GLOBAL);
    G.insfree = (ov->align_type == AADP_LOCAL || ov->align_type == AADP_SEMI_LOCAL || ov->align_type == AADP_GLOBAL_LOCAL);
    G.local = ov->align_type == AADP_LOCAL;
    if (ov->flags & AADP_CLAMP_ON) G.local = 1;   // dpmatrix.h:155: the constructor's align_t, not the evaluator's
    if (ov->flags & AADP_CLAMP_OFF) G.local = 0;
    G.repro_rev_bug = (ov->flags & AADP_REPRO_REV_BUG) ? 1 : 0;
    G.simov = ov->d_sim;
    G.A = 1;
    if (ov->d_del) {
      G.del_tab = ov->d_del;
      G.del_tabT = ov->d_delT;
      G.ins_tab = ov->d_ins;
      G.del_off = ov->d_del_off;
      G.ins_off = ov->d_ins_off;
      G.delfree = G.insfree = 0;  // free end gaps are whatever the tables say
      G.local = ov->tab_local;
    }
  }
  const bool tab = ov && ov->d_del;
  G.residues = c->residues.as<uint8_t>();
  G.seq_off = c->seq_off.as<int64_t>();
  G.pair_q = c->pair_q.as<int32_t>();
  G.pair_t = c->pair_t.as<int32_t>();
  G.items = nullptr;
  G.item0 = (int)p0;
  int nd = 0;
  for (int d = 0; d < 2; ++d) {
    if (!(dirmask & (1 << d))) continue;
    if (c->gg_score[d].reserve(std::max<size_t>((size_t)cells * 4, 16))) return 1;
    if (tb && (c->gg_pq[d].reserve(std::max<size_t>((size_t)cells * 4, 16)) || c->gg_pt[d].reserve(std::max<size_t>((size_t)cells * 4, 16)))) return 1;
    G.dirs[nd] = d;
    G.score[nd] = c->gg_score[d].as<float>();
    G.prevq[nd] = tb ? c->gg_pq[d].as<int32_t>() : nullptr;
    G.prevt[nd] = tb ? c->gg_pt[d].as<int32_t>() : nullptr;
    G.fin[nd] = d ? d_fin_rev : d_fin_fwd;
    G.pmcol[nd] = nullptr;
    if (use_rec || (c->gg_prune && prune_pays && !(ov && ov->d_del) && G.gi >= 0.f && G.ge >= 0.f)) {  // the pruning needs pen(len) to grow with len; the record kernel keeps its column links here
      if (c->gg_pm[d].reserve(std::max<size_t>((size_t)cells * 4, 16))) return 1;
      G.pmcol[nd] = c->gg_pm[d].as<float>();
    }
    ++nd;
  }
  if (nd == 0) return 0;
  CK(cudaStreamSynchronize(c->stream));  // the pinned pool may still feed an earlier copy
  if (pin_reserve(c, (size_t)(n + 1) * 8 + (rect ? (size_t)n * 16 : 0) + (ids ? (size_t)n * 4 : 0) + 4096)) return 1;
  if (upload_vec(c, c->gg_off, off)) return 1;
  G.dense_off = c->gg_off.as<int64_t>();
  if (ids) {
    std::vector<int32_t> it32((size_t)n);
    for (int64_t k = 0; k < n; ++k) it32[(size_t)k] = (int32_t)ids[k];
    if (upload_vec(c, c->gg_items, it32)) return 1;
    G.items = c->gg_items.as<int32_t>();
  }
  if (rect) {  // build_subdpm: one rectangle per item of this launch (4 ints each)
    std::vector<int32_t> r(rect, rect + 4 * n);
    if (upload_vec(c, c->gg_rect, r)) return 1;
    G.rects = c->gg_rect.as<int4>();
  }
  G.compact = compact ? 1 : 0;      // compact batches (aadp_fill_subpair_batch) keep only the rectangles and
  G.fin_by_item = compact ? 1 : 0;  // index the final scores by item: several items may share one pair
  const int width = rect ? std::max(1, maxNt) : maxNt;  // threads own columns: of the matrix, or of the widest rectangle
  double cu = 0;
  if (rect) {
    for (int64_t k = 0; k < n; ++k)
      cu += (double)(rect[4 * k + 2] - rect[4 * k] - 1) * (double)(rect[4 * k + 3] - rect[4 * k + 1] - 1);
  } else {
    for (int64_t k = 0; k < n; ++k) {
      const int64_t p = ids ? ids[k] : p0 + k;
      const int qs = b.pair_q[p], ts = b.pair_t[p];
      cu += (double)(b.seq_off[qs + 1] - b.seq_off[qs]) * (double)(b.seq_off[ts + 1] - b.seq_off[ts]);
    }
  }
  // few CTAs (single pairs): latency counts, one column per thread; many CTAs: smaller CTAs hide each other's barriers
  const int tcap = n * nd < 296 ? 512 : c->gg_threads_cap;
  const int threads = std::max(compact ? 32 : 64, std::min(tcap, (width + 31) / 32 * 32));
  const bool wide = maxNt > 1024;  // record-list kernel: more than 32 key columns per lane
  static const char* const kFrecNames[2][2] = {{"frec_fill_kernel<TB=0>", "frec_fill_kernel<TB=0,WIDE=1>"},
                                               {"frec_fill_kernel<TB=1>", "frec_fill_kernel<TB=1,WIDE=1>"}};
  c->prof_begin(use_rec ? kFrecNames[tb][wide]
                        : tab ? "general_fill_kernel<TB=1,TAB=1>" : tb ? "general_fill_kernel<TB=1>" : "general_fill_kernel<TB=0>", cu * nd);
  if (use_rec) {
    // (measurement aid: AADP_FREC_SMEM_PAD extra bytes per warp lower the resident warps per SM)
    const size_t rsm = frec_smem_bytes(rec_cap) + (getenv("AADP_FREC_SMEM_PAD") ? (size_t)atoi(getenv("AADP_FREC_SMEM_PAD")) : 0);
    const dim3 grid((unsigned)n, (unsigned)nd);
#define AADP_FREC_LAUNCH(TB_, WIDE_)                                                      \
    do {                                                                                  \
      CK(cached_max_smem((const void*)frec_fill_kernel<TB_, WIDE_>, rsm));               \
      frec_fill_kernel<TB_, WIDE_><<<grid, 32, rsm, c->stream>>>(G, rec_cap);            \
    } while (0)
    if (tb) { if (wide) AADP_FREC_LAUNCH(1, 1); else AADP_FREC_LAUNCH(1, 0); }
    else { if (wide) AADP_FREC_LAUNCH(0, 1); else AADP_FREC_LAUNCH(0, 0); }
#undef AADP_FREC_LAUNCH
  } else if (tab) {
    CK(cached_max_smem((const void*)general_fill_kernel<1, 1>, (size_t)(std::max<size_t>(smem, 1024))));
    general_fill_kernel<1, 1><<<dim3((unsigned)n, (unsigned)nd), threads, smem, c->stream>>>(G);
  } else if (tb) {
    CK(cached_max_smem((const void*)general_fill_kernel<1>, (size_t)(std::max<size_t>(smem, 1024))));
    general_fill_kernel<1><<<dim3((unsigned)n, (unsigned)nd), threads, smem, c->stream>>>(G);
  } else {
    CK(cached_max_smem((const void*)general_fill_kernel<0>, (size_t)(std::max<size_t>(smem, 1024))));
    general_fill_kernel<0><<<dim3((unsigned)n, (unsigned)nd), threads, smem, c->stream>>>(G);
  }
  c->prof_end();
  CK(cudaGetLastError());
  c->launches++;
  return 0;
}

static int gg_mask(aadp_ctx* c, int64_t p0, int64_t n, float delta_ratio, const float* d_fin_fwd, bool dense_mask,
                   int64_t cells, float* d_threshold, int64_t* d_count, bool listed = false) {
  // listed: the items are the pairs gg_fill was given as a list (c->gg_items still holds them)
  GeneralMaskParams M{};
  M.A = c->sc.A;
  M.subf = c->subf.as<float>();
  M.residues = c->residues.as<uint8_t>();
  M.seq_off = c->seq_off.as<int64_t>();
  M.pair_q = c->pair_q.as<int32_t>();
  M.pair_t = c->pair_t.as<int32_t>();
  M.items = listed ? c->gg_items.as<int32_t>() : nullptr;
  M.item0 = (int)p0;
  M.dense_off = c->gg_off.as<int64_t>();
  M.F = c->gg_score[0].as<float>();
  M.R = c->gg_score[1].as<float>();
  M.fin_fwd = d_fin_fwd;
  M.delta_ratio = delta_ratio;
  if (dense_mask && c->gg_mask.reserve(std::max<size_t>((size_t)cells, 16))) return 1;
  M.mask = dense_mask ? c->gg_mask.as<uint8_t>() : nullptr;
  M.threshold = d_threshold;
  M.count = reinterpret_cast<long long*>(d_count);
  c->prof_begin("general_mask_kernel", 0);
  general_mask_kernel<<<(unsigned)n, 256, 0, c->stream>>>(M);
  c->prof_end();
  CK(cudaGetLastError());
  c->launches++;
  return 0;
}

// Batch run in exact-float mode: per-pair scalars only; the dense matrices live in scratch for the
// duration of a chunk (aadp_batch_fetch_pair recomputes the pair it is asked for).
static int gg_run_batch(aadp_ctx* c, uint32_t what, float delta_ratio, float* d_fwd_score, float* d_rev_score,
                        float* d_threshold, int64_t* d_nearopt_count) {
  Batch& b = c->b;
  const int64_t np = b.npairs;
  const int dirmask = ((what & AADP_W_FWD) ? 1 : 0) | ((what & AADP_W_REV) ? 2 : 0);
  float* ffwd = d_fwd_score;
  if ((what & AADP_W_MASK) && !ffwd) {
    if (c->gg_fin[0].reserve(std::max<size_t>((size_t)np * 4, 16))) return 1;
    ffwd = c->gg_fin[0].as<float>();
  }
  // Chunks of pairs of SIMILAR template length: the record-list kernel sizes its shared memory (and with it the warps
  // per SM) by the longest template of a launch, and a launch ends with its longest pair.  Results are per pair id.
  std::vector<int64_t> order((size_t)np);
  std::iota(order.begin(), order.end(), (int64_t)0);
  auto len_t = [&](int64_t p) { const int ts = b.pair_t[p]; return b.seq_off[ts + 1] - b.seq_off[ts]; };
  // (inside a shared-memory class the pairs with the most cells come first: the blocks of a launch start in this order)
  auto len_q = [&](int64_t p) { const int qs = b.pair_q[p]; return b.seq_off[qs + 1] - b.seq_off[qs]; };
  if (c->gg_records)
    std::stable_sort(order.begin(), order.end(), [&](int64_t x, int64_t y) {
      const int64_t cx = (len_t(x) + 63) / 64, cy = (len_t(y) + 63) / 64;
      if (cx != cy) return cx > cy;
      return len_q(x) * len_t(x) > len_q(y) * len_t(y);
    });
  std::vector<int64_t> off;
  for (int64_t p0 = 0; p0 < np;) {
    off.assign(1, 0);
    int64_t p1 = p0;
    const int64_t lt0 = len_t(order[(size_t)p0]);
    while (p1 < np) {
      const int64_t p = order[(size_t)p1];
      const int qs = b.pair_q[p], ts = b.pair_t[p];
      const int64_t cl = (b.seq_off[qs + 1] - b.seq_off[qs] + 2) * (b.seq_off[ts + 1] - b.seq_off[ts] + 2);
      if (p1 > p0 && off.back() + cl > c->gg_budget_cells) break;
      // a new launch when the templates have become a shared-memory class (64 columns) shorter -- but not for a handful of pairs
      if (c->gg_records && p1 - p0 >= 2048 && (lt0 + 63) / 64 != (len_t(p) + 63) / 64) break;
      off.push_back(off.back() + cl);
      ++p1;
    }
    if (gg_fill(c, 0, p1 - p0, dirmask, false, off, ffwd, d_rev_score, nullptr, nullptr, false, order.data() + p0)) return 1;
    if ((what & AADP_W_MASK) && gg_mask(c, 0, p1 - p0, delta_ratio, ffwd, false, off.back(), d_threshold, d_nearopt_count, true)) return 1;
    p0 = p1;
  }
  c->last_delta = delta_ratio;
  b.ran_what = what;
  return 0;
}

// Dense, reference-shaped matrices of pair p in exact-float mode (recomputed on demand).
static int gg_fetch_pair(aadp_ctx* c, int64_t p, float* score_fwd, int32_t* prevq_fwd, int32_t* prevt_fwd, float* score_rev,
                         int32_t* prevq_rev, int32_t* prevt_rev, uint8_t* nearopt) {
  Batch& b = c->b;
  const int qs = b.pair_q[p], ts = b.pair_t[p];
  const int64_t n = (b.seq_off[qs + 1] - b.seq_off[qs] + 2) * (b.seq_off[ts + 1] - b.seq_off[ts] + 2);
  int dirmask = ((score_fwd || prevq_fwd || prevt_fwd) ? 1 : 0) | ((score_rev || prevq_rev || prevt_rev) ? 2 : 0);
  if (nearopt) {
    if (!(b.ran_what & AADP_W_MASK)) return fail("near-optimal mask was not computed (run with AADP_W_MASK)");
    dirmask = 3;
  }
  if (!dirmask) return 0;
  std::vector<int64_t> off = {0, n};
  if (c->gg_fin[0].reserve(std::max<size_t>((size_t)b.npairs * 4, 16))) return 1;
  if (gg_fill(c, p, 1, dirmask, true, off, c->gg_fin[0].as<float>(), nullptr)) return 1;
  if (nearopt) {
    if (gg_mask(c, p, 1, c->last_delta, c->gg_fin[0].as<float>(), true, n, nullptr, nullptr)) return 1;
    CK(cudaMemcpyAsync(nearopt, c->gg_mask.p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  }
  if (score_fwd) CK(cudaMemcpyAsync(score_fwd, c->gg_score[0].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prevq_fwd) CK(cudaMemcpyAsync(prevq_fwd, c->gg_pq[0].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prevt_fwd) CK(cudaMemcpyAsync(prevt_fwd, c->gg_pt[0].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (score_rev) CK(cudaMemcpyAsync(score_rev, c->gg_score[1].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prevq_rev) CK(cudaMemcpyAsync(prevq_rev, c->gg_pq[1].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prevt_rev) CK(cudaMemcpyAsync(prevt_rev, c->gg_pt[1].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

}  // extern "C"

// Buffers and work counters of a run (everything the first kernel launch needs).
static int run_prepare(aadp_ctx* c, uint32_t what) {
  Batch& b = c->b;
  c->launches = 0;
  if (c->counter.reserve(256)) return 1;
  CK(cudaMemsetAsync(c->counter.p, 0, 256, c->stream));
  if ((what & AADP_W_MASK) && c->mask.reserve(std::max<size_t>((size_t)b.mask_off[b.npairs] * 4, 16))) return 1;
  if ((what & AADP_W_FWD) && reserve_direction(c, 0, what)) return 1;
  if ((what & AADP_W_REV) && reserve_direction(c, 1, what)) return 1;
  return 0;
}

// The launches of a run.  fwd_packed_done: run_prepare and the forward packed kernels of every chunk were already
// issued (interleaved with the host scheduling, aadp_fill_batch).
static int run_batch_impl(aadp_ctx* c, uint32_t what, float delta_ratio, float* d_fwd_score, float* d_rev_score,
                          float* d_threshold, int64_t* d_nearopt_count, bool fwd_packed_done) {
  Batch& b = c->b;
  const int64_t np = b.npairs;
  if (!fwd_packed_done && run_prepare(c, what)) return 1;
  if (what & AADP_W_MASK) c->last_delta = delta_ratio;  // the delta the resident near-optimal set belongs to
  const int threads = 256;
  const int g1 = (int)std::min<int64_t>((np + threads - 1) / threads, 148 * 8);
  if (what & AADP_W_FWD) {
    if (!fwd_packed_done && launch_packed_chunk(c, 0, what, delta_ratio, d_threshold, d_nearopt_count, kAllChunks)) return 1;
    if (run_direction_int32(c, 0, what)) return 1;
    if (d_fwd_score) {
      scores_to_float_kernel<<<g1, threads, 0, c->stream>>>(c->fin_score[0].as<int32_t>(), d_fwd_score, np, c->sc.scale_log2);
      CK(cudaGetLastError());
      c->launches++;
    }
  }
  if (what & AADP_W_REV) {
    if (launch_packed_chunk(c, 1, what, delta_ratio, d_threshold, d_nearopt_count, kAllChunks)) return 1;
    if (run_direction_int32(c, 1, what)) return 1;
    if (d_rev_score) {
      scores_to_float_kernel<<<g1, threads, 0, c->stream>>>(c->fin_score[1].as<int32_t>(), d_rev_score, np, c->sc.scale_log2);
      CK(cudaGetLastError());
      c->launches++;
    }
  }
  if (run_wave_pairs(c, what)) return 1;
  if (!b.wave_pairs.empty()) {  // their scalar outputs (the launches above came after the conversions)
    if ((what & AADP_W_FWD) && d_fwd_score) {
      scores_to_float_kernel<<<g1, threads, 0, c->stream>>>(c->fin_score[0].as<int32_t>(), d_fwd_score, np, c->sc.scale_log2);
      c->launches++;
    }
    if ((what & AADP_W_REV) && d_rev_score) {
      scores_to_float_kernel<<<g1, threads, 0, c->stream>>>(c->fin_score[1].as<int32_t>(), d_rev_score, np, c->sc.scale_log2);
      c->launches++;
    }
    CK(cudaGetLastError());
  }
  if ((what & AADP_W_MASK) && (!b.order[0].empty() || !b.order[1].empty() || !b.wave_pairs.empty())) {
    MaskParams M{};
    M.fmt = c->fmt.as<uint8_t>();
    M.want_fmt = 0;
    M.only_pair = -1;
    M.sc = c->sc;
    M.sub8 = c->sub8.as<int8_t>();
    M.residues = c->residues.as<uint8_t>();
    M.seq_off = c->seq_off.as<int64_t>();
    M.pair_q = c->pair_q.as<int32_t>();
    M.pair_t = c->pair_t.as<int32_t>();
    M.n_pairs = (int)np;
    M.st_mode = b.st_mode;
    M.scF = c->scb[0].p;
    M.scR = c->scb[1].p;
    M.sc_off = c->sc_off.as<int64_t>();
    M.fin_fwd = c->fin_score[0].as<int32_t>();
    M.delta_ratio = delta_ratio;
    M.mask = c->mask.as<uint32_t>();
    M.mask_off = c->mask_off.as<int64_t>();
    M.threshold = d_threshold;
    M.count = reinterpret_cast<long long*>(d_nearopt_count);
    if (!b.order[0].empty() || !b.order[1].empty()) {
      c->prof_begin(c->prof_mode ? "mask_kernel<PRO=1>" : "mask_kernel", 0);
      if (c->prof_mode) mask_kernel<1><<<(int)np, 256, 0, c->stream>>>(M, c->prof_dev());
      else mask_kernel<0><<<(int)np, 256, 0, c->stream>>>(M, c->prof_dev());
      c->prof_end();
      CK(cudaGetLastError());
      c->launches++;
    }
    for (int32_t p : b.wave_pairs) {  // long pairs: rows of one pair split over many blocks
      M.want_fmt = 2;
      M.only_pair = p;
      if (d_nearopt_count) CK(cudaMemsetAsync(d_nearopt_count + p, 0, 8, c->stream));
      c->prof_begin(c->prof_mode ? "mask_kernel<PRO=1>(long pair)" : "mask_kernel(long pair)", 0);
      if (c->prof_mode) mask_kernel<1><<<dim3(1, 2368), 256, 0, c->stream>>>(M, c->prof_dev());
      else mask_kernel<0><<<dim3(1, 2368), 256, 0, c->stream>>>(M, c->prof_dev());
      c->prof_end();
      CK(cudaGetLastError());
      c->launches++;
    }
  }
  b.ran_what = what;
  return 0;
}

extern "C" {

int aadp_run_batch(aadp_ctx* c, uint32_t what, float delta_ratio, float* d_fwd_score, float* d_rev_score,
                   float* d_threshold, int64_t* d_nearopt_count) {
  if (check_ctx(c, true)) return 1;
  Batch& b = c->b;
  if (!b.sched_ok || !b.have_seqs)
    return fail("aadp_run_batch: no valid resident batch (the batch must be uploaded again after aadp_set_scoring or "
                "after a single-pair / general-gap / tabulated call reused the context)");
  if ((what & ~b.uploaded_what) & (AADP_W_TB | AADP_W_SCORES | AADP_W_MASK))
    return fail("aadp_run_batch asks for products the batch was not uploaded for");
  if ((what & AADP_W_MASK) && (what & (AADP_W_FWD | AADP_W_REV)) != (AADP_W_FWD | AADP_W_REV))
    return fail("AADP_W_MASK needs both AADP_W_FWD and AADP_W_REV");
  if (!(what & (AADP_W_FWD | AADP_W_REV))) return fail("nothing to do: neither AADP_W_FWD nor AADP_W_REV");
  c->launches = 0;
  if (b.npairs == 0) { b.ran_what = what; return 0; }
  if (c->float_mode) return gg_run_batch(c, what, delta_ratio, d_fwd_score, d_rev_score, d_threshold, d_nearopt_count);
  return run_batch_impl(c, what, delta_ratio, d_fwd_score, d_rev_score, d_threshold, d_nearopt_count, false);
}

// wait = false (aadp_fill_batch_submit): everything is enqueued, the final synchronisation -- and, for batches of
// packed pairs only, the look at the residue validation flag -- is left to aadp_fill_batch_wait.
static int fill_batch_impl(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq, const int32_t* pair_q,
                           const int32_t* pair_t, int64_t npairs, uint32_t what, float delta_ratio, float* fwd_score,
                           float* rev_score, float* threshold, int64_t* nearopt_count, bool wait) {
  if (check_ctx(c, true)) return 1;
  if (nseq < 0 || npairs < 0 || npairs > 0x7fffffff) return fail("bad batch size");
  if (!seq_off || (npairs && (!pair_q || !pair_t))) return fail("null input");
  if (seq_off[0] < 0) return fail("sequence offsets must start at a non-negative offset");
  if (nseq && !residues && seq_off[nseq] > seq_off[0]) return fail("null input");
  if ((what & AADP_W_MASK) && (what & (AADP_W_FWD | AADP_W_REV)) != (AADP_W_FWD | AADP_W_REV))
    return fail("AADP_W_MASK needs both AADP_W_FWD and AADP_W_REV");
  if (!(what & (AADP_W_FWD | AADP_W_REV))) return fail("nothing to do: neither AADP_W_FWD nor AADP_W_REV");
  const size_t nb = std::max<size_t>((size_t)npairs * 4, 16);
  float *df = nullptr, *dr = nullptr, *dt = nullptr;
  int64_t* dc = nullptr;
  if (fwd_score) { if (c->fscore[0].reserve(nb)) return 1; df = c->fscore[0].as<float>(); }
  if (rev_score) { if (c->fscore[1].reserve(nb)) return 1; dr = c->fscore[1].as<float>(); }
  if (threshold) { if (c->thr.reserve(nb)) return 1; dt = c->thr.as<float>(); }
  if (nearopt_count) { if (c->count.reserve(nb * 2)) return 1; dc = c->count.as<int64_t>(); }
  Batch& b = c->b;
  const bool timing = getenv("AADP_TIMING") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto ms_since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
  double t_seq = 0, t_chunk[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t_launched = 0;
  // Large batches are pipelined: the packed task list is built in chunks and the forward kernel of a chunk is
  // launched as soon as its tasks are on their way, so the GPU computes while the host schedules the next chunk.
  const bool pipelined = !c->float_mode && npairs >= 32768 && (what & AADP_W_FWD) && c->pipeline_chunks > 1;
  if (!pipelined) {
    if (aadp_upload_batch(c, residues, seq_off, nseq, pair_q, pair_t, npairs, what)) return 1;
    if (npairs && aadp_run_batch(c, what, delta_ratio, df, dr, dt, dc)) return 1;
  } else {
    if (pin_reserve(c, (size_t)(nseq + 1) * 12 + pairs_pin_bytes(npairs))) return 1;
    c->h2d_bytes = 0;
    c->d2h_bytes = 0;
    b.piece_waited = 0;
    g_marks.start();
    if (upload_sequences_impl(c, residues, seq_off, nseq, 2 * c->pipeline_chunks)) return 1;
    g_marks.mark("seq");
    t_seq = ms_since();
    const std::function<int(size_t)> on_chunk = [&](size_t k) -> int {
      if (k == 0 && run_prepare(c, what)) return 1;
      g_marks.mark("prep");
      if (wait_for_sequences(c, b.chunk_max_seq[k])) return 1;  // only the residue pieces this chunk references
      const int rc = launch_packed_chunk(c, 0, what, delta_ratio, dt, dc, k);
      g_marks.mark("launch");
      if (k < 8) t_chunk[k] = ms_since();
      return rc;
    };
    if (set_pairs_impl(c, pair_q, pair_t, npairs, what, c->pipeline_chunks, &on_chunk)) return 1;
    if (wait_for_sequences(c, nseq)) return 1;  // everything that follows may read any sequence
    // the residue validation flag came back long ago (it was queued right after the arena kernel); the int32 and
    // wavefront kernels read the raw residues, so they are only launched on validated input
    g_marks.mark("sched");
    // the packed kernels read the device-built arenas, in which arena_kernel has replaced an invalid code by 0 (in-bounds
    // garbage that the flag voids afterwards); only the int32 / wavefront kernels index tables with raw residues
    const bool raw_readers = !b.order[0].empty() || !b.order[1].empty() || !b.wave_pairs.empty();
    c->flag_deferred = !wait && !raw_readers;
    if (!c->flag_deferred) {
      CK(cudaEventSynchronize(c->ev_flag));
      g_marks.mark("flag");
      if (*c->pin_flag) {
        CK(cudaStreamSynchronize(c->stream));
        b.have_seqs = false;
        return fail("residue code outside the substitution alphabet");
      }
    }
    if (run_batch_impl(c, what, delta_ratio, df, dr, dt, dc, true)) return 1;
    g_marks.mark("all");
    t_launched = ms_since();
  }
  if (npairs) {
    if (fwd_score && (what & AADP_W_FWD)) { CK(cudaMemcpyAsync(fwd_score, df, npairs * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += npairs * 4; }
    if (rev_score && (what & AADP_W_REV)) { CK(cudaMemcpyAsync(rev_score, dr, npairs * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += npairs * 4; }
    if (threshold && (what & AADP_W_MASK)) { CK(cudaMemcpyAsync(threshold, dt, npairs * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += npairs * 4; }
    if (nearopt_count && (what & AADP_W_MASK)) { CK(cudaMemcpyAsync(nearopt_count, dc, npairs * 8, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += npairs * 8; }
  }
  if (!wait) { c->pending = true; return 0; }
  CK(cudaStreamSynchronize(c->stream));
  if (timing && pipelined)
    fprintf(stderr, "[aadp] fill_batch host timeline (ms): sequences enqueued %.2f, fwd chunk launches %.2f %.2f %.2f, all launched %.2f, done %.2f\n",
            t_seq, t_chunk[0], t_chunk[1], t_chunk[2], t_launched, ms_since());
  if (timing && pipelined) fprintf(stderr, "[aadp] marks:%s\n", g_marks.log.c_str());
  return 0;
}

int aadp_fill_batch(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq, const int32_t* pair_q,
                    const int32_t* pair_t, int64_t npairs, uint32_t what, float delta_ratio, float* fwd_score,
                    float* rev_score, float* threshold, int64_t* nearopt_count) {
  return fill_batch_impl(c, residues, seq_off, nseq, pair_q, pair_t, npairs, what, delta_ratio, fwd_score, rev_score,
                         threshold, nearopt_count, true);
}

int aadp_fill_batch_submit(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq, const int32_t* pair_q,
                           const int32_t* pair_t, int64_t npairs, uint32_t what, float delta_ratio, float* fwd_score,
                           float* rev_score, float* threshold, int64_t* nearopt_count) {
  return fill_batch_impl(c, residues, seq_off, nseq, pair_q, pair_t, npairs, what, delta_ratio, fwd_score, rev_score,
                         threshold, nearopt_count, false);
}

int aadp_fill_batch_wait(aadp_ctx* c) {
  if (!c) return fail("null context");
  if (!c->pending) return 0;
  c->pending = false;
  if (check_ctx(c, false)) return 1;
  CK(cudaStreamSynchronize(c->stream));
  if (c->flag_deferred) {
    c->flag_deferred = false;
    CK(cudaEventSynchronize(c->ev_flag));
    if (*c->pin_flag) {
      c->b.have_seqs = false;
      c->b.ran_what = 0;
      return fail("residue code outside the substitution alphabet");
    }
  }
  return 0;
}

int64_t aadp_batch_resident_bytes(aadp_ctx* c, uint32_t which) {
  if (!c) return 0;
  const Batch& b = c->b;
  if (b.tb_off.empty() || c->float_mode) return 0;
  const int ndir = ((b.ran_what & AADP_W_FWD) ? 1 : 0) + ((b.ran_what & AADP_W_REV) ? 1 : 0);
  if (which == AADP_W_TB) return (b.ran_what & AADP_W_TB) ? b.tb_off[b.npairs] * ndir : 0;
  if (which == AADP_W_SCORES) {
    // score blobs that are really kept (reserve_direction): both directions with AADP_W_SCORES; with AADP_W_MASK alone the
    // forward one only -- the packed reverse pass fuses the near-optimal test and writes no scores -- unless int32 /
    // wavefront pairs need the reverse matrix for their separate mask pass
    const bool have_v1 = !b.order[0].empty() || !b.order[1].empty() || !b.wave_pairs.empty();
    int blobs = 0;
    for (int dir = 0; dir < 2; ++dir) {
      if (!(b.ran_what & (dir ? AADP_W_REV : AADP_W_FWD))) continue;
      if ((b.ran_what & AADP_W_SCORES) || ((b.ran_what & AADP_W_MASK) && (dir == 0 || have_v1))) ++blobs;
    }
    return b.sc_off[b.npairs] * 2 * blobs;
  }
  if (which == AADP_W_MASK) return (b.ran_what & AADP_W_MASK) ? b.mask_off[b.npairs] * 4 : 0;
  return 0;
}

int64_t aadp_last_launch_count(aadp_ctx* c) { return c ? c->launches : 0; }
int64_t aadp_last_h2d_bytes(aadp_ctx* c) { return c ? c->h2d_bytes : 0; }
int64_t aadp_last_d2h_bytes(aadp_ctx* c) { return c ? c->d2h_bytes : 0; }

int aadp_set_profiling(aadp_ctx* c, int on) {
  if (!c) return fail("null context");
  c->profiling = on != 0;
  c->prof.clear();  // (re)arming resets the log; runs append to it
  c->ev_used = 0;
  return 0;
}

int aadp_profile_count(aadp_ctx* c) { return c ? (int)c->prof.size() : 0; }

int aadp_profile_get(aadp_ctx* c, int idx, char* name, int name_cap, float* ms, double* cells) {
  if (check_ctx(c, false)) return 1;
  if (idx < 0 || idx >= (int)c->prof.size()) return fail("profile index out of range");
  const aadp_ctx::Prof& p = c->prof[idx];
  CK(cudaEventSynchronize(p.e1));
  float t = 0.f;
  CK(cudaEventElapsedTime(&t, p.e0, p.e1));
  if (ms) *ms = t;
  if (cells) *cells = p.cells;
  if (name && name_cap > 0) { strncpy(name, p.name.c_str(), name_cap - 1); name[name_cap - 1] = 0; }
  return 0;
}

double aadp_last_cross_cell_updates(aadp_ctx* c) { return c ? c->x_cells : 0; }

double aadp_last_cell_updates(aadp_ctx* c) {
  if (!c) return 0;
  const int ndir = ((c->b.ran_what & AADP_W_FWD) ? 1 : 0) + ((c->b.ran_what & AADP_W_REV) ? 1 : 0);
  return c->b.cells * ndir;
}

int aadp_batch_fetch_pair(aadp_ctx* c, int64_t p, float* score_fwd, int32_t* prevq_fwd, int32_t* prevt_fwd,
                          float* score_rev, int32_t* prevq_rev, int32_t* prevt_rev, uint8_t* nearopt) {
  if (check_ctx(c, true)) return 1;
  if (p < 0 || p >= c->b.npairs) return fail("pair index out of range");
  if ((score_fwd || prevq_fwd || prevt_fwd) && !(c->b.ran_what & AADP_W_FWD)) return fail("forward fill was not run");
  if ((score_rev || prevq_rev || prevt_rev) && !(c->b.ran_what & AADP_W_REV)) return fail("reverse fill was not run");
  if (c->float_mode) return gg_fetch_pair(c, p, score_fwd, prevq_fwd, prevt_fwd, score_rev, prevq_rev, prevt_rev, nearopt);
  if (dense_pair(c, p, 0, score_fwd, prevq_fwd, prevt_fwd)) return 1;
  if (dense_pair(c, p, 1, score_rev, prevq_rev, prevt_rev)) return 1;
  if (dense_mask(c, p, nearopt)) return 1;
  return 0;
}

int aadp_fill_pair(aadp_ctx* c, const uint8_t* q, int Lq, const uint8_t* t, int Lt, int direction, float delta_ratio,
                   float* score_fwd, int32_t* prevq_fwd, int32_t* prevt_fwd, float* score_rev, int32_t* prevq_rev,
                   int32_t* prevt_rev, uint8_t* nearopt, float* threshold) {
  if (check_ctx(c, true)) return 1;
  if (c->prof_mode)
    return fail("aadp_fill_pair: profile scoring selects the similarity by template sequence id, which a single pair does not "
                "have; use a one-pair batch (aadp_fill_batch + aadp_batch_fetch_pair)");
  if (Lq < 0 || Lt < 0) return fail("Illegal bounds building DPM");  // dpmatrix.h:360-361
  if (direction < 1 || direction > 3) return fail("bad direction");
  std::vector<uint8_t> res((size_t)Lq + Lt + 1);
  if (Lq) memcpy(res.data(), q, Lq);
  if (Lt) memcpy(res.data() + Lq, t, Lt);
  const int64_t off[3] = {0, Lq, (int64_t)Lq + Lt};
  const int32_t pq = 0, pt = 1;
  uint32_t what = (direction & 1 ? AADP_W_FWD : 0) | (direction & 2 ? AADP_W_REV : 0);
  if (prevq_fwd || prevt_fwd || prevq_rev || prevt_rev) what |= AADP_W_TB;
  if (score_fwd || score_rev || c->sc.local) what |= AADP_W_SCORES;
  const bool want_mask = (nearopt || threshold) && delta_ratio >= 0.f;
  if (want_mask) {
    if (direction != 3) return fail("the near-optimal cell set needs direction 3 (fwd+rev)");
    what |= AADP_W_MASK;
  }
  float* dthr = nullptr;
  if (want_mask) { if (c->thr.reserve(16)) return 1; dthr = c->thr.as<float>(); }
  if (aadp_upload_batch(c, res.data(), off, 2, &pq, &pt, 1, what)) return 1;
  if (aadp_run_batch(c, what, delta_ratio, nullptr, nullptr, dthr, nullptr)) return 1;
  if (aadp_batch_fetch_pair(c, 0, (direction & 1) ? score_fwd : nullptr, (direction & 1) ? prevq_fwd : nullptr,
                            (direction & 1) ? prevt_fwd : nullptr, (direction & 2) ? score_rev : nullptr,
                            (direction & 2) ? prevq_rev : nullptr, (direction & 2) ? prevt_rev : nullptr,
                            want_mask ? nearopt : nullptr))
    return 1;
  if (threshold && want_mask) {
    CK(cudaMemcpyAsync(threshold, dthr, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

int64_t aadp_tb_row_bytes(int Lt) { return tb_row_bytes(Lt); }

int64_t aadp_batch_tb_bytes(aadp_ctx* c, int64_t p) {
  if (!c || p < 0 || p >= c->b.npairs || c->b.tb_off.empty()) return 0;
  return c->b.tb_off[p + 1] - c->b.tb_off[p];
}

int aadp_batch_fetch_tb(aadp_ctx* c, int64_t p, int direction, uint8_t* tb, int64_t tb_bytes, int32_t* final_rec) {
  if (check_ctx(c, true)) return 1;
  Batch& b = c->b;
  if (p < 0 || p >= b.npairs) return fail("pair index out of range");
  if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
  const int dir = direction - 1;
  if (!(b.ran_what & (dir ? AADP_W_REV : AADP_W_FWD))) return fail("that direction was not run");
  if (c->float_mode) return fail("exact-float mode keeps no packed traceback; use aadp_batch_fetch_pair / aadp_batch_optimal");
  if (tb) {
    if (!(b.ran_what & AADP_W_TB)) return fail("traceback was not kept (run with AADP_W_TB)");
    const int64_t need = b.tb_off[p + 1] - b.tb_off[p];
    if (tb_bytes < need) return fail("traceback buffer too small");
    if (need) CK(cudaMemcpyAsync(tb, c->tb[dir].as<uint8_t>() + b.tb_off[p], need, cudaMemcpyDeviceToHost, c->stream));
  }
  if (final_rec) {
    CK(cudaMemcpyAsync(&final_rec[0], c->fin_score[dir].as<int32_t>() + p, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&final_rec[1], c->fin_kind[dir].as<int32_t>() + p, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&final_rec[2], c->fin_k[dir].as<int32_t>() + p, 4, cudaMemcpyDeviceToHost, c->stream));
    final_rec[3] = c->sc.scale_log2;
    {
      const int ts = b.pair_t[p];
      const int Lt = (int)(b.seq_off[ts + 1] - b.seq_off[ts]);
      final_rec[4] = (b.fmt[p] == 1 && dir == 0) ? ((Lt + 15) / 16) * 16 - Lt : 0;  // leading pad columns of the layout
      final_rec[5] = b.fmt[p];                                                       // layout class: 0 words, 1 diagonal-major, 2 nibble groups
    }
  }
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int aadp_decode_cell(const uint8_t* tb, int Lq, int Lt, int direction, int align_type, uint32_t flags,
                     const int32_t* final_rec, int i, int j, int32_t* prev_q, int32_t* prev_t) {
  if (!tb || !prev_q || !prev_t) return fail("null argument");
  const int rev = (direction == AADP_REV);
  const int a = rev ? Lq + 1 - i : i, b = rev ? Lt + 1 - j : j;
  int pa = -1, pb = -1;
  bool is_final = false;
  Layout L = make_layout(Lq, Lt, final_rec ? final_rec[5] : 0, rev);
  if (final_rec) L.sig = final_rec[4];
  if (a >= 1 && a <= Lq && b >= 1 && b <= Lt) decode_prev(tb, L, a, b, &pa, &pb);
  else if (a == Lq + 1 && b == Lt + 1) {
    if (!final_rec) return fail("final_rec needed for the final cell");
    decode_final(tb, L, final_rec[1], final_rec[2], &pa, &pb);
    is_final = true;
  }
  if (pa < 0) { *prev_q = -1; *prev_t = -1; return 0; }
  *prev_q = rev ? Lq + 1 - pa : pa;
  *prev_t = rev ? Lt + 1 - pb : pb;
  if (is_final && rev && align_type != AADP_LOCAL && (flags & AADP_REPRO_REV_BUG) && final_rec[1] == 2 && Lq > 0 && Lt > 0)
    *prev_t = Lt;  // dpmatrix.h:868
  return 0;
}

int aadp_batch_optimal(aadp_ctx* c, int64_t p, int direction, int32_t* pairs, int32_t max_pairs, int32_t* npairs,
                       float* score) {
  if (check_ctx(c, true)) return 1;
  Batch& b = c->b;
  if (p < 0 || p >= b.npairs) return fail("pair index out of range");
  const int qs = b.pair_q[p], ts = b.pair_t[p];
  const int Lq = (int)(b.seq_off[qs + 1] - b.seq_off[qs]), Lt = (int)(b.seq_off[ts + 1] - b.seq_off[ts]);
  if (c->sc.local) {
    // Optimal::enumerate_local + find_max (optimal.h:76-124) / Optimal_Rev (optimal_rev.h:79-131) over the dense view of
    // this one pair (either exactness class); whole batches: aadp_batch_optimal_all traces them on the GPU
    if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
    const bool rev = direction == AADP_REV;
    const int sz1 = Lq + 2, sz2 = Lt + 2;
    const size_t n = (size_t)sz1 * sz2;
    std::vector<float> sc(n);
    std::vector<int32_t> pq(n), pt(n);
    if (aadp_batch_fetch_pair(c, p, rev ? nullptr : sc.data(), rev ? nullptr : pq.data(), rev ? nullptr : pt.data(),
                              rev ? sc.data() : nullptr, rev ? pq.data() : nullptr, rev ? pt.data() : nullptr, nullptr)) return 1;
    auto D = [&](int i, int j) { return sc[(size_t)i * sz2 + j]; };
    std::vector<int32_t> path;  // in walk order, framed afterwards
    int i, j;
    float s;
    if (!rev) {  // optimal.h:107-124
      i = sz1 - 2; j = sz2 - 2; s = D(i, j);
      for (int a = 0; a < sz1 - 1; ++a)
        for (int bb = 0; bb < sz2 - 1; ++bb)
          if (s < D(a, bb)) { i = a; j = bb; s = D(a, bb); }
    } else {     // optimal_rev.h:114-131
      i = 0; j = 0; s = D(0, 0);
      for (int a = sz1 - 1; a > 0; --a)
        for (int bb = sz2 - 1; bb > 0; --bb)
          if (s < D(a, bb)) { i = a; j = bb; s = D(a, bb); }
    }
    if (score) *score = s;
    path.push_back(i);
    path.push_back(j);
    int guard = 0;
    while (rev ? (i < sz1 - 1) : (i > 0)) {
      const int32_t pi = pq[(size_t)i * sz2 + j], pj = pt[(size_t)i * sz2 + j];
      i = pi;
      j = pj;
      if (i < 0 || j < 0 || ++guard > Lq + Lt + 4) break;
      if (D(i, j) <= 0.f) break;
      path.push_back(i);
      path.push_back(j);
    }
    const bool frame = rev ? (i != sz1 - 1 && j != sz2 - 1) : (i != 0 && j != 0);  // optimal.h:105, optimal_rev.h:111
    std::vector<int32_t> ali;  // front to back in matrix order
    const int nw = (int)path.size() / 2;
    if (!rev) {
      if (frame) { ali.push_back(0); ali.push_back(0); }
      for (int k = nw - 1; k >= 0; --k) { ali.push_back(path[2 * k]); ali.push_back(path[2 * k + 1]); }
      ali.push_back(sz1 - 1);
      ali.push_back(sz2 - 1);
    } else {
      ali.push_back(0);
      ali.push_back(0);
      for (int k = 0; k < nw; ++k) { ali.push_back(path[2 * k]); ali.push_back(path[2 * k + 1]); }
      if (frame) { ali.push_back(sz1 - 1); ali.push_back(sz2 - 1); }
    }
    const int n2 = (int)ali.size() / 2;
    if (npairs) *npairs = n2;
    for (int k = 0; k < n2 && k < max_pairs; ++k) { pairs[2 * k] = ali[2 * k]; pairs[2 * k + 1] = ali[2 * k + 1]; }
    return 0;
  }
  if (c->float_mode) {
    // exact-float mode: dense predecessors of this pair are recomputed, then optimal.h:57-74 / optimal_rev.h:57-76
    if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
    const bool rev = direction == AADP_REV;
    if (!(b.ran_what & (rev ? AADP_W_REV : AADP_W_FWD))) return fail("that direction was not run");
    const int sz2 = Lt + 2;
    const size_t n = (size_t)(Lq + 2) * sz2;
    std::vector<float> sc(n);
    std::vector<int32_t> pq(n), pt(n);
    if (gg_fetch_pair(c, p, rev ? nullptr : sc.data(), rev ? nullptr : pq.data(), rev ? nullptr : pt.data(),
                      rev ? sc.data() : nullptr, rev ? pq.data() : nullptr, rev ? pt.data() : nullptr, nullptr)) return 1;
    int i = rev ? 0 : Lq + 1, j = rev ? 0 : Lt + 1;
    const int ei = rev ? Lq + 1 : 0, ej = rev ? Lt + 1 : 0;
    if (score) *score = sc[(size_t)i * sz2 + j];
    std::vector<int32_t> path = {i, j};
    int guard = 0;
    while (rev ? (i < ei) : (i > 0)) {
      const int32_t pi = pq[(size_t)i * sz2 + j], pj = pt[(size_t)i * sz2 + j];
      i = pi;
      j = pj;
      path.push_back(i);
      path.push_back(j);
      if (i < 0 || j < 0 || ++guard > Lq + Lt + 4) break;
    }
    const int n2 = (int)path.size() / 2;
    if (npairs) *npairs = n2;
    for (int k = 0; k < n2 && k < max_pairs; ++k) {
      const int src = rev ? k : n2 - 1 - k;
      pairs[2 * k] = path[2 * src];
      pairs[2 * k + 1] = path[2 * src + 1];
    }
    if (i != ei || j != ej) { g_err = "Illegal alignment start pair"; return 3; }
    return 0;
  }
  std::vector<uint8_t> tb((size_t)std::max<int64_t>(b.tb_off[p + 1] - b.tb_off[p], 1));
  int32_t fin[6];
  if (aadp_batch_fetch_tb(c, p, direction, tb.data(), (int64_t)tb.size(), fin)) return 1;
  if (score) *score = (float)fin[0] / (float)(1 << fin[3]);
  // optimal.h:57-74 / optimal_rev.h:57-76: follow prev_* from the final cell to the anchor
  const int rev = (direction == AADP_REV);
  int i = rev ? 0 : Lq + 1, j = rev ? 0 : Lt + 1;
  const int ei = rev ? Lq + 1 : 0, ej = rev ? Lt + 1 : 0;
  std::vector<int32_t> path;
  path.push_back(i);
  path.push_back(j);
  int guard = 0;
  while (rev ? (i < ei) : (i > 0)) {
    int32_t pi, pj;
    if (aadp_decode_cell(tb.data(), Lq, Lt, direction, c->align_type, c->flags, fin, i, j, &pi, &pj)) return 1;
    i = pi;
    j = pj;
    path.push_back(i);
    path.push_back(j);
    if (i < 0 || j < 0 || ++guard > Lq + Lt + 4) break;
  }
  const int n = (int)path.size() / 2;
  if (npairs) *npairs = n;
  for (int k = 0; k < n && k < max_pairs; ++k) {
    const int src = rev ? k : n - 1 - k;  // forward alignments are built with prepend()
    pairs[2 * k] = path[2 * src];
    pairs[2 * k + 1] = path[2 * src + 1];
  }
  if (i != ei || j != ej) {
    g_err = "Illegal alignment start pair";  // optimal.h:74
    return 3;
  }
  return 0;
}

}  // extern "C"

// packs the capacity-sized alignment slots of a batch front to back: one warp per pair
__global__ void compact_alignments_kernel(const int2* __restrict__ slots, const int64_t* __restrict__ cap_off,
                                          const int32_t* __restrict__ n, const int64_t* __restrict__ out_off, int64_t npairs,
                                          int2* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  for (int64_t p = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; p < npairs; p += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const int2* src = slots + cap_off[p];
    int2* dst = out + out_off[p];
    for (int k = lane; k < n[p]; k += 32) dst[k] = src[k];
  }
}

// compact_off != nullptr: aadp_batch_optimal_all_compact
static int optimal_all_impl(aadp_ctx* c, int direction, int64_t* ali_off, int32_t* pairs, int64_t pairs_cap, int32_t* n_out,
                            int32_t* status, int64_t* compact_off) {
  if (check_ctx(c, true)) return 1;
  Batch& b = c->b;
  if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
  const int dir = direction - 1;
  // exact-float mode keeps no resident traceback: the forward optimal alignments (Optimal::enumerate, optimal.h:47-75) of
  // the whole batch are produced chunk by chunk -- dense fill with predecessors (record-list kernel), then one thread per
  // pair follows DPCell::prev_* from the final cell.  Reverse and local tracebacks go through aadp_batch_optimal.
  const bool float_all = c->float_mode;
  if (float_all && (dir != 0 || c->sc.local))
    return fail("aadp_batch_optimal_all: exact-float mode traces forward, non-local alignments only (use aadp_batch_optimal)");
  if (!float_all) {
    if (!(b.ran_what & (dir ? AADP_W_REV : AADP_W_FWD))) return fail("that direction was not run");
    if (!(b.ran_what & AADP_W_TB)) return fail("traceback was not kept (run with AADP_W_TB)");
  }
  if (c->sc.local && !(b.ran_what & AADP_W_SCORES)) return fail("local tracebacks need AADP_W_SCORES (find_max, optimal.h:107-124)");
  const int64_t np = b.npairs;
  std::vector<int64_t> cap((size_t)np + 1, 0);
  for (int64_t p = 0; p < np; ++p) {
    const int qs = b.pair_q[p], ts = b.pair_t[p];
    cap[(size_t)p + 1] = cap[(size_t)p] + (b.seq_off[qs + 1] - b.seq_off[qs]) + (b.seq_off[ts + 1] - b.seq_off[ts]) + 2;
  }
  if (ali_off) memcpy(ali_off, cap.data(), (size_t)(np + 1) * 8);
  if (np == 0) return 0;
  if (!compact_off && !pairs && !n_out && !status) return 0;  // a size query: the offsets are all the caller asked for
  if (!compact_off && pairs && pairs_cap < cap[(size_t)np]) return fail("aadp_batch_optimal_all: pairs buffer too small (needs 2*ali_off[npairs] ints)");
  CK(cudaStreamSynchronize(c->stream));
  if (pin_reserve(c, (size_t)(np + 1) * 8 + 4096)) return 1;
  if (upload_vec(c, c->ali_cap, cap)) return 1;
  if (c->ali_out.reserve((size_t)cap[(size_t)np] * 8) || c->ali_n.reserve((size_t)np * 4) || c->ali_status.reserve((size_t)np * 4)) return 1;
  if (float_all) {
    std::vector<int64_t> off;
    std::vector<int32_t> rects;
    c->launches = 0;
    for (int64_t p0 = 0; p0 < np;) {
      off.assign(1, 0);
      int64_t p1 = p0;
      while (p1 < np) {
        const int qs = b.pair_q[p1], ts = b.pair_t[p1];
        const int64_t cl = (b.seq_off[qs + 1] - b.seq_off[qs] + 2) * (b.seq_off[ts + 1] - b.seq_off[ts] + 2);
        if (p1 > p0 && off.back() + cl > c->gg_budget_cells / 4) break;  // scores + two predecessor matrices + links
        off.push_back(off.back() + cl);
        ++p1;
      }
      const int64_t m = p1 - p0;
      if (c->gg_fin[0].reserve(std::max<size_t>((size_t)np * 4, 16))) return 1;
      if (gg_fill(c, p0, m, 1, true, off, c->gg_fin[0].as<float>(), nullptr)) return 1;
      rects.resize((size_t)m * 4);
      for (int64_t k = p0; k < p1; ++k) {
        const int qs = b.pair_q[k], ts = b.pair_t[k];
        rects[(size_t)(k - p0) * 4] = 0;
        rects[(size_t)(k - p0) * 4 + 1] = 0;
        rects[(size_t)(k - p0) * 4 + 2] = (int32_t)(b.seq_off[qs + 1] - b.seq_off[qs]) + 1;
        rects[(size_t)(k - p0) * 4 + 3] = (int32_t)(b.seq_off[ts + 1] - b.seq_off[ts]) + 1;
      }
      CK(cudaStreamSynchronize(c->stream));
      if (pin_reserve(c, (size_t)m * 16 + 4096)) return 1;
      if (upload_vec(c, c->gg_rect, rects)) return 1;
      SubTraceParams S{};
      S.PQ = c->gg_pq[0].as<int32_t>();
      S.PT = c->gg_pt[0].as<int32_t>();
      S.D = c->gg_score[0].as<float>();
      S.dense_off = c->gg_off.as<int64_t>();
      S.rects = c->gg_rect.as<int4>();
      S.cap_off = c->ali_cap.as<int64_t>();
      S.item0 = (int)p0;
      S.n = (int)m;
      S.out = c->ali_out.as<int2>();
      S.out_n = c->ali_n.as<int32_t>();
      S.out_status = c->ali_status.as<int32_t>();
      S.out_score = nullptr;
      c->prof_begin("subali_trace_kernel", 0);
      subali_trace_kernel<<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(S);
      c->prof_end();
      CK(cudaGetLastError());
      c->launches++;
      CK(cudaStreamSynchronize(c->stream));  // the next chunk recycles the dense scratch and the pinned pool
      p0 = p1;
    }
  }
  TraceParams T{};
  T.tb = c->tb[dir].as<uint8_t>();
  T.tb_off = c->tb_off.as<int64_t>();
  T.fmt = c->fmt.as<uint8_t>();
  T.seq_off = c->seq_off.as<int64_t>();
  T.pair_q = c->pair_q.as<int32_t>();
  T.pair_t = c->pair_t.as<int32_t>();
  T.fin_kind = c->fin_kind[dir].as<int32_t>();
  T.fin_k = c->fin_k[dir].as<int32_t>();
  T.n_pairs = (int)np;
  T.rev = dir;
  T.repro_rev_bug = (c->flags & AADP_REPRO_REV_BUG) ? 1 : 0;
  T.cap_off = c->ali_cap.as<int64_t>();
  T.out = c->ali_out.as<int2>();
  T.out_n = c->ali_n.as<int32_t>();
  T.out_status = c->ali_status.as<int32_t>();
  if (float_all) {
    // (traced above)
  } else if (c->sc.local) {  // Optimal[_Rev]::enumerate_local + find_max: one warp per pair
    LocalTraceParams Q{};
    Q.t = T;
    Q.sc_blob = c->scb[dir].p;
    Q.sc_off = c->sc_off.as<int64_t>();
    Q.st_mode_v1 = b.st_mode;
    Q.bias16 = kBias16;
    Q.fin_score = c->fin_score[dir].as<int32_t>();
    Q.inv_scale = 1.f / (float)(1 << c->sc.scale_log2);
    Q.out_score = nullptr;
    c->prof_begin(dir ? "local_traceback_kernel rev" : "local_traceback_kernel fwd", 0);
    local_traceback_kernel<<<(unsigned)((np * 32 + 127) / 128), 128, 0, c->stream>>>(Q);
    c->prof_end();
  } else {
    c->prof_begin(dir ? "traceback_kernel rev" : "traceback_kernel fwd", 0);
    traceback_kernel<<<(unsigned)((np + 127) / 128), 128, 0, c->stream>>>(T);
    c->prof_end();
  }
  CK(cudaGetLastError());
  if (!float_all) c->launches = 1;
  c->d2h_bytes = 0;
  if (compact_off) {
    // compact form: only the aligned pairs that exist travel.  The lengths come back first (4 bytes per pair), the host
    // turns them into offsets, a gather kernel packs the slots front to back, and one copy brings the packed pairs.
    std::vector<int32_t> nn((size_t)np);
    CK(cudaMemcpyAsync(nn.data(), c->ali_n.p, (size_t)np * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->d2h_bytes += np * 4;
    compact_off[0] = 0;
    for (int64_t p = 0; p < np; ++p) compact_off[p + 1] = compact_off[p] + nn[(size_t)p];
    const int64_t total = compact_off[np];
    if (pairs && pairs_cap < total) return fail("aadp_batch_optimal_all_compact: pairs buffer too small");
    if (pairs && total > 0) {
      std::vector<int64_t> offv(compact_off, compact_off + np + 1);
      if (pin_reserve(c, (size_t)(np + 1) * 8 + 4096)) return 1;
      if (upload_vec(c, c->scratch_a, offv)) return 1;
      if (c->scratch_b.reserve((size_t)total * 8)) return 1;
      compact_alignments_kernel<<<(unsigned)std::min<int64_t>((np * 32 + 255) / 256, 148 * 16), 256, 0, c->stream>>>(
          c->ali_out.as<int2>(), c->ali_cap.as<int64_t>(), c->ali_n.as<int32_t>(), c->scratch_a.as<int64_t>(), np, c->scratch_b.as<int2>());
      CK(cudaGetLastError());
      c->launches++;
      CK(cudaMemcpyAsync(pairs, c->scratch_b.p, (size_t)total * 8, cudaMemcpyDeviceToHost, c->stream));
      c->d2h_bytes += total * 8;
    }
    if (n_out) memcpy(n_out, nn.data(), (size_t)np * 4);
  } else {
    if (pairs) { CK(cudaMemcpyAsync(pairs, c->ali_out.p, (size_t)cap[(size_t)np] * 8, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += cap[(size_t)np] * 8; }
    if (n_out) { CK(cudaMemcpyAsync(n_out, c->ali_n.p, (size_t)np * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += np * 4; }
  }
  if (status) { CK(cudaMemcpyAsync(status, c->ali_status.p, (size_t)np * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += np * 4; }
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" {

int aadp_batch_optimal_all(aadp_ctx* c, int direction, int64_t* ali_off, int32_t* pairs, int64_t pairs_cap, int32_t* n_out,
                           int32_t* status) {
  return optimal_all_impl(c, direction, ali_off, pairs, pairs_cap, n_out, status, nullptr);
}

int aadp_batch_optimal_all_compact(aadp_ctx* c, int direction, int64_t* ali_off, int32_t* pairs, int64_t pairs_cap,
                                   int32_t* n_out, int32_t* status) {
  if (!ali_off) return fail("aadp_batch_optimal_all_compact: ali_off is required");
  return optimal_all_impl(c, direction, nullptr, pairs, pairs_cap, n_out, status, ali_off);
}

}  // extern "C"

// UnconstrainedNearOptimal (cno = 0) / ConstrainedNearOptimal (cno = 1, flags = SuboptFlags per template position of
// every listed pair, flag_off = n+1 offsets; flags == nullptr: all true) of the listed pairs.
static int near_optimal_impl(aadp_ctx* c, int cno, const uint8_t* flags, const int64_t* flag_off, const int64_t* pair_ids,
                             int64_t n, float delta_ratio, int32_t max_alignments, int32_t* n_ali, int32_t* status, float* scores,
                             int32_t* ali_len, int64_t* path_off, int32_t* paths, int64_t paths_cap, float* threshold) {
  if (check_ctx(c, true)) return 1;
  Batch& b = c->b;
  if (n < 0 || (n && !pair_ids)) return fail("null input");
  if (max_alignments < 1) return fail("max_alignments must be positive");
  if (c->sc.local) return fail("aadp_batch_near_optimal: not for local alignments");
  if (!(b.ran_what & AADP_W_FWD)) return fail("forward fill was not run");
  if (!c->float_mode && !(b.ran_what & (AADP_W_SCORES | AADP_W_MASK))) return fail("score matrices were not kept (run with AADP_W_SCORES or AADP_W_MASK)");
  if (cno && !c->float_mode && !(b.ran_what & AADP_W_TB)) return fail("the constrained enumeration follows the optimal predecessors: run with AADP_W_TB");
  if (flags && !flag_off) return fail("null input");
  std::vector<int64_t> poff((size_t)n + 1, 0), soff((size_t)n + 1, 0);
  for (int64_t k = 0; k < n; ++k) {
    const int64_t p = pair_ids[k];
    if (p < 0 || p >= b.npairs) return fail("pair index out of range");
    const int64_t Lq = b.seq_off[b.pair_q[p] + 1] - b.seq_off[b.pair_q[p]];
    poff[(size_t)k + 1] = poff[(size_t)k] + (int64_t)max_alignments * (Lq + 2);  // an alignment has at most Lq+2 pairs
    soff[(size_t)k + 1] = soff[(size_t)k] + (Lq + 2);
    if (flags) {
      const int64_t Lt = b.seq_off[b.pair_t[p] + 1] - b.seq_off[b.pair_t[p]];
      if (flag_off[k + 1] - flag_off[k] != Lt + 2) return fail("SuboptFlags: one flag per template position including both sentinels");
    }
  }
  if (path_off) memcpy(path_off, poff.data(), (size_t)(n + 1) * 8);
  if (n == 0 || (!n_ali && !status && !scores && !ali_len && !paths && !threshold)) return 0;
  if (paths && paths_cap < poff[(size_t)n]) return fail("aadp_batch_near_optimal: paths buffer too small (needs 2*path_off[n] ints)");
  CK(cudaStreamSynchronize(c->stream));
  const size_t nflag = flags ? (size_t)(flag_off[n] - flag_off[0]) : 0;
  if (pin_reserve(c, (size_t)(n + 1) * 32 + nflag + 4096)) return 1;
  std::vector<int64_t> ids(pair_ids, pair_ids + n);
  if (upload_vec(c, c->ucw_ids, ids) || upload_vec(c, c->ucw_path_off, poff) || upload_vec(c, c->ucw_stack_off, soff)) return 1;
  if (flags) {
    std::vector<int64_t> fo((size_t)n + 1);
    for (int64_t k = 0; k <= n; ++k) fo[(size_t)k] = flag_off[k] - flag_off[0];
    std::vector<uint8_t> fl(flags + flag_off[0], flags + flag_off[n]);
    if (upload_vec(c, c->ucw_flag_off, fo) || upload_vec(c, c->ucw_flags, fl)) return 1;
  }
  if (c->ucw_plen.reserve(std::max<size_t>((size_t)soff[(size_t)n] * 4, 16)) || c->ucw_pathbuf.reserve(std::max<size_t>((size_t)soff[(size_t)n] * 8, 16))) return 1;
  if (c->ucw_paths.reserve(std::max<size_t>((size_t)poff[(size_t)n] * 8, 16)) || c->ucw_stack.reserve(std::max<size_t>((size_t)soff[(size_t)n] * 16, 16)) ||
      c->ucw_len.reserve((size_t)n * max_alignments * 4) || c->ucw_scores.reserve((size_t)n * max_alignments * 4) ||
      c->ucw_n.reserve((size_t)n * 4) || c->ucw_status.reserve((size_t)n * 4) || c->ucw_thr.reserve((size_t)n * 4)) return 1;
  UcwParams U{};
  U.A = c->sc.A;
  U.subf = c->subf.as<float>();
  U.gi = c->gi_f;
  U.ge = c->ge_f;
  U.delfree = c->sc.delfree;
  U.insfree = c->sc.insfree;
  U.inv_scale = 1.f / (float)(1 << c->sc.scale_log2);
  U.residues = c->residues.as<uint8_t>();
  U.seq_off = c->seq_off.as<int64_t>();
  U.pair_q = c->pair_q.as<int32_t>();
  U.pair_t = c->pair_t.as<int32_t>();
  U.fmt = c->fmt.as<uint8_t>();
  U.sc_blob = c->scb[0].p;
  U.sc_off = c->sc_off.as<int64_t>();
  U.st_mode_v1 = b.st_mode;
  U.bias16 = kBias16;
  U.fin_score = c->fin_score[0].as<int32_t>();
  U.tb = (!c->float_mode && (b.ran_what & AADP_W_TB)) ? c->tb[0].as<uint8_t>() : nullptr;
  U.tb_off = c->tb_off.as<int64_t>();
  // the resident near-optimal set prunes the deletion scans when it was built with the same delta_ratio (option
  // "enum_mask_prune", default 1)
  const bool prune = c->enum_mask_prune && !c->float_mode && (b.ran_what & AADP_W_MASK) && delta_ratio == c->last_delta;
  U.mask = prune ? c->mask.as<uint32_t>() : nullptr;
  U.mask_off = c->mask_off.as<int64_t>();
  U.subopt = flags ? c->ucw_flags.as<uint8_t>() : nullptr;
  U.subopt_off = flags ? c->ucw_flag_off.as<int64_t>() : nullptr;
  U.frame_plen = c->ucw_plen.as<int32_t>();
  U.pathbuf = c->ucw_pathbuf.as<int2>();
  U.ids = c->ucw_ids.as<int64_t>();
  U.n = (int)n;
  U.delta_ratio = delta_ratio;
  U.max_ali = max_alignments;
  U.user_limit = cno ? c->cw_user_limit : c->ucw_user_limit;
  U.path_off = c->ucw_path_off.as<int64_t>();
  U.paths = c->ucw_paths.as<int2>();
  U.ali_len = c->ucw_len.as<int32_t>();
  U.scores = c->ucw_scores.as<float>();
  U.n_ali = c->ucw_n.as<int32_t>();
  U.status = c->ucw_status.as<int32_t>();
  U.threshold = c->ucw_thr.as<float>();
  U.stack_off = c->ucw_stack_off.as<int64_t>();
  U.stack = c->ucw_stack.as<int4>();
  c->launches = 0;
  if (!c->float_mode) {
    const unsigned grid = (unsigned)((n * 32 + 127) / 128);
    if (c->prof_mode) {
      c->prof_begin(cno ? "ucw_enum_kernel<CNO=1,PRO=1>" : "ucw_enum_kernel<CNO=0,PRO=1>", 0);
      if (cno) ucw_enum_kernel<1, 1><<<grid, 128, 0, c->stream>>>(U, c->prof_dev());
      else ucw_enum_kernel<0, 1><<<grid, 128, 0, c->stream>>>(U, c->prof_dev());
    } else {
      c->prof_begin(cno ? "ucw_enum_kernel<CNO=1>" : "ucw_enum_kernel<CNO=0>", 0);
      if (cno) ucw_enum_kernel<1, 0><<<grid, 128, 0, c->stream>>>(U, c->prof_dev());
      else ucw_enum_kernel<0, 0><<<grid, 128, 0, c->stream>>>(U, c->prof_dev());
    }
    c->prof_end();
    CK(cudaGetLastError());
    c->launches++;
  } else {
    // exact-float mode keeps no resident matrices: refill the listed pairs with the exact general-gap kernel (dense fp32
    // scores + predecessors in scratch), a chunk of the scratch budget at a time, and walk those
    if (c->gg_fin[0].reserve(std::max<size_t>((size_t)b.npairs * 4, 16))) return 1;
    std::vector<int64_t> doff;
    for (int64_t k0 = 0; k0 < n;) {
      doff.assign(1, 0);
      int64_t k1 = k0;
      while (k1 < n) {
        const int64_t p = pair_ids[k1];
        const int64_t cl = (b.seq_off[b.pair_q[p] + 1] - b.seq_off[b.pair_q[p]] + 2) * (b.seq_off[b.pair_t[p] + 1] - b.seq_off[b.pair_t[p]] + 2);
        if (k1 > k0 && doff.back() + cl > c->gg_budget_cells / 4) break;  // scores + two predecessor matrices (+ prefix maxima)
        doff.push_back(doff.back() + cl);
        ++k1;
      }
      const int64_t m = k1 - k0;
      if (gg_fill(c, 0, m, 1, true, doff, c->gg_fin[0].as<float>(), nullptr, nullptr, nullptr, false, pair_ids + k0)) return 1;
      UcwParams V = U;
      V.denseF = c->gg_score[0].as<float>();
      V.densePQ = c->gg_pq[0].as<int32_t>();
      V.densePT = c->gg_pt[0].as<int32_t>();
      V.dense_off = c->gg_off.as<int64_t>();
      V.n = (int)m;
      V.ids = U.ids + k0;
      V.path_off = U.path_off + k0;
      V.stack_off = U.stack_off + k0;
      V.ali_len = U.ali_len + k0 * max_alignments;
      V.scores = U.scores + k0 * max_alignments;
      V.n_ali = U.n_ali + k0;
      V.status = U.status + k0;
      V.threshold = U.threshold + k0;
      if (flags) V.subopt_off = U.subopt_off + k0;
      c->prof_begin("ucw_enum_kernel (exact float)", 0);
      if (cno) ucw_enum_kernel<1, 0><<<(unsigned)((m * 32 + 127) / 128), 128, 0, c->stream>>>(V, c->prof_dev());
      else ucw_enum_kernel<0, 0><<<(unsigned)((m * 32 + 127) / 128), 128, 0, c->stream>>>(V, c->prof_dev());
      c->prof_end();
      CK(cudaGetLastError());
      c->launches++;
      k0 = k1;
    }
  }
  c->d2h_bytes = 0;
  auto back = [&](void* dst, const DevBuf& src, size_t bytes) {
    if (!dst || !bytes) return 0;
    if (cudaMemcpyAsync(dst, src.p, bytes, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return 1;
    c->d2h_bytes += (int64_t)bytes;
    return 0;
  };
  if (back(n_ali, c->ucw_n, (size_t)n * 4) || back(status, c->ucw_status, (size_t)n * 4) ||
      back(scores, c->ucw_scores, (size_t)n * max_alignments * 4) || back(ali_len, c->ucw_len, (size_t)n * max_alignments * 4) ||
      back(threshold, c->ucw_thr, (size_t)n * 4))
    return fail("device to host copy failed");
  if (paths) {
    // only the slots that hold an alignment travel: the budget is usually far larger than what a pair emits
    std::vector<int32_t> cnt((size_t)n);
    CK(cudaMemcpyAsync(cnt.data(), c->ucw_n.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int64_t k = 0; k < n; ++k) {
      const int64_t slot = (poff[(size_t)k + 1] - poff[(size_t)k]) / max_alignments;
      const size_t bytes = (size_t)cnt[(size_t)k] * (size_t)slot * 8;
      if (!bytes) continue;
      CK(cudaMemcpyAsync(paths + 2 * poff[(size_t)k], c->ucw_paths.as<int2>() + poff[(size_t)k], bytes, cudaMemcpyDeviceToHost, c->stream));
      c->d2h_bytes += (int64_t)bytes;
    }
  }
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" {

int aadp_batch_near_optimal(aadp_ctx* c, const int64_t* pair_ids, int64_t n, float delta_ratio, int32_t max_alignments,
                            int32_t* n_ali, int32_t* status, float* scores, int32_t* ali_len, int64_t* path_off, int32_t* paths,
                            int64_t paths_cap, float* threshold) {
  return near_optimal_impl(c, 0, nullptr, nullptr, pair_ids, n, delta_ratio, max_alignments, n_ali, status, scores, ali_len,
                           path_off, paths, paths_cap, threshold);
}

int aadp_batch_near_optimal_pruned(aadp_ctx* c, int64_t pair_id, int variant, const uint8_t* subopt_flags, float delta_ratio,
                                   uint32_t k_limit, uint32_t sort_limit, float max_overlap, uint32_t user_limit,
                                   int32_t max_alignments, int32_t* n_ali, int32_t* status, float* scores, int32_t* ali_len,
                                   int32_t* paths, int64_t paths_cap, float* threshold) {
  if (check_ctx(c, true)) return 1;
  Batch& b = c->b;
  if (variant != AADP_PRUNE_KSORTED && variant != AADP_PRUNE_REDUNDANCY) return fail("unknown pruning variant");
  if (pair_id < 0 || pair_id >= b.npairs) return fail("pair index out of range");
  if (max_alignments < 1 || !n_ali || !status) return fail("bad output arguments");
  if (k_limit < 1 || sort_limit < 1) return fail("k_limit and sort_limit must be positive");
  if (c->sc.local) return fail("near-optimal enumeration of local alignments is not defined by the reference");
  if (!(b.ran_what & AADP_W_FWD)) return fail("forward fill was not run");
  if (!c->float_mode && (!(b.ran_what & AADP_W_TB) || !(b.ran_what & (AADP_W_SCORES | AADP_W_MASK))))
    return fail("the pruned enumerators walk the forward scores and the optimal predecessors: run with AADP_W_TB and AADP_W_SCORES");
  const int qs = b.pair_q[(size_t)pair_id], ts = b.pair_t[(size_t)pair_id];
  const int Lq = (int)(b.seq_off[qs + 1] - b.seq_off[qs]), Lt = (int)(b.seq_off[ts + 1] - b.seq_off[ts]);
  const size_t ncell = (size_t)(Lq + 2) * (Lt + 2);
  std::vector<float> F(ncell), sim(ncell, 0.f);
  std::vector<int32_t> pq(ncell), pt(ncell);
  if (aadp_batch_fetch_pair(c, pair_id, F.data(), pq.data(), pt.data(), nullptr, nullptr, nullptr, nullptr)) return 1;
  // SimilarityMatrix (simmatrix.h:40-73): interior = substitution score of the two residues, borders 0
  std::vector<uint8_t> qr((size_t)Lq + 1), tr((size_t)Lt + 1);
  if (!b.have_seqs) return fail("the batch has no resident residues");
  if (Lq) CK(cudaMemcpyAsync(qr.data(), c->residues.as<uint8_t>() + b.seq_off[qs], (size_t)Lq, cudaMemcpyDeviceToHost, c->stream));
  if (Lt) CK(cudaMemcpyAsync(tr.data(), c->residues.as<uint8_t>() + b.seq_off[ts], (size_t)Lt, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const int A = c->sc.A;
  for (int i = 1; i <= Lq; ++i)
    for (int j = 1; j <= Lt; ++j)
      sim[(size_t)i * (Lt + 2) + j] = c->prof_mode ? c->proff_h[(size_t)(c->proff_off_h[(size_t)ts] + (int64_t)(j - 1) * A + qr[(size_t)i - 1])]
                                                   : c->subf_h[(size_t)qr[(size_t)i - 1] * A + tr[(size_t)j - 1]];
  PrunedParams Q;
  Q.Lq = Lq; Q.Lt = Lt;
  Q.F = F.data(); Q.pq = pq.data(); Q.pt = pt.data(); Q.sim = sim.data();
  Q.flags = subopt_flags;
  Q.gi = c->gi_f; Q.ge = c->ge_f;
  Q.delfree = c->sc.delfree; Q.insfree = c->sc.insfree;
  Q.delta_ratio = delta_ratio;
  Q.k_limit = k_limit; Q.sort_limit = sort_limit; Q.user_limit = user_limit; Q.max_overlap = max_overlap;
  Q.max_alignments = max_alignments;
  PrunedWalk W(Q);
  if (variant == AADP_PRUNE_KSORTED) W.run_ksorted(); else W.run_controlled();
  if (threshold) *threshold = W.threshold;
  *status = W.overflow ? 1 : 0;
  const size_t n_out = std::min<size_t>(W.as.size(), (size_t)max_alignments);
  *n_ali = (int32_t)n_out;
  int64_t at = 0;
  for (size_t k = 0; k < n_out; ++k) {
    const PrunedAlignment& a = W.as[k];
    if (scores) scores[k] = a.score;
    if (ali_len) ali_len[k] = (int32_t)a.back.size();
    if (paths) {
      if (at + (int64_t)a.back.size() > paths_cap) return fail("aadp_batch_near_optimal_pruned: paths buffer too small");
      for (size_t m = 0; m < a.back.size(); ++m) {  // front to back: (0,0) first
        const std::pair<int, int>& pr = a.back[a.back.size() - 1 - m];
        paths[2 * (at + (int64_t)m)] = pr.first;
        paths[2 * (at + (int64_t)m) + 1] = pr.second;
      }
    }
    at += (int64_t)a.back.size();
  }
  return 0;
}

int aadp_batch_near_optimal_constrained(aadp_ctx* c, const int64_t* pair_ids, int64_t n, const uint8_t* subopt_flags,
                                        const int64_t* flag_off, float delta_ratio, int32_t max_alignments, int32_t* n_ali,
                                        int32_t* status, float* scores, int32_t* ali_len, int64_t* path_off, int32_t* paths,
                                        int64_t paths_cap, float* threshold) {
  return near_optimal_impl(c, 1, subopt_flags, flag_off, pair_ids, n, delta_ratio, max_alignments, n_ali, status, scores, ali_len,
                           path_off, paths, paths_cap, threshold);
}

int aadp_fill_subpair(aadp_ctx* c, const uint8_t* q, int Lq, const uint8_t* t, int Lt, int q1_end, int t1_end, int q2_beg,
                      int t2_beg, int direction, float* score, int32_t* prev_q, int32_t* prev_t) {
  if (check_ctx(c, true)) return 1;
  if (c->prof_mode)
    return fail("aadp_fill_subpair: sub-rectangle fills run on the exact fp32 kernels, which profile scoring does not drive; use "
                "aadp_fill_pair_general with a rectangle and the profile's similarity matrix");
  if (Lq < 0 || Lt < 0) return fail("Illegal bounds building DPM");
  if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
  // dpmatrix.h:360-361 (and the matrix limits the reference does not check)
  if (q2_beg <= q1_end || t2_beg <= t1_end) return fail("Illegal bounds building DPM");
  if (q1_end < 0 || t1_end < 0 || q2_beg > Lq + 1 || t2_beg > Lt + 1) return fail("sub-rectangle anchors outside the matrix");
  std::vector<uint8_t> res((size_t)Lq + Lt + 1);
  if (Lq) memcpy(res.data(), q, Lq);
  if (Lt) memcpy(res.data() + Lq, t, Lt);
  const int64_t off[3] = {0, Lq, (int64_t)Lq + Lt};
  const int32_t pq = 0, pt = 1;
  if (aadp_upload_batch(c, res.data(), off, 2, &pq, &pt, 1, 0)) return 1;
  const int64_t n = (int64_t)(Lq + 2) * (Lt + 2);
  const std::vector<int64_t> doff = {0, n};
  const int rect[4] = {q1_end, t1_end, q2_beg, t2_beg};
  const int d = direction - 1;
  c->launches = 0;
  if (gg_fill(c, 0, 1, 1 << d, true, doff, nullptr, nullptr, rect)) return 1;
  if (score) CK(cudaMemcpyAsync(score, c->gg_score[d].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prev_q) CK(cudaMemcpyAsync(prev_q, c->gg_pq[d].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prev_t) CK(cudaMemcpyAsync(prev_t, c->gg_pt[d].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->b.ran_what = 0;
  return 0;
}

int aadp_fill_subpair_batch(aadp_ctx* c, const uint8_t* residues, const int64_t* seq_off, int64_t nseq, const int32_t* item_q,
                            const int32_t* item_t, const int32_t* rects, int64_t nitems, int direction, float* score,
                            int64_t* ali_off, int32_t* pairs, int64_t pairs_cap, int32_t* n_out, int32_t* status) {
  if (check_ctx(c, true)) return 1;
  if (c->prof_mode)
    return fail("aadp_fill_subpair_batch: sub-rectangle fills run on the exact fp32 kernels, which profile scoring does not drive; "
                "use aadp_fill_pair_general with a rectangle and the profile's similarity matrix");
  if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
  if (nitems < 0 || nitems > 0x7fffffff) return fail("bad batch size");
  if (nitems && (!item_q || !item_t || !rects || !seq_off)) return fail("null input");
  if (direction == AADP_REV && (pairs || n_out || status))
    return fail("aadp_fill_subpair_batch: sub-alignments are traced over forward fills only (optimal_subali.h:59-83)");
  // bounds (dpmatrix.h:360-361 and the matrix limits), slots and compact cell offsets
  std::vector<int64_t> cap((size_t)nitems + 1, 0), cells((size_t)nitems, 0);
  for (int64_t k = 0; k < nitems; ++k) {
    const int32_t* r = rects + 4 * k;
    if (item_q[k] < 0 || item_q[k] >= nseq || item_t[k] < 0 || item_t[k] >= nseq) return fail("sequence id out of range");
    const int64_t Lq = seq_off[item_q[k] + 1] - seq_off[item_q[k]], Lt = seq_off[item_t[k] + 1] - seq_off[item_t[k]];
    if (r[2] <= r[0] || r[3] <= r[1]) return fail("Illegal bounds building DPM");
    if (r[0] < 0 || r[1] < 0 || r[2] > Lq + 1 || r[3] > Lt + 1) return fail("sub-rectangle anchors outside the matrix");
    cap[(size_t)k + 1] = cap[(size_t)k] + (r[2] - r[0] + 1);
    cells[(size_t)k] = (int64_t)(r[2] - r[0] + 1) * (r[3] - r[1] + 1);
  }
  if (ali_off) memcpy(ali_off, cap.data(), (size_t)(nitems + 1) * 8);
  if (nitems == 0 || (!score && !pairs && !n_out && !status)) return 0;
  if (pairs && pairs_cap < cap[(size_t)nitems]) return fail("aadp_fill_subpair_batch: pairs buffer too small (needs 2*ali_off[nitems] ints)");
  if (aadp_upload_batch(c, residues, seq_off, nseq, item_q, item_t, nitems, 0)) return 1;
  const int d = direction - 1;
  const bool trace = d == 0 && (pairs || n_out || status);
  c->launches = 0;
  if (c->gg_fin[d].reserve((size_t)nitems * 4)) return 1;
  if (trace) {
    if (pin_reserve(c, (size_t)(nitems + 1) * 8 + 4096)) return 1;
    if (upload_vec(c, c->ali_cap, cap)) return 1;
    if (c->ali_out.reserve((size_t)cap[(size_t)nitems] * 8) || c->ali_n.reserve((size_t)nitems * 4) ||
        c->ali_status.reserve((size_t)nitems * 4)) return 1;
  }
  std::vector<int64_t> off;
  for (int64_t p0 = 0; p0 < nitems;) {
    off.assign(1, 0);
    int64_t p1 = p0;
    while (p1 < nitems && (p1 == p0 || off.back() + cells[(size_t)p1] <= c->gg_budget_cells)) {
      off.push_back(off.back() + cells[(size_t)p1]);
      ++p1;
    }
    const int64_t n = p1 - p0;
    if (gg_fill(c, p0, n, 1 << d, trace, off, d ? nullptr : c->gg_fin[0].as<float>(), d ? c->gg_fin[1].as<float>() : nullptr,
                rects + 4 * p0, nullptr, true)) return 1;
    if (trace) {
      SubTraceParams T{};
      T.PQ = c->gg_pq[0].as<int32_t>();
      T.PT = c->gg_pt[0].as<int32_t>();
      T.D = c->gg_score[0].as<float>();
      T.dense_off = c->gg_off.as<int64_t>();
      T.rects = c->gg_rect.as<int4>();
      T.cap_off = c->ali_cap.as<int64_t>();
      T.item0 = (int)p0;
      T.n = (int)n;
      T.out = c->ali_out.as<int2>();
      T.out_n = c->ali_n.as<int32_t>();
      T.out_status = c->ali_status.as<int32_t>();
      T.out_score = nullptr;
      c->prof_begin("subali_trace_kernel", 0);
      subali_trace_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(T);
      c->prof_end();
      CK(cudaGetLastError());
      c->launches++;
    }
    p0 = p1;
  }
  c->d2h_bytes = 0;
  if (score) { CK(cudaMemcpyAsync(score, c->gg_fin[d].p, (size_t)nitems * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += nitems * 4; }
  if (pairs) { CK(cudaMemcpyAsync(pairs, c->ali_out.p, (size_t)cap[(size_t)nitems] * 8, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += cap[(size_t)nitems] * 8; }
  if (n_out) { CK(cudaMemcpyAsync(n_out, c->ali_n.p, (size_t)nitems * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += nitems * 4; }
  if (status) { CK(cudaMemcpyAsync(status, c->ali_status.p, (size_t)nitems * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += nitems * 4; }
  CK(cudaStreamSynchronize(c->stream));
  c->b.ran_what = 0;
  return 0;
}

int aadp_fill_pair_general(aadp_ctx* c, const float* sim, int Lq, int Lt, float gi, float ge, int align_type, uint32_t flags,
                           int direction, const int* rect, float* score, int32_t* prev_q, int32_t* prev_t) {
  if (check_ctx(c, false)) return 1;
  if (Lq < 0 || Lt < 0) return fail("Illegal bounds building DPM");
  if (!sim) return fail("null argument");
  if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
  if (align_type < 0 || align_type > 4) return fail("Illegal gap style");
  if (!(gi >= 0.f) || !(ge >= 0.f)) return fail("gap penalties must be non-negative");
  if (rect) {
    if (rect[2] <= rect[0] || rect[3] <= rect[1]) return fail("Illegal bounds building DPM");
    if (rect[0] < 0 || rect[1] < 0 || rect[2] > Lq + 1 || rect[3] > Lt + 1) return fail("sub-rectangle anchors outside the matrix");
  }
  // a one-pair batch without residues: the similarity matrix carries everything the fill needs
  Batch& b = c->b;
  b.nseq = 2;
  b.npairs = 1;
  b.seq_off = {0, Lq, (int64_t)Lq + Lt};
  b.pair_q = {0};
  b.pair_t = {1};
  b.have_seqs = false;
  b.ran_what = 0;
  b.uploaded_what = 0;
  b.sched_ok = false;
  b.tb_off.clear();
  CK(cudaStreamSynchronize(c->stream));
  if (pin_reserve(c, 4096)) return 1;
  if (upload_vec(c, c->seq_off, b.seq_off) || upload_vec(c, c->pair_q, b.pair_q) || upload_vec(c, c->pair_t, b.pair_t)) return 1;
  if (c->residues.reserve((size_t)Lq + Lt + 16)) return 1;
  CK(cudaMemsetAsync(c->residues.p, 0, (size_t)Lq + Lt + 16, c->stream));
  const int64_t n = (int64_t)(Lq + 2) * (Lt + 2);
  if (c->scratch_d.reserve((size_t)n * 4)) return 1;
  CK(cudaMemcpyAsync(c->scratch_d.p, sim, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));  // gg_fill recycles the pinned pool; the caller's sim buffer is free again
  const std::vector<int64_t> doff = {0, n};
  GeneralOverride ov{gi, ge, align_type, flags, c->scratch_d.as<float>(), nullptr, nullptr, nullptr, 0, nullptr, nullptr};
  const int d = direction - 1;
  c->launches = 0;
  if (gg_fill(c, 0, 1, 1 << d, true, doff, nullptr, nullptr, rect, &ov)) return 1;
  if (score) CK(cudaMemcpyAsync(score, c->gg_score[d].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prev_q) CK(cudaMemcpyAsync(prev_q, c->gg_pq[d].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prev_t) CK(cudaMemcpyAsync(prev_t, c->gg_pt[d].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int aadp_fill_pair_tabulated(aadp_ctx* c, const float* sim, int Lq, int Lt, const float* del_tab, const float* ins_tab,
                             int is_local, uint32_t flags, int direction, float* score, int32_t* prev_q, int32_t* prev_t) {
  if (check_ctx(c, false)) return 1;
  if (Lq < 0 || Lt < 0) return fail("Illegal bounds building DPM");
  if (!sim || !del_tab || !ins_tab) return fail("null argument");
  if (direction != AADP_FWD && direction != AADP_REV) return fail("bad direction");
  const int sz1 = Lq + 2, sz2 = Lt + 2;
  // every evaluator of the reference returns 0 for adjacent positions (aasubalib.h:36,62; hmap_eval.h:69,95;
  // gn2_eval.h:104,138) and the kernel relies on it for the final cell; refuse a table that says otherwise
  for (int k = 0; k + 1 < sz2; ++k)
    if (del_tab[(size_t)k * sz2 + k + 1] != 0.f) return fail("tabulated gap model: deletion between adjacent positions must be 0");
  for (int j = 0; j < sz2; ++j)
    if (ins_tab[j] != 0.f) return fail("tabulated gap model: insertion between adjacent positions must be 0");
  Batch& b = c->b;
  b.nseq = 2;
  b.npairs = 1;
  b.seq_off = {0, Lq, (int64_t)Lq + Lt};
  b.pair_q = {0};
  b.pair_t = {1};
  b.have_seqs = false;
  b.ran_what = 0;
  b.uploaded_what = 0;
  b.sched_ok = false;
  b.tb_off.clear();
  CK(cudaStreamSynchronize(c->stream));
  if (pin_reserve(c, 4096)) return 1;
  if (upload_vec(c, c->seq_off, b.seq_off) || upload_vec(c, c->pair_q, b.pair_q) || upload_vec(c, c->pair_t, b.pair_t)) return 1;
  if (c->residues.reserve((size_t)Lq + Lt + 16)) return 1;
  CK(cudaMemsetAsync(c->residues.p, 0, (size_t)Lq + Lt + 16, c->stream));
  const int64_t n = (int64_t)sz1 * sz2, nd = (int64_t)sz2 * sz2, ni = (int64_t)(Lq + 1) * sz2;
  std::vector<float> delT((size_t)nd);
  for (int x = 0; x < sz2; ++x)
    for (int y = 0; y < sz2; ++y) delT[(size_t)y * sz2 + x] = del_tab[(size_t)x * sz2 + y];
  // one scratch block: sim | del | del^T | ins
  if (c->scratch_d.reserve((size_t)(n + 2 * nd + ni) * 4)) return 1;
  float* d = c->scratch_d.as<float>();
  CK(cudaMemcpyAsync(d, sim, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(d + n, del_tab, (size_t)nd * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(d + n + nd, delT.data(), (size_t)nd * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(d + n + 2 * nd, ins_tab, (size_t)ni * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const std::vector<int64_t> doff = {0, n};
  GeneralOverride ov{0.f, 0.f, is_local ? AADP_LOCAL : AADP_GLOBAL, flags, d, d + n, d + n + nd, d + n + 2 * nd, is_local ? 1 : 0, nullptr, nullptr};
  const int dd = direction - 1;
  c->launches = 0;
  if (gg_fill(c, 0, 1, 1 << dd, true, doff, nullptr, nullptr, nullptr, &ov)) return 1;
  if (score) CK(cudaMemcpyAsync(score, c->gg_score[dd].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prev_q) CK(cudaMemcpyAsync(prev_q, c->gg_pq[dd].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prev_t) CK(cudaMemcpyAsync(prev_t, c->gg_pt[dd].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int aadp_fill_batch_tabulated(aadp_ctx* c, int64_t n, const int32_t* Lq, const int32_t* Lt, const float* sim, const int64_t* sim_off,
                              const float* del_tab, const int64_t* del_off, const float* ins_tab, const int64_t* ins_off,
                              int is_local, uint32_t flags, int direction, float* fwd_score, float* rev_score, int64_t* ali_off,
                              int32_t* pairs, int64_t pairs_cap, int32_t* n_out, int32_t* status) {
  if (check_ctx(c, false)) return 1;
  if (n < 0 || n > 0x3fffffff) return fail("bad batch size");
  if (n && (!Lq || !Lt || !sim || !sim_off || !del_tab || !del_off || !ins_tab || !ins_off)) return fail("null argument");
  if (direction < 1 || direction > 3) return fail("bad direction");
  const bool want_ali = pairs || n_out || status;
  if (want_ali && (is_local || !(direction & 1))) return fail("aadp_fill_batch_tabulated: optimal alignments are traced over non-local forward fills");
  std::vector<int64_t> cap((size_t)n + 1, 0), cells((size_t)n);
  for (int64_t k = 0; k < n; ++k) {
    if (Lq[k] < 0 || Lt[k] < 0) return fail("Illegal bounds building DPM");
    const int sz2 = Lt[k] + 2;
    const float* dt = del_tab + del_off[k];
    const float* it = ins_tab + ins_off[k];
    for (int x = 0; x + 1 < sz2; ++x)
      if (dt[(size_t)x * sz2 + x + 1] != 0.f) return fail("tabulated gap model: deletion between adjacent positions must be 0");
    for (int j = 0; j < sz2; ++j)
      if (it[j] != 0.f) return fail("tabulated gap model: insertion between adjacent positions must be 0");
    cap[(size_t)k + 1] = cap[(size_t)k] + Lq[k] + 2;
    cells[(size_t)k] = (int64_t)(Lq[k] + 2) * sz2;
  }
  if (ali_off) memcpy(ali_off, cap.data(), (size_t)(n + 1) * 8);
  if (n == 0 || (!fwd_score && !rev_score && !want_ali)) return 0;
  if (pairs && pairs_cap < cap[(size_t)n]) return fail("aadp_fill_batch_tabulated: pairs buffer too small (needs 2*ali_off[n] ints)");
  // a batch without residues: item k is the pair of sequences 2k (Lq[k] positions) and 2k+1 (Lt[k] positions)
  Batch& b = c->b;
  b.nseq = 2 * n;
  b.npairs = n;
  b.seq_off.assign((size_t)(2 * n + 1), 0);
  b.pair_q.resize((size_t)n);
  b.pair_t.resize((size_t)n);
  for (int64_t k = 0; k < n; ++k) {
    b.seq_off[(size_t)(2 * k + 1)] = b.seq_off[(size_t)(2 * k)] + Lq[k];
    b.seq_off[(size_t)(2 * k + 2)] = b.seq_off[(size_t)(2 * k + 1)] + Lt[k];
    b.pair_q[(size_t)k] = (int32_t)(2 * k);
    b.pair_t[(size_t)k] = (int32_t)(2 * k + 1);
  }
  b.have_seqs = false;
  b.ran_what = 0;
  b.uploaded_what = 0;
  b.sched_ok = false;
  b.tb_off.clear();
  CK(cudaStreamSynchronize(c->stream));
  if (pin_reserve(c, (size_t)(2 * n + 1) * 8 + (size_t)n * 8 + (size_t)(n + 1) * 8 + 4096)) return 1;
  if (upload_vec(c, c->seq_off, b.seq_off) || upload_vec(c, c->pair_q, b.pair_q) || upload_vec(c, c->pair_t, b.pair_t)) return 1;
  const size_t nres = (size_t)b.seq_off.back() + 16;
  if (c->residues.reserve(nres)) return 1;
  CK(cudaMemsetAsync(c->residues.p, 0, nres, c->stream));
  if (want_ali) {
    if (upload_vec(c, c->ali_cap, cap)) return 1;
    if (c->ali_out.reserve((size_t)cap[(size_t)n] * 8) || c->ali_n.reserve((size_t)n * 4) || c->ali_status.reserve((size_t)n * 4)) return 1;
  }
  if (c->gg_fin[0].reserve((size_t)n * 4) || c->gg_fin[1].reserve((size_t)n * 4)) return 1;
  CK(cudaStreamSynchronize(c->stream));
  c->launches = 0;
  c->h2d_bytes = 0;
  const int dirmask = direction;
  std::vector<int64_t> off, doff, ioff;
  std::vector<int32_t> rects;
  for (int64_t p0 = 0; p0 < n;) {
    // one chunk: dense outputs + sim share the offsets `off`; the tables are packed next to each other
    off.assign(1, 0);
    doff.clear();
    ioff.clear();
    int64_t nd_cells = 0, ni_cells = 0, p1 = p0;
    while (p1 < n && (p1 == p0 || off.back() + cells[(size_t)p1] <= c->gg_budget_cells / 4)) {
      off.push_back(off.back() + cells[(size_t)p1]);
      doff.push_back(nd_cells);
      ioff.push_back(ni_cells);
      nd_cells += (int64_t)(Lt[p1] + 2) * (Lt[p1] + 2);
      ni_cells += (int64_t)(Lq[p1] + 1) * (Lt[p1] + 2);
      ++p1;
    }
    const int64_t m = p1 - p0;
    if (c->scratch_d.reserve((size_t)off.back() * 4) || c->tb_del.reserve((size_t)nd_cells * 4) || c->tb_ins.reserve((size_t)ni_cells * 4)) return 1;
    for (int64_t k = p0; k < p1; ++k) {
      const int64_t sz2 = Lt[k] + 2;
      CK(cudaMemcpyAsync(c->scratch_d.as<float>() + off[(size_t)(k - p0)], sim + sim_off[k], (size_t)cells[(size_t)k] * 4, cudaMemcpyHostToDevice, c->stream));
      CK(cudaMemcpyAsync(c->tb_del.as<float>() + doff[(size_t)(k - p0)], del_tab + del_off[k], (size_t)(sz2 * sz2) * 4, cudaMemcpyHostToDevice, c->stream));
      CK(cudaMemcpyAsync(c->tb_ins.as<float>() + ioff[(size_t)(k - p0)], ins_tab + ins_off[k], (size_t)((Lq[k] + 1) * sz2) * 4, cudaMemcpyHostToDevice, c->stream));
      c->h2d_bytes += (cells[(size_t)k] + sz2 * sz2 + (Lq[k] + 1) * sz2) * 4;
    }
    CK(cudaStreamSynchronize(c->stream));
    if (pin_reserve(c, (size_t)m * 16 + 4096)) return 1;
    if (upload_vec(c, c->tb_del_off, doff) || upload_vec(c, c->tb_ins_off, ioff)) return 1;
    CK(cudaStreamSynchronize(c->stream));  // gg_fill recycles the pinned pool
    GeneralOverride ov{0.f, 0.f, is_local ? AADP_LOCAL : AADP_GLOBAL, flags, c->scratch_d.as<float>(), c->tb_del.as<float>(), nullptr,
                       c->tb_ins.as<float>(), is_local ? 1 : 0, c->tb_del_off.as<int64_t>(), c->tb_ins_off.as<int64_t>()};
    if (gg_fill(c, p0, m, dirmask, true, off, c->gg_fin[0].as<float>(), c->gg_fin[1].as<float>(), nullptr, &ov)) return 1;
    if (want_ali) {  // Optimal::enumerate (optimal.h:47-75) = the sub-alignment walk over the whole matrix
      rects.resize((size_t)m * 4);
      for (int64_t k = p0; k < p1; ++k) {
        rects[(size_t)(k - p0) * 4] = 0;
        rects[(size_t)(k - p0) * 4 + 1] = 0;
        rects[(size_t)(k - p0) * 4 + 2] = Lq[k] + 1;
        rects[(size_t)(k - p0) * 4 + 3] = Lt[k] + 1;
      }
      CK(cudaStreamSynchronize(c->stream));
      if (pin_reserve(c, (size_t)m * 16 + 4096)) return 1;
      if (upload_vec(c, c->gg_rect, rects)) return 1;
      SubTraceParams T{};
      T.PQ = c->gg_pq[0].as<int32_t>();
      T.PT = c->gg_pt[0].as<int32_t>();
      T.D = c->gg_score[0].as<float>();
      T.dense_off = c->gg_off.as<int64_t>();
      T.rects = c->gg_rect.as<int4>();
      T.cap_off = c->ali_cap.as<int64_t>();
      T.item0 = (int)p0;
      T.n = (int)m;
      T.out = c->ali_out.as<int2>();
      T.out_n = c->ali_n.as<int32_t>();
      T.out_status = c->ali_status.as<int32_t>();
      T.out_score = nullptr;
      c->prof_begin("subali_trace_kernel", 0);
      subali_trace_kernel<<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(T);
      c->prof_end();
      CK(cudaGetLastError());
      c->launches++;
      CK(cudaStreamSynchronize(c->stream));
    }
    p0 = p1;
  }
  c->d2h_bytes = 0;
  if (fwd_score && (direction & 1)) { CK(cudaMemcpyAsync(fwd_score, c->gg_fin[0].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += n * 4; }
  if (rev_score && (direction & 2)) { CK(cudaMemcpyAsync(rev_score, c->gg_fin[1].p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += n * 4; }
  if (pairs) { CK(cudaMemcpyAsync(pairs, c->ali_out.p, (size_t)cap[(size_t)n] * 8, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += cap[(size_t)n] * 8; }
  if (n_out) { CK(cudaMemcpyAsync(n_out, c->ali_n.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += n * 4; }
  if (status) { CK(cudaMemcpyAsync(status, c->ali_status.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream)); c->d2h_bytes += n * 4; }
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

}  // extern "C"
