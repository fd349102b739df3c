// libb200snark: C-ABI entry points (include/b200snark.h) and the host-side
// orchestration of the CUDA kernels.  Device-only: there is no CPU fallback —
// every entry point fails with B200_ENODEVICE when no CUDA device is usable.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>
#include <algorithm>

#include "b200snark.h"
#include "msm.cuh"
#include "bucket_affine.cuh"
#include "poly_host.cuh"
#include "qap.cuh"
#include "qap_sparse.cuh"
#include "comm.cuh"
#include "shard_partition.h"
#include "glv.cuh"
#ifndef B200_NO_PAIRING
#include "pairing.cuh"
#include "pairing_warp.cuh"
#include "verify_batch.cuh"
#include "verify_batch_pinocchio.cuh"
#endif

using namespace b200;

namespace {

std::mutex g_mu;
std::string g_err;
bool g_init = false;
int g_device = -1;
cudaStream_t g_stream = nullptr;
cudaStream_t g_side[4] = {nullptr, nullptr, nullptr, nullptr};  // side streams: independent MSMs of one proof overlap
// Second prove context (B200_CFG_PK_CONTEXT): a proving key loaded under context 1 runs on its own side streams and
// polynomial workspace, so a proof on it can be in flight beside a proof on a context-0 key (two proofs pipelined on two
// caller streams: the latency-bound sort / tail / product chains of one overlap the accumulation of the other).
cudaStream_t g_side1[4] = {nullptr, nullptr, nullptr, nullptr};
cudaStream_t g_stream1 = nullptr;   // context 1's main stream (host-pointer entry points)
int g_pk_ctx = 0;
int g_pairing_kernel = 0;   // B200_CFG_PAIRING_KERNEL: 0 auto, 1 one thread per pairing, 2 one warp per pairing
int* g_d_err = nullptr;  // device error flags (bit0: coordinate >= q, bit1: scalar >= r, bit2: zero leading coeff)
std::unique_ptr<PolyCtx> g_poly, g_poly1;

Comm g_comm;  // NCCL communicator of this process (b200_comm_init); world 1 = none

// b200_config: bucket-accumulation kernel of base sets / proving keys created afterwards
// (0 auto: batched affine where the bucket population and the shard size amortise its rounds, else XYZZ; 1, 2 force)
int g_acc_mode = 0;
// partition tuning (b200_config keys 10..13; defaults = the measured best, profiles/r2_notes.md §8)
int g_w_ab = 100, g_w_g2 = 280, g_aff_min_g1 = 700000, g_aff_min_g2 = 400000;
int g_tma_staging = 0;   // B200_CFG_TMA_STAGING: 1 staged backward pass in every round, 2 only in the contiguous rounds (>= 2)

// ---- instrumentation (bench.py): kernel-launch counter and optional CUDA-event
// timing of the dominant kernel (k_accumulate), per group.
unsigned long long g_launches = 0;
bool g_prof = false;
bool g_serial = false;  // measurement mode: issue every MSM of a proof on the caller's stream (exclusive kernel timings)
struct ProfRec { cudaEvent_t e0, e1; int group; size_t terms; };
std::vector<ProfRec> g_prof_recs;
std::vector<cudaEvent_t> g_event_pool;
cudaEvent_t prof_event() {
  if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CU(call)                                                                             \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return fail(e_ == cudaErrorMemoryAllocation ? B200_ENOMEM : B200_ECUDA, "%s:%d %s: %s", \
                  __FILE__, __LINE__, #call, cudaGetErrorString(e_));                        \
  } while (0)

#define NEED_INIT()                                                                      \
  do {                                                                                   \
    if (!g_init) {                                                                       \
      int rc_ = init_locked(-1);                                                         \
      if (rc_) return rc_;                                                               \
    } else {                                                                             \
      cudaSetDevice(g_device);                                                           \
    }                                                                                    \
  } while (0)

int init_locked(int device) {
  if (g_init) {
    if (device >= 0 && device != g_device) return fail(B200_EINVAL, "already initialised on device %d", g_device);
    return B200_OK;
  }
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(B200_ENODEVICE, "no CUDA device (%s); libb200snark has no CPU fallback",
                e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
  if (device < 0) {
    if (cudaGetDevice(&device) != cudaSuccess) device = 0;
  }
  if (device >= count) return fail(B200_EINVAL, "device %d out of range (%d devices)", device, count);
  CU(cudaSetDevice(device));
  CU(cudaStreamCreateWithFlags(&g_stream, cudaStreamNonBlocking));
  for (auto& sd : g_side) CU(cudaStreamCreateWithFlags(&sd, cudaStreamNonBlocking));  // (stream priorities: no measurable effect)
  CU(cudaMalloc(&g_d_err, sizeof(int)));
  CU(cudaMemset(g_d_err, 0, sizeof(int)));
  for (auto& sd : g_side1) CU(cudaStreamCreateWithFlags(&sd, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&g_stream1, cudaStreamNonBlocking));
  g_poly = std::make_unique<PolyCtx>();
  g_poly->launch_counter = &g_launches;
  g_poly1 = std::make_unique<PolyCtx>();
  g_poly1->launch_counter = &g_launches;
  g_device = device;
  g_init = true;
  return B200_OK;
}

inline unsigned nblocks(size_t n, unsigned bs) { return nblk(n, bs); }

int pick_window_bits(size_t n) {
  // cost model: nwin*n bucket adds (~10 M) + 2*2^(c-1) reduction adds (~14 M), see DESIGN.md §3
  int best = 8;
  double best_cost = 1e300;
  for (int c = 8; c <= 18; c++) {
    double nwin = (255 + c - 1) / c;
    double cost = nwin * (double)n * 10.0 + 2.0 * (double)(1u << (c - 1)) * 14.0 * 4.0;
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}

// Output of the digit-recode / counting-sort front end for one scalar vector.  It depends only on the
// scalars and the window shape, so base sets that consume the SAME scalars (A, B1, B2 of a Groth16
// proof) share one SortScratch read-only.
struct SortScratch {
  MsmShape sh{};            // shape it was allocated for (n = capacity)
  DevBuf counts, offsets, cursor, entries, slice_off, slice_start, slice_end;
  uint32_t max_slices = 0;
  uint32_t slice_S = 0;     // > 0: fixed-size slices of S slots (batched-affine mode)
  SliceTables tables() const { return SliceTables{slice_off.as<uint32_t>(), slice_start.as<uint32_t>(), slice_end.as<uint32_t>()}; }
};

struct Bases {
  int group = 0;  // 1: G1 (Fq), 2: G2 (Fq2)
  size_t n = 0;
  MsmShape sh{};
  DevBuf table;    // [nwin][n] Affine<F>
  // per-base-set scratch of the bucket phase (different base sets may run concurrently)
  DevBuf scalars;  // n * 32 B (host-scalar entry points)
  DevBuf slice_out, buckets, partials, result, out_std;
  SortScratch sort;  // own front-end scratch (stand-alone MSMs)
  uint32_t nseg = 0, seg = 0;
  // batched-affine accumulation (affine_S > 0): ping-pong node buffers, prefix products, per-thread / per-block products
  uint32_t affine_S = 0;
  DevBuf nodeA, nodeB, aff_pre, aff_others, aff_btot, aff_ids;
};

int sort_alloc(SortScratch& ss, const MsmShape& sh, uint32_t slice_S) {
  ss.sh = sh;
  ss.slice_S = slice_S;
  size_t entries = (size_t)sh.nwin * sh.n;
  CU(ss.counts.alloc((sh.nbuckets + 2) * sizeof(uint32_t)));
  CU(ss.offsets.alloc((sh.nbuckets + 3) * sizeof(uint32_t)));
  CU(ss.cursor.alloc((sh.nbuckets + 2) * sizeof(uint32_t)));
  CU(ss.entries.alloc(entries * sizeof(uint32_t)));
  // slices: every bucket owns >= 1; a bucket above cap = 2*mean entries is cut => at most B + B/2 + 1
  ss.max_slices = sh.nbuckets + sh.nbuckets / 2 + 2;
  if (slice_S) ss.max_slices = sh.nbuckets + (uint32_t)((entries + slice_S - 1) / slice_S) + 2;
  CU(ss.slice_off.alloc((sh.nbuckets + 3) * sizeof(uint32_t)));
  CU(ss.slice_start.alloc((size_t)ss.max_slices * sizeof(uint32_t)));
  CU(ss.slice_end.alloc((size_t)ss.max_slices * sizeof(uint32_t)));
  return B200_OK;
}

std::map<uint64_t, std::unique_ptr<Bases>> g_bases;
uint64_t g_next_handle = 1;

// Reads the device error flags behind everything queued on `st` and waits for the stream.  With `lk` (the library mutex,
// held by the caller) the wait itself runs UNLOCKED, so a second host thread can enqueue a proof on the other prove
// context meanwhile (two host-pointer proofs in flight, B200_CFG_PK_CONTEXT).
template <class F>
int check_err_flag(const char* what, cudaStream_t st = nullptr, std::unique_lock<std::mutex>* lk = nullptr, int* pinned = nullptr) {
  if (!st) st = g_stream;
  int h_local = 0;
  int* hp = pinned ? pinned : &h_local;   // `pinned`: a page-locked word, so the copy does not block the host under the mutex
  *hp = 0;
  CU(cudaMemcpyAsync(hp, g_d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
  if (lk) lk->unlock();
  cudaError_t se = cudaStreamSynchronize(st);
  if (lk) lk->lock();
  CU(se);
  const int h = *hp;
  if (h) {
    CU(cudaMemset(g_d_err, 0, sizeof(int)));
    if (h & 16) return fail(B200_EINVAL, "%s: tau is one of the interpolation points 1..n", what);
    if (h & 8) return fail(B200_EINVAL, "%s: q1[2] != Fq2.One() (G2 point at infinity; the reference panics, bn128.go:238-241)", what);
    if (h & 4) return fail(B200_EDIVZERO, "%s: divisor has a zero leading coefficient", what);
    return fail(B200_ERANGE, "%s: %s", what, (h & 1) ? "point coordinate >= q" : "scalar / coefficient >= r");
  }
  return B200_OK;
}

// prefer_affine: batched-affine bucket accumulation (6 multiplies per add instead of 10) whenever the buckets are
// populated enough to amortise its per-round launches; since the per-round inversion became a binary-Euclid warp
// (182 -> ~45 us) it also wins for a stand-alone MSM (2^20: G1 4.40 vs 4.46 ms, G2 9.26 vs 11.80 ms XYZZ).  A proving-key
// shard that leaves a rank only a small MSM passes false (prove_host.cuh); B200_ACC_MODE=xyzz|affine forces either.
template <class F>
int bases_create(const uint64_t* pts, size_t n, int c, int group, std::unique_ptr<Bases>& out_b, bool prefer_affine = true) {
  if (!pts || n == 0 || n > (1u << 26)) return fail(B200_EINVAL, "bases_load: bad arguments");
  if (c == 0) c = pick_window_bits(n);
  if (c < 2 || c > 24) return fail(B200_EINVAL, "window_bits must be in [2,24]");
  auto b = std::make_unique<Bases>();
  b->group = group;
  b->n = n;
  MsmShape& sh = b->sh;
  sh.n = (uint32_t)n;
  sh.c = (uint32_t)c;
  sh.nwin = (255 + c - 1) / c;
  sh.nbuckets = 1u << (c - 1);
  sh.table_stride = (uint32_t)n;
  if ((uint64_t)sh.nwin * n >= (1ull << 31)) return fail(B200_EINVAL, "nwin*n exceeds 2^31 entries");
  size_t entries = (size_t)sh.nwin * n;
  CU(b->table.alloc(entries * sizeof(Affine<F>)));
  CU(b->scalars.alloc(n * sizeof(Fr)));
  CU(b->buckets.alloc((size_t)sh.nbuckets * sizeof(XYZZ<F>)));
  {
    // accumulation mode: batched affine (6.5 multiplies per add, 3 launches per round) where the buckets are populated
    // enough to amortise the rounds, else XYZZ mixed adds (10 multiplies, one launch); b200_config forces either
    const bool xyzz_mode = g_acc_mode == 2 || (g_acc_mode == 0 && !prefer_affine);
    uint32_t S = 0;
    uint64_t mean = ((uint64_t)sh.nwin * n) / sh.nbuckets;
    const uint64_t min_mean = g_acc_mode == 1 ? 16 : 96;
    if (!xyzz_mode && mean >= min_mean) {
      S = 8;
      while (S < 128 && (uint64_t)S * 2 * 6 <= mean) S *= 2;   // largest power of two <= mean/6, in [8, 128]
    }
    b->affine_S = S;
    int rc_ = sort_alloc(b->sort, sh, S);
    if (rc_) return rc_;
    if (S) {
      size_t nsl = b->sort.max_slices;
      CU(b->nodeA.alloc(nsl * (S / 2) * sizeof(Affine<F>)));
      CU(b->nodeB.alloc(nsl * (S / 4 ? S / 4 : 1) * sizeof(Affine<F>)));
      CU(b->aff_pre.alloc(nsl * (S / 2) * sizeof(F)));
      CU(b->aff_ids.alloc(nsl * (S / 2) * sizeof(uint2)));
      size_t nblk_max = (nsl * (S / 2) + kAffBlock * kAffPairs - 1) / (kAffBlock * kAffPairs);
      CU(b->aff_others.alloc(nblk_max * kAffBlock * sizeof(F)));
      CU(b->aff_btot.alloc(nblk_max * sizeof(F)));
    }
  }
  CU(b->slice_out.alloc((size_t)(b->affine_S ? 1 : b->sort.max_slices) * sizeof(XYZZ<F>)));
  // short latency chain: 4-bucket segments (8 adds + one small scalar mul per thread), then a two-level tree sum
  b->seg = sh.nbuckets >= 256 ? 4 : 1;
  b->nseg = (sh.nbuckets + b->seg - 1) / b->seg;
  CU(b->partials.alloc(((size_t)b->nseg + 1024) * sizeof(XYZZ<F>)));
  CU(b->result.alloc(sizeof(XYZZ<F>)));
  CU(b->out_std.alloc(3 * sizeof(F)));

  // upload + normalise + window precompute
  DevBuf staging, state;
  CU(staging.alloc(n * 3 * sizeof(F)));
  CU(state.alloc(n * sizeof(XYZZ<F>)));
  CU(cudaMemcpyAsync(staging.p, pts, n * 3 * sizeof(F), cudaMemcpyHostToDevice, g_stream));
  Affine<F>* table = b->table.as<Affine<F>>();
  k_load_bases<F><<<nblocks(n, 128), 128, 0, g_stream>>>(staging.as<F>(), n, table, g_d_err);
  k_affine_to_xyzz<F><<<nblocks(n, 128), 128, 0, g_stream>>>(table, state.as<XYZZ<F>>(), n);
  for (uint32_t w = 1; w < sh.nwin; w++) {
    k_window_step<F><<<nblocks(n, 128), 128, 0, g_stream>>>(state.as<XYZZ<F>>(), n, c);
    constexpr int K = 8;
    k_batch_to_affine<F, K><<<nblocks((n + K - 1) / K, 128), 128, 0, g_stream>>>(state.as<XYZZ<F>>(), table + (size_t)w * n, n);
  }
  CU(cudaGetLastError());
  int rc = check_err_flag<F>("bases_load");
  if (rc) return rc;
  out_b = std::move(b);
  return B200_OK;
}

template <class F>
int bases_load(const uint64_t* pts, size_t n, int c, int group, b200_bases_t* out) {
  if (!out) return fail(B200_EINVAL, "bases_load: null handle pointer");
  std::unique_ptr<Bases> b;
  int rc = bases_create<F>(pts, n, c, group, b);
  if (rc) return rc;
  uint64_t h = g_next_handle++;
  g_bases[h] = std::move(b);
  *out = h;
  return B200_OK;
}

Bases* find_bases(b200_bases_t h, int group) {
  auto it = g_bases.find(h);
  if (it == g_bases.end()) return nullptr;
  if (group && it->second->group != group) return nullptr;
  return it->second.get();
}

// Enqueue one MSM on `st`; result XYZZ written to d_out (device).
// Accumulate launch: LPB lanes per bucket slice (2 / 4 / 8 by mean bucket population).  Register budget:
// G1 runs at 128 regs (4 CTAs/SM); occupancy / prefetch variants measured within 2% of each other
// (profiles/r1_notes.md) — the kernel is bound by the IMAD.WIDE issue rate, not by latency hiding.
template <class F, int LPB>
void launch_accumulate_l(const Affine<F>* table, const uint32_t* entries, SliceTables stb, uint32_t m,
                         XYZZ<F>* out, uint32_t max_slices, cudaStream_t st) {
  unsigned grid = nblocks((size_t)max_slices * LPB, 128);
  if constexpr (sizeof(F) == sizeof(Fq)) {
    k_accumulate<F, LPB, 4><<<grid, 128, 0, st>>>(table, entries, stb, m, out);
  } else {
    k_accumulate<F, LPB, 1><<<grid, 128, 0, st>>>(table, entries, stb, m, out);
  }
}
template <class F>
void launch_accumulate(int lpb, const Affine<F>* table, const uint32_t* entries, SliceTables stb, uint32_t m,
                       XYZZ<F>* out, uint32_t max_slices, cudaStream_t st) {
  switch (lpb) {
    case 2: launch_accumulate_l<F, 2>(table, entries, stb, m, out, max_slices, st); break;
    case 4: launch_accumulate_l<F, 4>(table, entries, stb, m, out, max_slices, st); break;
    default: launch_accumulate_l<F, 8>(table, entries, stb, m, out, max_slices, st); break;
  }
}

constexpr int kLPB = 8;

// d_out[0] = sum of partials[0..n): one block if small, else 512 inputs per first-level block + a final block.
// `partials` must have room for n + ceil(n/512) records.
template <class F>
void launch_tree_sum(XYZZ<F>* partials, uint32_t n, XYZZ<F>* d_out, cudaStream_t st) {
  if (n <= 1024) {
    k_sum_points<F><<<1, 256, 0, st>>>(partials, n, n, d_out);
    g_launches += 1;
    return;
  }
  uint32_t nb = (n + 511) / 512;
  k_sum_points<F><<<nb, 256, 0, st>>>(partials, n, 512, partials + n);
  k_sum_points<F><<<1, 256, 0, st>>>(partials + n, nb, nb, d_out);
  g_launches += 2;
}

// sum_b b * S_b over the bucket array -> one XYZZ record (msm.cuh: rows / columns, bit planes, Horner).  `scratch` holds
// H + K + (c - 1) + 1 records.  Tiny bucket sets keep the segment kernel.
template <class F>
void launch_bucket_tail(const XYZZ<F>* buckets, uint32_t c, XYZZ<F>* scratch, XYZZ<F>* d_out, cudaStream_t st) {
  const uint32_t bits = c - 1, kl = (bits + 1) / 2, kh = bits - kl, K = 1u << kl, H = 1u << kh;
  XYZZ<F>* R = scratch;
  XYZZ<F>* C = scratch + H;
  XYZZ<F>* planes = C + K;
  k_tail_rowcol<F><<<nblocks((size_t)(H + K) * 32, 128), 128, 0, st>>>(buckets, kl, H, R, C);
  k_tail_planes<F><<<nblocks((size_t)(bits + 1) * 32, 128), 128, 0, st>>>(R, C, kl, kh, planes);
  k_tail_horner<F><<<1, 32, 0, st>>>(planes, bits, d_out);
  g_launches += 3;
}

// Front end: signed-digit recode + counting sort of n scalars into bucket order (3 launches).
int msm_sort(SortScratch& ss, const MsmShape& shape, const Fr* d_scalars, size_t n, int mont, cudaStream_t st) {
  if (n > ss.sh.n || shape.c != ss.sh.c || shape.table_stride != ss.sh.table_stride)
    return fail(B200_EINVAL, "msm_sort: shape mismatch");
  MsmShape sh = shape;
  sh.n = (uint32_t)n;
  uint32_t m = sh.nbuckets + 1;  // counts[0] unused (digit 0), buckets 1..B
  // slice cap: twice the mean bucket population (uniform scalars never split), at least 4 per lane
  uint64_t mean = ((uint64_t)sh.nwin * n + sh.nbuckets - 1) / sh.nbuckets;
  uint32_t cap = (uint32_t)(2 * mean < 4 * kLPB ? 4 * kLPB : 2 * mean);
  int fixed = 0;
  if (ss.slice_S) {
    cap = ss.slice_S;
    fixed = 1;
  }
  uint32_t* counts = ss.counts.as<uint32_t>();
  CU(cudaMemsetAsync(counts, 0, (m + 1) * sizeof(uint32_t), st));
  if (n) k_digits_count<<<nblocks(n, 256), 256, 0, st>>>(d_scalars, sh, mont, counts, g_d_err);
  k_scan<<<1, 1024, 0, st>>>(counts, m, cap, fixed, ss.offsets.as<uint32_t>(), ss.cursor.as<uint32_t>(), ss.tables());
  k_fill_slices<<<nblocks(m, 256), 256, 0, st>>>(counts, ss.offsets.as<uint32_t>(), m, cap, fixed, ss.tables());
  if (n) k_digits_scatter<<<nblocks(n, 256), 256, 0, st>>>(d_scalars, sh, mont, ss.cursor.as<uint32_t>(),
                                                           ss.entries.as<uint32_t>(), g_d_err);
  g_launches += n ? 4 : 2;
  CU(cudaGetLastError());
  return B200_OK;
}

// Back end: bucket accumulation over the sorted entries of `ss`, slice merge, weighted bucket
// reduction and final tree sum -> one XYZZ record in d_out (4 launches).
template <class F>
int msm_buckets(Bases* b, const SortScratch& ss, size_t n_terms, XYZZ<F>* d_out, cudaStream_t st) {
  const MsmShape& sh = b->sh;
  if (ss.sh.c != sh.c || ss.sh.table_stride != sh.table_stride || ss.max_slices != b->sort.max_slices ||
      ss.slice_S != b->sort.slice_S)
    return fail(B200_EINVAL, "msm_buckets: sort scratch does not match the base set");
  uint32_t m = sh.nbuckets + 1;
  XYZZ<F>* buckets = b->buckets.as<XYZZ<F>>();
  XYZZ<F>* partials = b->partials.as<XYZZ<F>>();
  SliceTables stb = ss.tables();
  // The out-of-line F_q multiply wins here: the fully inlined madd body (~38 KB of SASS) thrashes the
  // instruction caches (measured 5.85 ms vs 4.80 ms at 2^20, profiles/r1_notes.md).
  ProfRec pr{};
  if (g_prof) {
    pr = ProfRec{prof_event(), prof_event(), b->group, n_terms};
    cudaEventRecord(pr.e0, st);
  }
  if (b->affine_S) {
    if (ss.slice_S != b->affine_S) return fail(B200_EINVAL, "msm_buckets: slice size mismatch");
    const uint32_t S = b->affine_S;
    uint32_t R = 0;
    while ((1u << R) < S) R++;
    // host-side bound on the live slice count for this call (the exact count lives on the device)
    uint64_t total = (uint64_t)sh.nwin * n_terms;
    uint64_t nsl_bound = (uint64_t)sh.nbuckets + (total + S - 1) / S + 2;
    if (nsl_bound > ss.max_slices) nsl_bound = ss.max_slices;
    AffineRound<F> ar{};
    ar.table = b->table.as<Affine<F>>();
    ar.entries = ss.entries.as<uint32_t>();
    ar.slice_start = stb.slice_start;
    ar.slice_end = stb.slice_end;
    ar.nslices_ptr = stb.slice_off + m;
    ar.pre = b->aff_pre.as<F>();
    ar.others = b->aff_others.as<F>();
    ar.btot = b->aff_btot.as<F>();
    ar.pair_ids = g_tma_staging == 1 ? b->aff_ids.as<uint2>() : nullptr;
    // node buffers, x- and y-coordinates in separate halves (bucket_affine.cuh NodeBuf)
    const size_t capA = (size_t)ss.max_slices * (S / 2), capB = (size_t)ss.max_slices * (S / 4 ? S / 4 : 1);
    NodeBuf<F> bufs[2] = {{b->nodeA.as<F>(), b->nodeA.as<F>() + capA}, {b->nodeB.as<F>(), b->nodeB.as<F>() + capB}};
    NodeBuf<F> prev{nullptr, nullptr};
    // all R rounds affine: inside a proof the per-round inversion latency is hidden by the other MSMs' streams
    for (uint32_t r = 1; r <= R; r++) {
      ar.round = r;
      ar.q_log = R - r;
      ar.prev = prev;
      ar.out = bufs[(r - 1) & 1];
      uint64_t npairs_max = nsl_bound << ar.q_log;
      unsigned nb = (unsigned)((npairs_max + kAffBlock * kAffPairs - 1) / (kAffBlock * kAffPairs));
      // CTAs/SM bounds = register caps (ptxas -v: forward 64 / 128 registers, backward 96 / 128, G1 / G2; measured
      // sweep in profiles/r1_notes.md: forward 8 + backward 5 CTAs/SM for G1, 4 + 4 for G2)
      if (sizeof(F) == 32) {
        k_affine_forward<F, kAffPairs, 8><<<nb, kAffBlock, 0, st>>>(ar);
        k_affine_invert<F><<<nblocks((size_t)nb * 32, 128), 128, 0, st>>>(ar.btot, nb);
        if (g_tma_staging == 1 || (g_tma_staging == 2 && r >= 2)) k_affine_backward_staged<F, kAffPairs, 5><<<nb, kAffBlock, AffStageLayout<F>::kSmem, st>>>(ar);
        else k_affine_backward<F, kAffPairs, 5><<<nb, kAffBlock, 0, st>>>(ar);
      } else {
        k_affine_forward<F, kAffPairs, 4><<<nb, kAffBlock, 0, st>>>(ar);
        k_affine_invert<F><<<nblocks((size_t)nb * 32, 128), 128, 0, st>>>(ar.btot, nb);
        if (g_tma_staging == 1 || (g_tma_staging == 2 && r >= 2)) k_affine_backward_staged<F, kAffPairs, 4><<<nb, kAffBlock, AffStageLayout<F>::kSmem, st>>>(ar);
        else k_affine_backward<F, kAffPairs, 4><<<nb, kAffBlock, 0, st>>>(ar);
      }
      prev = ar.out;
      g_launches += 3;
    }
    if (g_prof) {
      cudaEventRecord(pr.e1, st);
      g_prof_recs.push_back(pr);
    }
    k_merge_slices_affine<F><<<nblocks(sh.nbuckets, 128), 128, 0, st>>>(prev, stb, sh.nbuckets, buckets);
    if (sh.c >= 7) {
      launch_bucket_tail<F>(buckets, sh.c, partials, d_out, st);
      g_launches += 1;
    } else {
      k_bucket_reduce<F><<<nblocks(b->nseg, 128), 128, 0, st>>>(buckets, sh.nbuckets, b->seg, partials, b->nseg);
      launch_tree_sum<F>(partials, b->nseg, d_out, st);
      g_launches += 2;
    }
    CU(cudaGetLastError());
    return B200_OK;
  }
  uint64_t mean = ((uint64_t)sh.nwin * n_terms + sh.nbuckets - 1) / sh.nbuckets;
  int lpb = mean >= 384 ? 8 : (mean >= 96 ? 4 : 2);
  launch_accumulate<F>(lpb, b->table.as<Affine<F>>(), ss.entries.as<uint32_t>(), stb, m,
                       b->slice_out.as<XYZZ<F>>(), ss.max_slices, st);
  if (g_prof) {
    cudaEventRecord(pr.e1, st);
    g_prof_recs.push_back(pr);
  }
  k_merge_slices<F><<<nblocks(sh.nbuckets, 128), 128, 0, st>>>(b->slice_out.as<XYZZ<F>>(), stb, sh.nbuckets, buckets);
  if (sh.c >= 7) {
    launch_bucket_tail<F>(buckets, sh.c, partials, d_out, st);
    g_launches += 1;
  } else {
    k_bucket_reduce<F><<<nblocks(b->nseg, 128), 128, 0, st>>>(buckets, sh.nbuckets, b->seg, partials, b->nseg);
    launch_tree_sum<F>(partials, b->nseg, d_out, st);
    g_launches += 3;
  }
  CU(cudaGetLastError());
  return B200_OK;
}

template <class F>
int msm_enqueue(Bases* b, const Fr* d_scalars, size_t n, int mont, XYZZ<F>* d_out, cudaStream_t st) {
  if (n > b->n) return fail(B200_EINVAL, "msm: n=%zu exceeds base set size %zu", n, b->n);
  int rc = msm_sort(b->sort, b->sh, d_scalars, n, mont, st);
  if (rc) return rc;
  return msm_buckets<F>(b, b->sort, n, d_out, st);
}

template <class F>
int msm_host(b200_bases_t h, int group, const uint64_t* scalars, size_t n, uint64_t* out) {
  Bases* b = find_bases(h, group);
  if (!b) return fail(B200_EINVAL, "msm: bad handle");
  if ((!scalars && n) || !out) return fail(B200_EINVAL, "msm: null pointer");
  if (n) CU(cudaMemcpyAsync(b->scalars.p, scalars, n * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  int rc = msm_enqueue<F>(b, b->scalars.as<Fr>(), n, 0, b->result.as<XYZZ<F>>(), g_stream);
  if (rc) return rc;
  k_finalize<F><<<1, 32, 0, g_stream>>>(b->result.as<XYZZ<F>>(), b->out_std.as<F>());
  CU(cudaMemcpyAsync(out, b->out_std.p, 3 * sizeof(F), cudaMemcpyDeviceToHost, g_stream));
  rc = check_err_flag<F>("msm");  // synchronises the stream
  return rc;
}

template <class F>
int sum_partials(const void* d_xyzz, size_t count, uint64_t* out, cudaStream_t st) {
  if (!d_xyzz || !out || count == 0 || count > (1u << 20)) return fail(B200_EINVAL, "sum_partials: bad arguments");
  DevBuf res, std_out;
  CU(res.alloc(sizeof(XYZZ<F>)));
  CU(std_out.alloc(3 * sizeof(F)));
  k_sum_points<F><<<1, 256, 0, st>>>(reinterpret_cast<const XYZZ<F>*>(d_xyzz), (uint32_t)count, (uint32_t)count, res.as<XYZZ<F>>());
  k_finalize<F><<<1, 32, 0, st>>>(res.as<XYZZ<F>>(), std_out.as<F>());
  CU(cudaMemcpyAsync(out, std_out.p, 3 * sizeof(F), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return B200_OK;
}

template <class F>
int mul_batch(const uint64_t* pts, int bcast, const uint64_t* scalars, size_t n, uint64_t* out) {
  if (!pts || !scalars || !out) return fail(B200_EINVAL, "mul_batch: null pointer");
  if (n == 0) return B200_OK;
  DevBuf dp, ds, dout;
  size_t np = bcast ? 1 : n;
  CU(dp.alloc(np * 3 * sizeof(F)));
  CU(ds.alloc(n * sizeof(Fr)));
  CU(dout.alloc(n * 3 * sizeof(F)));
  CU(cudaMemcpyAsync(dp.p, pts, np * 3 * sizeof(F), cudaMemcpyHostToDevice, g_stream));
  CU(cudaMemcpyAsync(ds.p, scalars, n * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  k_mul_batch_ref<F><<<nblocks(n, 128), 128, 0, g_stream>>>(dp.as<F>(), bcast, ds.as<Fr>(), n, dout.as<F>(), g_d_err);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, dout.p, n * 3 * sizeof(F), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<F>("mul_batch");
}

int poly_mul_host(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* out) {
  if (!a || !b || !out || na == 0 || nb == 0) return fail(B200_EINVAL, "poly_mul: bad arguments");
  if (na + nb - 1 > ((size_t)1 << 27)) return fail(B200_EINVAL, "poly_mul: product too long");
  DevBuf da, db, dout;
  CU(da.alloc(na * sizeof(Fr)));
  CU(db.alloc(nb * sizeof(Fr)));
  CU(dout.alloc((na + nb - 1) * sizeof(Fr)));
  CU(cudaMemcpyAsync(da.p, a, na * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  CU(cudaMemcpyAsync(db.p, b, nb * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  CU(poly_mul_device(*g_poly, da.as<Fr>(), na, 0, db.as<Fr>(), nb, 0, dout.as<Fr>(), g_d_err, g_stream));
  CU(cudaMemcpyAsync(out, dout.p, (na + nb - 1) * sizeof(Fr), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fr>("poly_mul");
}

int divisor_init(Divisor& dv, const uint64_t* b, size_t nb) {
  DevBuf tmp;
  CU(tmp.alloc(nb * sizeof(Fr)));
  CU(dv.b_mont.alloc(nb * sizeof(Fr)));
  CU(cudaMemcpyAsync(tmp.p, b, nb * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  k_poly_load<<<nblk(nb, 256), 256, 0, g_stream>>>(tmp.as<Fr>(), (uint32_t)nb, (uint32_t)nb, 0, 0, dv.b_mont.as<Fr>(),
                                                    (uint32_t)nb, g_d_err);
  CU(cudaStreamSynchronize(g_stream));
  dv.nb = nb;
  return B200_OK;
}

int poly_div_host(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* q, uint64_t* rem) {
  if (!a || !b || na == 0 || nb == 0) return fail(B200_EINVAL, "poly_div: bad arguments");
  if (na < nb) {  // reference: empty quotient, rem = a (r1csqap.go:70-84 loop never runs)
    if (rem) memcpy(rem, a, na * sizeof(Fr));
    return B200_OK;
  }
  if (!q) return fail(B200_EINVAL, "poly_div: null quotient buffer");
  Divisor dv;
  int rc = divisor_init(dv, b, nb);
  if (rc) return rc;
  size_t nq = na - nb + 1;
  DevBuf da, dq, dr;
  CU(da.alloc(na * sizeof(Fr)));
  CU(dq.alloc(nq * sizeof(Fr)));
  if (rem && nb > 1) CU(dr.alloc((nb - 1) * sizeof(Fr)));
  CU(cudaMemcpyAsync(da.p, a, na * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  CU(poly_div_device(*g_poly, dv, da.as<Fr>(), na, 0, dq.as<Fr>(), dr.as<Fr>(), g_d_err, g_stream));
  CU(cudaMemcpyAsync(q, dq.p, nq * sizeof(Fr), cudaMemcpyDeviceToHost, g_stream));
  if (rem && nb > 1) CU(cudaMemcpyAsync(rem, dr.p, (nb - 1) * sizeof(Fr), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fr>("poly_div");
}

#include "prove_host.cuh"

#include "qap_sparse_host.cuh"

// groth16.GenerateProofs fed from the witness: px = CombinePolynomials(w, R1CSToQAP(a, b, c)) is computed on the device
// from the resident sparse R1CS (never leaving HBM) and handed to the same prove pipeline.
int groth16_prove_witness(b200_pk_t h, b200_r1cs_t hr, const uint64_t* w, size_t nw, const uint64_t* r, const uint64_t* s,
                          uint64_t* pi_a, uint64_t* pi_b, uint64_t* pi_c) {
  ProvingKey* pk = find_pk(h, 1);
  R1cs* rc1 = find_r1cs(hr);
  if (!pk || !rc1) return fail(B200_EINVAL, "groth16_prove_witness: bad handle");
  if (!w || !r || !s || !pi_a || !pi_b || !pi_c) return fail(B200_EINVAL, "groth16_prove_witness: null pointer");
  if (nw != pk->m || nw != rc1->m) return fail(B200_EINVAL, "groth16_prove_witness: witness length %zu, NVars %zu, R1CS columns %zu", nw, pk->m, rc1->m);
  if (pk->world != 1) return fail(B200_EINVAL, "groth16_prove_witness: sharded key");
  cudaStream_t st = g_stream;
  CU(pk->w_stage.ensure(nw * sizeof(Fr)));
  CU(cudaMemcpyAsync(pk->w_stage.p, w, nw * sizeof(Fr), cudaMemcpyHostToDevice, st));
  // px is only consumed by the division, which groth16_enqueue runs on side stream 3: compute it THERE, so the QAP front
  // end (NTT passes, HBM-bound) overlaps the A / B1 / B2 bucket phases (multiply-bound) on the other streams
  cudaStream_t sq = g_serial ? st : g_side[2];
  if (sq != st) {
    CU(cudaEventRecord(pk->ev[0], st));
    CU(cudaStreamWaitEvent(sq, pk->ev[0], 0));
  }
  // h = (ax*bx - cx) / Z straight from the witness (no px): the shape the reference supports has Z = prod_{i<=n}(x - i)
  // (m = n + 2, SURVEY H5) — checked; anything else goes through px and the division.
  const bool h_direct = rc1->n >= 2 && pk->Z.nb == rc1->n + 1;
  int rc;
  Fq* o = pk->out_std.as<Fq>();
  if (h_direct) {
    CU(pk->h_full.ensure((pk->m + pk->n_h_bases + 4) * sizeof(Fr)));
    rc = qap_h_enqueue(rc1, pk->w_stage.as<Fr>(), pk->h_full.as<Fr>(), sq);
    if (rc) return rc;
    rc = groth16_enqueue(pk, pk->w_stage.as<Fr>(), nw, rc1->px_mont.as<Fr>(), 2 * rc1->n - 1, r, s, o, st, 1, pk->h_full.as<Fr>());
  } else {
    rc = qap_px_enqueue(rc1, pk->w_stage.as<Fr>(), nullptr, nullptr, sq);
    if (rc) return rc;
    rc = groth16_enqueue(pk, pk->w_stage.as<Fr>(), nw, rc1->px_mont.as<Fr>(), 2 * rc1->n - 1, r, s, o, st, /*px_mont=*/1);
  }
  if (rc) return rc;
  uint64_t host_out[48];
  CU(cudaMemcpyAsync(host_out, o, sizeof host_out, cudaMemcpyDeviceToHost, st));
  rc = check_err_flag<Fr>("groth16_prove_witness");
  if (rc) return rc;
  memcpy(pi_a, host_out, 12 * 8);
  memcpy(pi_c, host_out + 12, 12 * 8);
  memcpy(pi_b, host_out + 24, 24 * 8);
  return B200_OK;
}

// ---- dense QAP API (small n) -------------------------------------------------
int r1cs_to_qap_host(const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n, size_t m, uint64_t* alphas,
                     uint64_t* betas, uint64_t* gammas, uint64_t* z) {
  if (!a || !b || !c || !alphas || !betas || !gammas || !z) return fail(B200_EINVAL, "r1cs_to_qap: null pointer");
  if (n == 0 || m < 2 || n > 8191 || m > 8193) return fail(B200_EINVAL, "r1cs_to_qap: dense API supports 1 <= n <= 8191");
  cudaStream_t st = g_stream;
  DevBuf zn, L, M, out, zz;
  size_t nz = m - 2;  // Z = prod_{i=1}^{m-2} (x - i)   (r1csqap.go:177-186)
  size_t zmax = (n > nz ? n : nz) + 1;
  CU(zn.alloc(zmax * sizeof(Fr)));
  CU(L.alloc(n * n * sizeof(Fr)));
  CU(M.alloc(n * m * sizeof(Fr)));
  CU(out.alloc(m * n * sizeof(Fr)));
  CU(zz.alloc((nz + 1) * sizeof(Fr)));
  k_zero_poly<<<1, 1024, 0, st>>>(zn.as<Fr>(), (uint32_t)n);
  k_lagrange_basis<<<nblk(n, 128), 128, 0, st>>>(zn.as<Fr>(), (uint32_t)n, L.as<Fr>());
  const uint64_t* in[3] = {a, b, c};
  uint64_t* outs[3] = {alphas, betas, gammas};
  for (int k = 0; k < 3; k++) {
    CU(cudaMemcpyAsync(M.p, in[k], n * m * sizeof(Fr), cudaMemcpyHostToDevice, st));
    dim3 grid(nblk(n, 128), (unsigned)m);
    k_qap_interpolate<<<grid, 128, 0, st>>>(M.as<Fr>(), (uint32_t)n, (uint32_t)m, L.as<Fr>(), out.as<Fr>(), g_d_err);
    CU(cudaMemcpyAsync(outs[k], out.p, m * n * sizeof(Fr), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  k_zero_poly<<<1, 1024, 0, st>>>(zn.as<Fr>(), (uint32_t)nz);
  k_poly_store<<<nblk(nz + 1, 256), 256, 0, st>>>(zn.as<Fr>(), (uint32_t)(nz + 1), 0, 1, zz.as<Fr>());
  CU(cudaMemcpyAsync(z, zz.p, (nz + 1) * sizeof(Fr), cudaMemcpyDeviceToHost, st));
  CU(cudaGetLastError());
  return check_err_flag<Fr>("r1cs_to_qap");
}

int combine_polynomials_host(const uint64_t* r, size_t m, const uint64_t* ap, const uint64_t* bp, const uint64_t* cp,
                             size_t n, uint64_t* ax, uint64_t* bx, uint64_t* cx, uint64_t* px) {
  if (!r || !ap || !bp || !cp || !ax || !bx || !cx || !px || m == 0 || n == 0)
    return fail(B200_EINVAL, "combine_polynomials: bad arguments");
  cudaStream_t st = g_stream;
  DevBuf dr, dP, mont[3], stdv[3], prod;
  CU(dr.alloc(m * sizeof(Fr)));
  CU(dP.alloc(m * n * sizeof(Fr)));
  CU(prod.alloc((2 * n - 1) * sizeof(Fr)));
  CU(cudaMemcpyAsync(dr.p, r, m * sizeof(Fr), cudaMemcpyHostToDevice, st));
  const uint64_t* in[3] = {ap, bp, cp};
  uint64_t* outs[3] = {ax, bx, cx};
  for (int k = 0; k < 3; k++) {
    CU(mont[k].alloc(n * sizeof(Fr)));
    CU(stdv[k].alloc(n * sizeof(Fr)));
    CU(cudaMemcpyAsync(dP.p, in[k], m * n * sizeof(Fr), cudaMemcpyHostToDevice, st));
    k_combine<<<nblk(n, 128), 128, 0, st>>>(dr.as<Fr>(), (uint32_t)m, dP.as<Fr>(), (uint32_t)n, mont[k].as<Fr>(),
                                            stdv[k].as<Fr>(), g_d_err);
    CU(cudaMemcpyAsync(outs[k], stdv[k].p, n * sizeof(Fr), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  // px = ax*bx - cx   (r1csqap.go:208)
  CU(poly_mul_device(*g_poly, mont[0].as<Fr>(), n, 1, mont[1].as<Fr>(), n, 1, prod.as<Fr>(), g_d_err, st));
  k_poly_addsub<<<nblk(2 * n - 1, 256), 256, 0, st>>>(prod.as<Fr>(), (uint32_t)(2 * n - 1), stdv[2].as<Fr>(), (uint32_t)n, 1,
                                                      prod.as<Fr>(), g_d_err);
  CU(cudaMemcpyAsync(px, prod.p, (2 * n - 1) * sizeof(Fr), cudaMemcpyDeviceToHost, st));
  CU(cudaGetLastError());
  return check_err_flag<Fr>("combine_polynomials");
}

int poly_addsub_host(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, int sub, uint64_t* out) {
  size_t n = na > nb ? na : nb;
  if (n == 0) return B200_OK;
  if ((na && !a) || (nb && !b) || !out) return fail(B200_EINVAL, "poly_add/sub: null pointer");
  DevBuf da, db, dout;
  CU(da.alloc((na ? na : 1) * sizeof(Fr)));
  CU(db.alloc((nb ? nb : 1) * sizeof(Fr)));
  CU(dout.alloc(n * sizeof(Fr)));
  if (na) CU(cudaMemcpyAsync(da.p, a, na * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  if (nb) CU(cudaMemcpyAsync(db.p, b, nb * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  k_poly_addsub<<<nblk(n, 256), 256, 0, g_stream>>>(da.as<Fr>(), (uint32_t)na, db.as<Fr>(), (uint32_t)nb, sub, dout.as<Fr>(), g_d_err);
  CU(cudaMemcpyAsync(out, dout.p, n * sizeof(Fr), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fr>("poly_add/sub");
}

int poly_eval_host(const uint64_t* v, size_t n, const uint64_t* x, uint64_t* out) {
  if (!x || !out || (n && !v)) return fail(B200_EINVAL, "poly_eval: null pointer");
  DevBuf dv, dout;
  CU(dv.alloc((n ? n : 1) * sizeof(Fr)));
  CU(dout.alloc(sizeof(Fr)));
  if (n) CU(cudaMemcpyAsync(dv.p, v, n * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  Fr xs = fr_load_std(x);
  if (xs.geq_modulus()) return fail(B200_ERANGE, "poly_eval: x >= r");
  k_poly_eval<<<1, 256, 0, g_stream>>>(dv.as<Fr>(), (uint32_t)n, xs, dout.as<Fr>(), g_d_err);
  CU(cudaMemcpyAsync(out, dout.p, sizeof(Fr), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fr>("poly_eval");
}

int poly_eval_batch_host(const uint64_t* polys, size_t m, size_t n, const uint64_t* x, uint64_t* out) {
  if (!polys || !x || !out || m == 0 || n == 0) return fail(B200_EINVAL, "poly_eval_batch: bad arguments");
  Fr xs = fr_load_std(x);
  if (xs.geq_modulus()) return fail(B200_ERANGE, "poly_eval_batch: x >= r");
  DevBuf dp, dout;
  CU(dp.alloc(m * n * sizeof(Fr)));
  CU(dout.alloc(m * sizeof(Fr)));
  CU(cudaMemcpyAsync(dp.p, polys, m * n * sizeof(Fr), cudaMemcpyHostToDevice, g_stream));
  k_poly_eval_batch<<<(unsigned)m, 64, 0, g_stream>>>(dp.as<Fr>(), (uint32_t)n, xs, dout.as<Fr>(), g_d_err);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, dout.p, m * sizeof(Fr), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fr>("poly_eval_batch");
}

int zero_poly_host(size_t n, uint64_t* out) {   // coefficients of prod_{i=1..n} (x - i), n + 1 of them
  if (!out || n > ((size_t)1 << 26)) return fail(B200_EINVAL, "zero_poly: bad arguments (n <= 2^26)");
  DevBuf zn, zz;
  CU(zz.alloc((n + 1) * sizeof(Fr)));
  if (n <= 2048) {   // one-block schoolbook; above: Newton basis element n through the subproduct tree (qap_sparse.cuh)
    CU(zn.alloc((n + 1) * sizeof(Fr)));
    k_zero_poly<<<1, 1024, 0, g_stream>>>(zn.as<Fr>(), (uint32_t)n);
  } else {
    int rc = zero_poly_device(n, zn, g_stream);
    if (rc) return rc;
  }
  k_poly_store<<<nblk(n + 1, 256), 256, 0, g_stream>>>(zn.as<Fr>(), (uint32_t)(n + 1), 0, 1, zz.as<Fr>());
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, zz.p, (n + 1) * sizeof(Fr), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fr>("zero_poly");
}

#ifndef B200_NO_PAIRING
// ---- pairing / verification (SURVEY §8f row 2) -------------------------------------------------------
template <bool FAST_FE>
__device__ void pairing_from_jacobian(const Fq* g1, const Fq2* g2, F12& out, int* err) {
  bool bad = false;
  for (int k = 0; k < 3; k++) bad = bad || g1[k].geq_modulus() || g2[k].c0.geq_modulus() || g2[k].c1.geq_modulus();
  Jacobian<Fq> p{g1[0].to_mont(), g1[1].to_mont(), g1[2].to_mont()};
  Jacobian<Fq2> q{g2[0].to_mont(), g2[1].to_mont(), g2[2].to_mont()};
  if (bad || q.is_inf()) {  // G2 infinity: preComputeG2 panics "q1[2] != Fq2.One()" (bn128.go:238-241)
    atomicOr(err, bad ? 1 : 8);
    out = F12::one();
    return;
  }
  Affine<Fq> pa = jac_to_affine(p);                      // preComputeG1: G1.Affine, infinity -> (0, 0)
  Affine<Fq2> qa = jac_to_affine(q);
  F2::B px, py;
#pragma unroll
  for (int i = 0; i < 8; i++) { px.l[i] = pa.x.l[i]; py.l[i] = pa.y.l[i]; }
  out = pairing_affine_t<FAST_FE>(px, py, qa.x, qa.y);
}
__device__ void store_f12_std(const F12& f, Fq2* out) {
  out[0] = f.a.a.from_mont(); out[1] = f.a.b.from_mont(); out[2] = f.a.c.from_mont();
  out[3] = f.b.a.from_mont(); out[4] = f.b.b.from_mont(); out[5] = f.b.c.from_mont();
}
// out[i] = a[i] * b[i] in F_q^12 (fields/fq12.go:72-84), standard form in/out, [2][3][2] order
__global__ void __launch_bounds__(32) k_fq12_mul_batch(const Fq2* a, const Fq2* b, size_t n, Fq2* out, int* err) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  F12 x, y;
  Fq2* xs = &x.a.a;
  Fq2* ys = &y.a.a;
  bool bad = false;
  for (int k = 0; k < 6; k++) {
    Fq2 u = a[6 * i + k], v = b[6 * i + k];
    bad = bad || u.geq_modulus() || v.geq_modulus();
    xs[k] = u.to_mont();
    ys[k] = v.to_mont();
  }
  if (bad) atomicOr(err, 1);
  store_f12_std(f12_mul(x, y), out + 6 * i);
}
template <bool FAST_FE>
__global__ void __launch_bounds__(32) k_pairing_batch(const Fq* g1, const Fq2* g2, size_t n, Fq2* out, int* err) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  F12 f;
  pairing_from_jacobian<FAST_FE>(g1 + 3 * i, g2 + 3 * i, f, err);
  store_f12_std(f, out + 6 * i);
}
// ---- one warp per pairing (pairing_warp.cuh) ----------------------------------------------------------------------
constexpr int kPairWarps = 4;   // warps (pairings) per CTA: 4 x 9.5 KB of shared memory
// lane 0 validates and normalises the Jacobian inputs (preComputeG1 / G2.Affine); returns warp-uniformly whether a pairing
// is to be computed (false: out-of-range coordinate or G2 infinity — the reference panics, bn128.go:238-241 — result = one)
__device__ bool warp_pairing_inputs(wp::Ws& ws, const Fq* g1, const Fq2* g2, F2::B& px, F2::B& py, F2& qx, F2& qy, int* err) {
  int go = 1;
  if ((threadIdx.x & 31u) == 0) {
    bool bad = false;
    for (int k = 0; k < 3; k++) bad = bad || g1[k].geq_modulus() || g2[k].c0.geq_modulus() || g2[k].c1.geq_modulus();
    Jacobian<Fq> p{g1[0].to_mont(), g1[1].to_mont(), g1[2].to_mont()};
    Jacobian<Fq2> q{g2[0].to_mont(), g2[1].to_mont(), g2[2].to_mont()};
    if (bad || q.is_inf()) {
      atomicOr(err, bad ? 1 : 8);
      go = 0;
    } else {
      Affine<Fq> pa = jac_to_affine(p);
      Affine<Fq2> qa = jac_to_affine(q);
#pragma unroll
      for (int i = 0; i < 8; i++) { px.l[i] = pa.x.l[i]; py.l[i] = pa.y.l[i]; }
      qx = qa.x;
      qy = qa.y;
    }
  }
  (void)ws;
  return __shfl_sync(0xffffffffu, go, 0) != 0;
}
__global__ void __launch_bounds__(32 * kPairWarps) k_pairing_batch_warp(const Fq* g1, const Fq2* g2, size_t n, Fq2* out, int* err) {
  __shared__ wp::Ws wss[kPairWarps];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const size_t i = (size_t)blockIdx.x * kPairWarps + warp;
  if (i >= n) return;
  wp::Ws& ws = wss[warp];
  F2::B px, py;
  F2 qx, qy;
  if (warp_pairing_inputs(ws, g1 + 3 * i, g2 + 3 * i, px, py, qx, qy, err)) wp::pairing(ws, px, py, qx, qy);
  else wp::f12_set_one(ws, wp::RF);
  if (lane < 12) {  // standard form out, [2][3][2] order: one F_q component per lane
    const F2& c = ws.r[wp::RF][lane >> 1];
    F2::B v = ((lane & 1) ? c.c1 : c.c0).from_mont();
    Fq2* o = out + 6 * i + (lane >> 1);
    if (lane & 1) o->c1 = v;
    else o->c0 = v;
  }
}
// groth16.VerifyProof (groth16/groth16.go:281-305): e(A,B) == e(alpha,beta) * (e(icPubl,gamma) * e(C,delta)).
// Warp w pairs g1 with g2 (Jacobian standard form), in the order A/B, alpha/beta, icPubl/gamma, C/delta.  Four warps, one
// pairing each; warp 0 then forms the right-hand side with two warp-wide F_q^12 products and compares.
__device__ __forceinline__ void groth16_verify_block(wp::Ws (&wss)[4], const Fq* g1, const Fq2* g2, int* ok, int* err) {
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  wp::Ws& ws = wss[warp];
  F2::B px, py;
  F2 qx, qy;
  if (warp_pairing_inputs(ws, g1, g2, px, py, qx, qy, err)) wp::pairing(ws, px, py, qx, qy);
  else wp::f12_set_one(ws, wp::RF);
  __syncthreads();
  if (warp == 0) {
    if (lane < 6) {
      ws.r[2][lane] = wss[1].r[wp::RF][lane];
      ws.r[3][lane] = wss[2].r[wp::RF][lane];
      ws.r[4][lane] = wss[3].r[wp::RF][lane];
    }
    wp::wsync();
    wp::f12_mul(ws, 3, 3, 4);
    wp::f12_mul(ws, 2, 2, 3);
    const int same = lane < 6 ? (ws.r[0][lane] == ws.r[2][lane] ? 1 : 0) : 1;
    const unsigned all = __ballot_sync(0xffffffffu, same);
    if (lane == 0) *ok = all == 0xffffffffu ? 1 : 0;
  }
}
// pts1: A, alpha1, icPubl, C ; pts2: B, beta2, gamma2, delta2
__global__ void __launch_bounds__(128) k_groth16_verify(const Fq* pts1, const Fq2* pts2, int* ok, int* err) {
  __shared__ wp::Ws wss[4];
  const uint32_t warp = threadIdx.x >> 5;
  groth16_verify_block(wss, pts1 + 3 * warp, pts2 + 3 * warp, ok, err);
}
// The same check for proof idx[b] of a batch in block b: vk2 = beta2, gamma2, delta2; icp = the proofs' icPubl.
__global__ void __launch_bounds__(128) k_vb_verify_each(const Fq* A, const Fq2* B, const Fq* C, const Fq* icp, const Fq* alpha,
                                                        const Fq2* vk2, const uint32_t* idx, int* ok, int* err) {
  __shared__ wp::Ws wss[4];
  const uint32_t warp = threadIdx.x >> 5;
  const size_t i = idx[blockIdx.x];
  const Fq* g1 = warp == 0 ? A + 3 * i : (warp == 1 ? alpha : (warp == 2 ? icp + 3 * i : C + 3 * i));
  const Fq2* g2 = warp == 0 ? B + 3 * i : vk2 + 3 * (warp - 1);
  groth16_verify_block(wss, g1, g2, ok + blockIdx.x, err);
}
// icPubl = IC[0] + sum publicSignals[i] * IC[i+1] (groth16.go:283-286).  The products are independent: one half-warp each,
// with the GLV split of prove_host.cuh (128 doublings + ~12 additions deep instead of the 254 + ~127 of MulScalar's
// double-and-add; the same group element, which is all the pairing — it normalises its inputs — can see); the sum then runs
// in the reference's order with the reference's Add, so its degenerate cases (equal operands give Z = 0) are the reference's.
struct GlvScalar {
  uint64_t k[4];
  uint32_t neg[2];
};
__global__ void __launch_bounds__(32) k_ic_terms(const Fq* ic, const GlvScalar* gs, size_t npub, Jacobian<Fq>* terms, int* err) {
  const uint32_t t = threadIdx.x & 31u;
  const size_t i = (size_t)blockIdx.x * 2 + (t >> 4);
  const size_t ii = i < npub ? i : npub - 1;   // an odd count leaves the last half-warp a duplicate: every lane joins the shuffles
  const Fq* src = ic + 3 * (ii + 1);
  if (src[0].geq_modulus() || src[1].geq_modulus() || src[2].geq_modulus()) atomicOr(err, 1);
  Jacobian<Fq> p{src[0].to_mont(), src[1].to_mont(), src[2].to_mont()};
  GlvScalar g = gs[ii];
  Jacobian<Fq> r = glv_mul_halfwarp(p, g.k, g.neg, t);
  if (i < npub && (t & 15u) == 0) terms[i] = r;
}
__global__ void k_ic_sum(const Fq* ic, const Jacobian<Fq>* terms, size_t npub, Fq* out, int* err) {
  if (threadIdx.x | blockIdx.x) return;
  if (ic[0].geq_modulus() || ic[1].geq_modulus() || ic[2].geq_modulus()) atomicOr(err, 1);
  Jacobian<Fq> acc{ic[0].to_mont(), ic[1].to_mont(), ic[2].to_mont()};
  for (size_t i = 0; i < npub; i++) acc = jac_add_ref(acc, terms[i]);
  out[0] = acc.X.from_mont();
  out[1] = acc.Y.from_mont();
  out[2] = acc.Z.from_mont();
}

// Final exponentiation: Devegili-Scott-Dahab (easy part + hard part by the BN parameter), the SAME F_q^12 value as the
// reference's plain f^((q^12-1)/r) square-and-multiply (bn128.go:400-421) with ~13x fewer operations: validated on the
// GPU against the snarkjs golden vk_alfabeta_12 (K8), the bn128_test.go literal and the oracle (tests/test_gpu_verify.py,
// profiles/r2_notes.md).  The plain routine stays in pairing.cuh as the step-by-step restatement used by the host tests.
constexpr bool kFastFinalExp = true;
// n pairings of device inputs (Jacobian standard form) into out (standard form).  auto: a warp per pairing has the 5x shorter
// latency (3.4 vs 17 ms) and wins up to ~3 500 pairings per call; above that the thread-per-pairing kernel keeps more
// pairings resident and has twice the throughput (462 k vs 204 k pairings/s at 2^16)
void pairing_enqueue(const Fq* g1, const Fq2* g2, size_t n, Fq2* out, cudaStream_t st) {
  const bool thread_kernel = g_pairing_kernel == 1 || (g_pairing_kernel == 0 && n > 2048);
  if (thread_kernel) k_pairing_batch<kFastFinalExp><<<nblk(n, 32), 32, 0, st>>>(g1, g2, n, out, g_d_err);
  else k_pairing_batch_warp<<<nblk(n, kPairWarps), 32 * kPairWarps, 0, st>>>(g1, g2, n, out, g_d_err);
}
int pairing_batch_host(const uint64_t* g1, const uint64_t* g2, size_t n, uint64_t* out) {
  if (!g1 || !g2 || !out) return fail(B200_EINVAL, "pairing_batch: null pointer");
  if (n == 0) return B200_OK;
  DevBuf d1, d2, dout;
  CU(d1.alloc(n * 3 * sizeof(Fq)));
  CU(d2.alloc(n * 3 * sizeof(Fq2)));
  CU(dout.alloc(n * 6 * sizeof(Fq2)));
  CU(cudaMemcpyAsync(d1.p, g1, n * 3 * sizeof(Fq), cudaMemcpyHostToDevice, g_stream));
  CU(cudaMemcpyAsync(d2.p, g2, n * 3 * sizeof(Fq2), cudaMemcpyHostToDevice, g_stream));
  pairing_enqueue(d1.as<Fq>(), d2.as<Fq2>(), n, dout.as<Fq2>(), g_stream);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, dout.p, n * 6 * sizeof(Fq2), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fq>("pairing_batch");
}

int fq12_mul_batch_host(const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out) {
  if (!a || !b || !out) return fail(B200_EINVAL, "fq12_mul_batch: null pointer");
  if (n == 0) return B200_OK;
  DevBuf da, db, dout;
  size_t bytes = n * 6 * sizeof(Fq2);
  CU(da.alloc(bytes));
  CU(db.alloc(bytes));
  CU(dout.alloc(bytes));
  CU(cudaMemcpyAsync(da.p, a, bytes, cudaMemcpyHostToDevice, g_stream));
  CU(cudaMemcpyAsync(db.p, b, bytes, cudaMemcpyHostToDevice, g_stream));
  k_fq12_mul_batch<<<nblk(n, 32), 32, 0, g_stream>>>(da.as<Fq2>(), db.as<Fq2>(), n, dout.as<Fq2>(), g_d_err);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, dout.p, bytes, cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<Fq>("fq12_mul_batch");
}

int groth16_verify_host(const uint64_t* ic, size_t n_ic, const uint64_t* alpha1, const uint64_t* beta2,
                        const uint64_t* gamma2, const uint64_t* delta2, const uint64_t* pi_a, const uint64_t* pi_b,
                        const uint64_t* pi_c, const uint64_t* pub, size_t npub, int* ok) {
  if (!ic || !alpha1 || !beta2 || !gamma2 || !delta2 || !pi_a || !pi_b || !pi_c || !ok || (npub && !pub))
    return fail(B200_EINVAL, "groth16_verify: null pointer");
  if (n_ic < npub + 1) return fail(B200_EINVAL, "groth16_verify: len(IC) < len(publicSignals) + 1");
  // GLV split of every public signal on the host (they are the caller's host scalars anyway)
  std::vector<GlvScalar> gs(npub ? npub : 1);
  for (size_t i = 0; i < npub; i++) {
    Fr v = fr_load_std(pub + 4 * i);
    if (v.geq_modulus()) return fail(B200_ERANGE, "groth16_verify: scalar / coefficient >= r");
    if (glv_decompose(v, gs[i].k, gs[i].neg)) return fail(B200_EINVAL, "groth16_verify: GLV decomposition out of range");
  }
  DevBuf dic, dsig, dterms, d1, d2, dok;
  CU(dic.alloc(n_ic * 3 * sizeof(Fq)));
  CU(dsig.alloc(gs.size() * sizeof(GlvScalar)));
  CU(dterms.alloc(gs.size() * sizeof(Jacobian<Fq>)));
  CU(d1.alloc(4 * 3 * sizeof(Fq)));
  CU(d2.alloc(4 * 3 * sizeof(Fq2)));
  CU(dok.alloc(sizeof(int)));
  cudaStream_t st = g_stream;
  CU(cudaMemcpyAsync(dic.p, ic, n_ic * 3 * sizeof(Fq), cudaMemcpyHostToDevice, st));
  if (npub) CU(cudaMemcpyAsync(dsig.p, gs.data(), npub * sizeof(GlvScalar), cudaMemcpyHostToDevice, st));
  Fq* p1 = d1.as<Fq>();
  Fq2* p2 = d2.as<Fq2>();
  CU(cudaMemcpyAsync(p1, pi_a, 3 * sizeof(Fq), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(p1 + 3, alpha1, 3 * sizeof(Fq), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(p1 + 9, pi_c, 3 * sizeof(Fq), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(p2, pi_b, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(p2 + 3, beta2, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(p2 + 6, gamma2, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(p2 + 9, delta2, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, st));
  if (npub) k_ic_terms<<<(unsigned)((npub + 1) / 2), 32, 0, st>>>(dic.as<Fq>(), dsig.as<GlvScalar>(), npub, dterms.as<Jacobian<Fq>>(), g_d_err);
  k_ic_sum<<<1, 32, 0, st>>>(dic.as<Fq>(), dterms.as<Jacobian<Fq>>(), npub, p1 + 6, g_d_err);
  k_groth16_verify<<<1, 128, 0, st>>>(p1, p2, dok.as<int>(), g_d_err);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(ok, dok.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  return check_err_flag<Fq>("groth16_verify");
}

// groth16.VerifyProof for nproofs proofs under one key (include/b200snark.h b200_groth16_verify_batch).  The proofs the
// reference pairs bilinearly enter ONE aggregated check (N + 3 Miller loops, one final exponentiation); the others, and every
// proof of a batch whose aggregated check fails, run the four-pairing check of b200_groth16_verify one block per proof.
// A failed check verifies its proofs one by one rather than bisecting: that is the cost of the four-pairing route, paid
// only when a batch holds a bad proof, and every verdict is then the single verifier's own.
constexpr size_t kMillerThreads = 16384;   // chunk = ceil(pairs / this): longer chunks share one squaring among more pairs
int groth16_verify_batch_host(const uint64_t* ic, size_t n_ic, const uint64_t* alpha1, const uint64_t* beta2,
                              const uint64_t* gamma2, const uint64_t* delta2, size_t n, const uint64_t* pi_a,
                              const uint64_t* pi_b, const uint64_t* pi_c, const uint64_t* pub, size_t npub,
                              const uint64_t* rho, int* ok, uint64_t* stats) {
  if (!ic || !alpha1 || !beta2 || !gamma2 || !delta2 || !pi_a || !pi_b || !pi_c || !rho || !ok || (npub && !pub) || n == 0)
    return fail(B200_EINVAL, "groth16_verify_batch: null pointer or no proofs");
  if (n_ic < npub + 1) return fail(B200_EINVAL, "groth16_verify_batch: len(IC) < len(publicSignals) + 1");
  if (n > (1u << 26)) return fail(B200_EINVAL, "groth16_verify_batch: more than 2^26 proofs");
  for (size_t i = 0; i < n; i++)
    if (!rho[2 * i] && !rho[2 * i + 1]) return fail(B200_EINVAL, "groth16_verify_batch: rho[%zu] = 0", i);
  // the verification key, flagged as b200_groth16_verify flags it
  auto g1_range = [](const uint64_t* p) {
    for (int k = 0; k < 3; k++) {
      Fq v;
      std::memcpy(&v, p + 4 * k, sizeof v);
      if (v.geq_modulus()) return true;
    }
    return false;
  };
  auto g2_range = [&](const uint64_t* p) { return g1_range(p) || g1_range(p + 12); };
  auto g2_inf = [](const uint64_t* p) { return !(p[16] | p[17] | p[18] | p[19] | p[20] | p[21] | p[22] | p[23]); };
  int vkf = (g1_range(alpha1) || g2_range(beta2)) ? 1 : (g2_inf(beta2) ? 8 : 0);
  for (const uint64_t* g : {gamma2, delta2}) vkf |= g2_range(g) ? 1 : (g2_inf(g) ? 8 : 0);
  for (size_t j = 0; j <= npub; j++) vkf |= g1_range(ic + 12 * j) ? 1 : 0;
  if (vkf & 8) return fail(B200_EINVAL, "groth16_verify_batch: q1[2] != Fq2.One() (verification key G2 point at infinity)");
  if (vkf) return fail(B200_ERANGE, "groth16_verify_batch: verification key coordinate >= q");
  std::vector<int> st(n, 0);   // a public signal >= r: what b200_groth16_verify returns before any pairing
  for (size_t i = 0; i < n; i++)
    for (size_t j = 0; j < npub; j++)
      if (fr_load_std(pub + 4 * (i * npub + j)).geq_modulus()) st[i] = B200_ERANGE;
  const size_t np = n + 3;
  DevBuf dic, dalpha, dvk2, dA, dB, dC, dpub, drho, dst, dterms, dicp, dic_aff, dg2_aff, dbad, dpairs, drc, dric, dsum, dT, df,
      dfe, dres, dalpha_gs, dalpha_term;
  CU(dic.alloc((npub + 1) * 3 * sizeof(Fq)));
  CU(dalpha.alloc(2 * 3 * sizeof(Fq)));
  CU(dvk2.alloc(3 * 3 * sizeof(Fq2)));
  CU(dA.alloc(n * 3 * sizeof(Fq)));
  CU(dB.alloc(n * 3 * sizeof(Fq2)));
  CU(dC.alloc(n * 3 * sizeof(Fq)));
  CU(dpub.alloc(std::max<size_t>(n * npub, 1) * 4 * sizeof(uint64_t)));
  CU(drho.alloc(n * 2 * sizeof(uint64_t)));
  CU(dst.alloc(n * sizeof(int)));
  CU(dterms.alloc(std::max<size_t>(n * npub, 1) * sizeof(Jacobian<Fq>)));
  CU(dicp.alloc(n * 3 * sizeof(Fq)));
  CU(dic_aff.alloc((npub + 1) * sizeof(Affine<Fq>)));
  CU(dg2_aff.alloc(3 * sizeof(Affine<Fq2>)));
  CU(dbad.alloc(sizeof(int)));
  CU(dpairs.alloc(np * sizeof(vb::Pair)));
  CU(drc.alloc(n * sizeof(XYZZ<Fq>)));
  CU(dric.alloc(n * sizeof(XYZZ<Fq>)));
  cudaStream_t s = g_stream;
  CU(cudaMemcpyAsync(dic.p, ic, (npub + 1) * 3 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dalpha.p, alpha1, 3 * sizeof(Fq), cudaMemcpyHostToDevice, s));   // [alpha, alpha]: k_ic_terms reads slot 1
  CU(cudaMemcpyAsync(dalpha.as<Fq>() + 3, alpha1, 3 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk2.as<Fq2>(), beta2, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk2.as<Fq2>() + 3, gamma2, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk2.as<Fq2>() + 6, delta2, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dA.p, pi_a, n * 3 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dB.p, pi_b, n * 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dC.p, pi_c, n * 3 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  if (npub) CU(cudaMemcpyAsync(dpub.p, pub, n * npub * 4 * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(drho.p, rho, n * 2 * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dst.p, st.data(), n * sizeof(int), cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(dbad.p, 0, sizeof(int), s));
  // 1. per-proof preparation
  vb::k_vb_vk<<<1, 32, 0, s>>>(dic.as<Fq>(), (uint32_t)(npub + 1), dalpha.as<Fq>(), dvk2.as<Fq2>(), dic_aff.as<Affine<Fq>>(),
                               dg2_aff.as<Affine<Fq2>>(), dbad.as<int>());
  if (npub) vb::k_vb_ic_terms<<<nblk(n * npub, 64), 64, 0, s>>>(dic_aff.as<Affine<Fq>>(), dpub.as<uint64_t>(), n, npub, dterms.as<Jacobian<Fq>>());
  vb::k_vb_ic_sum<<<nblk(n, 64), 64, 0, s>>>(dic.as<Fq>(), dterms.as<Jacobian<Fq>>(), n, npub, dicp.as<Fq>());
  vb::k_vb_prepare<<<nblk(n, 64), 64, 0, s>>>(dA.as<Fq>(), dB.as<Fq2>(), dC.as<Fq>(), dicp.as<Fq>(), drho.as<uint64_t>(), n,
                                              dst.as<int>(), dpairs.as<vb::Pair>(), drc.as<XYZZ<Fq>>(), dric.as<XYZZ<Fq>>());
  CU(cudaGetLastError());
  int vk_bad = 0;
  CU(cudaMemcpyAsync(st.data(), dst.p, n * sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&vk_bad, dbad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (vk_bad) return fail(B200_EINVAL, "groth16_verify_batch: verification key point off the curve, or outside G2");
  std::vector<uint32_t> each;
  uint64_t rho_sum[4] = {0, 0, 0, 0};   // sum of < 2^26 128-bit values: < 2^154 < r, no reduction
  size_t n_agg = 0;
  for (size_t i = 0; i < n; i++) {
    if (st[i] == vb::kEach) each.push_back((uint32_t)i);
    if (st[i] != vb::kAgg) continue;
    n_agg++;
    unsigned __int128 c = (unsigned __int128)rho_sum[0] + rho[2 * i];
    rho_sum[0] = (uint64_t)c;
    c = (c >> 64) + rho_sum[1] + rho[2 * i + 1];
    rho_sum[1] = (uint64_t)c;
    c = (c >> 64) + rho_sum[2];
    rho_sum[2] = (uint64_t)c;
  }
  uint64_t st_stats[4] = {n_agg, 0, 0, 0};
  bool agg_ok = false;
  if (n_agg) {
    // 2. reductions: -(sum rho) alpha by the GLV half-warp of k_ic_terms, sum rho C and sum rho icPubl by tree sums
    static const uint64_t kR[4] = {0x43e1f593f0000001ULL, 0x2833e84879b97091ULL, 0xb85045b68181585dULL, 0x30644e72e131a029ULL};
    uint64_t neg[4];
    unsigned __int128 br = 0;
    for (int k = 0; k < 4; k++) {
      unsigned __int128 d = (unsigned __int128)kR[k] - rho_sum[k] - (uint64_t)br;
      neg[k] = (uint64_t)d;
      br = (d >> 64) & 1;
    }
    GlvScalar gs;
    if (glv_decompose(fr_load_std(neg), gs.k, gs.neg)) return fail(B200_EINVAL, "groth16_verify_batch: GLV decomposition out of range");
    CU(dalpha_gs.alloc(sizeof(GlvScalar)));
    CU(dalpha_term.alloc(sizeof(Jacobian<Fq>)));
    CU(cudaMemcpyAsync(dalpha_gs.p, &gs, sizeof(GlvScalar), cudaMemcpyHostToDevice, s));
    k_ic_terms<<<1, 32, 0, s>>>(dalpha.as<Fq>(), dalpha_gs.as<GlvScalar>(), 1, dalpha_term.as<Jacobian<Fq>>(), g_d_err);
    const uint32_t kSum = 32;
    size_t levels = 0;   // every level of both sums gets its own slots
    for (size_t m = n; m > 1; m = nblk(m, kSum)) levels += nblk(m, kSum);
    CU(dsum.alloc(std::max<size_t>(2 * levels, 1) * sizeof(XYZZ<Fq>)));
    XYZZ<Fq>* sums[2] = {dric.as<XYZZ<Fq>>(), drc.as<XYZZ<Fq>>()};
    XYZZ<Fq>* slot = dsum.as<XYZZ<Fq>>();
    for (int k = 0; k < 2; k++)
      for (size_t m = n; m > 1; m = nblk(m, kSum)) {
        vb::k_vb_sum<<<nblk(nblk(m, kSum), 64), 64, 0, s>>>(sums[k], m, kSum, slot);
        sums[k] = slot;
        slot += nblk(m, kSum);
      }
    CU(dres.alloc(2 * sizeof(int)));
    vb::k_vb_tail<<<1, 32, 0, s>>>(dalpha_term.as<Jacobian<Fq>>(), sums[0], sums[1], dg2_aff.as<Affine<Fq2>>(),
                                   dpairs.as<vb::Pair>() + n, dres.as<int>());
    // 3. multi-Miller loop, 4. product tree and one final exponentiation
    const uint32_t chunk = (uint32_t)std::max<size_t>(1, nblk(np, kMillerThreads));
    const size_t nth = nblk(np, chunk);
    CU(dT.alloc(np * sizeof(Jacobian<Fq2>)));
    CU(df.alloc(nth * sizeof(F12)));
    CU(dfe.alloc(nblk(nth, 2) * sizeof(F12)));
    vb::k_vb_miller<<<nblk(nth, 64), 64, 0, s>>>(dpairs.as<vb::Pair>(), np, chunk, dT.as<Jacobian<Fq2>>(), df.as<F12>());
    F12 *a = df.as<F12>(), *b = dfe.as<F12>();
    for (size_t m = nth; m > 1; m = nblk(m, 2)) {
      vb::k_vb_f12_tree<<<nblk(nblk(m, 2), 64), 64, 0, s>>>(a, m, b);
      std::swap(a, b);
    }
    vb::k_vb_final_exp<<<1, 32, 0, s>>>(a, dres.as<int>() + 1, nullptr);
    CU(cudaGetLastError());
    int res[2] = {0, 0};
    CU(cudaMemcpyAsync(res, dres.p, sizeof res, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    agg_ok = res[1] == 1;
    st_stats[2] = 1;
    st_stats[3] = n_agg + (uint64_t)res[0];
    if (!agg_ok)
      for (size_t i = 0; i < n; i++)
        if (st[i] == vb::kAgg) each.push_back((uint32_t)i);
  }
  std::vector<int> each_ok(each.size(), 0);
  if (!each.empty()) {
    DevBuf didx, dok, derr;
    CU(didx.alloc(each.size() * sizeof(uint32_t)));
    CU(dok.alloc(each.size() * sizeof(int)));
    CU(derr.alloc(sizeof(int)));   // inputs validated above: no flag can be raised
    CU(cudaMemcpyAsync(didx.p, each.data(), each.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    k_vb_verify_each<<<(unsigned)each.size(), 128, 0, s>>>(dA.as<Fq>(), dB.as<Fq2>(), dC.as<Fq>(), dicp.as<Fq>(), dalpha.as<Fq>(),
                                                         dvk2.as<Fq2>(), didx.as<uint32_t>(), dok.as<int>(), derr.as<int>());
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(each_ok.data(), dok.p, each.size() * sizeof(int), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    st_stats[1] = each.size();
    st_stats[3] += 4 * (uint64_t)each.size();
  }
  for (size_t i = 0; i < n; i++) ok[i] = st[i] < 0 ? st[i] : (st[i] == vb::kAgg && agg_ok ? 1 : 0);
  for (size_t k = 0; k < each.size(); k++) ok[each[k]] = each_ok[k];
  if (stats) std::memcpy(stats, st_stats, sizeof st_stats);
  return B200_OK;
}

// ---- Pinocchio verification (snark.VerifyProof, snark.go:292-372): one proof, and N proofs under one key ----
// the generator of G2 (bn128.go:57-83), Jacobian standard form
constexpr uint64_t kG2Gen[24] = {
    0x46debd5cd992f6edULL, 0x674322d4f75edaddULL, 0x426a00665e5c4479ULL, 0x1800deef121f1e76ULL,
    0x97e485b7aef312c2ULL, 0xf1aa493335a9e712ULL, 0x7260bfb731fb5d25ULL, 0x198e9393920d483aULL,
    0x4ce6cc0166fa7daaULL, 0xe3d1e7690c43d37bULL, 0x4aab71808dcb408fULL, 0x12c85ea5db8c6debULL,
    0x55acdadcd122975bULL, 0xbc4b313370b38ef3ULL, 0xec9e99ad690c3395ULL, 0x090689d0585ff075ULL,
    1, 0, 0, 0, 0, 0, 0, 0};
bool fq_any_geq_q(const uint64_t* p, size_t nfe) {
  for (size_t k = 0; k < nfe; k++) {
    Fq v;
    std::memcpy(&v, p + 4 * k, sizeof v);
    if (v.geq_modulus()) return true;
  }
  return false;
}
bool g2_at_infinity(const uint64_t* p) { return !(p[16] | p[17] | p[18] | p[19] | p[20] | p[21] | p[22] | p[23]); }
// The verification key's code: a G2 point at infinity (B200_EINVAL, before anything else) or a coordinate >= q (B200_ERANGE)
// among IC[0..npub], vk_g1 and vk_g2.
int pv_vk_code(const uint64_t* ic, size_t npub, const uint64_t* vk_g1, const uint64_t* vk_g2) {
  for (int k = 0; k < 5; k++)
    if (g2_at_infinity(vk_g2 + 24 * k)) return B200_EINVAL;
  if (fq_any_geq_q(ic, 3 * (npub + 1)) || fq_any_geq_q(vk_g1, 6) || fq_any_geq_q(vk_g2, 30)) return B200_ERANGE;
  return B200_OK;
}
// The twelve pairings and five checks of snark.VerifyProof for m proofs on the device: proof idx[b] (b when idx is null).
// P, B: the proofs' G1 points and PiB; vkx: their IC sums; vk1, vk2 as k_pv_pairs reads them.  failed (host, m ints): 0 or
// the first failing check.  Inputs are validated by the caller.
int pv_check(const Fq* P, const Fq2* B, const Fq* vkx, const Fq* vk1, const Fq2* vk2, const uint32_t* idx, size_t m,
             int* failed) {
  DevBuf d1, d2, de, df;
  CU(d1.alloc(12 * m * 3 * sizeof(Fq)));
  CU(d2.alloc(12 * m * 3 * sizeof(Fq2)));
  CU(de.alloc(12 * m * 6 * sizeof(Fq2)));
  CU(df.alloc(m * sizeof(int)));
  cudaStream_t s = g_stream;
  pv::k_pv_pairs<<<nblk(m, 64), 64, 0, s>>>(P, B, vkx, vk1, vk2, idx, m, d1.as<Fq>(), d2.as<Fq2>());
  pairing_enqueue(d1.as<Fq>(), d2.as<Fq2>(), 12 * m, de.as<Fq2>(), s);
  pv::k_pv_compare<<<nblk(m, 64), 64, 0, s>>>(de.as<Fq2>(), m, df.as<int>());
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(failed, df.p, m * sizeof(int), cudaMemcpyDeviceToHost, s));
  return check_err_flag<Fq>("pinocchio_verify");
}

int pinocchio_verify_host(const uint64_t* ic, size_t n_ic, const uint64_t* vk_g1, const uint64_t* vk_g2,
                          const uint64_t* proof_g1, const uint64_t* pi_b, const uint64_t* pub, size_t npub, int* ok,
                          int* failed_check) {
  if (!ic || !vk_g1 || !vk_g2 || !proof_g1 || !pi_b || !ok || (npub && !pub)) return fail(B200_EINVAL, "pinocchio_verify: null pointer");
  if (n_ic < npub + 1) return fail(B200_EINVAL, "pinocchio_verify: len(IC) < len(publicSignals) + 1");
  const int vkc = pv_vk_code(ic, npub, vk_g1, vk_g2);
  if (vkc == B200_EINVAL || g2_at_infinity(pi_b))
    return fail(B200_EINVAL, "pinocchio_verify: q1[2] != Fq2.One() (G2 point at infinity; the reference panics, bn128.go:238-241)");
  if (vkc || fq_any_geq_q(proof_g1, 21) || fq_any_geq_q(pi_b, 6)) return fail(B200_ERANGE, "pinocchio_verify: point coordinate >= q");
  std::vector<GlvScalar> gs(npub ? npub : 1);
  for (size_t i = 0; i < npub; i++) {
    Fr v = fr_load_std(pub + 4 * i);
    if (v.geq_modulus()) return fail(B200_ERANGE, "pinocchio_verify: scalar / coefficient >= r");
    if (glv_decompose(v, gs[i].k, gs[i].neg)) return fail(B200_EINVAL, "pinocchio_verify: GLV decomposition out of range");
  }
  DevBuf dic, dsig, dterms, dvkx, dP, dB, dvk1, dvk2;
  CU(dic.alloc((npub + 1) * 3 * sizeof(Fq)));
  CU(dsig.alloc(gs.size() * sizeof(GlvScalar)));
  CU(dterms.alloc(gs.size() * sizeof(Jacobian<Fq>)));
  CU(dvkx.alloc(3 * sizeof(Fq)));
  CU(dP.alloc(21 * sizeof(Fq)));
  CU(dB.alloc(3 * sizeof(Fq2)));
  CU(dvk1.alloc(6 * sizeof(Fq)));
  CU(dvk2.alloc(18 * sizeof(Fq2)));
  cudaStream_t s = g_stream;
  CU(cudaMemcpyAsync(dic.p, ic, (npub + 1) * 3 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  if (npub) CU(cudaMemcpyAsync(dsig.p, gs.data(), npub * sizeof(GlvScalar), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dP.p, proof_g1, 21 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dB.p, pi_b, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk1.p, vk_g1, 6 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk2.p, kG2Gen, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk2.as<Fq2>() + 3, vk_g2, 15 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  if (npub) k_ic_terms<<<(unsigned)((npub + 1) / 2), 32, 0, s>>>(dic.as<Fq>(), dsig.as<GlvScalar>(), npub, dterms.as<Jacobian<Fq>>(), g_d_err);
  k_ic_sum<<<1, 32, 0, s>>>(dic.as<Fq>(), dterms.as<Jacobian<Fq>>(), npub, dvkx.as<Fq>(), g_d_err);
  int failed = -1;
  if (int rc = pv_check(dP.as<Fq>(), dB.as<Fq2>(), dvkx.as<Fq>(), dvk1.as<Fq>(), dvk2.as<Fq2>(), nullptr, 1, &failed)) return rc;
  *ok = failed == 0 ? 1 : 0;
  if (failed_check) *failed_check = failed;
  return B200_OK;
}

// snark.VerifyProof for nproofs proofs under one key (include/b200snark.h b200_pinocchio_verify_batch).  The proofs the
// reference pairs bilinearly enter ONE aggregated check (N + 6 Miller loops, one final exponentiation, verify_batch_pinocchio.cuh);
// the others, and every proof of a batch whose aggregated check fails, run the twelve pairings of b200_pinocchio_verify.
// As for Groth16, a failed check verifies its proofs one by one rather than bisecting.
int pinocchio_verify_batch_host(const uint64_t* ic, size_t n_ic, const uint64_t* vk_g1, const uint64_t* vk_g2, size_t n,
                                const uint64_t* proofs_g1, const uint64_t* pi_b, const uint64_t* pub, size_t npub,
                                const uint64_t* rho, int* ok, uint64_t* stats) {
  if (!ic || !vk_g1 || !vk_g2 || !proofs_g1 || !pi_b || !rho || !ok || (npub && !pub) || n == 0)
    return fail(B200_EINVAL, "pinocchio_verify_batch: null pointer or no proofs");
  if (n_ic < npub + 1) return fail(B200_EINVAL, "pinocchio_verify_batch: len(IC) < len(publicSignals) + 1");
  if (n > (1u << 26)) return fail(B200_EINVAL, "pinocchio_verify_batch: more than 2^26 proofs");
  for (size_t k = 0; k < 5 * n; k++)
    if (!rho[2 * k] && !rho[2 * k + 1]) return fail(B200_EINVAL, "pinocchio_verify_batch: rho[%zu][%zu] = 0", k / 5, k % 5);
  const int vkc = pv_vk_code(ic, npub, vk_g1, vk_g2);
  if (vkc == B200_EINVAL) return fail(B200_EINVAL, "pinocchio_verify_batch: q1[2] != Fq2.One() (verification key G2 point at infinity)");
  if (vkc) return fail(B200_ERANGE, "pinocchio_verify_batch: verification key coordinate >= q");
  std::vector<int> st(n, 0);   // a public signal >= r: B200_ERANGE unless k_pv_prepare finds PiB at infinity
  for (size_t i = 0; i < n; i++)
    for (size_t j = 0; j < npub; j++)
      if (fr_load_std(pub + 4 * (i * npub + j)).geq_modulus()) st[i] = B200_ERANGE;
  const size_t np = n + 6;
  DevBuf dic, dvk1, dvk2, dP, dB, dpub, drho, dst, dterms, dvkx, dic_aff, dg1_aff, dg2_aff, dbad, dpts, dqb, dpairs, dsums, dsum,
      dT, df, dfe, dres;
  CU(dic.alloc((npub + 1) * 3 * sizeof(Fq)));
  CU(dvk1.alloc(6 * sizeof(Fq)));
  CU(dvk2.alloc(18 * sizeof(Fq2)));
  CU(dP.alloc(n * 21 * sizeof(Fq)));
  CU(dB.alloc(n * 3 * sizeof(Fq2)));
  CU(dpub.alloc(std::max<size_t>(n * npub, 1) * 4 * sizeof(uint64_t)));
  CU(drho.alloc(n * 10 * sizeof(uint64_t)));
  CU(dst.alloc(n * sizeof(int)));
  CU(dterms.alloc(std::max<size_t>(n * npub, 1) * sizeof(Jacobian<Fq>)));
  CU(dvkx.alloc(n * 3 * sizeof(Fq)));
  CU(dic_aff.alloc((npub + 1) * sizeof(Affine<Fq>)));
  CU(dg1_aff.alloc(pv::kVkG1 * sizeof(Affine<Fq>)));
  CU(dg2_aff.alloc(pv::kVkG2 * sizeof(Affine<Fq2>)));
  CU(dbad.alloc(sizeof(int)));
  CU(dpts.alloc(n * pv::kPts * sizeof(Affine<Fq>)));
  CU(dqb.alloc(n * sizeof(Affine<Fq2>)));
  cudaStream_t s = g_stream;
  CU(cudaMemcpyAsync(dic.p, ic, (npub + 1) * 3 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk1.p, vk_g1, 6 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk2.p, kG2Gen, 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dvk2.as<Fq2>() + 3, vk_g2, 15 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dP.p, proofs_g1, n * 21 * sizeof(Fq), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dB.p, pi_b, n * 3 * sizeof(Fq2), cudaMemcpyHostToDevice, s));
  if (npub) CU(cudaMemcpyAsync(dpub.p, pub, n * npub * 4 * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(drho.p, rho, n * 10 * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dst.p, st.data(), n * sizeof(int), cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(dbad.p, 0, sizeof(int), s));
  // 1. the key, vkx_i, per-proof preparation
  pv::k_pv_vk<<<1, 32, 0, s>>>(dic.as<Fq>(), (uint32_t)(npub + 1), dvk1.as<Fq>(), dvk2.as<Fq2>(), dic_aff.as<Affine<Fq>>(),
                               dg1_aff.as<Affine<Fq>>(), dg2_aff.as<Affine<Fq2>>(), dbad.as<int>());
  if (npub) vb::k_vb_ic_terms<<<nblk(n * npub, 64), 64, 0, s>>>(dic_aff.as<Affine<Fq>>(), dpub.as<uint64_t>(), n, npub, dterms.as<Jacobian<Fq>>());
  vb::k_vb_ic_sum<<<nblk(n, 64), 64, 0, s>>>(dic.as<Fq>(), dterms.as<Jacobian<Fq>>(), n, npub, dvkx.as<Fq>());
  pv::k_pv_prepare<<<nblk(n, 64), 64, 0, s>>>(dP.as<Fq>(), dB.as<Fq2>(), dvkx.as<Fq>(), n, dst.as<int>(), dpts.as<Affine<Fq>>(),
                                              dqb.as<Affine<Fq2>>());
  CU(cudaGetLastError());
  int vk_bad = 0;
  CU(cudaMemcpyAsync(st.data(), dst.p, n * sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&vk_bad, dbad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (vk_bad) return fail(B200_EINVAL, "pinocchio_verify_batch: verification key point at infinity, off the curve, or outside G2");
  std::vector<uint32_t> each;
  size_t n_agg = 0;
  for (size_t i = 0; i < n; i++) {
    if (st[i] == vb::kEach) each.push_back((uint32_t)i);
    if (st[i] == vb::kAgg) n_agg++;
  }
  uint64_t st_stats[4] = {n_agg, 0, 0, 0};
  bool agg_ok = false;
  if (n_agg) {
    // 2. the seven products per proof, tree sums of the six arrays, the six fixed-G2 pairs
    CU(dpairs.alloc(np * sizeof(vb::Pair)));
    CU(dsums.alloc(6 * n * sizeof(XYZZ<Fq>)));
    CU(dres.alloc(2 * sizeof(int)));
    CU(cudaMemsetAsync(dres.p, 0, 2 * sizeof(int), s));
    pv::k_pv_products<<<nblk(pv::kProducts * n, 64), 64, 0, s>>>(dpts.as<Affine<Fq>>(), dqb.as<Affine<Fq2>>(), dg1_aff.as<Affine<Fq>>(),
                                                                 drho.as<uint64_t>(), dst.as<int>(), n, dsums.as<XYZZ<Fq>>(),
                                                                 dpairs.as<vb::Pair>(), dres.as<int>());
    const uint32_t kSum = 32;
    size_t levels = 0;   // every level of every sum gets its own slots
    for (size_t m = n; m > 1; m = nblk(m, kSum)) levels += nblk(m, kSum);
    CU(dsum.alloc(std::max<size_t>(6 * levels, 1) * sizeof(XYZZ<Fq>)));
    pv::Sums6 sums;
    XYZZ<Fq>* slot = dsum.as<XYZZ<Fq>>();
    for (int k = 0; k < 6; k++) {
      const XYZZ<Fq>* cur = dsums.as<XYZZ<Fq>>() + k * n;
      for (size_t m = n; m > 1; m = nblk(m, kSum)) {
        vb::k_vb_sum<<<nblk(nblk(m, kSum), 64), 64, 0, s>>>(cur, m, kSum, slot);
        cur = slot;
        slot += nblk(m, kSum);
      }
      sums.s[k] = cur;
    }
    pv::k_pv_tail<<<1, 32, 0, s>>>(sums, dg2_aff.as<Affine<Fq2>>(), dpairs.as<vb::Pair>() + n, dres.as<int>());
    // 3. multi-Miller loop, 4. product tree and one final exponentiation
    const uint32_t chunk = (uint32_t)std::max<size_t>(1, nblk(np, kMillerThreads));
    const size_t nth = nblk(np, chunk);
    CU(dT.alloc(np * sizeof(Jacobian<Fq2>)));
    CU(df.alloc(nth * sizeof(F12)));
    CU(dfe.alloc(nblk(nth, 2) * sizeof(F12)));
    vb::k_vb_miller<<<nblk(nth, 64), 64, 0, s>>>(dpairs.as<vb::Pair>(), np, chunk, dT.as<Jacobian<Fq2>>(), df.as<F12>());
    F12 *a = df.as<F12>(), *b = dfe.as<F12>();
    for (size_t m = nth; m > 1; m = nblk(m, 2)) {
      vb::k_vb_f12_tree<<<nblk(nblk(m, 2), 64), 64, 0, s>>>(a, m, b);
      std::swap(a, b);
    }
    vb::k_vb_final_exp<<<1, 32, 0, s>>>(a, dres.as<int>() + 1, nullptr);
    CU(cudaGetLastError());
    int res[2] = {0, 0};
    CU(cudaMemcpyAsync(res, dres.p, sizeof res, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    agg_ok = res[1] == 1;
    st_stats[2] = 1;
    st_stats[3] = (uint64_t)res[0];
    if (!agg_ok)
      for (size_t i = 0; i < n; i++)
        if (st[i] == vb::kAgg) each.push_back((uint32_t)i);
  }
  std::vector<int> failed(each.size(), 0);
  if (!each.empty()) {
    DevBuf didx;
    CU(didx.alloc(each.size() * sizeof(uint32_t)));
    CU(cudaMemcpyAsync(didx.p, each.data(), each.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    if (int rc = pv_check(dP.as<Fq>(), dB.as<Fq2>(), dvkx.as<Fq>(), dvk1.as<Fq>(), dvk2.as<Fq2>(), didx.as<uint32_t>(), each.size(),
                          failed.data()))
      return rc;
    st_stats[1] = each.size();
    st_stats[3] += 12 * (uint64_t)each.size();
  }
  for (size_t i = 0; i < n; i++) ok[i] = st[i] < 0 ? st[i] : (st[i] == vb::kAgg && agg_ok ? 1 : 0);
  for (size_t k = 0; k < each.size(); k++) ok[each[k]] = failed[k] == 0 ? 1 : 0;
  if (stats) std::memcpy(stats, st_stats, sizeof st_stats);
  return B200_OK;
}

#else  // experiment builds without the verifier side (ptxas 12.9 crashes on the pairing kernels under -DB200_KARATSUBA)
int pairing_batch_host(const uint64_t*, const uint64_t*, size_t, uint64_t*) { return fail(B200_EINVAL, "pairing: not in this build variant"); }
int fq12_mul_batch_host(const uint64_t*, const uint64_t*, size_t, uint64_t*) { return fail(B200_EINVAL, "fq12_mul: not in this build variant"); }
int groth16_verify_host(const uint64_t*, size_t, const uint64_t*, const uint64_t*, const uint64_t*, const uint64_t*, const uint64_t*,
                        const uint64_t*, const uint64_t*, const uint64_t*, size_t, int*) {
  return fail(B200_EINVAL, "groth16_verify: not in this build variant");
}
int groth16_verify_batch_host(const uint64_t*, size_t, const uint64_t*, const uint64_t*, const uint64_t*, const uint64_t*, size_t,
                              const uint64_t*, const uint64_t*, const uint64_t*, const uint64_t*, size_t, const uint64_t*, int*,
                              uint64_t*) {
  return fail(B200_EINVAL, "groth16_verify_batch: not in this build variant");
}
int pinocchio_verify_host(const uint64_t*, size_t, const uint64_t*, const uint64_t*, const uint64_t*, const uint64_t*,
                          const uint64_t*, size_t, int*, int*) {
  return fail(B200_EINVAL, "pinocchio_verify: not in this build variant");
}
int pinocchio_verify_batch_host(const uint64_t*, size_t, const uint64_t*, const uint64_t*, size_t, const uint64_t*,
                                const uint64_t*, const uint64_t*, size_t, const uint64_t*, int*, uint64_t*) {
  return fail(B200_EINVAL, "pinocchio_verify_batch: not in this build variant");
}
#endif

template <class F>
int group_op_host(int op, const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out) {
  if (!p || !out || (op == 0 && !q)) return fail(B200_EINVAL, "group op: null pointer");
  if (n == 0) return B200_OK;
  DevBuf dp, dq, dout;
  size_t out_fe = op == 3 ? 2 : 3;
  CU(dp.alloc(n * 3 * sizeof(F)));
  CU(dout.alloc(n * out_fe * sizeof(F)));
  CU(cudaMemcpyAsync(dp.p, p, n * 3 * sizeof(F), cudaMemcpyHostToDevice, g_stream));
  if (op == 0) {
    CU(dq.alloc(n * 3 * sizeof(F)));
    CU(cudaMemcpyAsync(dq.p, q, n * 3 * sizeof(F), cudaMemcpyHostToDevice, g_stream));
  }
  if (op == 3)
    k_group_affine<F><<<nblk(n, 128), 128, 0, g_stream>>>(dp.as<F>(), n, dout.as<F>(), g_d_err);
  else
    k_group_op<F><<<nblk(n, 128), 128, 0, g_stream>>>(op, dp.as<F>(), dq.as<F>(), n, dout.as<F>(), g_d_err);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, dout.p, n * out_fe * sizeof(F), cudaMemcpyDeviceToHost, g_stream));
  return check_err_flag<F>("group op");
}

}  // namespace

// On an error return, work already queued on the library's streams is drained first: no entry point leaves kernels in
// flight that still read the caller's (or the library's soon-to-be-reused) buffers.
inline int drain_on_error(int rc) {
  if (rc != B200_OK && g_init) cudaDeviceSynchronize();
  return rc;
}
extern "C" {

int b200_groth16_pk_load(const uint64_t* at, const uint64_t* b1, const uint64_t* b2, const uint64_t* bacdelta,
                         size_t m, const uint64_t* ptd, size_t n_ptd, const uint64_t* z, size_t nz,
                         const uint64_t alpha1[12], const uint64_t beta1[12], const uint64_t delta1[12],
                         const uint64_t beta2[24], const uint64_t delta2[24], size_t npublic, int window_bits,
                         b200_pk_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return groth16_pk_load(at, b1, b2, bacdelta, m, ptd, n_ptd, z, nz, alpha1, beta1, delta1, beta2, delta2, npublic,
                         window_bits, 0, 1, out);
}
int b200_groth16_pk_load_shard(const uint64_t* at, const uint64_t* b1, const uint64_t* b2, const uint64_t* bacdelta,
                               size_t m, const uint64_t* ptd, size_t n_ptd, const uint64_t* z, size_t nz,
                               const uint64_t alpha1[12], const uint64_t beta1[12], const uint64_t delta1[12],
                               const uint64_t beta2[24], const uint64_t delta2[24], size_t npublic, int window_bits,
                               int rank, int world, b200_pk_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return groth16_pk_load(at, b1, b2, bacdelta, m, ptd, n_ptd, z, nz, alpha1, beta1, delta1, beta2, delta2, npublic,
                         window_bits, rank, world, out);
}
int b200_groth16_finalize_device(b200_pk_t pk, const void* d_parts, int nparts, const uint64_t r[4],
                                 const uint64_t s[4], void* d_out, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  ProvingKey* p = find_pk(pk, 1);
  if (!p || !d_parts || nparts < 1 || !r || !s || !d_out) return fail(B200_EINVAL, "groth16_finalize_device: bad arguments");
  return drain_on_error(groth16_finalize_enqueue(p, (const uint8_t*)d_parts, nparts, r, s, (Fq*)d_out,
                                  stream ? (cudaStream_t)stream : g_stream));
}
int b200_groth16_prove(b200_pk_t pk, const uint64_t* w, size_t nw, const uint64_t* px, size_t npx,
                       const uint64_t r[4], const uint64_t s[4], uint64_t pi_a[12], uint64_t pi_b[24],
                       uint64_t pi_c[12]) {
  std::unique_lock<std::mutex> lk(g_mu);
  NEED_INIT();
  return drain_on_error(groth16_prove(pk, w, nw, px, npx, r, s, pi_a, pi_b, pi_c, &lk));
}
int b200_pinocchio_pk_load(const uint64_t* a, const uint64_t* ap, const uint64_t* b2, const uint64_t* bp,
                           const uint64_t* c, const uint64_t* cp, const uint64_t* kp, size_t m,
                           const uint64_t* g1t, size_t n_g1t, const uint64_t* z, size_t nz, size_t npublic,
                           int window_bits, b200_pk_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return pinocchio_pk_load(a, ap, b2, bp, c, cp, kp, m, g1t, n_g1t, z, nz, npublic, window_bits, 0, 1, out);
}
int b200_pinocchio_pk_load_shard(const uint64_t* a, const uint64_t* ap, const uint64_t* b2, const uint64_t* bp,
                                 const uint64_t* c, const uint64_t* cp, const uint64_t* kp, size_t m,
                                 const uint64_t* g1t, size_t n_g1t, const uint64_t* z, size_t nz, size_t npublic,
                                 int window_bits, int rank, int world, b200_pk_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return pinocchio_pk_load(a, ap, b2, bp, c, cp, kp, m, g1t, n_g1t, z, nz, npublic, window_bits, rank, world, out);
}
int b200_pinocchio_prove_record_device(b200_pk_t pk, const uint64_t* w, size_t nw, const uint64_t* px, size_t npx, void* d_record) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  if (!d_record) return fail(B200_EINVAL, "pinocchio_prove_record_device: null record pointer");
  int rc = pinocchio_prove(pk, w, nw, px, npx, nullptr, nullptr, (uint8_t*)d_record);
  if (rc) return rc;
  return check_err_flag<Fr>("pinocchio_prove_record");
}
int b200_pinocchio_finalize_records(const void* d_records, int world, uint64_t* out_g1, uint64_t pi_b[24]) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return pinocchio_finalize_records((const uint8_t*)d_records, world, out_g1, pi_b);
}
int b200_pinocchio_prove(b200_pk_t pk, const uint64_t* w, size_t nw, const uint64_t* px, size_t npx,
                         uint64_t* out_g1 /* 7 x 12: PiA PiAp PiBp PiC PiCp PiH PiKp */, uint64_t pi_b[24]) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return drain_on_error(pinocchio_prove(pk, w, nw, px, npx, out_g1, pi_b));
}
int b200_groth16_prove_device(b200_pk_t pk, const void* d_w, size_t nw, const void* d_px, size_t npx,
                              const uint64_t r[4], const uint64_t s[4], void* d_out, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  ProvingKey* p = find_pk(pk, 1);
  if (!p || !d_w || !d_px || !r || !s || !d_out) return fail(B200_EINVAL, "groth16_prove_device: bad arguments");
  return drain_on_error(groth16_enqueue(p, (const Fr*)d_w, nw, (const Fr*)d_px, npx, r, s, (Fq*)d_out,
                         stream ? (cudaStream_t)stream : g_stream));
}
int b200_comm_unique_id(uint8_t out[128]) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!out) return fail(B200_EINVAL, "comm_unique_id: null pointer");
  if (const char* e = g_comm.api.load()) return fail(B200_ECOMM, "comm_unique_id: %s", e);
  ncclUniqueId id;
  ncclResult_t rc = g_comm.api.GetUniqueId(&id);
  if (rc != ncclSuccess) return fail(B200_ECOMM, "ncclGetUniqueId: %s", g_comm.api.GetErrorString(rc));
  memcpy(out, &id, 128);
  return B200_OK;
}
int b200_comm_init(const uint8_t id[128], int rank, int world) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  if (!id || world < 1 || rank < 0 || rank >= world) return fail(B200_EINVAL, "comm_init: bad arguments");
  if (g_comm.active()) return fail(B200_EINVAL, "comm_init: communicator already initialised (rank %d/%d)", g_comm.rank, g_comm.world);
  if (const char* e = g_comm.api.load()) return fail(B200_ECOMM, "comm_init: %s", e);
  ncclUniqueId uid;
  memcpy(&uid, id, 128);
  ncclResult_t rc = g_comm.api.CommInitRank(&g_comm.comm, world, uid, rank);
  if (rc != ncclSuccess) {
    g_comm.comm = nullptr;
    return fail(B200_ECOMM, "ncclCommInitRank: %s", g_comm.api.GetErrorString(rc));
  }
  g_comm.rank = rank;
  g_comm.world = world;
  // context 1's communicator (collective: every rank is inside b200_comm_init); older NCCL without ncclCommSplit: both
  // contexts share `comm` and only ONE host thread may prove on sharded keys
  g_comm.comm1 = nullptr;
  if (g_comm.api.CommSplit && world > 1) {
    rc = g_comm.api.CommSplit(g_comm.comm, 0, rank, &g_comm.comm1, nullptr);
    if (rc != ncclSuccess) g_comm.comm1 = nullptr;
  }
  return B200_OK;
}
int b200_comm_destroy(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_comm.active()) return B200_OK;
  cudaSetDevice(g_device);
  cudaDeviceSynchronize();
  if (g_comm.comm1) g_comm.api.CommDestroy(g_comm.comm1);
  g_comm.comm1 = nullptr;
  g_comm.api.CommDestroy(g_comm.comm);
  g_comm.comm = nullptr;
  g_comm.world = 1;
  g_comm.rank = 0;
  return B200_OK;
}
int b200_groth16_shard_info(b200_pk_t pk, uint64_t out[12]) {
  std::lock_guard<std::mutex> lk(g_mu);
  ProvingKey* p = find_pk(pk, 1);
  if (!p || !out) return fail(B200_EINVAL, "groth16_shard_info: bad arguments");
  const size_t l1 = p->npublic + 1, ncf = p->n_c_full;
  for (int k = 0; k < 3; k++) { out[2 * k] = p->lo[k]; out[2 * k + 1] = p->hi[k]; }
  size_t lo3 = p->lo[3], hi3 = p->hi[3];
  size_t c_lo = lo3 < ncf ? lo3 : ncf, c_hi = hi3 < ncf ? hi3 : ncf;
  out[6] = l1 + c_lo;                       // witness range feeding this rank's C part
  out[7] = l1 + c_hi;
  out[8] = hi3 > ncf ? 1 : 0;               // holds PowersTauDelta indices => needs px
  out[9] = (uint64_t)p->rank;
  out[10] = (uint64_t)p->world;
  out[11] = p->m;
  return B200_OK;
}
int b200_profile(int enable) {
  std::lock_guard<std::mutex> lk(g_mu);
  g_prof = (enable & 1) != 0;
  g_serial = (enable & 2) != 0;
  return B200_OK;
}
int b200_profile_read(double out[8]) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  if (!out) return fail(B200_EINVAL, "profile_read: null pointer");
  for (int i = 0; i < 8; i++) out[i] = 0;
  CU(cudaDeviceSynchronize());
  for (auto& r : g_prof_recs) {
    float ms = 0;
    cudaEventElapsedTime(&ms, r.e0, r.e1);
    int o = r.group == 1 ? 0 : 3;
    out[o] += ms;
    out[o + 1] += 1;
    out[o + 2] += (double)r.terms;
    g_event_pool.push_back(r.e0);
    g_event_pool.push_back(r.e1);
  }
  g_prof_recs.clear();
  out[6] = (double)g_launches;
  g_launches = 0;
  return B200_OK;
}
int b200_pk_free(b200_pk_t pk) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_init) return fail(B200_EINVAL, "not initialised");
  cudaSetDevice(g_device);
  cudaStreamSynchronize(g_stream);
  return g_pks.erase(pk) ? B200_OK : fail(B200_EINVAL, "pk_free: bad handle");
}

#define B200_API_BODY(expr)              \
  std::lock_guard<std::mutex> lk(g_mu);  \
  NEED_INIT();                           \
  return drain_on_error(expr);
int b200_r1cs_to_qap(const uint64_t* a, const uint64_t* b, const uint64_t* c, size_t n, size_t m, uint64_t* alphas,
                     uint64_t* betas, uint64_t* gammas, uint64_t* z) {
  B200_API_BODY(r1cs_to_qap_host(a, b, c, n, m, alphas, betas, gammas, z))
}
int b200_combine_polynomials(const uint64_t* r, size_t m, const uint64_t* ap, const uint64_t* bp, const uint64_t* cp,
                             size_t n, uint64_t* ax, uint64_t* bx, uint64_t* cx, uint64_t* px) {
  B200_API_BODY(combine_polynomials_host(r, m, ap, bp, cp, n, ax, bx, cx, px))
}
int b200_poly_add(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* out) { B200_API_BODY(poly_addsub_host(a, na, b, nb, 0, out)) }
int b200_poly_sub(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* out) { B200_API_BODY(poly_addsub_host(a, na, b, nb, 1, out)) }
int b200_poly_eval(const uint64_t* v, size_t n, const uint64_t x[4], uint64_t out[4]) { B200_API_BODY(poly_eval_host(v, n, x, out)) }
int b200_poly_eval_batch(const uint64_t* polys, size_t m, size_t n, const uint64_t x[4], uint64_t* out) { B200_API_BODY(poly_eval_batch_host(polys, m, n, x, out)) }
int b200_zero_poly(size_t n, uint64_t* out) { B200_API_BODY(zero_poly_host(n, out)) }
int b200_r1cs_load(size_t n, size_t m, const uint32_t* a_rowptr, const uint32_t* a_col, const uint64_t* a_val,
                   const uint32_t* b_rowptr, const uint32_t* b_col, const uint64_t* b_val, const uint32_t* c_rowptr,
                   const uint32_t* c_col, const uint64_t* c_val, b200_r1cs_t* out) {
  const uint32_t* const rp[3] = {a_rowptr, b_rowptr, c_rowptr};
  const uint32_t* const cl[3] = {a_col, b_col, c_col};
  const uint64_t* const vl[3] = {a_val, b_val, c_val};
  B200_API_BODY(r1cs_load(n, m, rp, cl, vl, out))
}
int b200_r1cs_free(b200_r1cs_t h) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_r1cs.erase(h)) return fail(B200_EINVAL, "r1cs_free: bad handle");
  return B200_OK;
}
int b200_qap_px(b200_r1cs_t h, const uint64_t* w, size_t nw, uint64_t* ax, uint64_t* bx, uint64_t* cx, uint64_t* px) {
  B200_API_BODY(qap_px_host(h, w, nw, ax, bx, cx, px))
}
int b200_qap_eval_at(b200_r1cs_t h, const uint64_t tau[4], size_t nz, uint64_t* at, uint64_t* bt, uint64_t* ct, uint64_t zt[4]) {
  B200_API_BODY(qap_eval_at_host(h, tau, nz, at, bt, ct, zt))
}
int b200_interpolate(const uint64_t* values, size_t n, uint64_t* coeffs) { B200_API_BODY(interpolate_host(values, n, coeffs)) }
int b200_groth16_prove_witness(b200_pk_t pk, b200_r1cs_t r1cs, const uint64_t* w, size_t nw, const uint64_t r[4],
                               const uint64_t s[4], uint64_t pi_a[12], uint64_t pi_b[24], uint64_t pi_c[12]) {
  B200_API_BODY(groth16_prove_witness(pk, r1cs, w, nw, r, s, pi_a, pi_b, pi_c))
}
int b200_fq12_mul_batch(const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out) { B200_API_BODY(fq12_mul_batch_host(a, b, n, out)) }
int b200_pairing_batch(const uint64_t* g1_jac, const uint64_t* g2_jac, size_t n, uint64_t* out) { B200_API_BODY(pairing_batch_host(g1_jac, g2_jac, n, out)) }
int b200_groth16_verify(const uint64_t* ic, size_t n_ic, const uint64_t alpha1[12], const uint64_t beta2[24],
                        const uint64_t gamma2[24], const uint64_t delta2[24], const uint64_t pi_a[12],
                        const uint64_t pi_b[24], const uint64_t pi_c[12], const uint64_t* public_signals, size_t n_public,
                        int* ok) {
  B200_API_BODY(groth16_verify_host(ic, n_ic, alpha1, beta2, gamma2, delta2, pi_a, pi_b, pi_c, public_signals, n_public, ok))
}
int b200_groth16_verify_batch(const uint64_t* ic, size_t n_ic, const uint64_t alpha1[12], const uint64_t beta2[24],
                              const uint64_t gamma2[24], const uint64_t delta2[24], size_t nproofs, const uint64_t* pi_a,
                              const uint64_t* pi_b, const uint64_t* pi_c, const uint64_t* public_signals, size_t n_public,
                              const uint64_t* rho, int* ok, uint64_t stats[4]) {
  B200_API_BODY(groth16_verify_batch_host(ic, n_ic, alpha1, beta2, gamma2, delta2, nproofs, pi_a, pi_b, pi_c, public_signals,
                                          n_public, rho, ok, stats))
}
int b200_pinocchio_verify(const uint64_t* ic, size_t n_ic, const uint64_t vk_g1[24], const uint64_t vk_g2[120],
                          const uint64_t proof_g1[84], const uint64_t pi_b[24], const uint64_t* public_signals,
                          size_t n_public, int* ok, int* failed_check) {
  B200_API_BODY(pinocchio_verify_host(ic, n_ic, vk_g1, vk_g2, proof_g1, pi_b, public_signals, n_public, ok, failed_check))
}
int b200_pinocchio_verify_batch(const uint64_t* ic, size_t n_ic, const uint64_t vk_g1[24], const uint64_t vk_g2[120],
                                size_t nproofs, const uint64_t* proofs_g1, const uint64_t* pi_b,
                                const uint64_t* public_signals, size_t n_public, const uint64_t* rho, int* ok,
                                uint64_t stats[4]) {
  B200_API_BODY(pinocchio_verify_batch_host(ic, n_ic, vk_g1, vk_g2, nproofs, proofs_g1, pi_b, public_signals, n_public, rho,
                                            ok, stats))
}
int b200_g1_add_batch(const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out) { B200_API_BODY(group_op_host<Fq>(0, p, q, n, out)) }
int b200_g1_double_batch(const uint64_t* p, size_t n, uint64_t* out) { B200_API_BODY(group_op_host<Fq>(1, p, nullptr, n, out)) }
int b200_g1_neg_batch(const uint64_t* p, size_t n, uint64_t* out) { B200_API_BODY(group_op_host<Fq>(2, p, nullptr, n, out)) }
int b200_g1_affine_batch(const uint64_t* p, size_t n, uint64_t* out_xy) { B200_API_BODY(group_op_host<Fq>(3, p, nullptr, n, out_xy)) }
int b200_g2_add_batch(const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out) { B200_API_BODY(group_op_host<Fq2>(0, p, q, n, out)) }
int b200_g2_double_batch(const uint64_t* p, size_t n, uint64_t* out) { B200_API_BODY(group_op_host<Fq2>(1, p, nullptr, n, out)) }
int b200_g2_neg_batch(const uint64_t* p, size_t n, uint64_t* out) { B200_API_BODY(group_op_host<Fq2>(2, p, nullptr, n, out)) }
int b200_g2_affine_batch(const uint64_t* p, size_t n, uint64_t* out_xy) { B200_API_BODY(group_op_host<Fq2>(3, p, nullptr, n, out_xy)) }

int b200_poly_mul(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return poly_mul_host(a, na, b, nb, out);
}
int b200_poly_div(const uint64_t* a, size_t na, const uint64_t* b, size_t nb, uint64_t* q, uint64_t* rem) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return poly_div_host(a, na, b, nb, q, rem);
}


int b200_version(void) { return 200; }
int b200_config(int key, int value) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (key == B200_CFG_ACC_MODE && value >= 0 && value <= 2) {
    g_acc_mode = value;
    return B200_OK;
  }
  if (key >= 10 && key <= 13 && value > 0) {   // shard-partition tuning (tools/shard_times.py sweeps them)
    (key == 10 ? g_w_ab : key == 11 ? g_w_g2 : key == 12 ? g_aff_min_g1 : g_aff_min_g2) = value;
    return B200_OK;
  }
  if (key == B200_CFG_PAIRING_KERNEL && value >= 0 && value <= 2) {
    g_pairing_kernel = value;
    return B200_OK;
  }
  if (key == B200_CFG_PK_CONTEXT && (value == 0 || value == 1)) {
    g_pk_ctx = value;
    return B200_OK;
  }
  if (key == B200_CFG_TMA_STAGING && value >= 0 && value <= 2) {
    g_tma_staging = value;
    return B200_OK;
  }
  return fail(B200_EINVAL, "b200_config: unknown key %d or bad value %d", key, value);
}

const char* b200_last_error(void) { return g_err.c_str(); }

int b200_init(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  return init_locked(device);
}

int b200_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_init) return B200_OK;
  cudaSetDevice(g_device);
  if (g_comm.active()) {
    cudaDeviceSynchronize();
    if (g_comm.comm1) g_comm.api.CommDestroy(g_comm.comm1);
    g_comm.comm1 = nullptr;
    g_comm.api.CommDestroy(g_comm.comm);
    g_comm.comm = nullptr;
    g_comm.world = 1;
  }
  g_bases.clear();
  g_pks.clear();
  g_r1cs.clear();
  g_domains.clear();
  g_poly.reset();
  g_poly1.reset();
  if (g_d_err) cudaFree(g_d_err);
  if (g_stream) cudaStreamDestroy(g_stream);
  for (auto& sd : g_side) { if (sd) cudaStreamDestroy(sd); sd = nullptr; }
  for (auto& sd : g_side1) { if (sd) cudaStreamDestroy(sd); sd = nullptr; }
  if (g_stream1) cudaStreamDestroy(g_stream1);
  g_stream1 = nullptr;
  g_d_err = nullptr;
  g_stream = nullptr;
  g_init = false;
  return B200_OK;
}

int b200_g1_bases_load(const uint64_t* p, size_t n, int c, b200_bases_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return bases_load<Fq>(p, n, c, 1, out);
}
int b200_g2_bases_load(const uint64_t* p, size_t n, int c, b200_bases_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return bases_load<Fq2>(p, n, c, 2, out);
}
int b200_bases_free(b200_bases_t h) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_init) return fail(B200_EINVAL, "not initialised");
  cudaSetDevice(g_device);
  cudaStreamSynchronize(g_stream);
  return g_bases.erase(h) ? B200_OK : fail(B200_EINVAL, "bases_free: bad handle");
}
int b200_bases_info(b200_bases_t h, size_t* n, int* group, int* window_bits, int* n_windows) {
  std::lock_guard<std::mutex> lk(g_mu);
  Bases* b = find_bases(h, 0);
  if (!b) return fail(B200_EINVAL, "bases_info: bad handle");
  if (n) *n = b->n;
  if (group) *group = b->group;
  if (window_bits) *window_bits = (int)b->sh.c;
  if (n_windows) *n_windows = (int)b->sh.nwin;
  return B200_OK;
}

int b200_bases_acc_mode(b200_bases_t h, int* mode) {
  std::lock_guard<std::mutex> lk(g_mu);
  Bases* b = find_bases(h, 0);
  if (!b || !mode) return fail(B200_EINVAL, "bases_acc_mode: bad handle");
  *mode = b->affine_S ? 1 : 2;
  return B200_OK;
}
int b200_g1_msm(b200_bases_t h, const uint64_t* s, size_t n, uint64_t out[12]) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return msm_host<Fq>(h, 1, s, n, out);
}
int b200_g2_msm(b200_bases_t h, const uint64_t* s, size_t n, uint64_t out[24]) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return msm_host<Fq2>(h, 2, s, n, out);
}

int b200_msm_device(b200_bases_t h, const void* d_scalars, size_t n, int mont, void* d_out, void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  Bases* b = find_bases(h, 0);
  if (!b || !d_out || (!d_scalars && n)) return fail(B200_EINVAL, "msm_device: bad arguments");
  cudaStream_t st = stream ? (cudaStream_t)stream : g_stream;
  if (b->group == 1) return msm_enqueue<Fq>(b, (const Fr*)d_scalars, n, mont, (XYZZ<Fq>*)d_out, st);
  return msm_enqueue<Fq2>(b, (const Fr*)d_scalars, n, mont, (XYZZ<Fq2>*)d_out, st);
}

int b200_g1_sum_partials(const void* d, size_t count, uint64_t out[12], void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return sum_partials<Fq>(d, count, out, stream ? (cudaStream_t)stream : g_stream);
}
int b200_g2_sum_partials(const void* d, size_t count, uint64_t out[24], void* stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return sum_partials<Fq2>(d, count, out, stream ? (cudaStream_t)stream : g_stream);
}

int b200_g1_mul_batch(const uint64_t* p, const uint64_t* s, size_t n, uint64_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return mul_batch<Fq>(p, 0, s, n, out);
}
int b200_g2_mul_batch(const uint64_t* p, const uint64_t* s, size_t n, uint64_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return mul_batch<Fq2>(p, 0, s, n, out);
}
int b200_g1_mul_batch_bcast(const uint64_t* p, const uint64_t* s, size_t n, uint64_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return mul_batch<Fq>(p, 1, s, n, out);
}
int b200_g2_mul_batch_bcast(const uint64_t* p, const uint64_t* s, size_t n, uint64_t* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  NEED_INIT();
  return mul_batch<Fq2>(p, 1, s, n, out);
}

}  // extern "C"
