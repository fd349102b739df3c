// CPU test vehicle for the Pinocchio verification kernels of verify_batch_pinocchio.cuh (g++, host_stub): the key check,
// the per-proof preparation and products, the tail's six fixed-G2 pairs through the multi-Miller loop, product tree and
// warp final exponentiation of verify_batch.cuh, and the single check's compare kernel.  Per-thread kernels run one
// emulated thread at a time, the warp kernel as 32 OS threads with a barrier for __syncwarp.  Test infrastructure only:
// never linked into libb200snark.
#include "host_stub/cuda_runtime.h"

#include <pthread.h>

#include <thread>
#include <vector>

#include "verify_batch_pinocchio.cuh"

using namespace b200;

namespace {
pthread_barrier_t g_warp_bar;
bool g_warp_mode = false;
}  // namespace
void stub_syncwarp() {
  if (g_warp_mode) pthread_barrier_wait(&g_warp_bar);
}
void stub_syncthreads() { stub_abort("__syncthreads"); }
uint32_t stub_shfl(uint32_t, int, int, int) { stub_abort("warp shuffle"); }
unsigned stub_ballot(int) { stub_abort("__ballot_sync"); }

namespace {
template <class K>
void run_warp(K kernel) {
  pthread_barrier_init(&g_warp_bar, nullptr, 32);
  g_warp_mode = true;
  std::vector<std::thread> th;
  for (unsigned t = 0; t < 32; t++)
    th.emplace_back([=] {
      threadIdx.x = t;
      blockIdx.x = 0;
      blockDim.x = 32;
      kernel();
    });
  for (auto& x : th) x.join();
  g_warp_mode = false;
  pthread_barrier_destroy(&g_warp_bar);
}
// every thread of a 1-D grid, one at a time (blockDim 1)
template <class K>
void run_threads(size_t n, K kernel) {
  for (size_t t = 0; t < n; t++) {
    blockIdx.x = (unsigned)t;
    blockDim.x = 1;
    threadIdx.x = 0;
    kernel();
  }
}
template <class F>
void store_std(uint32_t* p, const F& v) {
  F s = v.from_mont();
  std::memcpy(p, &s, sizeof(F));
}
void store_xyzz_affine(uint32_t* p, const XYZZ<Fq>& s) {
  const Affine<Fq> a = xyzz_to_affine(s);
  store_std(p, a.x);
  store_std(p + 8, a.y);
}

// The batch pipeline up to the products.  ic: n_ic G1, vk1: Vkb, G1Kbg; vk2: the generator, Vka, Vkc, Vkz, G2Kbg, G2Kg;
// P: n x 7 G1, B: n PiB (Jacobian standard form, 24 / 48 u32 per point); pub: n x npub x 8 u32; rho: n x 5 x 2 u64.
struct Batch {
  size_t n;
  std::vector<Affine<Fq>> ic_aff, g1_aff, pts;
  std::vector<Affine<Fq2>> g2_aff, qb;
  std::vector<Jacobian<Fq>> terms;
  std::vector<Fq> vkx;
  std::vector<int> status;
  std::vector<XYZZ<Fq>> sums;
  std::vector<vb::Pair> pairs;
  int bad = 0, n_active = 0;
  Batch(const uint32_t* ic, uint32_t npub, const uint32_t* vk1, const uint32_t* vk2, size_t n_, const uint32_t* P,
        const uint32_t* B, const uint32_t* pub, const uint64_t* rho)
      : n(n_), ic_aff(npub + 1), g1_aff(2), pts(n * pv::kPts), g2_aff(6), qb(n), terms(std::max<size_t>(n * npub, 1)),
        vkx(3 * n), status(n, 0), sums(6 * n), pairs(n + 6) {
    const Fq* icq = reinterpret_cast<const Fq*>(ic);
    run_threads(1, [&] { pv::k_pv_vk(icq, npub + 1, reinterpret_cast<const Fq*>(vk1), reinterpret_cast<const Fq2*>(vk2),
                                     ic_aff.data(), g1_aff.data(), g2_aff.data(), &bad); });
    if (npub)
      run_threads(n * npub, [&] { vb::k_vb_ic_terms(ic_aff.data(), reinterpret_cast<const uint64_t*>(pub), n, npub, terms.data()); });
    run_threads(n, [&] { vb::k_vb_ic_sum(icq, terms.data(), n, npub, vkx.data()); });
    run_threads(n, [&] { pv::k_pv_prepare(reinterpret_cast<const Fq*>(P), reinterpret_cast<const Fq2*>(B), vkx.data(), n,
                                          status.data(), pts.data(), qb.data()); });
    run_threads(pv::kProducts * n, [&] { pv::k_pv_products(pts.data(), qb.data(), g1_aff.data(), rho, status.data(), n,
                                                           sums.data(), pairs.data(), &n_active); });
  }
};
}  // namespace

extern "C" {
// Preparation and products.  status: n ints; pairs_g1: n x 16 u32 (the PiB pair's G1 side, affine standard form, (0, 0)
// when inactive); sums: 6 x n x 16 u32 (the six per-proof products, affine); returns the key check's bad flag.
int t_prepare(const uint32_t* ic, uint32_t npub, const uint32_t* vk1, const uint32_t* vk2, uint32_t n, const uint32_t* P,
              const uint32_t* B, const uint32_t* pub, const uint64_t* rho, int* status, uint32_t* pairs_g1, uint32_t* sums) {
  Batch b(ic, npub, vk1, vk2, n, P, B, pub, rho);
  for (uint32_t i = 0; i < n; i++) {
    status[i] = b.status[i];
    const vb::Pair& pr = b.pairs[i];
    Fq x, y;
    std::memcpy(&x, &pr.px, sizeof x);
    std::memcpy(&y, &pr.py, sizeof y);
    if (!pr.active) x = y = Fq::zero();
    store_std(pairs_g1 + 16 * i, x);
    store_std(pairs_g1 + 16 * i + 8, y);
  }
  for (size_t t = 0; t < 6 * (size_t)n; t++) store_xyzz_affine(sums + 16 * t, b.sums[t]);
  return b.bad;
}
// The whole aggregated check: preparation, products, k_vb_sum trees, k_pv_tail, k_vb_miller (chunk pairs per thread),
// k_vb_f12_tree, k_vb_final_exp.  Returns 1 when the product is one, 0 when not; *n_active = the Miller loops run.
int t_aggregate(const uint32_t* ic, uint32_t npub, const uint32_t* vk1, const uint32_t* vk2, uint32_t n, const uint32_t* P,
                const uint32_t* B, const uint32_t* pub, const uint64_t* rho, uint32_t chunk, int* n_active) {
  Batch b(ic, npub, vk1, vk2, n, P, B, pub, rho);
  const uint32_t k = 4;
  pv::Sums6 s6;
  std::vector<std::vector<XYZZ<Fq>>> lv;
  lv.reserve(64);
  for (int c = 0; c < 6; c++) {
    const XYZZ<Fq>* cur = b.sums.data() + c * n;
    for (size_t m = n; m > 1; m = (m + k - 1) / k) {
      lv.emplace_back((m + k - 1) / k);
      XYZZ<Fq>* out = lv.back().data();
      run_threads((m + k - 1) / k, [&] { vb::k_vb_sum(cur, m, k, out); });
      cur = out;
    }
    s6.s[c] = cur;
  }
  run_warp([&] { pv::k_pv_tail(s6, b.g2_aff.data(), b.pairs.data() + n, &b.n_active); });
  const size_t np = n + 6, nth = (np + chunk - 1) / chunk;
  std::vector<Jacobian<Fq2>> T(np);
  std::vector<F12> f(nth), g(nth);
  run_threads(nth, [&] { vb::k_vb_miller(b.pairs.data(), np, chunk, T.data(), f.data()); });
  for (size_t m = nth; m > 1; m = (m + 1) / 2) {
    run_threads((m + 1) / 2, [&] { vb::k_vb_f12_tree(f.data(), m, g.data()); });
    std::swap(f, g);
  }
  int ok = -1;
  run_warp([&] { vb::k_vb_final_exp(f.data(), &ok, nullptr); });
  *n_active = b.n_active;
  return ok;
}
// k_pv_compare on one proof's twelve F_q^12 values (standard form, 96 u32 each, the [2][3][2] order)
int t_compare(const uint32_t* e) {
  int failed = -1;
  run_threads(1, [&] { pv::k_pv_compare(reinterpret_cast<const Fq2*>(e), 1, &failed); });
  return failed;
}
}
