// CPU test vehicle for the batch-verification kernels of verify_batch.cuh (g++, host_stub): the multi-Miller loop with its
// chunks and inactive pairs, the F_q^12 product tree and the warp final exponentiation; the G1 / G2 curve and subgroup
// predicates; the XYZZ tree sum.  Per-thread kernels run one emulated thread at a time, the warp kernel as 32 OS threads
// with a barrier for __syncwarp.  Test infrastructure only: never linked into libb200snark.
#include "host_stub/cuda_runtime.h"

#include <pthread.h>

#include <thread>
#include <vector>

#include "verify_batch.cuh"

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
F load_std(const uint32_t* p) {
  F v;
  std::memcpy(&v, p, sizeof(F));
  return v.to_mont();
}
template <class F>
void store_std(uint32_t* p, const F& v) {
  F s = v.from_mont();
  std::memcpy(p, &s, sizeof(F));
}
Affine<Fq> g1_load(const uint32_t* p) { return Affine<Fq>{load_std<Fq>(p), load_std<Fq>(p + 8)}; }
Affine<Fq2> g2_load(const uint32_t* p) { return Affine<Fq2>{load_std<Fq2>(p), load_std<Fq2>(p + 16)}; }
}  // namespace

extern "C" {
// prod_k Miller(g1[k], g2[k]) through k_vb_miller (chunk pairs per thread; an inactive pair is put after every active one)
// -> k_vb_f12_tree -> k_vb_final_exp.  g1: k affine points (x, y), g2: k affine twist points (x.c0, x.c1, y.c0, y.c1),
// standard form.  out: the F_q^12 value in the reference's [2][3][2] order.  Returns the final kernel's ok flag.
int t_multi_pairing(const uint32_t* g1, const uint32_t* g2, uint32_t k, uint32_t chunk, uint32_t* out) {
  std::vector<vb::Pair> pairs;
  for (uint32_t i = 0; i < k; i++) {
    Affine<Fq> p = g1_load(g1 + 16 * i);
    Affine<Fq2> q = g2_load(g2 + 32 * i);
    pairs.push_back(vb::Pair{vb::as_b(p.x), vb::as_b(p.y), q.x, q.y, 1});
    pairs.push_back(vb::Pair{vb::as_b(p.y), vb::as_b(p.x), q.y, q.x, 0});   // inactive: must contribute one
  }
  const size_t np = pairs.size(), nth = (np + chunk - 1) / chunk;
  std::vector<Jacobian<Fq2>> T(np);
  std::vector<F12> f(nth), g(nth);
  run_threads(nth, [&] { vb::k_vb_miller(pairs.data(), np, chunk, T.data(), f.data()); });
  for (size_t m = nth; m > 1; m = (m + 1) / 2) {
    run_threads((m + 1) / 2, [&] { vb::k_vb_f12_tree(f.data(), m, g.data()); });
    std::swap(f, g);
  }
  int ok = -1;
  F12 res;
  run_warp([&] { vb::k_vb_final_exp(f.data(), &ok, &res); });
  const F2* parts[6] = {&res.a.a, &res.a.b, &res.a.c, &res.b.a, &res.b.b, &res.b.c};
  for (int c = 0; c < 6; c++) store_std(out + 16 * c, *parts[c]);
  return ok;
}
// G1: y^2 = x^3 + 3 on an affine standard-form point
int t_g1_on_curve(const uint32_t* p) { return vb::g1_on_curve(g1_load(p)) ? 1 : 0; }
// G2: bit 0 on the twist, bit 1 psi(Q) == [6 u^2] Q
int t_g2_predicates(const uint32_t* q) {
  Affine<Fq2> a = g2_load(q);
  return (vb::g2_on_twist(a) ? 1 : 0) | (vb::g2_in_subgroup(a) ? 2 : 0);
}
// sum of n affine G1 points ((0, 0) = infinity) by k_vb_sum levels of k; out: affine standard form, (0, 0) for infinity
void t_g1_tree_sum(const uint32_t* pts, uint32_t n, uint32_t k, uint32_t* out) {
  std::vector<XYZZ<Fq>> a(n), b(n);
  for (uint32_t i = 0; i < n; i++) a[i] = XYZZ<Fq>::from_affine(g1_load(pts + 16 * i));
  for (size_t m = n; m > 1; m = (m + k - 1) / k) {
    run_threads((m + k - 1) / k, [&] { vb::k_vb_sum(a.data(), m, k, b.data()); });
    std::swap(a, b);
  }
  Affine<Fq> r = xyzz_to_affine(a[0]);
  store_std(out, r.x);
  store_std(out + 8, r.y);
}
}
