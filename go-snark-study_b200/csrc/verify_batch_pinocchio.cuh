// Pinocchio verification (snark.VerifyProof, snark.go:292-372) for one proof and for N proofs under one key
// (b200_pinocchio_verify, b200_pinocchio_verify_batch): the device side.
//
// The five checks of proof i, each written as a product of pairings that must be one:
//   1  e(PiA, Vka) e(PiAp, g2)^-1                      2  e(Vkb, PiB) e(PiBp, g2)^-1
//   3  e(PiC, Vkc) e(PiCp, g2)^-1                      4  e(VkxA, PiB) e(PiH, Vkz)^-1 e(PiC, g2)^-1
//   5  e(VkxAC, G2Kbg) e(G1Kbg, PiB) e(PiKp, G2Kg)^-1
// with vkx = IC[0] + sum s_j IC[j+1], VkxA = Add(vkx, PiA), VkxAC = Add(VkxA, PiC) (the reference's Add, in its order).
// Check k of proof i is raised to the caller's secret 128-bit rho_ik and the factors are grouped by their G2 point:
//   PiB_i  rho2 Vkb + rho4 VkxA + rho5 G1Kbg             (one Miller loop per proof)
//   g2     -sum_i (rho1 PiAp + rho2 PiBp + rho3 PiCp + rho4 PiC)
//   Vka    sum_i rho1 PiA           Vkc    sum_i rho3 PiC          Vkz   -sum_i rho4 PiH
//   G2Kbg  sum_i rho5 VkxAC         G2Kg  -sum_i rho5 PiKp
// N + 6 Miller loops, one product tree and one final exponentiation (verify_batch.cuh's k_vb_miller, k_vb_f12_tree,
// k_vb_final_exp, unchanged).
//
//   k_pv_vk        verification-key points: affine form, on-curve / twist / G2-subgroup predicates
//   k_pv_prepare   one thread per proof: status word, VkxA and VkxAC, the predicates, the affine points the products read
//   k_pv_products  one thread per (proof, product): the seven multi-scalar products above, one shared doubling chain each
//   k_pv_tail      the six fixed-G2 pairs from the tree sums (k_vb_sum) of the six per-proof arrays
//   k_pv_pairs     the single check's twelve pairings of a proof, as pairing-kernel inputs
//   k_pv_compare   the single check's two F_q^12 products and the first failing check
//
// Host/device: tests/host/host_pinocchio_verify_batch_test.cpp runs these kernels through the carry-flag emulation.
#pragma once
#include "verify_batch.cuh"

namespace b200 {
namespace pv {

using vb::Pair;
// proof G1 points in b200_pinocchio_prove's out_g1 order, then the two sums prepared per proof
enum : int { kPiA, kPiAp, kPiBp, kPiC, kPiCp, kPiH, kPiKp, kVkxA, kVkxAC, kPts };
constexpr int kProofG1 = kVkxA;   // G1 points of a proof
constexpr int kProducts = 7;   // six arrays summed over the batch (fixed G2 points) + the PiB pair's G1 side
// verification-key G2 points on the device: the generator first, then vk_g2's order
enum : int { kG2, kVka, kVkc, kVkz, kG2Kbg, kG2Kg, kVkG2 };
// G1 key points: Vkb, G1Kbg
enum : int { kVkb, kG1Kbg, kVkG1 };

// Affine form of n Jacobian points (none at infinity) with one inversion: Montgomery's simultaneous inversion.
template <int N>
HD void jac_to_affine_n(const Jacobian<Fq>* p, Affine<Fq>* out) {
  Fq pre[N];
  pre[0] = p[0].Z;
#pragma unroll
  for (int k = 1; k < N; k++) pre[k] = pre[k - 1] * p[k].Z;
  Fq inv = pre[N - 1].inverse();
#pragma unroll
  for (int k = N - 1; k >= 0; k--) {
    const Fq zi = k ? inv * pre[k - 1] : inv;
    if (k) inv = inv * p[k].Z;
    const Fq zi2 = zi.sqr();
    out[k] = Affine<Fq>{p[k].X * zi2, p[k].Y * (zi2 * zi)};
  }
}

// sum_j k_j P_j over m <= 4 points and 128-bit scalars (two words each): one MSB-first doubling chain shared by all terms
HD XYZZ<Fq> mul_words_multi(const Affine<Fq>* p, const uint64_t* const* k, int m) {
  XYZZ<Fq> acc = XYZZ<Fq>::inf();
  for (int w = 1; w >= 0; w--)
    for (int b = 63; b >= 0; b--) {
      acc = xyzz_dbl(acc);
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (j < m && ((k[j][w] >> b) & 1)) xyzz_madd(acc, p[j]);
    }
  return acc;
}

// g1 = Vkb, G1Kbg; g2 = the generator, Vka, Vkc, Vkz, G2Kbg, G2Kg; ic[0..n_ic) (Jacobian standard form).  Writes the affine
// Montgomery forms and sets *bad when Vkb or G1Kbg is at infinity or off the curve, an IC point is off the curve, or a G2
// point is off the twist or outside G2.  Coordinates < q and G2 points != infinity are the caller's precondition.
__global__ void k_pv_vk(const Fq* ic, uint32_t n_ic, const Fq* g1, const Fq2* g2, Affine<Fq>* ic_aff, Affine<Fq>* g1_aff,
                        Affine<Fq2>* g2_aff, int* bad) {
  for (uint32_t t = threadIdx.x; t < n_ic + kVkG2 + kVkG1; t += blockDim.x) {
    bool ok;
    if (t < kVkG2) {
      const Affine<Fq2> q = jac_to_affine(vb::jac_load_std(g2 + 3 * t));
      ok = vb::g2_on_twist(q) && vb::g2_in_subgroup(q);
      g2_aff[t] = q;
    } else if (t < kVkG2 + kVkG1) {
      const Jacobian<Fq> p = vb::jac_load_std(g1 + 3 * (t - kVkG2));
      const Affine<Fq> a = jac_to_affine(p);
      ok = !p.is_inf() && vb::g1_on_curve(a);
      g1_aff[t - kVkG2] = a;
    } else {
      const Affine<Fq> a = jac_to_affine(vb::jac_load_std(ic + 3 * (t - kVkG2 - kVkG1)));
      ok = a.is_inf() || vb::g1_on_curve(a);
      ic_aff[t - kVkG2 - kVkG1] = a;
    }
    if (!ok) atomicOr(bad, 1);
  }
}

// One thread per proof.  P: n x 7 G1 points, B: n x PiB (Jacobian standard form); vkx: the proofs' IC sums (k_vb_ic_sum).
// status[i] arrives as 0 or B200_ERANGE for a public signal >= r.  PiB at infinity gives B200_EINVAL whatever else is
// wrong (the reference panics, bn128.go:238-241); otherwise a coordinate >= q or that signal gives B200_ERANGE: the codes of
// b200_pinocchio_verify.  A proof the reference pairs in a non-bilinear way (one of its G1 points, VkxA or VkxAC at
// infinity, a G1 point off the curve, PiB off the twist or outside G2) gets vb::kEach, the others vb::kAgg and their
// affine Montgomery points: pts[9 i + kPiA .. kVkxAC], qb[i] = PiB.
__global__ void k_pv_prepare(const Fq* P, const Fq2* B, const Fq* vkx, size_t n, int* status, Affine<Fq>* pts,
                             Affine<Fq2>* qb) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Fq* p = P + 3 * kProofG1 * i;
  const Fq2* b = B + 3 * i;
  if (b[2].is_zero()) {
    status[i] = -3;   // B200_EINVAL
    return;
  }
  bool range = status[i] < 0 || b[0].geq_modulus() || b[1].geq_modulus() || b[2].geq_modulus();
  for (int k = 0; k < 3 * kProofG1; k++) range = range || p[k].geq_modulus();
  if (range) {
    status[i] = -4;   // B200_ERANGE
    return;
  }
  Jacobian<Fq> j[kPts];
  bool inf = false;
#pragma unroll
  for (int k = 0; k < kProofG1; k++) {
    j[k] = vb::jac_load_std(p + 3 * k);
    inf = inf || j[k].is_inf();
  }
  j[kVkxA] = jac_add_ref(vb::jac_load_std(vkx + 3 * i), j[kPiA]);
  j[kVkxAC] = jac_add_ref(j[kVkxA], j[kPiC]);
  if (inf || j[kVkxA].is_inf() || j[kVkxAC].is_inf()) {
    status[i] = vb::kEach;
    return;
  }
  Affine<Fq> a[kPts];
  jac_to_affine_n<kPts>(j, a);
  bool on = true;
#pragma unroll
  for (int k = 0; k < kProofG1; k++) on = on && vb::g1_on_curve(a[k]);
  const Affine<Fq2> q = jac_to_affine(vb::jac_load_std(b));
  if (!on || !vb::g2_on_twist(q) || !vb::g2_in_subgroup(q)) {
    status[i] = vb::kEach;
    return;
  }
  status[i] = vb::kAgg;
#pragma unroll
  for (int k = 0; k < kPts; k++) pts[kPts * i + k] = a[k];
  qb[i] = q;
}

// Thread t = c n + i computes product c of proof i (product-major, so a warp runs one product shape):
//   c = 0 .. 5  sums[c n + i] = rho1 PiAp + ... + rho4 PiC (g2), rho1 PiA (Vka), rho3 PiC (Vkc), rho4 PiH (Vkz), rho5 VkxAC (G2Kbg),
//               rho5 PiKp (G2Kg): the six arrays k_vb_sum reduces; signs are applied by k_pv_tail
//   c = 6       pairs[i] = (rho2 Vkb + rho4 VkxA + rho5 G1Kbg, PiB), inactive when the G1 side is infinity
// A proof outside the aggregated check contributes infinity and an inactive pair.  *n_active counts the active pairs.
// rho: n x 5 x 2 words.
__global__ void k_pv_products(const Affine<Fq>* pts, const Affine<Fq2>* qb, const Affine<Fq>* g1_aff, const uint64_t* rho,
                              const int* status, size_t n, XYZZ<Fq>* sums, Pair* pairs, int* n_active) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (t >= kProducts * n) return;
  const int c = (int)(t / n);
  const size_t i = t - c * n;
  if (status[i] != vb::kAgg) {
    if (c < kProducts - 1) sums[t] = XYZZ<Fq>::inf();
    else pairs[i].active = 0;
    return;
  }
  const Affine<Fq>* a = pts + kPts * i;
  const uint64_t* r = rho + 10 * i;   // rho_k of check k at r + 2 (k - 1)
  Affine<Fq> p[4];
  const uint64_t* k[4];
  int m = 1;
  switch (c) {
    case 0:
      p[0] = a[kPiAp], p[1] = a[kPiBp], p[2] = a[kPiCp], p[3] = a[kPiC];
      k[0] = r, k[1] = r + 2, k[2] = r + 4, k[3] = r + 6;
      m = 4;
      break;
    case 1: p[0] = a[kPiA], k[0] = r; break;
    case 2: p[0] = a[kPiC], k[0] = r + 4; break;
    case 3: p[0] = a[kPiH], k[0] = r + 6; break;
    case 4: p[0] = a[kVkxAC], k[0] = r + 8; break;
    case 5: p[0] = a[kPiKp], k[0] = r + 8; break;
    default:
      p[0] = g1_aff[kVkb], p[1] = a[kVkxA], p[2] = g1_aff[kG1Kbg];
      k[0] = r + 2, k[1] = r + 6, k[2] = r + 8;
      m = 3;
  }
  const XYZZ<Fq> s = mul_words_multi(p, k, m);
  if (c < kProducts - 1) {
    sums[t] = s;
    return;
  }
  const Affine<Fq> g = xyzz_to_affine(s);
  const bool on = !g.is_inf();
  pairs[i] = Pair{vb::as_b(g.x), vb::as_b(g.y), qb[i].x, qb[i].y, on ? 1 : 0};
  if (on) atomicAdd(n_active, 1);
}

struct Sums6 {
  const XYZZ<Fq>* s[kVkG2];   // the reduced sums in k_pv_products' order: g2, Vka, Vkc, Vkz, G2Kbg, G2Kg
};
// Thread k < 6: pairs[k] = (+-sum k, G2 point k), negated for g2, Vkz and G2Kg; inactive when the G1 side is infinity
// (e(O, Q) = 1).  Adds the active ones to *n_active.
__global__ void k_pv_tail(Sums6 sums, const Affine<Fq2>* g2_aff, Pair* pairs, int* n_active) {
  const uint32_t k = threadIdx.x;
  if (blockIdx.x || k >= kVkG2) return;
  const bool neg = k == kG2 || k == kVkz || k == kG2Kg;
  const Affine<Fq> g = xyzz_to_affine(neg ? sums.s[k]->neg() : *sums.s[k]);
  const bool on = !g.is_inf();
  pairs[k] = Pair{vb::as_b(g.x), vb::as_b(g.y), g2_aff[k].x, g2_aff[k].y, on ? 1 : 0};
  if (on) atomicAdd(n_active, 1);
}

// The twelve pairings of snark.go:292-372 for proof idx[b] (b when idx is null), one thread per proof, as inputs of the
// pairing kernels (Jacobian standard form): g1[12 b + e], g2[12 b + e] in the order
//   PiA/Vka, PiAp/g2, Vkb/PiB, PiBp/g2, PiC/Vkc, PiCp/g2, VkxA/PiB, PiH/Vkz, PiC/g2, VkxAC/G2Kbg, G1Kbg/PiB, PiKp/G2Kg.
// vk1 = Vkb, G1Kbg; vk2 = the generator, Vka, Vkc, Vkz, G2Kbg, G2Kg; vkx[i]: the proof's IC sum.
__global__ void k_pv_pairs(const Fq* P, const Fq2* B, const Fq* vkx, const Fq* vk1, const Fq2* vk2, const uint32_t* idx,
                           size_t m, Fq* g1, Fq2* g2) {
  const size_t bi = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (bi >= m) return;
  const size_t i = idx ? idx[bi] : bi;
  const Fq* p = P + 3 * kProofG1 * i;
  const Jacobian<Fq> vka = jac_add_ref(vb::jac_load_std(vkx + 3 * i), vb::jac_load_std(p + 3 * kPiA));
  const Jacobian<Fq> vkac = jac_add_ref(vka, vb::jac_load_std(p + 3 * kPiC));
  const Fq sums[6] = {vka.X.from_mont(), vka.Y.from_mont(), vka.Z.from_mont(),
                      vkac.X.from_mont(), vkac.Y.from_mont(), vkac.Z.from_mont()};
  const Fq* src1[12] = {p + 3 * kPiA, p + 3 * kPiAp, vk1 + 3 * kVkb, p + 3 * kPiBp, p + 3 * kPiC, p + 3 * kPiCp,
                        sums, p + 3 * kPiH, p + 3 * kPiC, sums + 3, vk1 + 3 * kG1Kbg, p + 3 * kPiKp};
  const Fq2* pib = B + 3 * i;
  const Fq2* src2[12] = {vk2 + 3 * kVka, vk2, pib, vk2, vk2 + 3 * kVkc, vk2, pib, vk2 + 3 * kVkz, vk2, vk2 + 3 * kG2Kbg,
                         pib, vk2 + 3 * kG2Kg};
  for (int e = 0; e < 12; e++)
    for (int c = 0; c < 3; c++) {
      g1[3 * (12 * bi + e) + c] = src1[e][c];
      g2[3 * (12 * bi + e) + c] = src2[e][c];
    }
}

HD F12 f12_load_std(const Fq2* p) {
  return F12{F6{p[0].to_mont(), p[1].to_mont(), p[2].to_mont()}, F6{p[3].to_mont(), p[4].to_mont(), p[5].to_mont()}};
}
HD bool f12_eq(const F12& x, const F12& y) {
  return x.a.a == y.a.a && x.a.b == y.a.b && x.a.c == y.a.c && x.b.a == y.b.a && x.b.b == y.b.b && x.b.c == y.b.c;
}
// One thread per proof: e = its twelve pairing values in k_pv_pairs' order (standard form, 6 Fq2 each).  failed[b] = 0 when
// the five checks hold, else the first that fails (1..5), in the reference's order.
__global__ void k_pv_compare(const Fq2* e, size_t m, int* failed) {
  const size_t b = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (b >= m) return;
  const Fq2* v = e + 72 * b;
  auto at = [&](int k) { return f12_load_std(v + 6 * k); };
  int f = 0;
  if (!f12_eq(at(0), at(1))) f = 1;
  else if (!f12_eq(at(2), at(3))) f = 2;
  else if (!f12_eq(at(4), at(5))) f = 3;
  else if (!f12_eq(at(6), f12_mul(at(7), at(8)))) f = 4;
  else if (!f12_eq(f12_mul(at(9), at(10)), at(11))) f = 5;
  failed[b] = f;
}

}  // namespace pv
}  // namespace b200
