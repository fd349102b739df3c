// Batch Groth16 verification under one verification key (b200_groth16_verify_batch): the device side.
//
// N proofs are checked with one random linear combination (rho_i: the caller's secret 128-bit scalars)
//     prod_i e(rho_i A_i, B_i) * e(-(sum rho_i) alpha, beta) * e(-sum rho_i icPubl_i, gamma) * e(-sum rho_i C_i, delta) == 1
// i.e. N + 3 Miller loops whose F_q^12 values are multiplied together, and ONE final exponentiation.  The final
// exponentiation is a homomorphism, so the product equals the product of the reference's pairing values bit for bit.
//
//   k_vb_vk        verification-key points: affine form, on-curve / G2-subgroup predicates
//   k_vb_ic_terms  publicSignals[i][j] * IC[j+1], one thread per (proof, signal)
//   k_vb_ic_sum    icPubl_i = IC[0] + terms in the reference's Add order (jac_add_ref: its P + P = infinity quirk kept)
//   k_vb_prepare   one thread per proof: status word, rho_i A_i (affine, paired with B_i), rho_i C_i, rho_i icPubl_i
//   k_vb_sum       tree sum of XYZZ points (complete additions)
//   k_vb_tail      the three vk pairs from the sums
//   k_vb_miller    multi-Miller loop: a thread owns a chunk of pairs and one F_q^12 accumulator, which it squares ONCE per
//                  iteration for the whole chunk
//   k_vb_f12_tree  pairwise F_q^12 products of the partial accumulators
//   k_vb_final_exp one warp: wp::final_exp and the compare against one
//
// Host/device: tests/host/host_verify_batch_test.cpp runs these kernels through the carry-flag emulation on the CPU.
#pragma once
#include "pairing_warp.cuh"

namespace b200 {
namespace vb {

enum : int { kEach = 1, kAgg = 2 };   // status word of a proof: aggregated check / verified alone; < 0: B200_E* code
// 6 u^2 = q - r: on G2, psi (untwist-Frobenius-twist) acts as multiplication by q = 6 u^2 (mod r)
constexpr uint64_t kSixU2Lo = 0xf83e9682e87cfd46ULL, kSixU2Hi = 0x6f4d8248eeb859fbULL;

struct Pair {   // one Miller loop: affine Montgomery P in G1, Q on the twist; active = 0 contributes one
  F2::B px, py;
  F2 qx, qy;
  int active;
};

HD F2::B as_b(const Fq& x) {
  F2::B r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = x.l[i];
  return r;
}
template <class F>
HD Jacobian<F> jac_load_std(const F* p) { return Jacobian<F>{p[0].to_mont(), p[1].to_mont(), p[2].to_mont()}; }
template <class F>
HD bool jac_geq_modulus(const F* p) { return p[0].geq_modulus() || p[1].geq_modulus() || p[2].geq_modulus(); }

// y^2 = x^3 + 3
HD bool g1_on_curve(const Affine<Fq>& p) {
  const Fq three = Fq::one() + Fq::one() + Fq::one();
  return p.y.sqr() == p.x.sqr() * p.x + three;
}
// y^2 = x^3 + 3 / (9 + u)
HD bool g2_on_twist(const Affine<Fq2>& q) { return q.y.sqr() == q.x.sqr() * q.x + B200_F2_CONST(TWIST_COEF_B); }
// psi(Q) = (x^q * TWIST_MUL_BY_Q_X, y^q * TWIST_MUL_BY_Q_Y): the q1 of the Miller loop's last steps
HD Affine<Fq2> g2_psi(const Affine<Fq2>& q) {
  const F2 tqx = B200_F2_CONST(TWIST_MUL_BY_Q_X), tqy = B200_F2_CONST(TWIST_MUL_BY_Q_Y);
  return Affine<Fq2>{tqx * F2{q.x.c0, q.x.c1.neg()}, tqy * F2{q.y.c0, q.y.c1.neg()}};
}
// k * P, MSB-first double-and-add over the nwords 64-bit words of k, complete XYZZ formulas (P may be infinity)
template <class F>
HD XYZZ<F> mul_words(const Affine<F>& p, const uint64_t* k, int nwords) {
  XYZZ<F> acc = XYZZ<F>::inf();
  for (int w = nwords - 1; w >= 0; w--)
    for (int b = 63; b >= 0; b--) {
      acc = xyzz_dbl(acc);
      if ((k[w] >> b) & 1) xyzz_madd(acc, p);
    }
  return acc;
}
template <class F>
HD bool xyzz_eq_affine(const XYZZ<F>& a, const Affine<F>& p) { return !a.is_inf() && a.X == p.x * a.ZZ && a.Y == p.y * a.ZZZ; }
// Q (on the twist, not infinity) is in the order-r subgroup G2 iff psi(Q) == [6 u^2] Q
HD bool g2_in_subgroup(const Affine<Fq2>& q) {
  const uint64_t k[2] = {kSixU2Lo, kSixU2Hi};
  return xyzz_eq_affine(mul_words(q, k, 2), g2_psi(q));
}

// vk points: g2 = beta, gamma, delta (Jacobian standard form); ic[0..n_ic) and alpha.  Writes the affine Montgomery forms
// and sets *bad when alpha is infinity or off the curve, an IC point is off the curve, or a G2 point is outside G2.
// Coordinates < q and G2 points != infinity are the caller's precondition.
__global__ void k_vb_vk(const Fq* ic, uint32_t n_ic, const Fq* alpha, const Fq2* g2, Affine<Fq>* ic_aff, Affine<Fq2>* g2_aff,
                        int* bad) {
  for (uint32_t t = threadIdx.x; t < n_ic + 4; t += blockDim.x) {
    bool ok;
    if (t < 3) {
      Affine<Fq2> q = jac_to_affine(jac_load_std(g2 + 3 * t));
      ok = g2_on_twist(q) && g2_in_subgroup(q);
      g2_aff[t] = q;
    } else if (t == 3) {
      Jacobian<Fq> p = jac_load_std(alpha);
      ok = !p.is_inf() && g1_on_curve(jac_to_affine(p));
    } else {
      Affine<Fq> p = jac_to_affine(jac_load_std(ic + 3 * (t - 4)));
      ok = p.is_inf() || g1_on_curve(p);
      ic_aff[t - 4] = p;
    }
    if (!ok) atomicOr(bad, 1);
  }
}

// terms[i * npub + j] = pub[i][j] * IC[j + 1] (Montgomery Jacobian); the scalars are standard-form, < r
__global__ void k_vb_ic_terms(const Affine<Fq>* ic_aff, const uint64_t* pub, size_t n, size_t npub, Jacobian<Fq>* terms) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (t >= n * npub) return;
  terms[t] = xyzz_to_jacobian(mul_words(ic_aff[t % npub + 1], pub + 4 * t, 4));
}
// icp[i] = IC[0] + terms[i][0] + ... in groth16.go:283-286's order with the reference's Add (standard-form Jacobian out)
__global__ void k_vb_ic_sum(const Fq* ic, const Jacobian<Fq>* terms, size_t n, size_t npub, Fq* icp) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Jacobian<Fq> acc = jac_load_std(ic);
  for (size_t j = 0; j < npub; j++) acc = jac_add_ref(acc, terms[i * npub + j]);
  icp[3 * i] = acc.X.from_mont();
  icp[3 * i + 1] = acc.Y.from_mont();
  icp[3 * i + 2] = acc.Z.from_mont();
}

// One thread per proof.  status[i] arrives as 0 or a host-found error code (kept).  The codes follow the single verifier's
// flags: pairing (A, B) flags a coordinate >= q, else B at infinity; pairing (C, delta) flags C's coordinates; a B at
// infinity anywhere makes the call B200_EINVAL, a coordinate alone B200_ERANGE.  A proof the reference pairs in a
// non-bilinear way (A, C or icPubl at infinity, A or C off the curve, B off the twist or outside G2) gets kEach; the others
// kAgg and their terms of the combination.
__global__ void k_vb_prepare(const Fq* A, const Fq2* B, const Fq* C, const Fq* icp, const uint64_t* rho, size_t n, int* status,
                             Pair* pairs, XYZZ<Fq>* rho_c, XYZZ<Fq>* rho_ic) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  pairs[i].active = 0;
  rho_c[i] = XYZZ<Fq>::inf();
  rho_ic[i] = XYZZ<Fq>::inf();
  if (status[i] < 0) return;
  const Fq *a = A + 3 * i, *c = C + 3 * i;
  const Fq2* b = B + 3 * i;
  const bool b_range = b[0].geq_modulus() || b[1].geq_modulus() || b[2].geq_modulus();
  const bool b_inf = b[2].is_zero();
  int flags = (jac_geq_modulus(a) || b_range) ? 1 : (b_inf ? 8 : 0);
  if (jac_geq_modulus(c)) flags |= 1;
  if (flags) {
    status[i] = (flags & 8) ? -3 /* B200_EINVAL */ : -4 /* B200_ERANGE */;
    return;
  }
  const Jacobian<Fq> ja = jac_load_std(a), jc = jac_load_std(c), jic = jac_load_std(icp + 3 * i);
  if (ja.is_inf() || jc.is_inf() || jic.is_inf()) {
    status[i] = kEach;
    return;
  }
  const Affine<Fq> pa = jac_to_affine(ja), pc = jac_to_affine(jc), pic = jac_to_affine(jic);
  const Affine<Fq2> qb = jac_to_affine(jac_load_std(b));
  if (!g1_on_curve(pa) || !g1_on_curve(pc) || !g2_on_twist(qb) || !g2_in_subgroup(qb)) {
    status[i] = kEach;
    return;
  }
  status[i] = kAgg;
  const uint64_t* r = rho + 2 * i;
  const Affine<Fq> ra = xyzz_to_affine(mul_words(pa, r, 2));   // rho < r and A of order r: never infinity
  pairs[i] = Pair{as_b(ra.x), as_b(ra.y), qb.x, qb.y, 1};
  rho_c[i] = mul_words(pc, r, 2);
  rho_ic[i] = mul_words(pic, r, 2);
}

// out[t] = in[k t] + ... + in[k t + k - 1] (the last group may be short)
__global__ void k_vb_sum(const XYZZ<Fq>* in, size_t n, uint32_t k, XYZZ<Fq>* out) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (t * k >= n) return;
  XYZZ<Fq> acc = in[t * k];
  for (size_t j = t * k + 1; j < n && j < t * k + k; j++) xyzz_add(acc, in[j]);
  out[t] = acc;
}

// pairs[0..3) = (alpha_term, beta), (-sum_ic, gamma), (-sum_c, delta); alpha_term = -(sum rho) alpha already.  A G1 side at
// infinity leaves its pair inactive (e(O, Q) = 1).  *n_active = the number of pairs written.
__global__ void k_vb_tail(const Jacobian<Fq>* alpha_term, const XYZZ<Fq>* sum_ic, const XYZZ<Fq>* sum_c, const Affine<Fq2>* g2_aff,
                          Pair* pairs, int* n_active) {
  if (threadIdx.x | blockIdx.x) return;
  Affine<Fq> g1[3] = {jac_to_affine(*alpha_term), xyzz_to_affine(sum_ic->neg()), xyzz_to_affine(sum_c->neg())};
  int cnt = 0;
  for (int k = 0; k < 3; k++) {
    const bool on = !g1[k].is_inf();
    pairs[k] = Pair{as_b(g1[k].x), as_b(g1[k].y), g2_aff[k].x, g2_aff[k].y, on ? 1 : 0};
    cnt += on;
  }
  *n_active = cnt;
}

// Multi-Miller loop (bn128.go:354-372 for every pair at once): thread t owns pairs [t chunk, t chunk + chunk) and writes the
// product of their Miller-loop values to out[t].  T: the running G2 point of every pair (scratch).
__global__ void __launch_bounds__(64) k_vb_miller(const Pair* pairs, size_t npairs, uint32_t chunk, Jacobian<Fq2>* T, F12* out) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const size_t lo = t * chunk;
  if (lo >= npairs) return;
  const size_t hi = lo + chunk < npairs ? lo + chunk : npairs;
  for (size_t p = lo; p < hi; p++) T[p] = Jacobian<Fq2>{pairs[p].qx, pairs[p].qy, F2::one()};
  F12 f = F12::one();
#pragma unroll 1
  for (int i = 63; i >= 0; i--) {
    f = f12_sqr(f);
#pragma unroll 1
    for (size_t p = lo; p < hi; p++) {
      const Pair& pr = pairs[p];
      if (!pr.active) continue;
      F2 X = T[p].X, Y = T[p].Y, Z = T[p].Z;
      f = pairing_line(f, pairing_doubling_step(X, Y, Z), pr.px, pr.py);
      if ((pc::LOOP_COUNT_LOW64 >> i) & 1) f = pairing_line(f, pairing_mixed_addition_step(pr.qx, pr.qy, X, Y, Z), pr.px, pr.py);
      T[p] = Jacobian<Fq2>{X, Y, Z};
    }
  }
  // q1 = pi(Q), q2 = -pi^2(Q)  (bn128.go:238-253, 331-346)
  const F2 tqx = B200_F2_CONST(TWIST_MUL_BY_Q_X), tqy = B200_F2_CONST(TWIST_MUL_BY_Q_Y);
#pragma unroll 1
  for (size_t p = lo; p < hi; p++) {
    const Pair& pr = pairs[p];
    if (!pr.active) continue;
    F2 X = T[p].X, Y = T[p].Y, Z = T[p].Z;
    const F2 q1x = tqx * F2{pr.qx.c0, pr.qx.c1.neg()}, q1y = tqy * F2{pr.qy.c0, pr.qy.c1.neg()};
    const F2 q2x = tqx * F2{q1x.c0, q1x.c1.neg()}, q2y = (tqy * F2{q1y.c0, q1y.c1.neg()}).neg();
    f = pairing_line(f, pairing_mixed_addition_step(q1x, q1y, X, Y, Z), pr.px, pr.py);
    f = pairing_line(f, pairing_mixed_addition_step(q2x, q2y, X, Y, Z), pr.px, pr.py);
  }
  out[t] = f;
}

// out[i] = in[2 i] * in[2 i + 1] (in[2 i] alone when n is odd)
__global__ void k_vb_f12_tree(const F12* in, size_t n, F12* out) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (2 * i >= n) return;
  out[i] = 2 * i + 1 < n ? f12_mul(in[2 * i], in[2 * i + 1]) : in[2 * i];
}

// One warp: *ok = (f^((q^12 - 1) / r) == 1); the exponentiated value to res (Montgomery) when res is not null.
__global__ void __launch_bounds__(32) k_vb_final_exp(const F12* f, int* ok, F12* res) {
  __shared__ wp::Ws ws;
  const uint32_t lane = wp::lane_id();
  const F2* src = &f->a.a;
  if (lane < 6) ws.r[wp::RF][lane] = src[lane];
  wp::wsync();
  wp::pairing_constants(ws);
  wp::final_exp(ws);
  if (lane == 0) {
    const F2* r = ws.r[wp::RF];
    bool one = r[0] == F2::one();
    for (int k = 1; k < 6; k++) one = one && r[k].is_zero();
    *ok = one ? 1 : 0;
    if (res) *res = F12{F6{r[0], r[1], r[2]}, F6{r[3], r[4], r[5]}};
  }
}

}  // namespace vb
}  // namespace b200
