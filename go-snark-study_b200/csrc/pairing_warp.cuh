// Optimal-ate pairing, ONE WARP per pairing (bn128/bn128.go:179-421; the thread-per-pairing restatement is pairing.cuh).
//
// A pairing is ~25 000 dependent F_q multiplications when one thread walks the tower; a dependent multiplication in a
// lone thread costs ~0.4 us, so a verification (groth16.go:281-305: four pairings) took ~20 ms however idle the GPU was.
// Here the F_q^12 accumulator and every temporary live in SHARED memory and the 32 lanes of a warp share the work of
// each tower operation:
//   F_q^12 product   Karatsuba over F_q^6 (3 products) x schoolbook inside F_q^6 (9 F_q^2 products each) = 27 F_q^2
//                    products, ONE per lane, in a single step; the reductions by v^3 = xi are folded into the operands
//                    (xi * y_j prepared beforehand with additions only: 9 = 2^3 + 1), and twelve lanes (one per F_q
//                    component) gather their sums of <= 9 products
//   line functions   the doubling / mixed-addition steps (bn128.go:262-330) level by level: independent F_q^2 products
//                    of one level on different lanes (5 + 1 + 4 and 2 + 4 + 3 + 4 products)
//   Frobenius, conjugation, packing   one coefficient per lane
// so the dependency chain of a pairing is ~1 400 F_q^2-product steps instead of ~25 000 F_q products.  Every intermediate
// is an exact field element: the result is bit-identical to pairing_affine_t (and to bn128.Pairing).
//
// Control flow is warp-uniform; lanes differ only in the operands they select.  Host/device: the CPU test vehicle runs a
// warp as 32 OS threads (tests/host/host_kernel_test.cpp).
#pragma once
#include "pairing.cuh"

namespace b200 {
namespace wp {

constexpr int kF12Regs = 12;
// F_q^12 registers hold the six F_q^2 coefficients in tower order: a.a, a.b, a.c, b.a, b.b, b.c
struct alignas(32) Ws {
  F2 r[kF12Regs][6];
  F2 T[27];    // the 27 products of a multiplication
  F2 S[6];     // a.A + a.B (3), b.A + b.B (3)
  F2 Xi[6];    // xi * y_j, j = 1, 2, of the three right-hand F_q^6 operands
  F2 P[3];     // the running G2 point X, Y, Z (bn128.go:262-330)
  F2 Q[6];     // affine Q, pi(Q), -pi^2(Q): x, y each
  F2 pt[13];   // scratch of the point steps
  F2 fc[15];   // Frobenius constants xi^(j (q^k - 1) / 6): [k - 1][j - 1]
  F2::B px, py;
};

DEV void wsync() {
#ifdef __CUDA_ARCH__
  __syncwarp();
#elif !defined(__CUDACC__)
  stub_syncwarp();
#endif
}
DEV uint32_t lane_id() { return threadIdx.x & 31u; }

// xi * a, xi = 9 + u, with additions only
HD F2::B fq_nine(const F2::B& x) { return x.dbl().dbl().dbl() + x; }
HD F2 f2_mul_xi(const F2& a) { return F2{fq_nine(a.c0) - a.c1, fq_nine(a.c1) + a.c0}; }
HD F2 f2_halve(const F2& a) {  // a / 2 (Montgomery form is linear: halve the representative)
  F2 r = a;
  F2::B::halve_mod(r.c0.l);
  F2::B::halve_mod(r.c1.l);
  return r;
}
HD const F2::B& comp(const F2& a, int c) { return c ? a.c1 : a.c0; }

// component c of coefficient k of the F_q^6 product held in T[9 g ..]: sum over i of T[3 i + (k - i mod 3)] — the
// reduction by v^3 = xi is already inside the products with i + j >= 3
DEV F2::B f6_coeff(const F2* T, int g, int k, int c) {
  const F2* t = T + 9 * g;
  F2::B s = comp(t[(k + 3) % 3], c);                       // i = 0
  s = s + comp(t[3 + (k + 2) % 3], c);                     // i = 1
  return s + comp(t[6 + (k + 1) % 3], c);                  // i = 2
}

// r[d] <- r[a] * r[b]   (fq12.go:72-84; d may alias a or b)
DEV void f12_mul(Ws& ws, int d, int a, int b) {
  const uint32_t lane = lane_id();
  const F2* A = ws.r[a];
  const F2* B = ws.r[b];
  if (lane < 6) ws.S[lane] = lane < 3 ? A[lane] + A[lane + 3] : B[lane - 3] + B[lane];
  wsync();
  if (lane < 6) {  // xi * y_j for the right-hand operands b.A, b.B, b.A + b.B (j = 1, 2)
    const int g = lane >> 1, j = 1 + (lane & 1);
    ws.Xi[lane] = f2_mul_xi(g == 0 ? B[j] : (g == 1 ? B[3 + j] : ws.S[3 + j]));
  }
  wsync();
  if (lane < 27) {
    const int g = lane / 9, i = (lane % 9) / 3, j = lane % 3;
    const F2 x = g == 0 ? A[i] : (g == 1 ? A[3 + i] : ws.S[i]);
    const F2 y = (i + j >= 3) ? ws.Xi[2 * g + j - 1] : (g == 0 ? B[j] : (g == 1 ? B[3 + j] : ws.S[3 + j]));
    ws.T[lane] = x * y;
  }
  wsync();
  // with P_g the three F_q^6 products: d.A = P0 + v P1 = (P0[0] + xi P1[2], P0[1] + P1[0], P0[2] + P1[1]), d.B = P2 - P0 - P1
  if (lane < 12) {
    const int o = lane >> 1, c = lane & 1;
    F2::B v;
    if (o == 0) {
      const F2::B p0 = f6_coeff(ws.T, 1, 2, 0), p1 = f6_coeff(ws.T, 1, 2, 1);
      v = f6_coeff(ws.T, 0, 0, c) + (c == 0 ? fq_nine(p0) - p1 : fq_nine(p1) + p0);
    } else if (o < 3) {
      v = f6_coeff(ws.T, 0, o, c) + f6_coeff(ws.T, 1, o - 1, c);
    } else {
      v = f6_coeff(ws.T, 2, o - 3, c) - f6_coeff(ws.T, 0, o - 3, c) - f6_coeff(ws.T, 1, o - 3, c);
    }
    if (c == 0) ws.r[d][o].c0 = v;
    else ws.r[d][o].c1 = v;
  }
  wsync();
}
DEV void f12_sqr(Ws& ws, int d, int a) { f12_mul(ws, d, a, a); }
DEV void f12_copy(Ws& ws, int d, int a) {
  const uint32_t lane = lane_id();
  if (lane < 6 && d != a) ws.r[d][lane] = ws.r[a][lane];
  wsync();
}
DEV void f12_set_one(Ws& ws, int d) {
  const uint32_t lane = lane_id();
  if (lane < 6) ws.r[d][lane] = lane == 0 ? F2::one() : F2::zero();
  wsync();
}
// x^(q^6): conjugation over F_q^6
DEV void f12_conj(Ws& ws, int d, int a) {
  const uint32_t lane = lane_id();
  if (lane < 6) ws.r[d][lane] = lane < 3 ? ws.r[a][lane] : ws.r[a][lane].neg();
  wsync();
}
// x^(q^K), K = 1, 2, 3 (pairing.cuh f12_frobenius): the coefficient of w^j is conjugated K times and multiplied by fc[K-1][j-1]
DEV void f12_frobenius(Ws& ws, int d, int a, int K) {
  const uint32_t lane = lane_id();
  if (lane < 6) {
    const int j = lane < 3 ? 2 * (int)lane : 2 * ((int)lane - 3) + 1;   // tower slot -> power of w
    F2 c = ws.r[a][lane];
    if (K & 1) c = F2{c.c0, c.c1.neg()};
    if (j > 0) c = c * ws.fc[5 * (K - 1) + (j - 1)];
    ws.r[d][lane] = c;
  }
  wsync();
}
// the inversion happens once per pairing: lane 0 walks the tower formulas of pairing.cuh
DEV void f12_inverse(Ws& ws, int d, int a) {
  if (lane_id() == 0) {
    F12 x{F6{ws.r[a][0], ws.r[a][1], ws.r[a][2]}, F6{ws.r[a][3], ws.r[a][4], ws.r[a][5]}};
    F12 y = b200::f12_inverse(x);
    ws.r[d][0] = y.a.a; ws.r[d][1] = y.a.b; ws.r[d][2] = y.a.c;
    ws.r[d][3] = y.b.a; ws.r[d][4] = y.b.b; ws.r[d][5] = y.b.c;
  }
  wsync();
}
// r[d] <- r[a]^u, MSB-first over the 63 bits of the BN parameter (d != a)
DEV void f12_exp_u(Ws& ws, int d, int a) {
  f12_copy(ws, d, a);
#pragma unroll 1
  for (int b = 61; b >= 0; b--) {
    f12_sqr(ws, d, d);
    if ((pc::BN_U >> b) & 1ULL) f12_mul(ws, d, d, a);
  }
}

// ---- line functions -------------------------------------------------------------------------------------------------
// The sparse line value ((ell0, 0, ellVV * px), (0, ellVW * py, 0)) is left in r[s] (bn128.go:402-416).
// Doubling step (bn128.go:262-294), three levels of independent products.
DEV void doubling_step(Ws& ws, int s) {
  const uint32_t lane = lane_id();
  F2* pt = ws.pt;
  const F2 &X = ws.P[0], &Y = ws.P[1], &Z = ws.P[2];
  if (lane < 5) {  // X Y, Y^2 (b), Z^2 (c), (Y + Z)^2, X^2 (j)
    const F2 u = lane == 0 ? X : (lane == 1 ? Y : (lane == 2 ? Z : (lane == 3 ? Y + Z : X)));
    const F2 v = lane == 0 ? Y : u;
    pt[lane] = u * v;
  }
  wsync();
  if (lane == 0) {  // e = twist_b * 3 c
    const F2 twist_b = B200_F2_CONST(TWIST_COEF_B);
    pt[5] = twist_b * (pt[2] + (pt[2] + pt[2]));
  }
  wsync();
  if (lane < 4) {  // X' = a (b - f), g^2, e^2, Z' = b h     with a = X Y / 2, f = 3 e, g = (b + f) / 2, h = (Y + Z)^2 - (b + c)
    const F2 b = pt[1], e = pt[5], f = e + (e + e);
    F2 u, v;
    if (lane == 0) { u = f2_halve(pt[0]); v = b - f; }
    else if (lane == 1) { u = f2_halve(b + f); v = u; }
    else if (lane == 2) { u = e; v = e; }
    else { u = b; v = pt[3] - (b + pt[2]); }
    pt[6 + lane] = u * v;
  }
  wsync();
  if (lane < 6) {
    const F2 b = pt[1], c = pt[2], e = pt[5], h = pt[3] - (b + c), j = pt[4];
    F2 out = F2::zero();
    if (lane == 0) out = f2_mul_xi(e - b);                                     // ell0 = (e - b) * twist
    else if (lane == 2) out = f2_scale(j + (j + j), ws.px);                    // ellVV * px
    else if (lane == 4) out = f2_scale(h.neg(), ws.py);                        // ellVW * py
    ws.r[s][lane] = out;
    if (lane == 1) ws.P[0] = pt[6];
    if (lane == 3) ws.P[1] = pt[7] - pt[8] - (pt[8] + pt[8]);                  // g^2 - 3 e^2
    if (lane == 5) ws.P[2] = pt[9];
  }
  wsync();
}
// Mixed addition step with the affine point Q[2 q], Q[2 q + 1] (bn128.go:296-330)
DEV void addition_step(Ws& ws, int s, int q) {
  const uint32_t lane = lane_id();
  F2* pt = ws.pt;
  const F2 x2 = ws.Q[2 * q], y2 = ws.Q[2 * q + 1];
  const F2 X = ws.P[0], Y = ws.P[1], Z = ws.P[2];
  if (lane < 2) pt[lane] = (lane == 0 ? X : Y) - (lane == 0 ? x2 : y2) * Z;   // d, e
  wsync();
  if (lane < 4) {  // f = d^2, g = e^2, e x2, d y2
    const F2 d = pt[0], e = pt[1];
    const F2 u = (lane == 0 || lane == 3) ? d : e;
    const F2 v = lane == 0 ? d : (lane == 1 ? e : (lane == 2 ? x2 : y2));
    pt[2 + lane] = u * v;
  }
  wsync();
  if (lane < 3) {  // h = d f, i = X f, Z g
    const F2 u = lane == 0 ? pt[0] : (lane == 1 ? X : Z);
    const F2 v = lane == 2 ? pt[3] : pt[2];
    pt[6 + lane] = u * v;
  }
  wsync();
  if (lane < 4) {  // j = h + Z g - 2 i;  d j, e (i - j), h Y, Z h  ->  pt[9..12]
    const F2 h = pt[6], i = pt[7], j = h + pt[8] - (i + i);
    const F2 u = lane == 0 ? pt[0] : (lane == 1 ? pt[1] : (lane == 2 ? h : Z));
    const F2 v = lane == 0 ? j : (lane == 1 ? i - j : (lane == 2 ? Y : h));
    pt[9 + lane] = u * v;
  }
  wsync();
  if (lane < 6) {
    const F2 d = pt[0], e = pt[1];
    F2 out = F2::zero();
    if (lane == 0) out = f2_mul_xi(pt[4] - pt[5]);                             // ell0 = (e x2 - d y2) * twist
    else if (lane == 2) out = f2_scale(e.neg(), ws.px);                        // ellVV * px
    else if (lane == 4) out = f2_scale(d, ws.py);                              // ellVW * py
    ws.r[s][lane] = out;
    if (lane == 1) ws.P[0] = pt[9];
    if (lane == 3) ws.P[1] = pt[10] - pt[11];
    if (lane == 5) ws.P[2] = pt[12];
  }
  wsync();
}

// the Frobenius constants (lane 0 writes them once per pairing)
DEV void pairing_constants(Ws& ws) {
  if (lane_id() == 0) {
    ws.fc[0] = B200_F2_CONST(FROB1_1); ws.fc[1] = B200_F2_CONST(FROB1_2); ws.fc[2] = B200_F2_CONST(FROB1_3);
    ws.fc[3] = B200_F2_CONST(FROB1_4); ws.fc[4] = B200_F2_CONST(FROB1_5);
    ws.fc[5] = B200_F2_CONST(FROB2_1); ws.fc[6] = B200_F2_CONST(FROB2_2); ws.fc[7] = B200_F2_CONST(FROB2_3);
    ws.fc[8] = B200_F2_CONST(FROB2_4); ws.fc[9] = B200_F2_CONST(FROB2_5);
    ws.fc[10] = B200_F2_CONST(FROB3_1); ws.fc[11] = B200_F2_CONST(FROB3_2); ws.fc[12] = B200_F2_CONST(FROB3_3);
    ws.fc[13] = B200_F2_CONST(FROB3_4); ws.fc[14] = B200_F2_CONST(FROB3_5);
  }
  wsync();
}

constexpr int RF = 0, RS = 1;   // accumulator, line value

// r[RF] <- r[RF]^((q^12 - 1) / r): Devegili-Scott-Dahab, the operations of pairing.cuh final_exp_fast.  Needs the Frobenius
// constants in ws.fc (pairing_constants) and uses registers 1..11 as scratch.
DEV void final_exp(Ws& ws) {
  enum { M = 2, MU = 3, MU2 = 4, MU3 = 5, Y0 = 6, Y2 = 7, Y3 = 8, Y4 = 9, Y6 = 10, T0 = 11, T1 = 1 };
  f12_inverse(ws, T0, RF);
  f12_conj(ws, M, RF);
  f12_mul(ws, M, M, T0);                 // f^(q^6 - 1)
  f12_frobenius(ws, T0, M, 2);
  f12_mul(ws, M, T0, M);                 // ^(q^2 + 1)
  f12_exp_u(ws, MU, M);
  f12_exp_u(ws, MU2, MU);
  f12_exp_u(ws, MU3, MU2);
  f12_frobenius(ws, Y0, M, 1);
  f12_frobenius(ws, T0, M, 2);
  f12_mul(ws, Y0, Y0, T0);
  f12_frobenius(ws, T0, M, 3);
  f12_mul(ws, Y0, Y0, T0);               // y0 = m^q m^(q^2) m^(q^3)
  f12_frobenius(ws, Y2, MU2, 2);         // y2
  f12_frobenius(ws, Y3, MU, 1);
  f12_conj(ws, Y3, Y3);                  // y3
  f12_frobenius(ws, T0, MU2, 1);
  f12_mul(ws, Y4, MU, T0);
  f12_conj(ws, Y4, Y4);                  // y4
  f12_frobenius(ws, T0, MU3, 1);
  f12_mul(ws, Y6, MU3, T0);
  f12_conj(ws, Y6, Y6);                  // y6
  f12_conj(ws, MU2, MU2);                // y5 = conj(mu2)   (mu2 itself is no longer needed)
  f12_conj(ws, M, M);                    // y1 = conj(m)     (likewise)
  // y0 * y1^2 * y2^6 * y3^12 * y4^18 * y5^30 * y6^36
  f12_sqr(ws, T0, Y6);
  f12_mul(ws, T0, T0, Y4);
  f12_mul(ws, T0, T0, MU2);              // t0 = y6^2 y4 y5
  f12_mul(ws, T1, Y3, MU2);
  f12_mul(ws, T1, T1, T0);               // t1 = y3 y5 t0
  f12_mul(ws, T0, T0, Y2);               // t0 = t0 y2
  f12_sqr(ws, T1, T1);
  f12_mul(ws, T1, T1, T0);
  f12_sqr(ws, T1, T1);                   // t1 = (t1^2 t0)^2
  f12_mul(ws, T0, T1, M);                // t0 = t1 y1
  f12_mul(ws, T1, T1, Y0);               // t1 = t1 y0
  f12_sqr(ws, T0, T0);
  f12_mul(ws, RF, T0, T1);
}

// Pairing of affine Montgomery-form inputs: the value of pairing_affine_t<true> in r[0] (all lanes call; px, py, qx, qy
// need only be valid on lane 0).
DEV void pairing(Ws& ws, const F2::B& px, const F2::B& py, const F2& qx, const F2& qy) {
  const uint32_t lane = lane_id();
  if (lane == 0) {
    ws.px = px;
    ws.py = py;
    ws.Q[0] = qx;
    ws.Q[1] = qy;
    ws.P[0] = qx;
    ws.P[1] = qy;
    ws.P[2] = F2::one();
    // q1 = pi(Q), q2 = -pi^2(Q)  (bn128.go:238-253, 331-346)
    const F2 tqx = B200_F2_CONST(TWIST_MUL_BY_Q_X), tqy = B200_F2_CONST(TWIST_MUL_BY_Q_Y);
    const F2 q1x = tqx * F2{qx.c0, qx.c1.neg()}, q1y = tqy * F2{qy.c0, qy.c1.neg()};
    ws.Q[2] = q1x;
    ws.Q[3] = q1y;
    ws.Q[4] = tqx * F2{q1x.c0, q1x.c1.neg()};
    ws.Q[5] = (tqy * F2{q1y.c0, q1y.c1.neg()}).neg();
  }
  wsync();
  pairing_constants(ws);
  f12_set_one(ws, RF);
  // Miller loop (bn128.go:354-372), the G2 precomputation fused with it
#pragma unroll 1
  for (int i = 63; i >= 0; i--) {
    doubling_step(ws, RS);
    f12_sqr(ws, RF, RF);
    f12_mul(ws, RF, RF, RS);
    if ((pc::LOOP_COUNT_LOW64 >> i) & 1) {
      addition_step(ws, RS, 0);
      f12_mul(ws, RF, RF, RS);
    }
  }
  addition_step(ws, RS, 1);
  f12_mul(ws, RF, RF, RS);
  addition_step(ws, RS, 2);
  f12_mul(ws, RF, RF, RS);
  final_exp(ws);
}

}  // namespace wp
}  // namespace b200
