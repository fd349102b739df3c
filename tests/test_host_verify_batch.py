"""CPU: the batch-verification kernels of csrc/verify_batch.cuh through the carry-flag emulation (tests/host/
host_verify_batch_test.cpp): the multi-Miller loop (chunks sharing one squaring, inactive pairs), the F_q^12 product tree and
the warp final exponentiation against the product of the oracle's bn128.Pairing values; the G1 on-curve, twist and G2
subgroup predicates; the XYZZ tree sum against the oracle's group sum."""
import ctypes
import random

import numpy as np
import pytest

import build as b200build
from oracle import ref_py as o

pytestmark = pytest.mark.slow
Q, R = o.Q, o.R
G1, G2, F2, F12 = o.BN.G1, o.BN.G2, o.BN.Fq2, o.BN.Fq12


@pytest.fixture(scope="module")
def lib():
    return ctypes.CDLL(b200build.build_host_verify_batch())


def _u32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype=np.uint32).copy()


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _g1(p):
    return list(p[:2])


def _g2(q):
    return [q[0][0], q[0][1], q[1][0], q[1][1]]


def _f2_pow(a, e):
    r = F2.one()
    while e:
        if e & 1:
            r = F2.mul(r, a)
        a = F2.square(a)
        e >>= 1
    return r


def _f2_sqrt(a):
    """Square root in F_q^2 = F_q[u]/(u^2 + 1), q = 3 mod 4 (Adj and Rodriguez-Henriquez, algorithm 9); None if a is not a square."""
    a1 = _f2_pow(a, (Q - 3) // 4)
    alpha = F2.mul(a1, F2.mul(a1, a))
    a0 = F2.mul(_f2_pow(alpha, Q), alpha)
    minus_one = (Q - 1, 0)
    if a0 == minus_one:
        return None
    x0 = F2.mul(a1, a)
    if alpha == minus_one:
        x = F2.mul((0, 1), x0)
    else:
        x = F2.mul(_f2_pow(F2.add(F2.one(), alpha), (Q - 1) // 2), x0)
    assert F2.square(x) == a
    return x


def _twist_point_outside_g2(rng):
    """A random point of y^2 = x^3 + 3/(9+u): in G2 with probability 1/cofactor (~2^-254)."""
    while True:
        x = (rng.randrange(Q), rng.randrange(Q))
        y = _f2_sqrt(F2.add(F2.mul(F2.square(x), x), o.BN.twist_coef_b))
        if y is not None:
            return x, y


def _multi(lib, g1s, g2s, chunk):
    a = _u32([c for p in g1s for c in _g1(p)])
    b = _u32([c for q in g2s for c in _g2(q)])
    out = np.zeros(96, dtype=np.uint32)
    ok = lib.t_multi_pairing(_ptr(a), _ptr(b), len(g1s), chunk, _ptr(out))
    raw = out.tobytes()
    v = [int.from_bytes(raw[32 * i:32 * (i + 1)], "little") for i in range(12)]
    return ok, tuple(tuple((v[6 * h + 2 * k], v[6 * h + 2 * k + 1]) for k in range(3)) for h in range(2))


@pytest.mark.parametrize("k", [1, 2, 5])
def test_multi_miller_loop_is_the_product_of_pairings(lib, k):
    """One final exponentiation of the chunked multi-Miller product == prod of BN.pairing (bn128.go:179-186) on the oracle."""
    rng = random.Random(100 + k)
    g1s = [G1.affine(G1.mul_scalar(G1.G, rng.randrange(1, R))) for _ in range(k)]
    g2s = [G2.affine(G2.mul_scalar(G2.G, rng.randrange(1, R))) for _ in range(k)]
    exp = F12.one()
    for p, q in zip(g1s, g2s):
        exp = F12.mul(exp, o.BN.pairing((p[0], p[1], 1), (q[0], q[1], (1, 0))))
    for chunk in sorted({1, 2, 2 * k + 1}):          # pairs per thread (every active pair is followed by an inactive one)
        ok, got = _multi(lib, g1s, g2s, chunk)
        assert got == exp, chunk
        assert ok == 0


def test_cancelling_pairs_give_one(lib):
    """e(aP, Q) * e(-aP, Q) * e(bP, cQ) * e(-cP, bQ) == 1: the final kernel's compare against one."""
    p = G1.affine(G1.mul_scalar(G1.G, 1234567))
    pn = (p[0], Q - p[1])
    q = G2.affine(G2.mul_scalar(G2.G, 89))
    b1 = G1.affine(G1.mul_scalar(G1.G, 5))
    c2 = G2.affine(G2.mul_scalar(G2.G, 7))
    c1 = G1.affine(G1.mul_scalar(G1.G, 7))
    c1 = (c1[0], Q - c1[1])
    b2 = G2.affine(G2.mul_scalar(G2.G, 5))
    ok, got = _multi(lib, [p, pn, b1, c1], [q, q, c2, b2], 3)
    assert ok == 1 and got == F12.one()


def test_curve_and_subgroup_predicates(lib):
    rng = random.Random(7)
    for _ in range(3):
        p = G1.affine(G1.mul_scalar(G1.G, rng.randrange(1, R)))
        assert lib.t_g1_on_curve(_ptr(_u32(_g1(p)))) == 1
        assert lib.t_g1_on_curve(_ptr(_u32([p[0], (p[1] + 1) % Q]))) == 0
        q = G2.affine(G2.mul_scalar(G2.G, rng.randrange(1, R)))
        assert lib.t_g2_predicates(_ptr(_u32(_g2(q)))) == 3                       # on the twist, in G2
        off = (q[0], ((q[1][0] + 1) % Q, q[1][1]))
        assert lib.t_g2_predicates(_ptr(_u32(_g2(off)))) & 1 == 0                  # off the twist
        t = _twist_point_outside_g2(rng)
        assert lib.t_g2_predicates(_ptr(_u32(_g2(t)))) == 1                       # on the twist, outside G2
    g = G2.affine(G2.G)
    assert lib.t_g2_predicates(_ptr(_u32(_g2(g)))) == 3


@pytest.mark.parametrize("n,k", [(1, 4), (5, 2), (37, 4), (70, 32)])
def test_tree_sum(lib, n, k):
    """k_vb_sum levels == the oracle's sum, with infinity, equal and opposite points among the inputs."""
    rng = random.Random(n)
    ks = [rng.randrange(1, R) for _ in range(n)]
    if n >= 5:
        ks[1] = ks[0]                 # a doubling
        ks[3] = R - ks[2]             # a cancellation
        ks[4] = 0                     # infinity
    pts = [(0, 0) if s == 0 else G1.affine(G1.mul_scalar(G1.G, s)) for s in ks]
    out = np.zeros(16, dtype=np.uint32)
    lib.t_g1_tree_sum(_ptr(_u32([c for p in pts for c in p[:2]])), n, k, _ptr(out))
    raw = out.tobytes()
    got = (int.from_bytes(raw[:32], "little"), int.from_bytes(raw[32:], "little"))
    tot = sum(ks) % R
    assert got == ((0, 0) if tot == 0 else G1.affine(G1.mul_scalar(G1.G, tot))[:2])
