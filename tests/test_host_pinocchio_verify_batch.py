"""CPU: the Pinocchio verification kernels of csrc/verify_batch_pinocchio.cuh through the carry-flag emulation (tests/host/
host_pinocchio_verify_batch_test.cpp): the per-proof preparation and products against the oracle's group arithmetic for
given rho, the status word of every bad-proof kind, the whole aggregated check (tail, multi-Miller loop, product tree, final
exponentiation) on a valid and a broken batch, and the single check's compare kernel on the oracle's twelve pairing values."""
import ctypes
import random

import numpy as np
import pytest

import build as b200build
from oracle import ref_py as o
from test_host_verify_batch import _twist_point_outside_g2

pytestmark = pytest.mark.slow
Q, R = o.Q, o.R
G1, G2, F12 = o.BN.G1, o.BN.G2, o.BN.Fq12
ORDER = ("PiA", "PiAp", "PiBp", "PiC", "PiCp", "PiH", "PiKp")


@pytest.fixture(scope="module")
def lib():
    return ctypes.CDLL(b200build.build_host_pinocchio_verify_batch())


def _u32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype=np.uint32).copy()


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _j1(ps):
    return _u32([c for p in ps for c in p])


def _j2(qs):
    return _u32([c for q in qs for xy in q for c in xy])


def instance(rng, n, npub):
    """A key and n valid proofs with known discrete logs (oracle-minted)."""
    rnd = lambda: rng.randrange(1, R)
    ka, kb, kc, kbg, kg, z = (rnd() for _ in range(6))
    ic = [rnd() for _ in range(npub + 1)]
    g1 = lambda k: G1.mul_scalar(G1.G, k % R)
    g2 = lambda k: G2.mul_scalar(G2.G, k % R)
    vk = {"Vka": g2(ka), "Vkb": g1(kb), "Vkc": g2(kc), "G1Kbg": g1(kbg), "G2Kbg": g2(kbg), "G2Kg": g2(kg), "Vkz": g2(z),
          "IC": [g1(k) for k in ic]}
    proofs, pubs = [], []
    for _ in range(n):
        s = [rnd() for _ in range(npub)]
        a, b, c = rnd(), rnd(), rnd()
        vkx = (ic[0] + sum(x * k for x, k in zip(s, ic[1:]))) % R
        h = ((vkx + a) * b - c) * pow(z, -1, R)
        kp = kbg * (vkx + a + c + b) * pow(kg, -1, R)
        proofs.append({"PiA": g1(a), "PiAp": g1(ka * a), "PiB": g2(b), "PiBp": g1(kb * b), "PiC": g1(c), "PiCp": g1(kc * c),
                       "PiH": g1(h), "PiKp": g1(kp)})
        pubs.append(s)
    return vk, proofs, pubs


def _args(vk, proofs, pubs, rho):
    npub = len(pubs[0])
    return [_j1(vk["IC"][:npub + 1]), npub, _j1([vk["Vkb"], vk["G1Kbg"]]),
            _j2([G2.G, vk["Vka"], vk["Vkc"], vk["Vkz"], vk["G2Kbg"], vk["G2Kg"]]), len(proofs),
            _j1([p[k] for p in proofs for k in ORDER]), _j2([p["PiB"] for p in proofs]),
            _u32([x for s in pubs for x in s] or [0]), np.array([[x & (2**64 - 1), x >> 64] for r in rho for x in r], dtype=np.uint64)]


def _call(fn, args, *extra):
    conv = [_ptr(a) if isinstance(a, np.ndarray) else a for a in args]
    return fn(*conv, *extra)


def _aff(p):
    return (0, 0) if G1.is_zero(p) else tuple(G1.affine(p)[:2])


def _words(raw, k):
    return [int.from_bytes(raw[32 * (2 * k + j):32 * (2 * k + j + 1)], "little") for j in range(2)]


def test_prepare_products_equal_the_oracle(lib):
    rng = random.Random(21)
    vk, proofs, pubs = instance(rng, 3, 2)
    rho = [[rng.randrange(1, 1 << 128) for _ in range(5)] for _ in proofs]
    n = len(proofs)
    status = np.zeros(n, dtype=np.int32)
    pairs = np.zeros(16 * n, dtype=np.uint32)
    sums = np.zeros(6 * n * 16, dtype=np.uint32)
    bad = _call(lib.t_prepare, _args(vk, proofs, pubs, rho), _ptr(status), _ptr(pairs), _ptr(sums))
    assert bad == 0 and list(status) == [2] * n
    pr, sr = pairs.tobytes(), sums.tobytes()
    mul = lambda p, k: G1.mul_scalar(p, k)
    for i, (p, s, r) in enumerate(zip(proofs, pubs, rho)):
        vkx = vk["IC"][0]
        for j, x in enumerate(s):
            vkx = G1.add(vkx, mul(vk["IC"][j + 1], x))
        vkxa = G1.add(vkx, p["PiA"])
        vkxac = G1.add(vkxa, p["PiC"])
        s0 = G1.add(G1.add(mul(p["PiAp"], r[0]), mul(p["PiBp"], r[1])), G1.add(mul(p["PiCp"], r[2]), mul(p["PiC"], r[3])))
        want = [s0, mul(p["PiA"], r[0]), mul(p["PiC"], r[2]), mul(p["PiH"], r[3]), mul(vkxac, r[4]), mul(p["PiKp"], r[4])]
        for c, w in enumerate(want):
            assert tuple(_words(sr, c * n + i)) == _aff(w), (i, c)
        side = G1.add(G1.add(mul(vk["Vkb"], r[1]), mul(vkxa, r[3])), mul(vk["G1Kbg"], r[4]))
        assert tuple(_words(pr, i)) == _aff(side), i


def test_status_word_of_every_bad_kind(lib):
    rng = random.Random(22)
    k = 0x1234567
    vk, proofs, pubs = instance(rng, 1, 1)
    vk["IC"] = [G1.mul_scalar(G1.G, k), G1.G]
    base, s = proofs[0], [5]
    vkx = G1.add(vk["IC"][0], G1.mul_scalar(G1.G, 5))
    a = G1.affine(base["PiH"])
    tx, ty = _twist_point_outside_g2(random.Random(3))
    q = base["PiB"]
    cases = [({}, 2)]
    cases += [({key: G1.zero3()}, 1) for key in ORDER]                                   # each G1 slot at infinity
    cases += [({"PiB": G2.zero3()}, -3),                                                  # PiB at infinity
              ({"PiC": (Q, 1, 1)}, -4),                                                   # a coordinate == q
              ({"PiB": (q[0], q[1], (Q, 0))}, -4),
              ({"PiB": G2.zero3(), "PiKp": (Q + 1, 1, 1)}, -3),                           # PiB at infinity wins
              ({"PiH": (a[0], (a[1] + 1) % Q, 1)}, 1),                                    # off the curve
              ({"PiB": (tx, ty, (1, 0))}, 1),                                             # on the twist, outside G2
              ({"PiB": (q[0], ((q[1][0] + 1) % Q, q[1][1]), q[2])}, 1),                   # off the twist
              ({"PiA": vkx}, 1),                                                          # VkxA = Add(vkx, vkx): infinity
              ({"PiC": G1.add(vkx, base["PiA"])}, 1)]                                     # VkxAC = Add(VkxA, VkxA)
    P = [dict(base, **chg) for chg, _ in cases]
    n = len(P)
    rho = [[1, 2, 3, 4, 5]] * n
    status = np.zeros(n, dtype=np.int32)
    bad = _call(lib.t_prepare, _args(vk, P, [s] * n, rho), _ptr(status), _ptr(np.zeros(16 * n, dtype=np.uint32)),
                _ptr(np.zeros(96 * n, dtype=np.uint32)))
    assert bad == 0
    assert list(status) == [w for _, w in cases]
    # the key check: Vkb off the curve, a vk G2 point outside G2
    st1 = np.zeros(1, dtype=np.int32)
    out = lambda: (_ptr(st1), _ptr(np.zeros(16, dtype=np.uint32)), _ptr(np.zeros(96, dtype=np.uint32)))
    vb = G1.affine(vk["Vkb"])
    for bad_vk in (dict(vk, Vkb=(vb[0], (vb[1] + 1) % Q, 1)), dict(vk, Vkz=(tx, ty, (1, 0))), dict(vk, G1Kbg=G1.zero3())):
        assert _call(lib.t_prepare, _args(bad_vk, [base], [s], rho[:1]), *out()) == 1


@pytest.mark.parametrize("chunk", [1, 3])
def test_aggregated_check_valid_and_broken(lib, chunk):
    rng = random.Random(23)
    vk, proofs, pubs = instance(rng, 2, 1)
    rho = [[rng.randrange(1, 1 << 128) for _ in range(5)] for _ in proofs]
    act = ctypes.c_int(-1)
    assert _call(lib.t_aggregate, _args(vk, proofs, pubs, rho), chunk, ctypes.byref(act)) == 1
    assert act.value == 2 + 6
    broken = [proofs[0], dict(proofs[1], PiH=G1.double(proofs[1]["PiH"]))]
    assert _call(lib.t_aggregate, _args(vk, broken, pubs, rho), chunk, ctypes.byref(act)) == 0


def _f12_u32(e):
    return _u32([c for f6 in e for f2 in f6 for c in f2])


def test_compare_kernel_on_the_oracles_pairings(lib):
    """The twelve values of snark.go:292-372 for a valid proof (the oracle's bn128.Pairing), then each check broken alone
    by a value from another check, and two broken at once: failed_check is the first failing one."""
    rng = random.Random(24)
    vk, proofs, pubs = instance(rng, 1, 1)
    p, s = proofs[0], pubs[0]
    vkx = G1.add(vk["IC"][0], G1.mul_scalar(vk["IC"][1], s[0]))
    vkxa = G1.add(vkx, p["PiA"])
    g1s = [p["PiA"], p["PiAp"], vk["Vkb"], p["PiBp"], p["PiC"], p["PiCp"], vkxa, p["PiH"], p["PiC"], G1.add(vkxa, p["PiC"]),
           vk["G1Kbg"], p["PiKp"]]
    g2s = [vk["Vka"], G2.G, p["PiB"], G2.G, vk["Vkc"], G2.G, p["PiB"], vk["Vkz"], G2.G, vk["G2Kbg"], p["PiB"], vk["G2Kg"]]
    e = [o.BN.pairing(a, b) for a, b in zip(g1s, g2s)]
    assert o.pinocchio_verify(vk, p, s) == (True, 0)
    t = lambda vals: lib.t_compare(_ptr(np.concatenate([_f12_u32(v) for v in vals])))
    assert t(e) == 0
    for k, slot in ((1, 1), (2, 3), (3, 5), (4, 6), (5, 11)):
        bad = list(e)
        bad[slot] = e[(slot + 2) % 12]
        assert t(bad) == k, k
    bad = list(e)
    bad[3], bad[8] = e[0], e[0]
    assert t(bad) == 2
