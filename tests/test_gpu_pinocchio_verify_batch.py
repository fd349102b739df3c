"""GPU: b200_pinocchio_verify / b200_pinocchio_verify_batch / snark.VerifyProofBatch.  The single call's verdict and first
failing check equal the oracle's snark.VerifyProof and the library's host-side snark.VerifyProof; every batch verdict equals
b200_pinocchio_verify on the proof alone; valid batches take the aggregated path (stats); invalid proofs that cancel without
the random rho are rejected; call-level errors leave ok[] alone."""
import ctypes
import json
import os
import random

import numpy as np
import pytest

from oracle import ref_py as o

pytestmark = pytest.mark.gpu
R, Q = o.R, o.Q
G1, G2 = o.BN.G1, o.BN.G2
ORDER = ("PiA", "PiAp", "PiBp", "PiC", "PiCp", "PiH", "PiKp")


@pytest.fixture(scope="module")
def gs():
    from gosnark_b200 import _lib, bn128, snark
    _lib.init()
    return _lib, bn128, snark


def _mint(bn128, ks, group):
    """k * G for every k, on the device (b200_g*_mul_batch_bcast: X,Y,Z-exact against the oracle)."""
    g = bn128.G1() if group == 1 else bn128.G2()
    return g.MulScalarBatch([g.G], [k % R for k in ks])


class Instance:
    """A Pinocchio key and n valid proofs with known discrete logs: PiH = ((vkx + a) b - c) / z G1 and
    PiKp = kbg (vkx + a + c + b) / kg G1, with vkx = ic_0 + sum s_j ic_{j+1}."""

    def __init__(self, bn128, n, npub, seed, ic_k=None):
        rng = random.Random(seed)
        rnd = lambda: rng.randrange(1, R)
        ka, kb, kc, kbg, kg, z = (rnd() for _ in range(6))
        self.ic_k = ic_k if ic_k is not None else [rnd() for _ in range(npub + 1)]
        self.pubs = [[rnd() for _ in range(npub)] for _ in range(n)]
        g1k = []
        b = []
        for i in range(n):
            a, bi, c = rnd(), rnd(), rnd()
            vkx = (self.ic_k[0] + sum(x * k for x, k in zip(self.pubs[i], self.ic_k[1:]))) % R
            h = ((vkx + a) * bi - c) * pow(z, -1, R)
            kp = kbg * (vkx + a + c + bi) * pow(kg, -1, R)
            g1k += [a, ka * a, kb * bi, c, kc * c, h, kp]
            b.append(bi)
        m = len(self.ic_k)
        g1 = _mint(bn128, self.ic_k + [kb, kbg] + g1k, 1)
        g2 = _mint(bn128, [ka, kc, z, kbg, kg] + b, 2)
        self.vk = {"IC": g1[:m], "Vkb": g1[m], "G1Kbg": g1[m + 1], "Vka": g2[0], "Vkc": g2[1], "Vkz": g2[2], "G2Kbg": g2[3],
                   "G2Kg": g2[4]}
        self.proofs = [dict(zip(ORDER, g1[m + 2 + 7 * i:m + 9 + 7 * i]), PiB=g2[5 + i]) for i in range(n)]


def _pub_limbs(lib_mod, pubs, npub):
    return lib_mod.ints_to_limbs([x for p in pubs for x in p]) if npub else np.zeros((1, 4), dtype=np.uint64)


def _vk_args(bn128, vk):
    return (bn128._flatten_g1(vk["IC"]), len(vk["IC"]), bn128._flatten_g1([vk["Vkb"], vk["G1Kbg"]]),
            bn128._flatten_g2([vk["Vka"], vk["Vkc"], vk["Vkz"], vk["G2Kbg"], vk["G2Kg"]]))


def batch(gs, vk, proofs, pubs, rho=None, n_ic=None):
    """(rc, ok list, stats) of b200_pinocchio_verify_batch."""
    _lib, bn128, _ = gs
    n, npub = len(proofs), len(pubs[0]) if pubs else 0
    rng = random.Random(len(proofs))
    rho = rho if rho is not None else [[rng.randrange(1, 1 << 128) for _ in range(5)] for _ in range(n)]
    ic, nic, vk1, vk2 = _vk_args(bn128, vk)
    ok = np.full(max(n, 1), 7, dtype=np.int32)
    st = np.zeros(4, dtype=np.uint64)
    pg1 = bn128._flatten_g1([p[k] for p in proofs for k in ORDER] or [G1.zero3()] * 7)
    pb = bn128._flatten_g2([p["PiB"] for p in proofs] or [G2.zero3()])
    rl = _lib.ints_to_limbs([x for r in rho for x in r] or [1] * 5, 2)
    rc = _lib.lib().b200_pinocchio_verify_batch(_lib.ptr(ic), nic if n_ic is None else n_ic, _lib.ptr(vk1), _lib.ptr(vk2), n,
                                                _lib.ptr(pg1), _lib.ptr(pb), _lib.ptr(_pub_limbs(_lib, pubs, npub)), npub,
                                                _lib.ptr(rl), _lib.ptr(ok), _lib.ptr(st))
    return rc, [int(v) for v in ok[:n]], [int(v) for v in st]


def single(gs, vk, proof, pub, n_ic=None):
    """b200_pinocchio_verify on one proof: (1 / 0 or its error code, failed_check)."""
    _lib, bn128, _ = gs
    ic, nic, vk1, vk2 = _vk_args(bn128, vk)
    ok, fc = ctypes.c_int(-100), ctypes.c_int(-100)
    rc = _lib.lib().b200_pinocchio_verify(_lib.ptr(ic), nic if n_ic is None else n_ic, _lib.ptr(vk1), _lib.ptr(vk2),
                                          _lib.ptr(bn128._flatten_g1([proof[k] for k in ORDER])),
                                          _lib.ptr(bn128._flatten_g2([proof["PiB"]])), _lib.ptr(_pub_limbs(_lib, [pub], len(pub))),
                                          len(pub), ctypes.byref(ok), ctypes.byref(fc))
    return (rc, None) if rc else (ok.value, fc.value)


@pytest.mark.parametrize("npub", [0, 1, 8])
@pytest.mark.parametrize("n", [1, 2, 3, 33, 1024])
def test_valid_batches_take_the_aggregated_path(gs, n, npub):
    inst = Instance(gs[1], n, npub, seed=1000 * n + npub)
    rc, ok, st = batch(gs, inst.vk, inst.proofs, inst.pubs)
    assert rc == 0 and ok == [1] * n
    assert st == [n, 0, 1, n + 6]


def test_each_check_fails_alone(gs):
    """Doubling PiAp, PiBp, PiCp, PiH or PiKp breaks check 1..5 alone: the single call, the oracle and snark.VerifyProof
    agree on it, and the batch rejects that proof only."""
    _, _, snark = gs
    inst = Instance(gs[1], 8, 1, seed=31)
    P, pubs = [dict(p) for p in inst.proofs], inst.pubs
    assert single(gs, inst.vk, P[0], pubs[0]) == (1, 0)
    assert o.pinocchio_verify(inst.vk, P[0], pubs[0]) == (True, 0)
    for k, key in enumerate(("PiAp", "PiBp", "PiCp", "PiH", "PiKp"), start=1):
        P[k] = dict(P[k], **{key: G1.double(P[k][key])})
        assert single(gs, inst.vk, P[k], pubs[k]) == (0, k), key
        assert o.pinocchio_verify(inst.vk, P[k], pubs[k]) == (False, k), key
        assert snark.VerifyProof(inst.vk, P[k], pubs[k]) is False
    rc, ok, st = batch(gs, inst.vk, P, pubs)
    assert rc == 0 and ok == [1, 0, 0, 0, 0, 0, 1, 1]
    assert st == [8, 8, 1, 14 + 12 * 8]


def _twist_point_outside_g2():
    from test_host_verify_batch import _twist_point_outside_g2 as tp
    x, y = tp(random.Random(3))
    return (x, y, (1, 0))


def test_mixed_batch_matches_the_single_verifier(gs):
    """Every kind of bad proof in one batch: ok[i] == b200_pinocchio_verify(proof i) for all i, and the oracle agrees on a
    few.  The key has IC[0] = k G, IC[1] = G, so the signal k makes the reference's vkx = Add(kG, kG) = infinity."""
    k = 0x1234567
    inst = Instance(gs[1], 22, 1, seed=5, ic_k=[k, 1])
    P, pubs = [dict(p) for p in inst.proofs], [list(s) for s in inst.pubs]
    for j, key in enumerate(ORDER):                                   # 1-7: each G1 slot at infinity
        P[1 + j][key] = G1.zero3()
    P[8]["PiB"] = G2.zero3()                                           # PiB at infinity: B200_EINVAL
    P[9]["PiCp"] = (Q, P[9]["PiCp"][1], P[9]["PiCp"][2])               # coordinate == q: B200_ERANGE
    P[10]["PiB"] = G2.zero3()                                          # PiB at infinity with a coordinate >= q: EINVAL
    P[10]["PiH"] = (Q + 5, 1, 1)
    a = G1.affine(P[11]["PiBp"])
    P[11]["PiBp"] = (a[0], (a[1] + 1) % Q, 1)                          # off the curve
    P[12]["PiB"] = _twist_point_outside_g2()                           # PiB on the twist, outside G2
    pubs[13][0] = k                                                    # vkx degenerate
    vkx14 = G1.add(inst.vk["IC"][0], G1.mul_scalar(inst.vk["IC"][1], pubs[14][0]))
    P[14]["PiA"] = vkx14                                               # VkxA = Add(vkx, vkx) degenerate
    pubs[15][0] = (pubs[15][0] + 1) % R                                # moved public signal
    pubs[16][0] = R + 3                                                # public signal >= r: B200_ERANGE
    P[17]["PiB"], P[18]["PiB"] = P[18]["PiB"], P[17]["PiB"]            # PiB swapped between two proofs
    rc, ok, st = batch(gs, inst.vk, P, pubs)
    assert rc == 0
    want = [single(gs, inst.vk, P[i], pubs[i])[0] for i in range(len(P))]
    assert ok == want
    assert want[0] == want[19] == want[20] == want[21] == 1
    assert want[8] == want[10] == -3 and want[9] == want[16] == -4
    assert all(want[i] == 0 for i in list(range(1, 8)) + [11, 12, 13, 14, 15, 17, 18])
    # aggregated: 0, 13, 15, 17-21; the check fails, so they run one by one with 1-7, 11, 12, 14
    assert st[0] == 8 and st[2] == 1 and st[1] == 8 + 10
    assert st[3] == 8 + 6 + 12 * st[1]
    for i in (0, 13, 15):
        assert o.pinocchio_verify(inst.vk, P[i], pubs[i])[0] == bool(want[i]), i


def test_cancelling_invalid_proofs_need_rho(gs):
    """PiH_1 + D and PiH_2 - D: their sum is right, so a check with every rho = 1 accepts both; random rho rejects both."""
    _, _, snark = gs
    inst = Instance(gs[1], 2, 1, seed=9)
    d = G1.mul_scalar(G1.G, 777)
    P = [dict(p) for p in inst.proofs]
    P[0]["PiH"] = G1.add(P[0]["PiH"], d)
    P[1]["PiH"] = G1.add(P[1]["PiH"], G1.neg(d))
    rc, ok, _ = batch(gs, inst.vk, P, inst.pubs, rho=[[1] * 5, [1] * 5])
    assert rc == 0 and ok == [1, 1]
    rc, ok, st = batch(gs, inst.vk, P, inst.pubs)
    assert rc == 0 and ok == [0, 0] and st == [2, 2, 1, 8 + 24]
    assert snark.VerifyProofBatch(inst.vk, P, inst.pubs) == [False, False]
    assert [snark.VerifyProof(inst.vk, p, s) for p, s in zip(P, inst.pubs)] == [False, False]


def _golden_vk_proof(g):
    """The Go binary's Pinocchio setup and proof (older JSON layout), as test_gpu_verify.py loads them."""
    st, pr = g["pinocchio_setup"], g["pinocchio_proofs"]
    t3 = lambda p: tuple(p)
    t2 = lambda p: tuple(tuple(c) for c in p)
    vk = {k: ([t3(p) for p in v] if k == "IC" else (t2(v) if isinstance(v[0], list) else t3(v))) for k, v in st["Vk"].items()}
    return vk, {k: (t2(v) if k == "PiB" else t3(v)) for k, v in pr.items()}


@pytest.mark.parametrize("name", ["mul", "x3x5", "chain21"])
def test_real_keys(gs, golden_dir, name):
    """snark.GenerateTrustedSetup + b200_pinocchio_prove, and the Go binary's own setup and proof: the batch verdicts equal
    snark.VerifyProof for the right public inputs and for moved ones."""
    from gosnark_b200 import r1csqap
    _, _, snark = gs
    g = json.load(open(os.path.join(golden_dir, f"gobin_{name}.json")))
    cc = g["compiledcircuit"]
    r1 = cc["R1CS"]
    pf = r1csqap.PolynomialField()
    alphas, betas, gammas, _ = pf.R1CSToQAP(r1["A"], r1["B"], r1["C"])
    setup = snark.GenerateTrustedSetup(len(g["witness"]), cc, alphas, betas, gammas)
    w = [int(x) for x in g["witness"]]
    _, _, _, px = pf.CombinePolynomials(w, alphas, betas, gammas)
    proof = snark.GenerateProofs(cc, setup["Pk"], w, px)
    pub = [int(x) for x in g["public"]]
    sigs = [pub, [pub[0] + 1], pub, [pub[0] + R], [pub[0] - 1]]
    gvk, gproof = _golden_vk_proof(g)
    for vk, pr in ((setup["Vk"], proof), (gvk, gproof)):
        want = [snark.VerifyProof(vk, pr, s) for s in sigs]
        assert want == [True, False, True, True, False]
        stats = []
        assert snark.VerifyProofBatch(vk, [pr] * len(sigs), sigs, stats=stats) == want
        assert stats[0] == 5 and stats[2] == 1


def test_one_bad_among_many_and_all_bad(gs):
    inst = Instance(gs[1], 4096, 1, seed=11)
    P = list(inst.proofs)
    P[2345] = dict(P[2345], PiH=G1.double(P[2345]["PiH"]))
    rc, ok, st = batch(gs, inst.vk, P, inst.pubs)
    assert rc == 0 and ok == [0 if i == 2345 else 1 for i in range(4096)]
    assert st == [4096, 4096, 1, 4102 + 12 * 4096]
    bad = [dict(p, PiKp=G1.double(p["PiKp"])) for p in inst.proofs[:64]]
    rc, ok, st = batch(gs, inst.vk, bad, inst.pubs[:64])
    assert rc == 0 and ok == [0] * 64
    assert st == [64, 64, 1, 70 + 12 * 64]


def test_call_level_errors(gs):
    _, _, snark = gs
    inst = Instance(gs[1], 3, 2, seed=13)
    rc, ok, _ = batch(gs, inst.vk, inst.proofs, inst.pubs, n_ic=2)          # len(IC) < n_public + 1
    assert rc == -3 and ok == [7, 7, 7]
    assert single(gs, inst.vk, inst.proofs[0], inst.pubs[0], n_ic=2)[0] == -3
    rho = [[5] * 5, [5, 6, 0, 7, 8], [9] * 5]                               # a rho equal to 0
    rc, ok, _ = batch(gs, inst.vk, inst.proofs, inst.pubs, rho=rho)
    assert rc == -3 and ok == [7, 7, 7]
    rc, _, _ = batch(gs, inst.vk, [], [])                                   # no proofs
    assert rc == -3
    vb = G1.affine(inst.vk["Vkb"])
    bad_keys = (
        (dict(inst.vk, Vkb=(Q, 1, 1)), -4, -4),                             # coordinate >= q
        (dict(inst.vk, IC=[inst.vk["IC"][0], (1, Q + 2, 1), inst.vk["IC"][2]]), -4, -4),
        (dict(inst.vk, Vkz=G2.zero3()), -3, -3),                            # a G2 point at infinity
        (dict(inst.vk, G2Kg=G2.zero3(), Vkb=(Q, 1, 1)), -3, -3),            # ... wins over a coordinate >= q
        (dict(inst.vk, Vkb=G1.zero3()), -3, None),                          # stricter than the single call
        (dict(inst.vk, G1Kbg=G1.zero3()), -3, None),
        (dict(inst.vk, Vkb=(vb[0], (vb[1] + 1) % Q, 1)), -3, None),
        (dict(inst.vk, IC=[inst.vk["IC"][0], G1.affine(inst.vk["IC"][1])[:1] + (5, 1), inst.vk["IC"][2]]), -3, None),
        (dict(inst.vk, Vka=_twist_point_outside_g2()), -3, None),
        (dict(inst.vk, Vkc=(G2.G[0], ((G2.G[1][0] + 1) % Q, G2.G[1][1]), G2.G[2])), -3, None),   # off the twist
    )
    for j, (vk, code, single_code) in enumerate(bad_keys):
        rc, ok, _ = batch(gs, vk, inst.proofs, inst.pubs)
        assert rc == code and ok == [7, 7, 7], j
        if single_code is not None:
            assert single(gs, vk, inst.proofs[0], inst.pubs[0])[0] == single_code, j
    with pytest.raises(ValueError):
        snark.VerifyProofBatch(inst.vk, inst.proofs, inst.pubs, rho=[[1] * 5, [1] * 5, [1, 2, 3, 0, 5]])
    with pytest.raises(ValueError):
        snark.VerifyProofBatch(inst.vk, inst.proofs, inst.pubs, rho=[[1] * 5, [1] * 5, [1] * 4])
    with pytest.raises(ValueError):
        snark.VerifyProofBatch(inst.vk, inst.proofs, inst.pubs, rho=[[1] * 5] * 2)
