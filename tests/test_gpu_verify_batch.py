"""GPU: b200_groth16_verify_batch / groth16.VerifyProofBatch.  Every verdict equals b200_groth16_verify on the proof alone
(and the oracle's groth16.VerifyProof on small cases), valid batches take the aggregated path (stats), a batch whose invalid
proofs cancel without the random rho is rejected, and call-level errors leave ok[] alone."""
import json
import os
import random

import numpy as np
import pytest

from oracle import ref_py as o

pytestmark = pytest.mark.gpu
R, Q = o.R, o.Q
G1, G2 = o.BN.G1, o.BN.G2


@pytest.fixture(scope="module")
def gs():
    from gosnark_b200 import _lib, bn128, groth16
    _lib.init()
    return _lib, bn128, groth16


def _mint(bn128, ks, group):
    """k * G for every k, on the device (b200_g*_mul_batch_bcast: X,Y,Z-exact against the oracle)."""
    g = bn128.G1() if group == 1 else bn128.G2()
    return g.MulScalarBatch([g.G], [k % R for k in ks])


class Instance:
    """A verification key and n proofs with known discrete logs: c = (a b - alpha beta - icPubl gamma) / delta."""

    def __init__(self, bn128, n, npub, seed, ic_k=None):
        rng = random.Random(seed)
        rnd = lambda: rng.randrange(1, R)
        self.al, self.be, self.ga, self.de = (rnd() for _ in range(4))
        self.ic_k = ic_k if ic_k is not None else [rnd() for _ in range(npub + 1)]
        self.pubs = [[rnd() for _ in range(npub)] for _ in range(n)]
        a = [rnd() for _ in range(n)]
        b = [rnd() for _ in range(n)]
        c = []
        for i in range(n):
            icp = (self.ic_k[0] + sum(p * k for p, k in zip(self.pubs[i], self.ic_k[1:]))) % R
            c.append((a[i] * b[i] - self.al * self.be - icp * self.ga) * pow(self.de, -1, R) % R)
        g1 = _mint(bn128, self.ic_k + [self.al] + a + c, 1)
        g2 = _mint(bn128, [self.be, self.ga, self.de] + b, 2)
        m = len(self.ic_k)
        self.vk = {"IC": g1[:m], "G1": {"Alpha": g1[m]}, "G2": {"Beta": g2[0], "Gamma": g2[1], "Delta": g2[2]}}
        self.proofs = [{"PiA": g1[m + 1 + i], "PiB": g2[3 + i], "PiC": g1[m + 1 + n + i]} for i in range(n)]


def _pub_limbs(lib_mod, pubs, npub):
    return lib_mod.ints_to_limbs([x for p in pubs for x in p]) if npub else np.zeros((1, 4), dtype=np.uint64)


def _vk_args(bn128, vk):
    return (bn128._flatten_g1(vk["IC"]), len(vk["IC"]), bn128._flatten_g1([vk["G1"]["Alpha"]]), bn128._flatten_g2([vk["G2"]["Beta"]]),
            bn128._flatten_g2([vk["G2"]["Gamma"]]), bn128._flatten_g2([vk["G2"]["Delta"]]))


def batch(gs, vk, proofs, pubs, rho=None, n_ic=None):
    """(rc, ok list, stats) of b200_groth16_verify_batch."""
    _lib, bn128, _ = gs
    n, npub = len(proofs), len(pubs[0]) if pubs else 0
    rng = random.Random(len(proofs))
    rho = rho if rho is not None else [rng.randrange(1, 1 << 128) for _ in range(n)]
    ic, nic, al, be, ga, de = _vk_args(bn128, vk)
    ok = np.full(max(n, 1), 7, dtype=np.int32)
    st = np.zeros(4, dtype=np.uint64)
    rc = _lib.lib().b200_groth16_verify_batch(
        _lib.ptr(ic), nic if n_ic is None else n_ic, _lib.ptr(al), _lib.ptr(be), _lib.ptr(ga), _lib.ptr(de), n,
        _lib.ptr(bn128._flatten_g1([p["PiA"] for p in proofs] or [G1.zero3()])),
        _lib.ptr(bn128._flatten_g2([p["PiB"] for p in proofs] or [G2.zero3()])),
        _lib.ptr(bn128._flatten_g1([p["PiC"] for p in proofs] or [G1.zero3()])), _lib.ptr(_pub_limbs(_lib, pubs, npub)), npub,
        _lib.ptr(_lib.ints_to_limbs(rho or [1], 2)), _lib.ptr(ok), _lib.ptr(st))
    return rc, [int(v) for v in ok[:n]], [int(v) for v in st]


def single(gs, vk, proof, pub):
    """b200_groth16_verify on one proof: 1 / 0, or its error code."""
    import ctypes
    _lib, bn128, _ = gs
    ic, nic, al, be, ga, de = _vk_args(bn128, vk)
    ok = ctypes.c_int(-100)
    rc = _lib.lib().b200_groth16_verify(_lib.ptr(ic), nic, _lib.ptr(al), _lib.ptr(be), _lib.ptr(ga), _lib.ptr(de),
                                         _lib.ptr(bn128._flatten_g1([proof["PiA"]])), _lib.ptr(bn128._flatten_g2([proof["PiB"]])),
                                         _lib.ptr(bn128._flatten_g1([proof["PiC"]])), _lib.ptr(_pub_limbs(_lib, [pub], len(pub))),
                                         len(pub), ctypes.byref(ok))
    return rc if rc else ok.value


@pytest.mark.parametrize("npub", [0, 1, 8])
@pytest.mark.parametrize("n", [1, 2, 3, 33, 1024])
def test_valid_batches_take_the_aggregated_path(gs, n, npub):
    inst = Instance(gs[1], n, npub, seed=1000 * n + npub)
    rc, ok, st = batch(gs, inst.vk, inst.proofs, inst.pubs)
    assert rc == 0 and ok == [1] * n
    assert st == [n, 0, 1, n + 3]


def _twist_point_outside_g2():
    from test_host_verify_batch import _twist_point_outside_g2 as tp
    x, y = tp(random.Random(3))
    return (x, y, (1, 0))


def test_mixed_batch_matches_the_single_verifier(gs):
    """Every kind of bad proof in one batch: ok[i] == b200_groth16_verify(proof i) for all i, and the oracle agrees on a few.
    The key has IC[0] = k G, IC[1] = G, so the signal k makes the reference's icPubl = Add(kG, kG) = infinity (SURVEY H6)."""
    k = 0x1234567
    inst = Instance(gs[1], 14, 1, seed=5, ic_k=[k, 1])
    P, pubs = [dict(p) for p in inst.proofs], [list(s) for s in inst.pubs]
    pubs[1][0] = (pubs[1][0] + 1) % R                                  # moved public signal
    P[2]["PiC"] = G1.double(P[2]["PiC"])                               # doubled C
    P[3]["PiB"], P[4]["PiB"] = P[4]["PiB"], P[3]["PiB"]                # B swapped between two proofs
    P[5]["PiA"] = G1.zero3()                                           # A at infinity
    P[6]["PiC"] = G1.zero3()                                           # C at infinity
    P[7]["PiB"] = G2.zero3()                                           # B at infinity: B200_EINVAL
    P[8]["PiA"] = (Q, P[8]["PiA"][1], P[8]["PiA"][2])                  # coordinate >= q: B200_ERANGE
    a = G1.affine(P[9]["PiA"])
    P[9]["PiA"] = (a[0], (a[1] + 1) % Q, 1)                            # A off the curve
    P[10]["PiB"] = _twist_point_outside_g2()                           # B on the twist, outside G2
    pubs[11][0] = k                                                    # icPubl degenerate
    P[12]["PiC"] = (Q + 1, 1, 1)                                       # C >= q together with B at infinity: EINVAL
    P[12]["PiB"] = G2.zero3()
    rc, ok, st = batch(gs, inst.vk, P, pubs)
    assert rc == 0
    want = [single(gs, inst.vk, P[i], pubs[i]) for i in range(len(P))]
    assert ok == want
    assert want[0] == want[13] == 1 and want[7] == want[12] == -3 and want[8] == -4
    assert all(want[i] == 0 for i in (1, 2, 3, 4))
    assert st[0] == 6 and st[2] == 1                                   # 0-4, 13 aggregated; the check failed ...
    assert st[1] == 6 + 5                                              # ... so they ran one by one, with 5, 6, 9, 10, 11
    for i in (0, 2):
        assert o.groth16_verify(inst.vk, P[i], pubs[i]) == bool(want[i]), i


def test_cancelling_invalid_proofs_need_rho(gs):
    """C_1 + D and C_2 - D: their sum is right, so a check without rho (rho = 1, 1) accepts both; random rho rejects both."""
    inst = Instance(gs[1], 2, 1, seed=9)
    d = G1.mul_scalar(G1.G, 777)
    P = [dict(p) for p in inst.proofs]
    P[0]["PiC"] = G1.add(P[0]["PiC"], d)
    P[1]["PiC"] = G1.add(P[1]["PiC"], G1.neg(d))
    rc, ok, _ = batch(gs, inst.vk, P, inst.pubs, rho=[1, 1])
    assert rc == 0 and ok == [1, 1]
    rc, ok, st = batch(gs, inst.vk, P, inst.pubs)
    assert rc == 0 and ok == [0, 0] and st == [2, 2, 1, 5 + 8]
    _, _, groth16 = gs
    assert groth16.VerifyProofBatch(inst.vk, P, inst.pubs) == [False, False]
    assert [groth16.VerifyProof(inst.vk, p, s) for p, s in zip(P, inst.pubs)] == [False, False]


def test_one_bad_among_many_and_all_bad(gs):
    inst = Instance(gs[1], 4096, 1, seed=11)
    P = list(inst.proofs)
    P[2345] = dict(P[2345], PiC=G1.double(P[2345]["PiC"]))
    rc, ok, st = batch(gs, inst.vk, P, inst.pubs)
    assert rc == 0 and ok == [0 if i == 2345 else 1 for i in range(4096)]
    assert st == [4096, 4096, 1, 4099 + 4 * 4096]
    bad = [dict(p, PiC=G1.double(p["PiC"])) for p in inst.proofs[:64]]
    rc, ok, _ = batch(gs, inst.vk, bad, inst.pubs[:64])
    assert rc == 0 and ok == [0] * 64


def test_real_crs_flow(gs):
    """CircuitGroth16 at 2^10 (the CRS of GenerateTrustedSetup): proofs by the library's prover with four blindings are
    accepted together, and a changed public signal is rejected at its index only."""
    _lib, bn128, groth16 = gs
    from gosnark_b200.synthetic import CircuitGroth16
    syn = CircuitGroth16(10)
    pk = syn.load_pk()
    proofs = []
    for j in range(4):
        r, s = _lib.ints_to_limbs([syn.r + j]), _lib.ints_to_limbs([syn.s + 3 * j])
        pa, pb, pc = np.zeros(12, dtype=np.uint64), np.zeros(24, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
        _lib.check(_lib.lib().b200_groth16_prove(pk, _lib.ptr(syn.w), syn.m, _lib.ptr(syn.px), syn.px.shape[0], _lib.ptr(r),
                                                 _lib.ptr(s), _lib.ptr(pa), _lib.ptr(pb), _lib.ptr(pc)))
        proofs.append({"PiA": bn128._unflatten_g1(pa)[0], "PiB": bn128._unflatten_g2(pb)[0], "PiC": bn128._unflatten_g1(pc)[0]})
    _lib.check(_lib.lib().b200_pk_free(pk))
    vk = {"IC": bn128._unflatten_g1(syn.ic), "G1": {"Alpha": bn128._unflatten_g1(syn.alpha1)[0]},
          "G2": {"Beta": bn128._unflatten_g2(syn.beta2)[0], "Gamma": bn128._unflatten_g2(syn.gamma2)[0],
                 "Delta": bn128._unflatten_g2(syn.delta2)[0]}}
    pub = list(syn.circuit.public_signals)
    stats = []
    assert groth16.VerifyProofBatch(vk, proofs, [pub] * 4, stats=stats) == [True] * 4
    assert stats == [4, 0, 1, 7]
    moved = [pub, pub, [pub[0] + 1], pub]
    assert groth16.VerifyProofBatch(vk, proofs, moved) == [True, True, False, True]


def test_snarkjs_golden_proof(gs, golden_dir):
    _, _, groth16 = gs
    c = json.load(open(os.path.join(golden_dir, "circom_groth16.json")))
    v, pr = c["vk"], c["proof"]
    i3 = lambda p: tuple(int(x) for x in p)
    i32 = lambda p: tuple(tuple(int(x) for x in q) for q in p)
    vk = {"IC": [i3(p) for p in v["IC"]], "G1": {"Alpha": i3(v["vk_alfa_1"])},
          "G2": {"Beta": i32(v["vk_beta_2"]), "Gamma": i32(v["vk_gamma_2"]), "Delta": i32(v["vk_delta_2"])}}
    proof = {"PiA": i3(pr["pi_a"]), "PiB": i32(pr["pi_b"]), "PiC": i3(pr["pi_c"])}
    public = [int(x) for x in c["public"]]
    sigs = [public, [public[0] + 1], public, [public[0] + R], public]
    want = [groth16.VerifyProof(vk, proof, s) for s in sigs]
    assert want == [True, False, True, True, True]
    assert groth16.VerifyProofBatch(vk, [proof] * len(sigs), sigs) == want


def test_call_level_errors(gs):
    _lib, _, groth16 = gs
    inst = Instance(gs[1], 3, 2, seed=13)
    rc, ok, _ = batch(gs, inst.vk, inst.proofs, inst.pubs, n_ic=2)          # len(IC) < n_public + 1
    assert rc == -3 and ok == [7, 7, 7]
    rc, ok, _ = batch(gs, inst.vk, inst.proofs, inst.pubs, rho=[5, 0, 6])   # a rho equal to 0
    assert rc == -3 and ok == [7, 7, 7]
    rc, _, _ = batch(gs, inst.vk, [], [])                                   # no proofs
    assert rc == -3
    bad_range = dict(inst.vk, G1={"Alpha": (Q, 1, 1)})
    bad_inf = dict(inst.vk, G2=dict(inst.vk["G2"], Gamma=G2.zero3()))
    bad_g2 = dict(inst.vk, G2=dict(inst.vk["G2"], Delta=_twist_point_outside_g2()))
    for vk, code in ((bad_range, -4), (bad_inf, -3), (bad_g2, -3)):
        rc, ok, _ = batch(gs, vk, inst.proofs, inst.pubs)
        assert rc == code and ok == [7, 7, 7]
    assert single(gs, bad_range, inst.proofs[0], inst.pubs[0]) == -4        # the single call's codes for the same keys
    assert single(gs, bad_inf, inst.proofs[0], inst.pubs[0]) == -3
    with pytest.raises(ValueError):
        groth16.VerifyProofBatch(inst.vk, inst.proofs, inst.pubs, rho=[1, 2, 0])
