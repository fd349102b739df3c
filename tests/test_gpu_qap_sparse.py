"""GPU parity tests for the sparse QAP front end (include/b200snark.h: b200_r1cs_load / b200_qap_px / b200_interpolate /
b200_qap_eval_at / b200_groth16_prove_witness) — the large-n form of r1csqap.R1CSToQAP + CombinePolynomials
(r1csqap/r1csqap.go:129-210) — against the oracle, the Go binary's goldens, and the dense GPU kernels."""
import json
import os
import random
import shutil
import tempfile

import numpy as np
import pytest

import gocli
from oracle import ref_py as o

pytestmark = pytest.mark.gpu
R = o.R


@pytest.fixture(scope="module")
def mods():
    from gosnark_b200 import _lib, r1csqap
    _lib.init()
    return r1csqap


def horner(c, x):
    acc = 0
    for v in reversed(c):
        acc = (acc * x + v) % R
    return acc


@pytest.mark.parametrize("n", [1, 2, 3, 7, 16, 21, 33, 100, 1000, 1024, 1500, 5000])
def test_interpolation_over_1_to_n(mods, n):
    """LagrangeInterpolation (r1csqap.go:150-158): the unique polynomial of degree < n through (j+1, v_j).  Equal to the
    oracle's coefficients for small n; checked by evaluation at every (sampled for large n) point beyond."""
    pf = mods.PolynomialField()
    rng = random.Random(n)
    v = [rng.randrange(R) for _ in range(n)]
    if n > 2:
        v[1] = 0                                   # zero and small values, like R1CS columns
        v[2] = 5
    c = pf.LagrangeInterpolation(v)
    assert len(c) == n
    if n <= 21:
        assert c == o.PF.lagrange_interpolation(v)
    pts = range(n) if n <= 1500 else rng.sample(range(n), 300)
    for j in pts:
        assert horner(c, j + 1) == v[j], (n, j)


def test_new_pol_zero_at_matches_oracle(mods):
    pf = mods.PolynomialField()
    for total, pos, h in ((4, 2, 7), (7, 7, R - 3), (21, 5, 1)):
        assert pf.NewPolZeroAt(pos, total, h) == o.PF.new_pol_zero_at(pos, total, h)


@pytest.mark.parametrize("n", [2049, 5000, 65536])
def test_zero_poly_large(mods, n):
    """Z = prod_{i=1..n}(x - i) (groth16.go:122-132) beyond the one-block kernel: monic, degree n, zero at 1..n, and
    the right value at a random point."""
    from gosnark_b200._lib import check, lib, limbs_to_ints, ptr
    z = np.zeros((n + 1, 4), dtype=np.uint64)
    check(lib().b200_zero_poly(n, ptr(z)))
    zc = limbs_to_ints(z)
    assert zc[n] == 1
    rng = random.Random(n)
    for x in rng.sample(range(1, n + 1), 40):
        assert horner(zc, x) == 0, x
    t = rng.randrange(R)
    exp = 1
    for i in range(1, n + 1):
        exp = exp * (t - i) % R
    assert horner(zc, t) == exp


@pytest.mark.parametrize("name", ["x3x5", "mul", "chain21"])
def test_sparse_combine_equals_go_binary_px(mods, golden_dir, name):
    """px, ax, bx, cx from (sparse R1CS, witness) == the Go binary's own px.json and the oracle's
    CombinePolynomials(w, R1CSToQAP(a, b, c)) (r1csqap.go:161-210)."""
    with open(os.path.join(golden_dir, f"gobin_{name}.json")) as f:
        g = json.load(f)
    cc = g["compiledcircuit"]
    a, b, c = cc["R1CS"]["A"], cc["R1CS"]["B"], cc["R1CS"]["C"]
    sp = mods.SparseR1CS(len(a), len(a[0]), (a, b, c))
    ax, bx, cx, px = sp.CombinePolynomials(g["witness"])
    assert px == [x % R for x in g["px"]]
    alphas, betas, gammas, _ = o.PF.r1cs_to_qap(a, b, c)
    eax, ebx, ecx, epx = o.PF.combine_polynomials(g["witness"], alphas, betas, gammas)
    assert (ax, bx, cx, px) == (eax, ebx, ecx, epx)
    # Eval(alphas[i], tau) for every signal, without the dense polynomials (groth16.go:164-205)
    tau = 0x1234567 + len(a)
    at, bt, ct, zt = sp.EvalAt(tau)
    from gosnark_b200._lib import limbs_to_ints
    assert limbs_to_ints(at) == [o.PF.eval(p, tau) for p in alphas]
    assert limbs_to_ints(bt) == [o.PF.eval(p, tau) for p in betas]
    assert limbs_to_ints(ct) == [o.PF.eval(p, tau) for p in gammas]
    exp_zt = 1
    for i in range(1, len(a[0]) - 1):
        exp_zt = exp_zt * (tau - i) % R
    assert zt == exp_zt
    sp.free()


@pytest.mark.parametrize("n", [5, 64, 1000, 1024])
def test_sparse_combine_equals_dense_kernels(mods, n):
    """Same result as the dense GPU path b200_r1cs_to_qap + b200_combine_polynomials on the synthetic chain circuit
    (different algorithms: per-column Lagrange basis vs Newton + subproduct tree)."""
    from gosnark_b200.synthetic import SyntheticCircuit
    circ = SyntheticCircuit(n)
    pf = mods.PolynomialField()
    a, b, c = circ.dense()
    alphas, betas, gammas, _ = pf.R1CSToQAP(a, b, c)
    exp = pf.CombinePolynomials(circ.witness, alphas, betas, gammas)
    sp = mods.SparseR1CS(n, n + 2, circ.csr)
    got = sp.CombinePolynomials(circ.witness)
    assert tuple(got) == tuple(exp)
    # a satisfied R1CS: px vanishes on 1..n  (K7: px == hx * Z, remainder 0; groth16_test.go:77-86)
    for x in range(1, min(n, 40) + 1):
        assert horner(got[3], x) == 0
    sp.free()


def test_r1cs_load_argument_errors(mods):
    from gosnark_b200 import _lib
    rp = np.array([0, 1, 2], dtype=np.uint32)
    with pytest.raises(_lib.B200Error):                                   # column index out of range
        mods.SparseR1CS(2, 3, [(rp, np.array([0, 3], dtype=np.uint32), [1, 1])] * 3)
    with pytest.raises(_lib.B200Error):                                   # coefficient >= r
        bad = np.zeros((2, 4), dtype=np.uint64)
        bad[:] = np.uint64(0xFFFFFFFFFFFFFFFF)
        mods.SparseR1CS(2, 3, [(rp, np.array([0, 1], dtype=np.uint32), bad)] * 3)
    sp = mods.SparseR1CS(2, 3, [(rp, np.array([0, 1], dtype=np.uint32), [1, 1])] * 3)
    with pytest.raises(_lib.B200Error):                                   # witness length != m
        sp.CombinePolynomials([1, 2])
    with pytest.raises(_lib.B200Error):                                   # tau inside the domain {1..n}
        sp.EvalAt(2)
    sp.free()


def go_groth16_verify(vk_json, proof_json, public):
    d = tempfile.mkdtemp(prefix="gsv_")
    try:
        # the prebuilt binary also opens compiledcircuit.json (unused by VerifyProof): an empty object will do
        for fname, obj in (("trustedsetup.json", {"Vk": vk_json}), ("publicInputs.json", public), ("proofs.json", proof_json),
                           ("compiledcircuit.json", {})):
            with open(os.path.join(d, fname), "w") as f:
                json.dump(obj, f)
        return gocli.run(d, "groth16", "verify")
    finally:
        shutil.rmtree(d)


@pytest.mark.parametrize("logn", [6, 10, 16])
def test_real_crs_witness_to_verified_proof(mods, logn):
    """Config 2 end to end with a REAL CRS (groth16.go:94-222 semantics, toxic values seeded): witness -> px on the device
    -> proof; the proof equals the one the reference's GenerateProofs would return (known discrete logs, from the QAP
    identity, independent of the GPU's px / h), verifies under the real Vk on the GPU (groth16.go:281-305) and — the
    reference's own Go code — under `go-snark-cli groth16 verify`; a wrong public input is rejected."""
    import ctypes
    from gosnark_b200._lib import check, ints_to_limbs, lib, limbs_to_ints, ptr
    from gosnark_b200.bn128 import _unflatten_g1, _unflatten_g2
    from gosnark_b200.synthetic import CircuitGroth16
    syn = CircuitGroth16(logn)
    pk = syn.load_pk()
    rr, ss = ints_to_limbs([syn.r]), ints_to_limbs([syn.s])
    outs = []
    for mode in ("px", "witness"):
        pa, pb, pc = np.zeros(12, dtype=np.uint64), np.zeros(24, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
        if mode == "px":
            check(lib().b200_groth16_prove(pk, ptr(syn.w), syn.m, ptr(syn.px), syn.px.shape[0], ptr(rr), ptr(ss), ptr(pa),
                                           ptr(pb), ptr(pc)))
        else:
            check(lib().b200_groth16_prove_witness(pk, syn.r1cs.handle, ptr(syn.w), syn.m, ptr(rr), ptr(ss), ptr(pa), ptr(pb),
                                                   ptr(pc)))
        outs.append((pa, pb, pc))
    # same group elements from both entry points (the Jacobian representatives may differ from run to run: the counting
    # sort scatters with atomics, so the order of additions inside a bucket is not fixed)
    assert o.BN.G1.affine(_unflatten_g1(outs[0][0])[0]) == o.BN.G1.affine(_unflatten_g1(outs[1][0])[0])
    assert o.BN.G2.affine(_unflatten_g2(outs[0][1])[0]) == o.BN.G2.affine(_unflatten_g2(outs[1][1])[0])
    assert o.BN.G1.affine(_unflatten_g1(outs[0][2])[0]) == o.BN.G1.affine(_unflatten_g1(outs[1][2])[0])
    pa, pb, pc = outs[1]
    a, b, c = syn.expected_dlogs()
    A, B, C = _unflatten_g1(pa)[0], _unflatten_g2(pb)[0], _unflatten_g1(pc)[0]
    assert o.BN.G1.affine(A) == o.BN.G1.affine(o.BN.G1.mul_scalar(o.BN.G1.G, a))
    assert o.BN.G2.affine(B) == o.BN.G2.affine(o.BN.G2.mul_scalar(o.BN.G2.G, b))
    assert o.BN.G1.affine(C) == o.BN.G1.affine(o.BN.G1.mul_scalar(o.BN.G1.G, c))
    assert syn.verify(pa, pb, pc)
    ok = ctypes.c_int(1)
    wrong = ints_to_limbs([(syn.circuit.public_signals[0] + 1) % R])
    check(lib().b200_groth16_verify(ptr(syn.ic), 2, ptr(syn.alpha1), ptr(syn.beta2), ptr(syn.gamma2), ptr(syn.delta2), ptr(pa),
                                    ptr(pb), ptr(pc), ptr(wrong), 1, ctypes.byref(ok)))
    assert ok.value == 0
    vk_json = {"IC": [list(p) for p in _unflatten_g1(syn.ic)], "G1": {"Alpha": list(_unflatten_g1(syn.alpha1)[0])},
               "G2": {k: [list(cc) for cc in _unflatten_g2(v)[0]] for k, v in
                      (("Beta", syn.beta2), ("Gamma", syn.gamma2), ("Delta", syn.delta2))}}
    out = go_groth16_verify(vk_json, {"PiA": list(A), "PiB": [list(cc) for cc in B], "PiC": list(C)}, syn.circuit.public_signals)
    assert "Proofs verified" in out and "not verified" not in out, out
    check(lib().b200_pk_free(pk))
    syn.r1cs.free()
