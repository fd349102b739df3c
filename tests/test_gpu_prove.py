"""GPU parity tests for the prove paths through the C ABI:
  snark.GenerateProofs   (snark.go:254-289)  — bit-exact (affine) vs the Go binary's proofs.json
  groth16.GenerateProofs (groth16.go:225-278) — vs the oracle with injected r,s, verified by the
                                               oracle's VerifyProof and by real Go code (tests/gocli.py)
"""
import json
import os
import random
import shutil
import tempfile

import pytest

import gocli
from oracle import ref_py as o

pytestmark = pytest.mark.gpu
G1, G2 = o.BN.G1, o.BN.G2


@pytest.fixture(scope="module")
def mods():
    from gosnark_b200 import _lib, groth16, snark
    _lib.init()
    return groth16, snark


def load(golden_dir, name):
    with open(os.path.join(golden_dir, name)) as f:
        return json.load(f)


def t3(p):
    return tuple(p)


def g2t(p):
    return tuple(tuple(c) for c in p)


def affeq(group, ours, ref):
    """H1: parity on affine coordinates (our Jacobian representative differs)."""
    return group.affine(ours) == group.affine(ref)


def pinocchio_pk(setup):
    pk = {k: [t3(p) for p in setup["Pk"][k]] for k in ("A", "C", "Kp", "Ap", "Bp", "Cp")}
    pk["B"] = [g2t(p) for p in setup["Pk"]["B"]]
    pk["Z"] = setup["Pk"]["Z"]
    pk["G1T"] = [t3(p) for p in setup["G1T"]]
    return pk


def groth_pk(setup):
    pk = setup["Pk"]
    return {"Z": pk["Z"], "BACDelta": [t3(p) for p in pk["BACDelta"]],
            "PowersTauDelta": [t3(p) for p in pk["PowersTauDelta"]],
            "G1": {"Alpha": t3(pk["G1"]["Alpha"]), "Beta": t3(pk["G1"]["Beta"]), "Delta": t3(pk["G1"]["Delta"]),
                   "At": [t3(p) for p in pk["G1"]["At"]], "BACGamma": [t3(p) for p in pk["G1"]["BACGamma"]]},
            "G2": {"Beta": g2t(pk["G2"]["Beta"]), "Delta": g2t(pk["G2"]["Delta"]),
                   "BACGamma": [g2t(p) for p in pk["G2"]["BACGamma"]]}}


def groth_vk(setup):
    vk = setup["Vk"]
    return {"IC": [t3(p) for p in vk["IC"]], "G1": {"Alpha": t3(vk["G1"]["Alpha"])},
            "G2": {k: g2t(vk["G2"][k]) for k in ("Beta", "Gamma", "Delta")}}


@pytest.mark.parametrize("name", ["x3x5", "mul", "chain21"])
def test_pinocchio_matches_go_binary(mods, golden_dir, name):
    """K5: the GPU proof equals the reference Go binary's proofs.json on affine
    coordinates for all 8 proof elements."""
    _, snark = mods
    g = load(golden_dir, f"gobin_{name}.json")
    cc = g["compiledcircuit"]
    proof = snark.GenerateProofs(cc, pinocchio_pk(g["pinocchio_setup"]), g["witness"], g["px"])
    ref = g["pinocchio_proofs"]
    for k in ("PiA", "PiAp", "PiBp", "PiC", "PiCp", "PiH", "PiKp"):
        assert affeq(G1, proof[k], t3(ref[k])), k
    assert affeq(G2, proof["PiB"], g2t(ref["PiB"]))


def go_verify(g, proof_json, cmd):
    """Have the reference's real Go code verify our proof (cli/main.go verify commands)."""
    d = tempfile.mkdtemp(prefix="gsv_")
    try:
        key = "groth16_setup" if cmd[0] == "groth16" else "pinocchio_setup"
        for fname, obj in (("trustedsetup.json", g[key]), ("compiledcircuit.json", g["compiledcircuit"]),
                           ("publicInputs.json", g["public"]), ("proofs.json", proof_json)):
            with open(os.path.join(d, fname), "w") as f:
                json.dump(obj, f)
        return gocli.run(d, *cmd)
    finally:
        shutil.rmtree(d)


@pytest.mark.parametrize("name", ["x3x5", "chain21"])
def test_groth16_vs_oracle_and_verifiers(mods, golden_dir, name):
    groth16, _ = mods
    g = load(golden_dir, f"gobin_{name}.json")
    cc = g["compiledcircuit"]
    pk = groth_pk(g["groth16_setup"])
    rng = random.Random(42)
    r, s = rng.randrange(1 << 240), rng.randrange(1 << 240)      # Fq.Rand range (H2)
    proof = groth16.GenerateProofs(cc, pk, g["witness"], g["px"], r=r, s=s)
    ref, _ = o.groth16_prove(cc["NVars"], cc["NPublic"], pk, g["witness"], g["px"], r, s)
    assert affeq(G1, proof["PiA"], ref["PiA"])
    assert affeq(G2, proof["PiB"], ref["PiB"])
    assert affeq(G1, proof["PiC"], ref["PiC"])
    # reference semantics: verifies for the right public input, not for a wrong one (groth16_test.go:100,106)
    if name == "x3x5":
        vk = groth_vk(g["groth16_setup"])
        assert o.groth16_verify(vk, proof, g["public"])
        assert not o.groth16_verify(vk, proof, [g["public"][0] - 1])
    out = go_verify(g, {"PiA": list(proof["PiA"]), "PiB": [list(c) for c in proof["PiB"]], "PiC": list(proof["PiC"])},
                    ["groth16", "verify"])
    assert "verification passed" in out, out
    # fresh randomness path (like the reference): still a valid proof, different every time
    p1 = groth16.GenerateProofs(cc, pk, g["witness"], g["px"])
    p2 = groth16.GenerateProofs(cc, pk, g["witness"], g["px"])
    assert G1.affine(p1["PiA"]) != G1.affine(p2["PiA"])


def test_pinocchio_go_binary_verifies_our_proof(mods, golden_dir):
    _, snark = mods
    g = load(golden_dir, "gobin_x3x5.json")
    proof = snark.GenerateProofs(g["compiledcircuit"], pinocchio_pk(g["pinocchio_setup"]), g["witness"], g["px"])
    pj = {k: (list(v) if k != "PiB" else [list(c) for c in v]) for k, v in proof.items()}
    out = go_verify(g, pj, ["verify"])
    assert "Proofs verified" in out and "❌" not in out, out


def test_prove_argument_errors(mods, golden_dir):
    from gosnark_b200 import _lib
    groth16, _ = mods
    g = load(golden_dir, "gobin_mul.json")
    cc = g["compiledcircuit"]
    pk = groth_pk(g["groth16_setup"])
    with pytest.raises(_lib.B200Error):                      # wrong witness length
        groth16.GenerateProofs(cc, pk, g["witness"][:-1], g["px"], r=1, s=1)
    with pytest.raises(_lib.B200Error):                      # len(hx) > len(PowersTauDelta): reference panics
        groth16.GenerateProofs(cc, pk, g["witness"], g["px"] + [0] * 8, r=1, s=1)
    for rr, ss in ((o.R - 1, o.R - 2), (1, o.R - 1), ((1 << 128) + 5, (1 << 64) - 1)):    # full-range / edge blinding scalars
        got = groth16.GenerateProofs(cc, pk, g["witness"], g["px"], r=rr, s=ss)
        exp, _ = o.groth16_prove(cc["NVars"], cc["NPublic"], pk, g["witness"], g["px"], rr, ss)
        assert affeq(G1, got["PiA"], exp["PiA"]) and affeq(G2, got["PiB"], exp["PiB"]) and affeq(G1, got["PiC"], exp["PiC"])
    ok = groth16.GenerateProofs(cc, pk, g["witness"], g["px"], r=0, s=0)       # r = s = 0: no blinding
    ref, _ = o.groth16_prove(cc["NVars"], cc["NPublic"], pk, g["witness"], g["px"], 0, 0)
    assert affeq(G1, ok["PiC"], ref["PiC"]) and affeq(G1, ok["PiA"], ref["PiA"])


def test_proofs_depend_only_on_the_quotient_of_px(mods, golden_dir):
    """hx = DivisorPolynomial(px, Z) keeps the quotient and drops the remainder (r1csqap.go:213-216), and the quotient is
    fixed by the top len(px) - len(Z) + 1 coefficients of px — the only ones the host-pointer entry points stage over
    PCIe (csrc/prove_host.cuh).  A px whose LOW coefficients are garbage (not a multiple of Z any more) must therefore
    give the same proof, on the device and in the oracle's restatement of the reference's long division."""
    groth16, snark = mods
    g = load(golden_dir, "gobin_chain21.json")
    cc = g["compiledcircuit"]
    px = list(g["px"])
    nq = len(px) - len(g["groth16_setup"]["Pk"]["Z"]) + 1
    rng = random.Random(7)
    bad = [rng.randrange(o.R) for _ in range(len(px) - nq)] + px[len(px) - nq:]
    assert bad != px and len(bad) == len(px)
    pk = groth_pk(g["groth16_setup"])
    got = groth16.GenerateProofs(cc, pk, g["witness"], bad, r=11, s=13)
    for ref_px in (px, bad):
        exp, _ = o.groth16_prove(cc["NVars"], cc["NPublic"], pk, g["witness"], ref_px, 11, 13)
        assert affeq(G1, got["PiA"], exp["PiA"]) and affeq(G2, got["PiB"], exp["PiB"]) and affeq(G1, got["PiC"], exp["PiC"])
    ppk = pinocchio_pk(g["pinocchio_setup"])
    nq_p = len(px) - len(ppk["Z"]) + 1
    bad_p = [rng.randrange(o.R) for _ in range(len(px) - nq_p)] + px[len(px) - nq_p:]
    proof = snark.GenerateProofs(cc, ppk, g["witness"], bad_p)
    assert affeq(G1, proof["PiH"], t3(g["pinocchio_proofs"]["PiH"]))


@pytest.mark.timeout(600)
@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("logn", [12, 16])
def test_groth16_prove_named_sizes_known_dlogs(mods, logn, mode):
    """BASELINE config 2 (2^16 constraints, 1 GPU) through the host-pointer C ABI b200_groth16_prove, with the proving
    key built for the batched-affine kernels (mode 1) and for the XYZZ kernels (mode 2): every proof element equals
    (known scalar)*G — the exact output of groth16.GenerateProofs (groth16.go:225-278) on the same key, witness, px, r, s."""
    import numpy as np
    from gosnark_b200 import _lib
    from gosnark_b200._lib import check, ints_to_limbs, lib, ptr
    from gosnark_b200.bn128 import _unflatten_g1, _unflatten_g2
    from gosnark_b200.synthetic import SyntheticGroth16
    syn = SyntheticGroth16(logn)
    check(lib().b200_config(_lib.CFG_ACC_MODE, mode))
    try:
        pk = syn.load_pk()
    finally:
        check(lib().b200_config(_lib.CFG_ACC_MODE, _lib.ACC_AUTO))
    pa, pb, pc = np.zeros(12, dtype=np.uint64), np.zeros(24, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
    rr, ss = ints_to_limbs([syn.r]), ints_to_limbs([syn.s])
    for _ in range(2):      # twice: scratch reuse across proofs
        check(lib().b200_groth16_prove(pk, ptr(syn.w), syn.m, ptr(syn.px), syn.px.shape[0], ptr(rr), ptr(ss), ptr(pa), ptr(pb),
                                       ptr(pc)))
        ea, eb, ec = syn.expected_dlogs()
        assert G1.affine(_unflatten_g1(pa)[0]) == G1.affine(G1.mul_scalar(G1.G, ea))
        assert G2.affine(_unflatten_g2(pb)[0]) == G2.affine(G2.mul_scalar(G2.G, eb))
        assert G1.affine(_unflatten_g1(pc)[0]) == G1.affine(G1.mul_scalar(G1.G, ec))
    check(lib().b200_pk_free(pk))


@pytest.mark.timeout(600)
@pytest.mark.parametrize("logn", [10, 14])
def test_two_proofs_in_flight_on_two_contexts(mods, logn):
    """B200_CFG_PK_CONTEXT: two proving keys loaded under contexts 0 and 1 prove DIFFERENT statements (different r, s)
    interleaved on two streams with no host synchronisation in between (what bench.py's `proofs_in_flight` does); every
    proof of every round equals its known-discrete-log expectation — groth16.GenerateProofs (groth16.go:225-278) on the
    same key, witness, px, r, s."""
    import numpy as np
    import torch
    from gosnark_b200 import _lib
    from gosnark_b200._lib import check, ints_to_limbs, lib, ptr
    from gosnark_b200.bn128 import _unflatten_g1, _unflatten_g2
    from gosnark_b200.synthetic import SyntheticGroth16
    syn = SyntheticGroth16(logn)
    L = lib()
    pks = []
    try:
        for k in range(2):
            check(L.b200_config(_lib.CFG_PK_CONTEXT, k))
            pks.append(syn.load_pk())
    finally:
        check(L.b200_config(_lib.CFG_PK_CONTEXT, 0))
    d_w = torch.from_numpy(syn.w.view(np.int64)).cuda()
    d_px = torch.from_numpy(syn.px.view(np.int64)).cuda()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    rounds = 4
    outs = [[torch.zeros(48, dtype=torch.int64, device="cuda") for _ in range(rounds)] for _ in range(2)]
    rs = [[(syn.r + 17 * (2 * j + k)) % o.R, (syn.s + 29 * (2 * j + k)) % o.R] for j in range(rounds) for k in range(2)]
    torch.cuda.synchronize()
    for j in range(rounds):
        for k in range(2):
            r_, s_ = rs[2 * j + k]
            rr, ss = ints_to_limbs([r_]), ints_to_limbs([s_])
            check(L.b200_groth16_prove_device(pks[k], d_w.data_ptr(), syn.m, d_px.data_ptr(), syn.px.shape[0], ptr(rr), ptr(ss),
                                              outs[k][j].data_ptr(), streams[k].cuda_stream))
    torch.cuda.synchronize()
    for j in range(rounds):
        for k in range(2):
            r_, s_ = rs[2 * j + k]
            ea, eb, ec = syn.expected_dlogs(r_, s_)
            out = outs[k][j].cpu().numpy().view(np.uint64)
            pa, pc = _unflatten_g1(out[:24])
            pb = _unflatten_g2(out[24:])[0]
            assert G1.affine(pa) == G1.affine(G1.mul_scalar(G1.G, ea)), (j, k)
            assert G2.affine(pb) == G2.affine(G2.mul_scalar(G2.G, eb)), (j, k)
            assert G1.affine(pc) == G1.affine(G1.mul_scalar(G1.G, ec)), (j, k)
    for pk in pks:
        check(L.b200_pk_free(pk))


@pytest.mark.timeout(600)
def test_two_host_threads_prove_on_two_contexts(mods):
    """The host-pointer entry point b200_groth16_prove from two threads, thread k on the context-k key: a call enqueues
    under the library mutex and waits for its proof with the mutex released, so the two proofs are in flight together;
    every proof equals the known-discrete-log expectation for its own (r, s)."""
    import threading
    import numpy as np
    from gosnark_b200 import _lib
    from gosnark_b200._lib import check, ints_to_limbs, lib, ptr
    from gosnark_b200.bn128 import _unflatten_g1, _unflatten_g2
    from gosnark_b200.synthetic import SyntheticGroth16
    syn = SyntheticGroth16(13)
    L = lib()
    pks = []
    try:
        for k in range(2):
            check(L.b200_config(_lib.CFG_PK_CONTEXT, k))
            pks.append(syn.load_pk())
    finally:
        check(L.b200_config(_lib.CFG_PK_CONTEXT, 0))
    rounds = 5
    results, errs = {}, []

    def worker(k):
        try:
            for j in range(rounds):
                r_, s_ = (syn.r + 101 * (2 * j + k)) % o.R, (syn.s + 103 * (2 * j + k)) % o.R
                pa, pb, pc = np.zeros(12, dtype=np.uint64), np.zeros(24, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
                check(L.b200_groth16_prove(pks[k], ptr(syn.w), syn.m, ptr(syn.px), syn.px.shape[0], ptr(ints_to_limbs([r_])),
                                           ptr(ints_to_limbs([s_])), ptr(pa), ptr(pb), ptr(pc)))
                results[(k, j)] = (r_, s_, pa, pb, pc)
        except Exception as e:
            errs.append(e)

    ths = [threading.Thread(target=worker, args=(k,)) for k in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    assert len(results) == 2 * rounds
    for (k, j), (r_, s_, pa, pb, pc) in results.items():
        ea, eb, ec = syn.expected_dlogs(r_, s_)
        assert G1.affine(_unflatten_g1(pa)[0]) == G1.affine(G1.mul_scalar(G1.G, ea)), (k, j)
        assert G2.affine(_unflatten_g2(pb)[0]) == G2.affine(G2.mul_scalar(G2.G, eb)), (k, j)
        assert G1.affine(_unflatten_g1(pc)[0]) == G1.affine(G1.mul_scalar(G1.G, ec)), (k, j)
    for pk in pks:
        check(L.b200_pk_free(pk))
