"""CPU: host logic of the Pinocchio setup / verify mirrors (SURVEY §8f rows 1-2: snark.go:98-251, 292-372) and of the
Groth16 VerifyProof mirror, run against an oracle-backed stand-in for the C ABI (tests/abi_standin.py).  What is
checked here is everything ABOVE the ABI: scalar derivation, batching order, struct layout, check order, error
behaviour.  The kernels underneath are covered by the -m gpu tests of the same mirrors."""
import json
import os
import shutil
import tempfile

import pytest

import abi_standin
import gocli
from oracle import ref_py as o

pytestmark = pytest.mark.slow
TOX = {"T": 0x1234567, "Ka": 0x1111, "Kb": 0x2222, "Kc": 0x3333, "Kbeta": 0x4444, "Kgamma": 0x5555, "RhoA": 0x6666,
       "RhoB": 0x7777}


def _lists(p):
    return [list(c) if isinstance(c, tuple) else c for c in p]


@pytest.fixture()
def flow(monkeypatch, golden_dir):
    abi_standin.install(monkeypatch)
    from gosnark_b200 import snark
    g = json.load(open(os.path.join(golden_dir, "gobin_x3x5.json")))
    cc = g["compiledcircuit"]
    r1 = cc["R1CS"]
    alphas, betas, gammas, _ = o.PF.r1cs_to_qap(r1["A"], r1["B"], r1["C"])
    return snark, g, cc, alphas, betas, gammas


def test_pinocchio_setup_equals_oracle_and_go_accepts_it(flow):
    snark, g, cc, alphas, betas, gammas = flow
    setup = snark.GenerateTrustedSetup(len(g["witness"]), cc, alphas, betas, gammas, toxic=TOX)
    opk, ovk = o.pinocchio_setup(cc["NVars"], cc["NPublic"], alphas, betas, gammas, TOX)
    for k in opk:
        assert setup["Pk"][k] == opk[k], k                      # Jacobian X,Y,Z identical, Z polynomial identical
    for k in ovk:
        assert setup["Vk"][k] == ovk[k], k
    assert setup["Toxic"]["RhoC"] == TOX["RhoA"] * TOX["RhoB"] % o.R
    w = [int(x) for x in g["witness"]]
    _, _, _, px = o.PF.combine_polynomials(w, alphas, betas, gammas)
    proof, _ = o.pinocchio_prove(cc["NVars"], cc["NPublic"], setup["Pk"], w, px)
    assert snark.VerifyProof(setup["Vk"], proof, [35])
    assert not snark.VerifyProof(setup["Vk"], proof, [34])
    d = tempfile.mkdtemp(prefix="pin_")                          # the reference's own verifier on the minted setup
    try:
        pk = setup["Pk"]
        js = {"Toxic": {k: None for k in setup["Toxic"]}, "G1T": [_lists(p) for p in pk["G1T"]], "G2T": None,
              "Pk": {k: ([_lists(p) for p in v] if k != "Z" else v) for k, v in pk.items() if k != "G1T"},
              "Vk": {k: ([_lists(p) for p in v] if k == "IC" else _lists(v)) for k, v in setup["Vk"].items()}}
        for name, obj in (("trustedsetup.json", js), ("proofs.json", {k: _lists(v) for k, v in proof.items()}),
                          ("compiledcircuit.json", cc), ("publicInputs.json", g["public"]),
                          ("privateInputs.json", g["private"])):
            json.dump(obj, open(os.path.join(d, name), "w"))
        out = gocli.run(d, "verify")
        assert "Proofs verified" in out and "❌" not in out, out
    finally:
        shutil.rmtree(d)


def test_pinocchio_verify_go_proof_check_order_and_messages(flow, capsys):
    snark, g, cc, *_ = flow
    st, pr = g["pinocchio_setup"], g["pinocchio_proofs"]
    t3 = lambda p: tuple(p)
    t2 = lambda p: tuple(tuple(c) for c in p)
    vk = {k: ([t3(p) for p in v] if k == "IC" else (t2(v) if isinstance(v[0], list) else t3(v))) for k, v in st["Vk"].items()}
    proof = {k: (t2(v) if k == "PiB" else t3(v)) for k, v in pr.items()}
    assert snark.VerifyProof(vk, proof, [int(x) for x in g["public"]], True)
    out = capsys.readouterr().out
    assert out.count("✓") == 5 and "❌" not in out
    assert [l[2:] for l in out.strip().splitlines()] == [l[2:] for l in g["pinocchio_verify_stdout"].strip().splitlines()[:5]]
    assert not snark.VerifyProof(vk, proof, [34], True)          # wrong public input: fails at the QAP check (4th)
    out = capsys.readouterr().out
    assert out.count("✓") == 3 and out.count("❌") == 1 and "QAP" in out.splitlines()[-1]
    bad = dict(proof, PiAp=o.BN.G1.double(proof["PiAp"]))         # broken knowledge commitment: first check
    assert not snark.VerifyProof(vk, bad, [35], True)
    out = capsys.readouterr().out
    assert out.count("✓") == 0 and out.count("❌") == 1
    with pytest.raises(IndexError):
        snark.VerifyProof(vk, proof, [35, 1, 2])


def test_groth16_verify_mirror_marshalling(monkeypatch, golden_dir):
    abi_standin.install(monkeypatch)
    from gosnark_b200 import groth16
    g = json.load(open(os.path.join(golden_dir, "gobin_mul.json")))
    vk, pr = g["groth16_setup"]["Vk"], g["groth16_proofs"]
    t3 = lambda p: tuple(p)
    t2 = lambda p: tuple(tuple(c) for c in p)
    vkd = {"IC": [t3(p) for p in vk["IC"]], "G1": {"Alpha": t3(vk["G1"]["Alpha"])},
           "G2": {k: t2(vk["G2"][k]) for k in ("Beta", "Gamma", "Delta")}}
    proof = {"PiA": t3(pr["PiA"]), "PiB": t2(pr["PiB"]), "PiC": t3(pr["PiC"])}
    assert groth16.VerifyProof(vkd, proof, [int(x) for x in g["public"]])
    assert not groth16.VerifyProof(vkd, proof, [int(g["public"][0]) + 1])
    with pytest.raises(Exception, match="len\\(IC\\)"):
        groth16.VerifyProof(vkd, proof, [1, 2, 3])


def test_verify_from_circom_files(monkeypatch, golden_dir, tmp_path, capsys):
    """externalVerif.VerifyFromCircom (circomVerifier.go:26-96; circomVerifier_test.go:9-13) over the snarkjs fixture."""
    abi_standin.install(monkeypatch)
    from gosnark_b200 import externalVerif
    c = json.load(open(os.path.join(golden_dir, "circom_groth16.json")))
    paths = {}
    for name, obj in (("verification_key.json", c["vk"]), ("proof.json", c["proof"]), ("public.json", c["public"])):
        paths[name] = str(tmp_path / name)
        json.dump(obj, open(paths[name], "w"))
    ok, err = externalVerif.VerifyFromCircom(paths["verification_key.json"], paths["proof.json"], paths["public.json"])
    assert ok and err is None
    out = capsys.readouterr().out
    assert "vk parsed:" in out and "proof parsed:" in out and "publicSignals parsed:" in out and "✓" in out
    json.dump([str(int(c["public"][0]) + 1)], open(paths["public.json"], "w"))
    ok, err = externalVerif.VerifyFromCircom(paths["verification_key.json"], paths["proof.json"], paths["public.json"])
    assert not ok and err is None
    ok, err = externalVerif.VerifyFromCircom(paths["verification_key.json"], str(tmp_path / "missing.json"), paths["public.json"])
    assert not ok and isinstance(err, OSError)
    json.dump(["12x"], open(paths["public.json"], "w"))
    ok, err = externalVerif.VerifyFromCircom(paths["verification_key.json"], paths["proof.json"], paths["public.json"])
    assert not ok and "error parsing px from pxString" in str(err)


@pytest.mark.parametrize("proto", ["groth16", "pinocchio"])
def test_cli_trustedsetup_files_feed_the_go_binary(monkeypatch, golden_dir, proto, capsys):
    """File-level interop in the other direction (cli/main.go:231-301, 407-453): OUR `trustedsetup` writes
    trustedsetup.json, the UNMODIFIED Go binary proves with it and verifies; our `verify` accepts the Go proof."""
    abi_standin.install(monkeypatch)
    from gosnark_b200 import cli
    gocli.seed_rand_fr(monkeypatch, 3)
    g = json.load(open(os.path.join(golden_dir, "gobin_x3x5.json")))
    d = tempfile.mkdtemp(prefix="clits_")
    cwd = os.getcwd()
    pre = ["groth16"] if proto == "groth16" else []
    try:
        for fname, key in (("compiledcircuit.json", "compiledcircuit"), ("privateInputs.json", "private"),
                           ("publicInputs.json", "public")):
            json.dump(g[key], open(os.path.join(d, fname), "w"))
        os.chdir(d)
        assert cli.main(pre + ["trustedsetup"] + (["wasm"] if proto == "pinocchio" else [])) == 0
        written = json.load(open("trustedsetup.json"))
        assert all(v is None for v in written["Toxic"].values())          # toxic waste is not written (main.go:273-277)
        out = gocli.run(d, *pre, "genproofs")
        assert os.path.exists("proofs.json"), out[-1000:]
        out = gocli.run(d, *pre, "verify")
        assert ("verification passed" in out) if proto == "groth16" else ("Proofs verified" in out and "❌" not in out), out
        capsys.readouterr()
        assert cli.main(pre + ["verify"]) == 0
        assert "Proofs verified" in capsys.readouterr().out
        if proto == "pinocchio":
            from gosnark_b200 import utils
            s = json.load(open("trustedsetupString.json"))
            assert utils.SetupFromString(s)["Vk"]["Vkb"] == tuple(written["Vk"]["Vkb"])
    finally:
        os.chdir(cwd)
        shutil.rmtree(d)
