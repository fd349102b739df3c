"""GPU: the format / tooling rows (SURVEY §8f row 4) end to end on the device — the same mirrors that
tests/test_snark_host_logic.py and tests/test_utils_parsers.py exercise on the CPU, here over the real library."""
import json
import os
import shutil
import tempfile

import pytest

import gocli
from oracle import ref_py as o
from test_utils_parsers import K5, K5_PIB

pytestmark = pytest.mark.gpu
G1, G2 = o.BN.G1, o.BN.G2


@pytest.fixture(scope="module", autouse=True)
def _init():
    from gosnark_b200 import _lib
    _lib.init()


def test_wasm_string_fixture_gives_the_k5_proof(golden_dir):
    """wasm/index.js:2-8 string-form circuit / setup / px -> snark.GenerateProofs on the GPU == the Go binary's proof."""
    from gosnark_b200 import snark, utils
    wasm = json.load(open(os.path.join(golden_dir, "wasm_index_strings.json")))
    circuit = utils.CircuitFromString(wasm["circuit"])
    setup = utils.SetupFromString(wasm["setup"])
    px = utils.ArrayStringToBigInt(wasm["px"])
    proof = snark.GenerateProofs(circuit, setup["Pk"], [1, 35, 3, 9, 27, 30, 35, 1], px)
    for k, v in K5.items():
        assert G1.affine(proof[k])[:2] == v, k
    assert G2.affine(proof["PiB"])[:2] == K5_PIB
    s = utils.ProofToString(proof)
    assert utils.ProofFromString(s) == proof and utils.ProofFromHex(utils.ProofToHex(proof)) == proof


def test_verify_from_circom_files(golden_dir, tmp_path):
    """externalVerif/circomVerifier_test.go:9-13."""
    from gosnark_b200 import externalVerif
    c = json.load(open(os.path.join(golden_dir, "circom_groth16.json")))
    paths = {}
    for name, obj in (("verification_key.json", c["vk"]), ("proof.json", c["proof"]), ("public.json", c["public"])):
        paths[name] = str(tmp_path / name)
        json.dump(obj, open(paths[name], "w"))
    ok, err = externalVerif.VerifyFromCircom(paths["verification_key.json"], paths["proof.json"], paths["public.json"])
    assert ok and err is None
    json.dump([str(int(c["public"][0]) + 1)], open(paths["public.json"], "w"))
    ok, err = externalVerif.VerifyFromCircom(paths["verification_key.json"], paths["proof.json"], paths["public.json"])
    assert not ok and err is None


@pytest.mark.parametrize("proto", ["groth16", "pinocchio"])
def test_cli_trustedsetup_prove_verify_with_go_in_the_loop(golden_dir, proto, capsys, monkeypatch):
    """Our `trustedsetup` (GPU-minted CRS) -> Go `genproofs` + `verify` accept it -> our `genproofs` overwrites
    proofs.json -> Go `verify` and our `verify` accept that too (cli/main.go:231-549)."""
    from gosnark_b200 import cli
    gocli.seed_rand_fr(monkeypatch, 2)
    g = json.load(open(os.path.join(golden_dir, "gobin_x3x5.json")))
    d = tempfile.mkdtemp(prefix="clizz_")
    cwd = os.getcwd()
    pre = ["groth16"] if proto == "groth16" else []
    ok_text = (lambda out: "verification passed" in out) if proto == "groth16" else \
        (lambda out: "Proofs verified" in out and "❌" not in out)
    try:
        for fname, key in (("compiledcircuit.json", "compiledcircuit"), ("privateInputs.json", "private"),
                           ("publicInputs.json", "public")):
            json.dump(g[key], open(os.path.join(d, fname), "w"))
        os.chdir(d)
        assert cli.main(pre + ["trustedsetup"]) == 0
        out = gocli.run(d, *pre, "genproofs")
        assert os.path.exists("proofs.json"), out[-800:]
        out = gocli.run(d, *pre, "verify")
        assert ok_text(out), out
        capsys.readouterr()
        assert cli.main(pre + ["verify"]) == 0                       # Go's proof, our verifier
        assert "Proofs verified" in capsys.readouterr().out
        assert cli.main(pre + ["genproofs"]) == 0                    # our proof under our setup
        out = gocli.run(d, *pre, "verify")
        assert ok_text(out), out
        capsys.readouterr()
        assert cli.main(pre + ["verify"]) == 0
        assert "Proofs verified" in capsys.readouterr().out
    finally:
        os.chdir(cwd)
        shutil.rmtree(d)
