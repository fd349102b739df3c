"""GPU: file-level interoperability with the reference's CLI (SURVEY §8f row 4): our prove commands read the
files `go-snark-cli compile` / `trustedsetup` wrote (tests/golden fixtures), write proofs.json, and the
UNMODIFIED Go binary's verify commands accept it."""
import json
import os
import shutil
import tempfile

import pytest

import gocli

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,proto", [("x3x5", "groth16"), ("chain21", "groth16"), ("x3x5", "pinocchio")])
def test_go_cli_verifies_files_we_write(golden_dir, name, proto, monkeypatch):
    from gosnark_b200 import cli
    gocli.seed_rand_fr(monkeypatch, 1)
    g = json.load(open(os.path.join(golden_dir, f"gobin_{name}.json")))
    d = tempfile.mkdtemp(prefix="clif_")
    cwd = os.getcwd()
    try:
        for fname, obj in (("compiledcircuit.json", g["compiledcircuit"]), ("privateInputs.json", g["private"]),
                           ("publicInputs.json", g["public"]),
                           ("trustedsetup.json", g["groth16_setup" if proto == "groth16" else "pinocchio_setup"])):
            with open(os.path.join(d, fname), "w") as f:
                json.dump(obj, f)
        os.chdir(d)
        assert cli.main(["groth16", "genproofs"] if proto == "groth16" else ["genproofs"]) == 0
        os.chdir(cwd)
        out = gocli.run(d, *(["groth16", "verify"] if proto == "groth16" else ["verify"]))
        assert ("verification passed" in out) if proto == "groth16" else ("Proofs verified" in out and "❌" not in out), out
    finally:
        os.chdir(cwd)
        shutil.rmtree(d)


@pytest.mark.parametrize("name", ["x3x5", "mul", "chain21"])
def test_our_verify_accepts_go_proofs(golden_dir, name, capsys):
    """The other direction: `groth16 verify` on the GPU accepts the proofs.json the Go binary wrote
    (cli/main.go:520-549) and rejects it for a different public input."""
    from gosnark_b200 import cli
    g = json.load(open(os.path.join(golden_dir, f"gobin_{name}.json")))
    d = tempfile.mkdtemp(prefix="cliv_")
    cwd = os.getcwd()
    try:
        for fname, obj in (("proofs.json", g["groth16_proofs"]), ("trustedsetup.json", g["groth16_setup"]),
                           ("publicInputs.json", g["public"])):
            with open(os.path.join(d, fname), "w") as f:
                json.dump(obj, f)
        os.chdir(d)
        assert cli.main(["groth16", "verify"]) == 0
        assert "Proofs verified" in capsys.readouterr().out
        with open("publicInputs.json", "w") as f:
            json.dump([int(g["public"][0]) + 1] + list(g["public"][1:]), f)
        assert cli.main(["groth16", "verify"]) == 0
        assert "ERROR: proofs not verified" in capsys.readouterr().out
    finally:
        os.chdir(cwd)
        shutil.rmtree(d)
