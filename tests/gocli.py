"""Runs of the reference's prebuilt Go CLI (go-snark-cli), replayed from tests/golden/gocli_runs.json.

The tests that have the reference's own Go code prove with or verify our files call `run(d, *args)`.  A run is keyed by
its arguments and by the JSON input files the CLI reads from `d`, with every curve point in them taken to affine form (the
Jacobian representative our library returns depends on the order of additions inside a bucket).  The replay writes the
files the Go binary wrote and returns its output; input files that differ from the ones the binary was run on have no
recorded run, and the test fails.

GOSNARK_GOCLI=<path to go-snark-cli> runs that binary instead and records each run into the file named by
GOSNARK_GOCLI_RECORD (default: the golden file), e.g. `GOSNARK_GOCLI=... python -m pytest tests -k "go_"`.
"""
import hashlib
import json
import os
import subprocess

from oracle import ref_py as o

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gocli_runs.json")
READS = ("compiledcircuit.json", "trustedsetup.json", "proofs.json", "publicInputs.json", "privateInputs.json")
_CURVES = ((o.BN.G1, 3), (o.BN.G2, o.BN.twist_coef_b))


def _point(v):
    """v as an affine point when it is a Jacobian point [x, y, z] of G1 or G2 (y^2 = x^3 + b z^6), else None."""
    if len(v) != 3:
        return None
    try:
        if all(isinstance(c, (int, str)) for c in v):
            G, b = _CURVES[0]
            p = tuple(int(c) % o.Q for c in v)
        elif all(isinstance(c, list) and len(c) == 2 for c in v):
            G, b = _CURVES[1]
            p = tuple((int(c[0]) % o.Q, int(c[1]) % o.Q) for c in v)
        else:
            return None
    except (TypeError, ValueError):
        return None
    F = G.F
    x, y, z = p
    z2 = F.square(z)
    if not F.equal(F.square(y), F.add(F.mul(F.square(x), x), F.mul(b, F.mul(F.square(z2), z2)))):
        return None
    return {"affine": G.affine(p)}


def _canon(v):
    if isinstance(v, dict):
        return {k: _canon(x) for k, x in v.items()}
    if isinstance(v, list):
        p = _point(v)
        return p if p is not None else [_canon(x) for x in v]
    return v


def _key(d, args):
    files = {}
    for name in READS:
        path = os.path.join(d, name)
        if os.path.exists(path):
            with open(path) as f:
                files[name] = _canon(json.load(f))
    return hashlib.sha256(json.dumps([list(args), files], sort_keys=True).encode()).hexdigest()


def _snapshot(d):
    out = {}
    for name in os.listdir(d):
        path = os.path.join(d, name)
        if os.path.isfile(path) and name.endswith(".json"):
            with open(path) as f:
                out[name] = f.read()
    return out


def seed_rand_fr(monkeypatch, seed):
    """Draw the Fq.Rand values of our CLI (proof blinding, toxic waste) from a seeded generator, so that the files it writes
    are the same from run to run."""
    import random

    from gosnark_b200 import groth16
    rng = random.Random(seed)
    monkeypatch.setattr(groth16, "rand_fr", lambda: rng.randrange(1 << 240) % o.R)


def run(d, *args):
    """stdout + stderr of `go-snark-cli *args` run in directory d; the files it wrote appear in d."""
    key = _key(d, args)
    binary = os.environ.get("GOSNARK_GOCLI")
    if binary:
        before = _snapshot(d)
        p = subprocess.run([os.path.abspath(binary), *args], cwd=d, capture_output=True, text=True, timeout=300)
        wrote = {k: v for k, v in _snapshot(d).items() if before.get(k) != v}
        record = os.environ.get("GOSNARK_GOCLI_RECORD", GOLDEN)
        runs = {}
        if os.path.exists(record):
            with open(record) as f:
                runs = json.load(f)
        runs[key] = {"args": list(args), "output": p.stdout + p.stderr, "wrote": wrote}
        with open(record, "w") as f:
            json.dump(runs, f, indent=0, sort_keys=True)
        return p.stdout + p.stderr
    with open(GOLDEN) as f:
        rec = json.load(f).get(key)
    assert rec is not None, (f"no recorded go-snark-cli {' '.join(args)} run on these input files: they differ from the files "
                             "the reference binary was run on")
    for name, text in rec["wrote"].items():
        with open(os.path.join(d, name), "w") as f:
            f.write(text)
    return rec["output"]
