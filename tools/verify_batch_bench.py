"""Throughput of batch Groth16 verification (b200_groth16_verify_batch) against the per-proof routes, on one GPU.

For N in --sizes and each public-signal count in --npub, N known-discrete-log proofs under one key are minted on the device
(b200_g1/g2_mul_batch_bcast) from a fixed seed.  Each JSON line reports, with the GPU's name and power limit:
  batch          the batch call: median ms of --reps synchronised calls after a warm-up, proofs/s, its stats array
  route4         the four-pairings-per-proof route: b200_pairing_batch over 4N pairs + two b200_fq12_mul_batch, compared on
                 the host (icPubl_i precomputed and not timed, so this route is timed optimistically)
  single_loop    N <= 64: a loop of b200_groth16_verify
  one_bad        the batch call with proof N/2 made invalid: the price of the failure path
Usage: python tools/verify_batch_bench.py [--sizes 1,64,1024,16384,65536] [--npub 1,8] [--reps 5] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import random
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from gosnark_b200 import _lib  # noqa: E402
from gosnark_b200._lib import check, ints_to_limbs, lib, ptr  # noqa: E402
from gosnark_b200.bn128 import G1, G2, R, _flatten_g1, _flatten_g2  # noqa: E402

G1_GEN, G2_GEN = _flatten_g1([G1.G]), _flatten_g2([G2.G])


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
        return name, power
    except Exception as e:  # the numbers below are still the device's; say that the card could not be named
        return f"unknown ({e})", "unknown"


def mint(group, ks):
    """k * G for every k (standard-form Jacobian limbs, n x 12 or n x 24)."""
    n = len(ks)
    out = np.zeros((n, 12 if group == 1 else 24), dtype=np.uint64)
    fn = lib().b200_g1_mul_batch_bcast if group == 1 else lib().b200_g2_mul_batch_bcast
    check(fn(ptr(G1_GEN if group == 1 else G2_GEN), ptr(ints_to_limbs(ks)), n, ptr(out)))
    return out


class Instance:
    def __init__(self, n, npub, seed):
        rng = random.Random(seed)
        rnd = lambda: rng.randrange(1, R)
        al, be, ga, de = (rnd() for _ in range(4))
        ic_k = [rnd() for _ in range(npub + 1)]
        self.pubs = [rnd() for _ in range(n * npub)]
        a = [rnd() for _ in range(n)]
        b = [rnd() for _ in range(n)]
        inv_de = pow(de, -1, R)
        icp = [(ic_k[0] + sum(self.pubs[i * npub + j] * ic_k[j + 1] for j in range(npub))) % R for i in range(n)]
        c = [(a[i] * b[i] - al * be - icp[i] * ga) * inv_de % R for i in range(n)]
        self.n, self.npub = n, npub
        self.ic = mint(1, ic_k)
        self.alpha = mint(1, [al])
        self.beta, self.gamma, self.delta = (mint(2, [k]) for k in (be, ga, de))
        self.A, self.B, self.C = mint(1, a), mint(2, b), mint(1, c)
        self.icp = mint(1, icp)
        self.pub = ints_to_limbs(self.pubs) if npub else np.zeros((1, 4), dtype=np.uint64)
        self.rho = ints_to_limbs([rng.randrange(1, 1 << 128) for _ in range(n)], 2)

    def batch(self, C=None):
        ok = np.zeros(self.n, dtype=np.int32)
        st = np.zeros(4, dtype=np.uint64)
        check(lib().b200_groth16_verify_batch(ptr(self.ic), self.npub + 1, ptr(self.alpha), ptr(self.beta), ptr(self.gamma),
                                              ptr(self.delta), self.n, ptr(self.A), ptr(self.B), ptr(self.C if C is None else C),
                                              ptr(self.pub), self.npub, ptr(self.rho), ptr(ok), ptr(st)))
        return ok, [int(x) for x in st]

    def route4(self):
        n = self.n
        g1 = np.concatenate([self.A, np.repeat(self.alpha, n, 0), self.icp, self.C])
        g2 = np.concatenate([self.B, np.repeat(self.beta, n, 0), np.repeat(self.gamma, n, 0), np.repeat(self.delta, n, 0)])
        e = np.zeros((4 * n, 48), dtype=np.uint64)
        check(lib().b200_pairing_batch(ptr(g1), ptr(g2), 4 * n, ptr(e)))
        t = np.zeros((n, 48), dtype=np.uint64)
        check(lib().b200_fq12_mul_batch(ptr(np.ascontiguousarray(e[n:2 * n])), ptr(np.ascontiguousarray(e[2 * n:3 * n])), n, ptr(t)))
        rhs = np.zeros((n, 48), dtype=np.uint64)
        check(lib().b200_fq12_mul_batch(ptr(t), ptr(np.ascontiguousarray(e[3 * n:])), n, ptr(rhs)))
        return (e[:n] == rhs).all(axis=1)

    def single_loop(self):
        res = []
        for i in range(self.n):
            ok = ctypes.c_int(0)
            check(lib().b200_groth16_verify(ptr(self.ic), self.npub + 1, ptr(self.alpha), ptr(self.beta), ptr(self.gamma),
                                            ptr(self.delta), ptr(self.A[i]), ptr(self.B[i]), ptr(self.C[i]),
                                            ptr(self.pub[i * self.npub:]) if self.npub else ptr(self.pub), self.npub,
                                            ctypes.byref(ok)))
            res.append(ok.value)
        return res


def timed(fn, reps):
    fn()                                          # warm-up (module load, allocations)
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()                                # every entry point ends in a stream synchronise
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,64,1024,16384,65536")
    ap.add_argument("--npub", default="1,8")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 5:
        ap.error("--reps must be >= 5")
    _lib.init(0)
    name, power = gpu_info()
    sink = open(args.out, "w") if args.out else None
    for npub in (int(x) for x in args.npub.split(",")):
        for n in (int(x) for x in args.sizes.split(",")):
            inst = Instance(n, npub, seed=n * 10 + npub)
            rec = {"gpu": name, "power_limit": power, "n": n, "npub": npub, "reps": args.reps}
            ms, (ok, st) = timed(inst.batch, args.reps)
            assert (ok == 1).all() and st == [n, 0, 1, n + 3], (st, ok[:8])
            rec.update(batch_ms=round(ms, 3), batch_proofs_per_s=round(n / ms * 1e3, 1), stats=st)
            ms, ok = timed(inst.route4, args.reps)
            assert ok.all()
            rec.update(route4_ms=round(ms, 3), route4_proofs_per_s=round(n / ms * 1e3, 1))
            if n <= 64:
                ms, ok = timed(inst.single_loop, args.reps)
                assert all(v == 1 for v in ok)
                rec.update(single_loop_ms=round(ms, 3), single_loop_proofs_per_s=round(n / ms * 1e3, 1))
            bad_c = inst.C.copy()
            bad_c[n // 2] = inst.A[n // 2]            # C_i := A_i: invalid
            ms, (ok, st) = timed(lambda: inst.batch(bad_c), args.reps)
            assert [i for i in range(n) if ok[i] != 1] == [n // 2], st
            rec.update(one_bad_ms=round(ms, 3), one_bad_proofs_per_s=round(n / ms * 1e3, 1), one_bad_stats=st)
            rec["batch_vs_route4"] = round(rec["route4_ms"] / rec["batch_ms"], 2)
            line = json.dumps(rec)
            print(line, flush=True)
            if sink:
                sink.write(line + "\n")
                sink.flush()


if __name__ == "__main__":
    main()
