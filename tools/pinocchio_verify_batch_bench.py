"""Throughput of batch Pinocchio verification (b200_pinocchio_verify_batch) against the per-proof routes, on one GPU.

For N in --sizes and each public-signal count in --npub, N known-discrete-log proofs under one key are minted on the device
(b200_g1/g2_mul_batch_bcast) from a fixed seed.  Each JSON line reports, with the GPU's name and power limit:
  batch          the batch call: median ms of --reps synchronised calls after a warm-up, proofs/s, its stats array
  route12        the twelve-pairings-per-proof route: b200_pairing_batch over 12N pairs + two b200_fq12_mul_batch, compared on
                 the host (vkx_i + PiA_i and vkx_i + PiA_i + PiC_i precomputed and not timed, so this route is timed
                 optimistically)
  single_loop    N <= 64: a loop of b200_pinocchio_verify
  python_loop    N <= 16: a loop of snark.VerifyProof (the host-side Python verifier)
  one_bad        the batch call with proof N/2 made invalid: the price of the failure path
Usage: python tools/pinocchio_verify_batch_bench.py [--sizes 1,64,1024,16384,65536] [--npub 1,8] [--reps 5] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import random
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from verify_batch_bench import gpu_info, mint, timed  # noqa: E402
from gosnark_b200 import _lib  # noqa: E402
from gosnark_b200._lib import check, ints_to_limbs, lib, ptr  # noqa: E402
from gosnark_b200.bn128 import R, _unflatten_g1, _unflatten_g2  # noqa: E402

ORDER = ("PiA", "PiAp", "PiBp", "PiC", "PiCp", "PiH", "PiKp")


class Instance:
    def __init__(self, n, npub, seed):
        rng = random.Random(seed)
        rnd = lambda: rng.randrange(1, R)
        ka, kb, kc, kbg, kg, z = (rnd() for _ in range(6))
        ic_k = [rnd() for _ in range(npub + 1)]
        self.pubs = [rnd() for _ in range(n * npub)]
        inv_z, inv_kg = pow(z, -1, R), pow(kg, -1, R)
        g1k, b, vkxa, vkxac = [], [], [], []
        for i in range(n):
            a, bi, c = rnd(), rnd(), rnd()
            vkx = (ic_k[0] + sum(self.pubs[i * npub + j] * ic_k[j + 1] for j in range(npub))) % R
            g1k += [a, ka * a % R, kb * bi % R, c, kc * c % R, ((vkx + a) * bi - c) * inv_z % R,
                    kbg * (vkx + a + c + bi) * inv_kg % R]
            b.append(bi)
            vkxa.append((vkx + a) % R)
            vkxac.append((vkx + a + c) % R)
        self.n, self.npub = n, npub
        self.ic = mint(1, ic_k)
        self.vk1 = mint(1, [kb, kbg])
        self.vk2 = mint(2, [ka, kc, z, kbg, kg])
        self.P = mint(1, g1k).reshape(n, 84)
        self.B = mint(2, b)
        self.pub = ints_to_limbs(self.pubs) if npub else np.zeros((1, 4), dtype=np.uint64)
        self.rho = ints_to_limbs([rng.randrange(1, 1 << 128) for _ in range(5 * n)], 2)
        # route12 inputs: pair e of proof i at [e][i]
        g = lambda k: self.P[:, 12 * k:12 * k + 12]
        rep1 = lambda p: np.repeat(p[None, :], n, 0)
        gen2 = np.repeat(mint(2, [1]), n, 0)
        vka, vkc, vkz, g2kbg, g2kg = (rep1(self.vk2[k]) for k in range(5))
        self.g1 = np.ascontiguousarray(np.concatenate([g(0), g(1), rep1(self.vk1[0]), g(2), g(3), g(4), mint(1, vkxa), g(5), g(3),
                                                       mint(1, vkxac), rep1(self.vk1[1]), g(6)]))
        self.g2 = np.ascontiguousarray(np.concatenate([vka, gen2, self.B, gen2, vkc, gen2, self.B, vkz, gen2, g2kbg, self.B, g2kg]))

    def batch(self, P=None):
        ok = np.zeros(self.n, dtype=np.int32)
        st = np.zeros(4, dtype=np.uint64)
        check(lib().b200_pinocchio_verify_batch(ptr(self.ic), self.npub + 1, ptr(self.vk1), ptr(self.vk2), self.n,
                                                ptr(self.P if P is None else P), ptr(self.B), ptr(self.pub), self.npub,
                                                ptr(self.rho), ptr(ok), ptr(st)))
        return ok, [int(x) for x in st]

    def route12(self):
        n = self.n
        e = np.zeros((12 * n, 48), dtype=np.uint64)
        check(lib().b200_pairing_batch(ptr(self.g1), ptr(self.g2), 12 * n, ptr(e)))
        e = e.reshape(12, n, 48)
        p0, p1 = np.zeros((n, 48), dtype=np.uint64), np.zeros((n, 48), dtype=np.uint64)
        check(lib().b200_fq12_mul_batch(ptr(np.ascontiguousarray(e[7])), ptr(np.ascontiguousarray(e[8])), n, ptr(p0)))
        check(lib().b200_fq12_mul_batch(ptr(np.ascontiguousarray(e[9])), ptr(np.ascontiguousarray(e[10])), n, ptr(p1)))
        eq = lambda x, y: (x == y).all(axis=1)
        return eq(e[0], e[1]) & eq(e[2], e[3]) & eq(e[4], e[5]) & eq(e[6], p0) & eq(p1, e[11])

    def single_loop(self):
        res = []
        for i in range(self.n):
            ok, fc = ctypes.c_int(0), ctypes.c_int(0)
            check(lib().b200_pinocchio_verify(ptr(self.ic), self.npub + 1, ptr(self.vk1), ptr(self.vk2), ptr(self.P[i]),
                                              ptr(self.B[i]), ptr(self.pub[i * self.npub:]) if self.npub else ptr(self.pub),
                                              self.npub, ctypes.byref(ok), ctypes.byref(fc)))
            res.append(ok.value)
        return res

    def python_loop(self):
        from gosnark_b200 import snark
        g1v, g2v = _unflatten_g1(self.vk1.reshape(-1)), _unflatten_g2(self.vk2.reshape(-1))
        vk = {"IC": _unflatten_g1(self.ic.reshape(-1)), "Vkb": g1v[0], "G1Kbg": g1v[1], "Vka": g2v[0], "Vkc": g2v[1],
              "Vkz": g2v[2], "G2Kbg": g2v[3], "G2Kg": g2v[4]}
        res = []
        for i in range(self.n):
            proof = dict(zip(ORDER, _unflatten_g1(self.P[i])), PiB=_unflatten_g2(self.B[i])[0])
            res.append(snark.VerifyProof(vk, proof, self.pubs[i * self.npub:(i + 1) * self.npub]))
        return res


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
            assert (ok == 1).all() and st == [n, 0, 1, n + 6], (st, ok[:8])
            rec.update(batch_ms=round(ms, 3), batch_proofs_per_s=round(n / ms * 1e3, 1), stats=st)
            ms, ok = timed(inst.route12, args.reps)
            assert ok.all()
            rec.update(route12_ms=round(ms, 3), route12_proofs_per_s=round(n / ms * 1e3, 1))
            if n <= 64:
                ms, ok = timed(inst.single_loop, args.reps)
                assert all(v == 1 for v in ok)
                rec.update(single_loop_ms=round(ms, 3), single_loop_proofs_per_s=round(n / ms * 1e3, 1))
            if n <= 16:
                ms, ok = timed(inst.python_loop, args.reps)
                assert all(ok)
                rec.update(python_loop_ms=round(ms, 3), python_loop_proofs_per_s=round(n / ms * 1e3, 1))
            bad = inst.P.copy()
            bad[n // 2, 60:72] = bad[n // 2, 0:12]      # PiH_i := PiA_i: invalid
            ms, (ok, st) = timed(lambda: inst.batch(bad), args.reps)
            assert [i for i in range(n) if ok[i] != 1] == [n // 2], st
            rec.update(one_bad_ms=round(ms, 3), one_bad_proofs_per_s=round(n / ms * 1e3, 1), one_bad_stats=st)
            rec["batch_vs_route12"] = round(rec["route12_ms"] / rec["batch_ms"], 2)
            line = json.dumps(rec)
            print(line, flush=True)
            if sink:
                sink.write(line + "\n")
                sink.flush()


if __name__ == "__main__":
    main()
