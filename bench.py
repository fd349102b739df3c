#!/usr/bin/env python3
"""bench.py — Groth16 prove throughput on B200 (the driver's contract).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload prove|g1msm|g2msm|verify]
                    [--logn L] [--with-qap] [--dump-outputs DIR]

Default workload (BASELINE.json's metric): one step = one groth16.GenerateProofs (groth16/groth16.go:225-278) on the
synthetic R1CS shape of SURVEY §8(d): n = 2^20 constraints, m = n+2 signals, NPublic = 1, full-width witness.

  value   proofs/s with witness, px and CRS resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e     proofs/s through the host-pointer C ABI b200_groth16_prove: pinned host buffers, H2D of the witness and px
          and D2H of the proof inside the timed region — at N > 1 too (the NCCL all-gather of the 1 KB partial records
          happens inside the library: b200_comm_init)
  N > 1   the four MSMs are sharded by cost over the ranks (strong scaling), one all-gather per proof

Other workloads (BASELINE.json configs 3 and 5; never the default line):
  --workload g1msm  BN128 G1 MSM, 2^20 random scalars/points, Mscalar-mul/s, roofline at 96 B/term
  --workload g2msm  BN128 G2 MSM, 2^22, sharded over the ranks (partial records + point sums), 160 B/term
  --workload verify batched bn128.Pairing (pairings/s) and groth16.VerifyProof calls
  --with-qap        the prove step starts from the WITNESS: px = CombinePolynomials(w, R1CSToQAP(..)) is computed on
                    the device from the sparse R1CS (b200_groth16_prove_witness), with a REAL CRS (trusted setup with
                    seeded toxic values) — the proof is verified on the GPU and by the reference's Go binary.

`--impl reference` times the reference's own algorithm (oracle/ref_c.c: per-term MSB-first double-and-add + add-2007-bl
accumulate, exactly groth16.go:243-271) on the host cores, on a fixed-size sample of the same workload; nothing of the
GPU library is loaded in that arm.

`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy in float64: prove -> PiA, PiB, PiC;
g1msm / g2msm -> msm; verify -> pairing (a seeded sample of at most 4096 results of the batch) and pairing_rows (their
indices).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.  Every
F_q value is stored as its eight little-endian 32-bit words (exact in float64).  Curve points are stored in affine form
(x, y): the Jacobian representative the library returns depends on the order of additions inside a bucket.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

G1_GEN = (1, 2, 1)
G2_GEN = ((10857046999023057135944570762232829481370756359578518086990519993285655852781,
           11559732032986387107991004021392285783925812861821192530917403151452391805634),
          (8495653923123431417604973247489272438418190587263600148770280649306958101930,
           4082367875863433681332203403145435568316851327593401208105741076214120093531), (1, 0))   # bn128.go:57-83
R_MOD = 21888242871839275222246405745257275088548364400416034343698204186575808495617


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="prove", choices=["prove", "g1msm", "g2msm", "verify"])
    ap.add_argument("--logn", type=int, default=None)
    ap.add_argument("--with-qap", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / side measurements")
    ap.add_argument("--profile-region", action="store_true",
                    help="cudaProfilerStart/Stop around the timed device-resident steps (ncu --profile-from-start off)")
    ap.add_argument("--acc-mode", type=int, default=None, choices=[0, 1, 2], help="A/B: bucket accumulation auto / batched affine / XYZZ")
    ap.add_argument("--in-flight", type=int, default=2, choices=[1, 2],
                    help="prove workload: independent proofs kept in flight (2 = two proving-key contexts on two streams, the "
                         "latency chains of one proof overlap the accumulation of the other; 1 = one proof at a time)")
    ap.add_argument("--pairing-kernel", type=int, default=None, choices=[0, 1, 2], help="A/B (verify workload): b200_pairing_batch with one thread (1) / one warp (2) per pairing")
    ap.add_argument("--tma-staging", type=int, default=None, choices=[0, 1, 2], help="A/B: staged backward pass off / all rounds / rounds >= 2")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float64, see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def _fq_words(vals):
    """F_q values -> their eight little-endian 32-bit words each."""
    from gosnark_b200._lib import ints_to_limbs
    return ints_to_limbs(vals).view(np.uint32)


def affine_words(group, p):
    """A Jacobian point of the oracle's G1 / G2 -> its affine x, y as 32-bit words: shape (2, 8) for G1, (2, 2, 8) for G2."""
    x, y = group.affine(p)[:2]
    if isinstance(x, tuple):
        return _fq_words([*x, *y]).reshape(2, 2, 8)
    return _fq_words([x, y]).reshape(2, 8)


def dump_outputs(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------- CPU reference arm
def host_cores():
    """Cores this process may actually use: the scheduler affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
            if q != "max":
                quota = max(1, int(float(q) / float(per)))
    except Exception:
        pass
    return (min(n, quota) if quota else n), {"affinity": n, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


def _limbs(vals, words=4):
    return np.frombuffer(b"".join(int(v).to_bytes(8 * words, "little") for v in vals), dtype=np.uint64).copy()


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class CpuReference:
    """The reference's hot loops (C restatement, oracle/ref_c.c) on a FIXED-SIZE sample of this workload: k1 G1 terms and
    k2 G2 terms per run, sized from the usable core count so a run takes a few seconds on any lease; sample points
    k_i*G are minted by the oracle itself (no GPU library in this arm); full-width scalars."""

    def __init__(self):
        import build as b200build
        self.oc = ctypes.CDLL(b200build.build_oracle())
        self.cores, self.core_info = host_cores()
        self.threads = max(1, min(self.cores, 256))
        rng = np.random.default_rng(0x5EED0006)

        def rnd(n):
            a = rng.integers(0, 1 << 63, size=(n, 4), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, 4), dtype=np.uint64)
            a[:, 3] &= np.uint64((1 << 61) - 1)
            return np.ascontiguousarray(a)

        pool = 1024
        self.k1 = max(pool, 1536 * self.threads)
        self.k2 = max(pool // 4, 384 * self.threads)
        g1 = _limbs(G1_GEN)
        g2 = _limbs([c for pt in G2_GEN for c in pt])
        p1 = np.zeros((pool, 12), dtype=np.uint64)
        p2 = np.zeros((pool // 4, 24), dtype=np.uint64)
        self.oc.oc_g1_mul_batch_bcast(_p(g1), _p(rnd(pool)), ctypes.c_long(pool), self.threads, _p(p1))
        self.oc.oc_g2_mul_batch_bcast(_p(g2), _p(rnd(pool // 4)), ctypes.c_long(pool // 4), self.threads, _p(p2))
        self.pts1 = np.ascontiguousarray(np.tile(p1, (self.k1 // pool + 1, 1))[: self.k1])
        self.pts2 = np.ascontiguousarray(np.tile(p2, (self.k2 // (pool // 4) + 1, 1))[: self.k2])
        self.sc1, self.sc2 = rnd(self.k1), rnd(self.k2)
        # one calibration probe: if the lease gives fewer effective cores than it reports, shrink the sample ONCE so a
        # run stays near 3 s per group; the size is then fixed for every repeat (no time-budgeted sampling)
        for grp in (1, 2):
            probe = 32 * self.threads if grp == 1 else 8 * self.threads
            t = self._run(grp, probe, self.threads) / probe
            cap = max(probe, int(3.0 / t))
            if grp == 1:
                self.k1 = min(self.k1, cap)
            else:
                self.k2 = min(self.k2, cap)

    def _run(self, group, k, threads):
        fn = self.oc.oc_g1_msm_loop if group == 1 else self.oc.oc_g2_msm_loop
        pts, sc = (self.pts1, self.sc1) if group == 1 else (self.pts2, self.sc2)
        out = np.zeros(24, dtype=np.uint64)
        t0 = time.perf_counter()
        fn(_p(pts), _p(sc), ctypes.c_long(k), threads, _p(out))
        return time.perf_counter() - t0

    def per_term(self, threads=None):
        """(seconds per G1 term, seconds per G2 term) with `threads` threads (all usable cores by default)."""
        th = self.threads if threads is None else threads
        k1 = self.k1 if threads is None else max(64, self.k1 // self.threads)
        k2 = self.k2 if threads is None else max(16, self.k2 // self.threads)
        return self._run(1, k1, th) / k1, self._run(2, k2, th) / k2

    def single_thread(self):
        t1, t2 = self.per_term(threads=1)
        return {"g1_us_per_term": t1 * 1e6, "g2_us_per_term": t2 * 1e6}


def workload_terms(workload, n):
    """(G1 terms, G2 terms) of the reference's loops for one unit of the workload."""
    if workload == "prove":
        m = n + 2
        return m + m + (m - 2) + (n - 1), m          # A, B1, C, H loops (groth16.go:243-250,269-271); B2
    if workload == "g1msm":
        return n, 0
    if workload == "g2msm":
        return 0, n
    return 0, 0


def reference_value(ref, workload, n, repeats):
    """Median over `repeats` fixed-size samples, extrapolated linearly in the term count (exact for full-width scalars)."""
    g1_terms, g2_terms = workload_terms(workload, n)
    vals, t1s, t2s = [], [], []
    for _ in range(repeats):
        t1, t2 = ref.per_term()
        t1s.append(t1); t2s.append(t2)
        vals.append(1.0 / (t1 * g1_terms + t2 * g2_terms))
    info = {"kind": "port", "cores": ref.threads, "core_detection": ref.core_info,
            "sample": f"reference double-and-add loops on a fixed sample of {ref.k1} G1 + {ref.k2} G2 terms of this workload per "
                      f"run (median of {repeats}), {ref.threads} threads, extrapolated linearly to {g1_terms} G1 + {g2_terms} G2 "
                      "terms; h = px/Z (O(n^3) in the reference, r1csqap.go:70-84) excluded in the CPU's favour",
            "g1_us_per_term": statistics.median(t1s) * 1e6, "g2_us_per_term": statistics.median(t2s) * 1e6,
            "spread": {"min": min(vals), "max": max(vals)}}
    return statistics.median(vals), info


def metric_of(workload):
    return {"prove": ("groth16_proofs_per_sec", "proofs/s"), "g1msm": ("g1_msm_mscalar_mul_per_sec", "Mscalar-mul/s"),
            "g2msm": ("g2_msm_mscalar_mul_per_sec", "Mscalar-mul/s"), "verify": ("bn128_pairings_per_sec", "pairings/s")}[workload]


def default_logn(workload):
    return {"prove": 20, "g1msm": 20, "g2msm": 22, "verify": 16}[workload]


def make_config(args, logn, world):
    n = 1 << logn
    if args.workload == "prove":
        src = ("REAL CRS from the sparse trusted setup of the chain circuit, px computed on the device from the witness "
               "(b200_groth16_prove_witness)") if args.with_qap else "px = h0*Z, CRS points k_i*G with known discrete logs"
        wl = f"synthetic R1CS 2^{logn} constraints Groth16 prove (m=n+2 signals, NPublic=1, full-width witness), {src}"
    elif args.workload in ("g1msm", "g2msm"):
        wl = f"BN128 {'G1' if args.workload == 'g1msm' else 'G2'} MSM 2^{logn} random scalars/points (P_i = k_i*G), device-resident"
    else:
        wl = f"bn128.Pairing batch of 2^{logn} (Miller loop + final exponentiation) and groth16.VerifyProof"
    fly = {} if args.workload == "verify" else {
        "in_flight": 1 if args.with_qap else args.in_flight,
        "in_flight_note": "independent proofs / MSMs the GPU arm keeps in flight (own key objects, streams, outputs); the K timed steps "
                          "are K complete proofs either way, and the one-at-a-time figures are reported beside `value` and `e2e`"}
    return {"workload": wl, "constraints" if args.workload == "prove" else "n": n, **fly,
            "parallelism": ((f"msm-cost-shard x{world}" + (" (A / B1 term 0.85, G2 term 2.75 of a C||PTD term)" if not args.with_qap and args.in_flight > 1 else "")
                             + ", all-gather inside libb200snark") if args.workload == "prove" else
                            f"index-shard x{world}") if world > 1 else "single-gpu",
            "l2": "inputs larger than L2 (>= 1 GB of precomputed CRS tables gathered per MSM)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    logn = args.logn if args.logn is not None else default_logn(args.workload)
    n = 1 << logn
    metric, unit = metric_of(args.workload)
    config = make_config(args, logn, args.gpus)
    if args.workload == "verify":
        print(json.dumps({"impl": "reference", "unavailable": "no CPU port of the pairing loop is timed (oracle/ref_py is pure Python)"}))
        return 0
    ref = CpuReference()
    for _ in range(args.warmup):
        ref.per_term()
    v, info = reference_value(ref, args.workload, n, args.steps)
    if args.workload != "prove":
        v = v * n / 1e6                      # MSMs per second -> Mscalar-mul/s
    info["value"], info["unit"] = v, unit
    info["single_thread"] = ref.single_thread()
    print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": unit,
                      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": (1e3 / v) if args.workload == "prove" else (n / (v * 1e6) * 1e3),
                      "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u256 (mod q/r)",
                      "data": "synthetic", "config": config, "cpu_baseline": info,
                      "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
    return 0


# --------------------------------------------------------------------------- GPU arm
class Ctx:
    pass


def setup_dist(args):
    import torch
    import torch.distributed as dist
    from gosnark_b200 import _lib
    c = Ctx()
    c.rank = int(os.environ.get("RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    c.torch, c.dist = torch, dist
    torch.cuda.set_device(c.local)
    if c.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", c.local))
    _lib.init(c.local)
    c.L = _lib.lib()
    if args.acc_mode is not None:
        _lib.check(c.L.b200_config(_lib.CFG_ACC_MODE, args.acc_mode))
    if args.tma_staging is not None:
        _lib.check(c.L.b200_config(_lib.CFG_TMA_STAGING, args.tma_staging))
    c.stream = torch.cuda.Stream()
    torch.cuda.set_stream(c.stream)
    c.st = c.stream.cuda_stream
    if c.world > 1:            # NCCL communicator INSIDE the library; torch.distributed only carries the 128-byte id
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if c.rank == 0:
            buf = np.zeros(128, dtype=np.uint8)
            _lib.check(c.L.b200_comm_unique_id(buf.ctypes.data_as(ctypes.c_void_p)))
            uid.copy_(torch.from_numpy(buf))
        dist.broadcast(uid, 0)
        ub = uid.cpu().numpy()
        _lib.check(c.L.b200_comm_init(ub.ctypes.data_as(ctypes.c_void_p), c.rank, c.world))
    return c


def barrier(c):
    c.torch.cuda.synchronize()
    if c.world > 1:
        c.dist.barrier()
    c.torch.cuda.synchronize()


def timed(c, fn, steps, wall=False, profile=False, extra_streams=()):
    """Device time of `steps` calls bracketed by barrier + synchronize, MAX over ranks.  wall=True for calls that
    synchronise internally on the library's own stream (the host-pointer C ABI).  extra_streams: further streams `fn`
    launches on (proofs in flight): they start after the opening event and the closing event waits for them."""
    torch = c.torch
    barrier(c)
    if profile:
        torch.cuda.profiler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(c.stream)
    for s_ in extra_streams:
        s_.wait_event(e0)
    for _ in range(steps):
        fn()
    for s_ in extra_streams:
        ev = torch.cuda.Event()
        ev.record(s_)
        c.stream.wait_event(ev)
    e1.record(c.stream)
    torch.cuda.synchronize()
    if profile:
        torch.cuda.profiler.stop()
    ms = (time.perf_counter() - t0) * 1e3 if wall else e0.elapsed_time(e1)
    if c.world > 1:
        t = torch.tensor([ms], device="cuda")
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
        ms = float(t.item())
    barrier(c)
    return ms


def peaks_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (of fallback)"


def measured_traffic():
    """Per-term DRAM bytes of the G1 accumulation phase from this round's ncu --set full capture (profiles/traffic.json,
    regenerated by tools/ncu_traffic.py from profiles/r2_ncu_*.csv); None when that capture does not exist."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


# measured on B200 with ncu (profiles/r2_notes.md): an IMAD.WIDE.U32 warp instruction occupies the fmaheavy pipe for 4
# cycles per SM sub-partition => 32 wide multiply-accumulates / clk / SM; 148 SMs at 1.965 GHz.
IMAD_WIDE_PEAK = 148 * 32 * 1.965e9


def _nwin(n):
    """Windows per scalar the library uses for an n-term base set (mirror of pick_window_bits, csrc/capi.cu)."""
    best, best_cost = 8, float("inf")
    for cbits in range(8, 19):
        cost = ((255 + cbits - 1) // cbits) * float(n) * 10.0 + 2.0 * float(1 << (cbits - 1)) * 14.0 * 4.0
        if cost < best_cost:
            best, best_cost = cbits, cost
    return (255 + best - 1) // best


def alu_model(terms_per_launch, ms_per_launch, fq_mults_per_add, wide_per_mult=137.5):
    macs = fq_mults_per_add * wide_per_mult * _nwin(terms_per_launch) * terms_per_launch / (ms_per_launch * 1e-3)
    return {"achieved": macs, "peak": IMAD_WIDE_PEAK, "unit": "32x32+64 multiply-accumulates/s", "frac": macs / IMAD_WIDE_PEAK,
            "windows_per_term": _nwin(terms_per_launch),
            "note": f"one bucket add per term and window; {fq_mults_per_add} F_q multiplies per batched-affine add x {wide_per_mult} "
                    "IMAD.WIDE-equivalent fmaheavy slots each (SASS of fp_mul_outlined, profiles/r2_sass_fp_mul.txt: 120 IMAD.WIDE x 4 cycles + 35 "
                    "IMAD / IMAD.HI / IMAD.X / IMAD.MOV x 2 cycles); peak = 32 "
                    "IMAD.WIDE / clk / SM (ncu: sm__pipe_fmaheavy_cycles_active, profiles/r2_notes.md) x 148 SMs x 1.965 GHz"}


def run_prove(args, c):
    torch, dist, L = c.torch, c.dist, c.L
    from gosnark_b200 import _lib
    from gosnark_b200._lib import check, ints_to_limbs, ptr
    from gosnark_b200.synthetic import CircuitGroth16, SyntheticGroth16
    rank, world, st = c.rank, c.world, c.st
    logn = args.logn if args.logn is not None else 20
    n = 1 << logn
    syn = CircuitGroth16(logn) if args.with_qap else SyntheticGroth16(logn)
    # proofs in flight: one proving-key context (own tables, scratch, side streams: B200_CFG_PK_CONTEXT) and one stream each
    n_fly = 1 if args.with_qap else max(1, args.in_flight)
    if n_fly > 1 and world > 1:    # latency hidden by the second proof: every shard takes the batched-affine tree (6 vs 10 multiplies per add)
        check(L.b200_config(_lib.CFG_SHARD_AFFINE_MIN_G1, 1))
        check(L.b200_config(_lib.CFG_SHARD_AFFINE_MIN_G2, 1))
        # partition weights for that mode (profiles/r2_notes.md section 16, every rank of the 2 / 4 / 8-way split timed on one GPU):
        # the C||PTD ranks also run the division, so their terms weigh more — A / B1 terms 0.85, G2 terms 2.75 of a C||PTD term
        check(L.b200_config(_lib.CFG_SHARD_W_AB, 85))
        check(L.b200_config(_lib.CFG_SHARD_W_G2, 275))
    pks = []
    for k in range(n_fly):
        check(L.b200_config(_lib.CFG_PK_CONTEXT, k))
        pks.append(syn.load_pk(rank, world))
    check(L.b200_config(_lib.CFG_PK_CONTEXT, 0))
    pk = pks[0]
    fly_streams = [c.stream] + [torch.cuda.Stream() for _ in range(n_fly - 1)]
    m, npx = syn.m, 2 * n - 1
    r_l, s_l = ints_to_limbs([syn.r]), ints_to_limbs([syn.s])
    d_w = torch.from_numpy(syn.w.view(np.int64)).cuda()
    d_px = torch.from_numpy(syn.px.view(np.int64)).cuda()
    d_outs = [torch.zeros(48, dtype=torch.int64, device="cuda") for _ in range(n_fly)]
    d_out = d_outs[0]
    torch.cuda.synchronize()
    h_w = torch.from_numpy(syn.w.view(np.int64)).pin_memory()
    h_px = torch.from_numpy(syn.px.view(np.int64)).pin_memory()
    host_out = (np.zeros(12, dtype=np.uint64), np.zeros(24, dtype=np.uint64), np.zeros(12, dtype=np.uint64))
    qap = args.with_qap and world == 1

    def step_device():      # with a communicator the all-gather + finalize run inside the call (csrc/prove_host.cuh)
        check(L.b200_groth16_prove_device(pk, d_w.data_ptr(), m, d_px.data_ptr(), npx, ptr(r_l), ptr(s_l), d_out.data_ptr(), st))

    fly_ctr = [0]

    def step_in_flight():    # proof k on context k mod n_fly: consecutive proofs overlap (independent keys, streams, outputs)
        k = fly_ctr[0] % n_fly
        fly_ctr[0] += 1
        check(L.b200_groth16_prove_device(pks[k], d_w.data_ptr(), m, d_px.data_ptr(), npx, ptr(r_l), ptr(s_l), d_outs[k].data_ptr(),
                                          fly_streams[k].cuda_stream))

    def step_e2e():          # the reference-facing call: host pointers in, proof out — on every rank
        if qap:
            check(L.b200_groth16_prove_witness(pk, syn.r1cs.handle, h_w.data_ptr(), m, ptr(r_l), ptr(s_l), ptr(host_out[0]),
                                               ptr(host_out[1]), ptr(host_out[2])))
        else:
            check(L.b200_groth16_prove(pk, h_w.data_ptr(), m, h_px.data_ptr(), npx, ptr(r_l), ptr(s_l), ptr(host_out[0]),
                                       ptr(host_out[1]), ptr(host_out[2])))

    info = np.zeros(12, dtype=np.uint64)
    check(L.b200_groth16_shard_info(pk, ptr(info)))
    ranges = []
    for lo, hi in sorted({(int(info[2 * k]), int(info[2 * k + 1])) for k in range(4)}):
        if lo < hi:
            if ranges and lo <= ranges[-1][1]:
                ranges[-1] = (ranges[-1][0], max(ranges[-1][1], hi))
            else:
                ranges.append((lo, hi))
    needs_px = bool(info[8])
    # the library stages only the top len(px) - len(Z) + 1 = n - 1 coefficients of px (all the quotient depends on; csrc/prove_host.cuh)
    px_staged = npx - n
    h2d_bytes = (32 * m + (0 if qap else 32 * px_staged)) if world == 1 else (sum(32 * (hi - lo) for lo, hi in ranges) + (32 * px_staged if needs_px else 0))

    # ---- correctness of what we time (every step function): proof == the known-discrete-log expectation
    from oracle import ref_py as o          # checker only
    from gosnark_b200.bn128 import _unflatten_g1, _unflatten_g2
    G1o, G2o = o.BN.G1, o.BN.G2
    ea, eb, ec = syn.expected_dlogs() if rank == 0 else (0, 0, 0)

    def matches(pa, pb, pc):
        return (G1o.affine(pa) == G1o.affine(G1o.mul_scalar(G1o.G, ea)) and G2o.affine(pb) == G2o.affine(G2o.mul_scalar(G2o.G, eb))
                and G1o.affine(pc) == G1o.affine(G1o.mul_scalar(G1o.G, ec)))

    for _ in range(n_fly):
        step_in_flight()
    torch.cuda.synchronize()
    step_e2e()
    parity, verified = None, None
    if rank == 0:
        parity = matches(_unflatten_g1(host_out[0])[0], _unflatten_g2(host_out[1])[0], _unflatten_g1(host_out[2])[0])
        for d_o in d_outs:                      # every context's device-resident proof
            out = d_o.cpu().numpy().view(np.uint64)
            pa, pc = _unflatten_g1(out[:24])
            parity = parity and matches(pa, _unflatten_g2(out[24:])[0], pc)
        if not parity:
            print(json.dumps({"error": "proof does not match the known-discrete-log expectation"}))
            return 1
        if args.with_qap:
            verified = bool(syn.verify(host_out[0], host_out[1], host_out[2]))       # groth16.VerifyProof on the GPU, real Vk
            if not verified:
                print(json.dumps({"error": "proof does not verify under the real verification key"}))
                return 1

    # ---- timed region: device-resident
    clocks = ClockSampler(c.local)
    if rank == 0:
        clocks.start()                         # sampled across warm-up + timed region (the region can be < 100 ms)
    for _ in range(args.warmup * n_fly):
        step_in_flight()
    torch.cuda.synchronize()
    check(L.b200_profile(1))
    prof0 = (ctypes.c_double * 8)()
    check(L.b200_profile_read(prof0))          # reset counters
    ms_total = timed(c, step_in_flight, args.steps, profile=args.profile_region, extra_streams=fly_streams[1:])
    last_out = d_outs[(fly_ctr[0] - 1) % n_fly].cpu().numpy().view(np.uint64) if args.dump_outputs and rank == 0 else None
    prof = (ctypes.c_double * 8)()
    check(L.b200_profile_read(prof))
    check(L.b200_profile(0))
    clk = clocks.stop() if rank == 0 else None
    ms_step = ms_total / args.steps
    value = 1e3 / ms_step
    # one proof at a time on one context (the latency of a proof; equals ms_step when n_fly == 1)
    ms_one = timed(c, step_device, args.steps) / args.steps if n_fly > 1 else ms_step

    # ---- exclusive timing of the dominant kernels: the same step with the MSMs serialised on one stream
    # (in the overlapped step above the bucket phases of the four MSMs share the SMs, so their event times overlap)
    check(L.b200_profile(3))
    check(L.b200_profile_read(prof0))
    for _ in range(2):
        step_device()
    torch.cuda.synchronize()
    check(L.b200_profile_read(prof0))
    ser_steps = args.steps
    ms_serial = timed(c, step_device, ser_steps) / ser_steps
    prof_x = (ctypes.c_double * 8)()
    check(L.b200_profile_read(prof_x))
    check(L.b200_profile(0))

    # ---- e2e through the host-pointer API (wall clock around the calls: they synchronise internally)
    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    e2e_one_ms = timed(c, step_e2e, args.steps, wall=True) / args.steps
    e2e_ms = e2e_one_ms
    if n_fly > 1:
        # the same K calls issued by n_fly host threads, thread k proving on context k's key: a call holds the library
        # mutex while it ENQUEUES and waits for its proof with the mutex released, so the next proof's staging copies and
        # latency chains overlap this one's accumulation (ctypes drops the GIL for the duration of a call)
        import threading
        host_outs = [host_out] + [(np.zeros(12, dtype=np.uint64), np.zeros(24, dtype=np.uint64), np.zeros(12, dtype=np.uint64))
                                  for _ in range(n_fly - 1)]
        errs = []

        def e2e_worker(k, count):
            try:
                ho = host_outs[k]
                for _ in range(count):
                    check(L.b200_groth16_prove(pks[k], h_w.data_ptr(), m, h_px.data_ptr(), npx, ptr(r_l), ptr(s_l), ptr(ho[0]), ptr(ho[1]),
                                               ptr(ho[2])))
            except Exception as e:      # surfaced after the join
                errs.append(e)

        def e2e_threads(total):
            ths = [threading.Thread(target=e2e_worker, args=(k, total // n_fly + (1 if k < total % n_fly else 0))) for k in range(n_fly)]
            for t in ths:
                t.daemon = True
                t.start()
            deadline = time.time() + 300.0
            for t in ths:
                t.join(max(0.0, deadline - time.time()))
            if any(t.is_alive() for t in ths):       # never leave the box hung: a stuck collective cannot be recovered in-process
                print(json.dumps({"error": "host-pointer proofs in flight did not finish within 300 s"}), flush=True)
                os._exit(3)
            if errs:
                raise errs[0]

        e2e_threads(2 * n_fly)                                   # warm-up of every context's host path
        e2e_ms = timed(c, lambda: e2e_threads(args.steps), 1, wall=True) / args.steps
        if rank == 0:
            for ho in host_outs:
                if not matches(_unflatten_g1(ho[0])[0], _unflatten_g2(ho[1])[0], _unflatten_g1(ho[2])[0]):
                    print(json.dumps({"error": "a host-pointer proof in flight does not match the known-discrete-log expectation"}))
                    return 1

    # ---- per-rank phase times (exclusive, ms per proof) so the limiter of the 1 -> N curve is visible
    mine = {"rank": rank, "g1_acc_ms": prof_x[0] / ser_steps, "g1_phases": prof_x[1] / ser_steps, "g1_terms": prof_x[2] / ser_steps,
            "g2_acc_ms": prof_x[3] / ser_steps, "g2_terms": prof_x[5] / ser_steps, "launches": prof_x[6] / ser_steps,
            "witness_ranges": ranges, "holds_px_division": needs_px}
    per_rank = [mine]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = gathered
        dist.barrier()
        check(L.b200_comm_destroy())
        dist.destroy_process_group()
    if rank != 0:
        return 0

    peak, peak_src = peaks_hbm()
    g1_ms, g1_l, g1_terms = prof_x[0], max(prof_x[1], 1), prof_x[2]      # exclusive (serialised) timings, this rank
    g2_ms, g2_l, g2_terms = prof_x[3], max(prof_x[4], 1), prof_x[5]
    ach = 96.0 * (g1_terms / g1_l) / (g1_ms / g1_l * 1e-3) / 1e9 if g1_ms > 0 else None
    tr = measured_traffic()
    per_term = (tr or {}).get("g1_accumulation_dram_bytes_per_term")
    traffic = per_term * (g1_terms / g1_l) if per_term and g1_ms > 0 else None
    metric, unit = metric_of("prove")
    line = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u256 (mod q/r)", "data": "synthetic",
        "config": make_config(args, logn, world),
        "constraints_per_sec": value * n, "parity_vs_known_dlog": parity,
        "proofs_in_flight": n_fly,
        "one_at_a_time": {"ms_per_step": ms_one, "value": 1e3 / ms_one, "unit": unit,
                          "note": "the same K steps with ONE proof in flight (device-resident, one context): the latency of a proof; "
                                  "`value` keeps `proofs_in_flight` independent proofs in flight on as many proving-key contexts"},
        "e2e": {"value": 1e3 / e2e_ms, "unit": unit, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 384,
                "proofs_in_flight": n_fly, "one_at_a_time_ms_per_step": e2e_one_ms,
                "note": ("b200_groth16_prove_witness: pinned witness in, px computed on the device, proof out" if qap else
                         "the host-pointer C ABI call b200_groth16_prove on every rank (pinned witness and px in, proof out; of px only the top "
                         "len(px) - len(Z) + 1 coefficients cross PCIe: the quotient depends on nothing else); at N > 1 "
                         "each rank stages only the witness ranges it reads (+ the top n - 1 coefficients of px on ranks holding PowersTauDelta) and the NCCL "
                         "all-gather of the 1 KB partial records runs inside the library; h2d bytes are rank 0's")},
        "gpu_launches": int(prof[6]),
        "clocks": clk,
        "roofline": {
            "bound": "hbm", "kernel": "G1 bucket accumulation phase (k_affine_forward / k_affine_invert / k_affine_backward<Fq> rounds; "
                                      "k_accumulate<Fq> below the affine threshold)",
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if ach else None, "peak_source": peak_src,
            "traffic": traffic,
            "traffic_source": (tr or {}).get("source", "not measured in this run: no profiles/traffic.json from this round's ncu capture"),
            "launches_per_step": prof_x[1] / ser_steps, "avg_launch_ms": g1_ms / g1_l,
            "timing": "CUDA events around each phase on its stream, measured with the proof's MSMs serialised on one stream "
                      f"(b200_profile(3)); serialised step = {ms_serial:.3f} ms, overlapped step = {ms_step:.3f} ms",
            "share_of_serial_step": (g1_ms / ser_steps) / ms_serial if ms_serial else None,
            "note": "bound by the integer multiply pipe (fmaheavy: IMAD.WIDE occupies it 4 cycles per warp; ncu on the dominant "
                    "kernel: sm__pipe_fmaheavy_cycles_active 76.7 %, DRAM 25 %), not by HBM: the HBM fraction is reported "
                    "because the contract asks for it (SURVEY H8)",
            "g2": {"avg_launch_ms": g2_ms / g2_l, "share_of_serial_step": (g2_ms / ser_steps) / ms_serial if ms_serial else None,
                   "achieved": 160.0 * (g2_terms / g2_l) / (g2_ms / g2_l * 1e-3) / 1e9 if g2_ms > 0 else None},
            "alu": alu_model(g1_terms / g1_l, g1_ms / g1_l, 6) if g1_ms > 0 else None,
            "overlapped": {"g1_avg_ms": prof[0] / max(prof[1], 1), "g2_avg_ms": prof[3] / max(prof[4], 1)}},
        "algorithmic_bytes_per_proof": syn.algorithmic_bytes(),
        "per_rank": per_rank,
    }
    if args.with_qap:
        line["verified_under_real_vk"] = verified
    if not args.no_extras and world == 1 and not args.with_qap:
        try:
            line["g1_msm_2p20"] = side_g1_msm(c, steps=args.steps, warmup=args.warmup)
        except Exception as e:   # a side measurement must never take the bench line down
            line["g1_msm_2p20"] = {"error": str(e)}
    if not args.no_extras and world == 1:
        try:
            ref = CpuReference()
            v, cinfo = reference_value(ref, "prove", n, 5)
            cinfo["value"], cinfo["unit"] = v, unit
            cinfo["single_thread"] = ref.single_thread()
            line["cpu_baseline"] = cinfo
        except Exception as e:   # the checker must never take the bench line down
            line["cpu_baseline"] = {"error": str(e)}
    if last_out is not None:
        pa, pc = _unflatten_g1(last_out[:24])
        dump_outputs(args.dump_outputs, {"PiA": affine_words(G1o, pa), "PiB": affine_words(G2o, _unflatten_g2(last_out[24:])[0]),
                                         "PiC": affine_words(G1o, pc)})
    print(json.dumps(line))
    return 0


def side_g1_msm(c, steps, warmup, logn=20):
    """The other half of BASELINE.json's metric inside the default line: a stand-alone BN128 G1 MSM of 2^logn random scalars /
    points (config 3), device-resident — two MSMs in flight on two base-set objects, and one at a time."""
    torch, L = c.torch, c.L
    from gosnark_b200 import _lib
    from gosnark_b200._lib import check, ptr
    from gosnark_b200.bn128 import _flatten_g1, _unflatten_g1
    from gosnark_b200.synthetic import SEED_POINTS, SEED_SCALARS, rand_limbs
    n = 1 << logn
    ks = rand_limbs(n, SEED_POINTS)
    ks[:, 0] |= np.uint64(1)
    ss = rand_limbs(n, SEED_SCALARS)
    pts = np.zeros((n, 12), dtype=np.uint64)
    check(L.b200_g1_mul_batch_bcast(ptr(_flatten_g1([G1_GEN])), ptr(ks), n, ptr(pts)))
    hbs = []
    for _ in range(2):
        h_ = _lib._h(0)
        check(L.b200_g1_bases_load(ptr(pts), n, 0, h_))
        hbs.append(h_)
    del pts
    d_s = torch.from_numpy(ss.view(np.int64)).cuda()
    d_parts = [torch.zeros(16, dtype=torch.int64, device="cuda") for _ in range(2)]
    streams = [c.stream, torch.cuda.Stream()]
    ctr = [0]
    torch.cuda.synchronize()

    def step2():
        k = ctr[0] % 2
        ctr[0] += 1
        check(L.b200_msm_device(hbs[k].value, d_s.data_ptr(), n, 0, d_parts[k].data_ptr(), streams[k].cuda_stream))

    def step1():
        check(L.b200_msm_device(hbs[0].value, d_s.data_ptr(), n, 0, d_parts[0].data_ptr(), c.st))

    for _ in range(2 * warmup):
        step2()
    torch.cuda.synchronize()
    ms2 = timed(c, step2, steps, extra_streams=streams[1:]) / steps
    ms1 = timed(c, step1, steps) / steps
    from oracle import ref_py as o          # checker only
    out = np.zeros(12, dtype=np.uint64)
    parity = True
    expect = sum(int(a) * int(b) for a, b in zip(_lib.limbs_to_ints(ks), _lib.limbs_to_ints(ss))) % R_MOD
    for d_p in d_parts:
        check(L.b200_g1_sum_partials(d_p.data_ptr(), 1, ptr(out), c.st))
        parity = parity and o.BN.G1.affine(_unflatten_g1(out)[0]) == o.BN.G1.affine(o.BN.G1.mul_scalar(o.BN.G1.G, expect))
    for h_ in hbs:
        check(L.b200_bases_free(h_.value))
    return {"n": n, "ms_per_msm": ms2, "mscalar_mul_per_sec": n / ms2 / 1e3, "msms_in_flight": 2,
            "one_at_a_time_ms": ms1, "one_at_a_time_mscalar_mul_per_sec": n / ms1 / 1e3, "parity_vs_known_dlog": bool(parity),
            "whole_msm_hbm_algorithmic_GBps": 96.0 * n / (ms2 * 1e-3) / 1e9,
            "note": "stand-alone G1 MSM (BASELINE config 3) measured in the same run; `bench.py --workload g1msm` is its full line"}


def run_msm(args, c):
    """Configs 3 / 5: stand-alone MSM, scalars and points device-resident, index range sharded over the ranks."""
    torch, dist, L = c.torch, c.dist, c.L
    from gosnark_b200 import _lib
    from gosnark_b200._lib import check, ptr
    from gosnark_b200.bn128 import _flatten_g1, _flatten_g2, _unflatten_g1, _unflatten_g2
    from gosnark_b200.synthetic import SEED_POINTS, SEED_SCALARS, rand_limbs
    rank, world, st = c.rank, c.world, c.st
    group = 1 if args.workload == "g1msm" else 2
    logn = args.logn if args.logn is not None else default_logn(args.workload)
    n = 1 << logn
    lo, hi = n * rank // world, n * (rank + 1) // world
    ks = rand_limbs(n, SEED_POINTS)[lo:hi]
    ks[:, 0] |= np.uint64(1)
    ss = rand_limbs(n, SEED_SCALARS)[lo:hi]
    words = 12 if group == 1 else 24
    gen = _flatten_g1([G1_GEN]) if group == 1 else _flatten_g2([G2_GEN])
    pts = np.zeros((hi - lo, words), dtype=np.uint64)
    check((L.b200_g1_mul_batch_bcast if group == 1 else L.b200_g2_mul_batch_bcast)(ptr(gen), ptr(ks), hi - lo, ptr(pts)))
    # MSMs in flight: independent base-set objects (own tables and scratch) on their own streams
    n_fly = max(1, args.in_flight)
    hbs = []
    for _ in range(n_fly):
        h_ = _lib._h(0)
        check((L.b200_g1_bases_load if group == 1 else L.b200_g2_bases_load)(ptr(pts), hi - lo, 0, h_))
        hbs.append(h_)
    hb = hbs[0]
    del pts
    rec = 128 if group == 1 else 256                                     # XYZZ partial record bytes
    d_s = torch.from_numpy(ss.view(np.int64)).cuda()
    d_parts = [torch.zeros(rec // 8, dtype=torch.int64, device="cuda") for _ in range(n_fly)]
    d_alls = [torch.zeros(rec // 8 * world, dtype=torch.int64, device="cuda") for _ in range(n_fly)]
    d_part, d_all = d_parts[0], d_alls[0]
    fly_streams = [c.stream] + [torch.cuda.Stream() for _ in range(n_fly - 1)]
    fly_ctr = [0]
    torch.cuda.synchronize()

    def step_in_flight():
        k = fly_ctr[0] % n_fly
        fly_ctr[0] += 1
        check(L.b200_msm_device(hbs[k].value, d_s.data_ptr(), hi - lo, 0, d_parts[k].data_ptr(), fly_streams[k].cuda_stream))
        if world > 1:
            with torch.cuda.stream(fly_streams[k]):
                dist.all_gather_into_tensor(d_alls[k], d_parts[k])
    h_s = torch.from_numpy(ss.view(np.int64)).pin_memory()
    out = np.zeros(words, dtype=np.uint64)

    def step_device():
        check(L.b200_msm_device(hb.value, d_s.data_ptr(), hi - lo, 0, d_part.data_ptr(), st))
        if world > 1:
            dist.all_gather_into_tensor(d_all, d_part)

    def finish():
        src = d_all if world > 1 else d_part
        check((L.b200_g1_sum_partials if group == 1 else L.b200_g2_sum_partials)(src.data_ptr(), world, ptr(out), st))

    def step_e2e():
        d_s.copy_(h_s, non_blocking=True)
        step_device()
        finish()

    step_e2e()
    parity = None
    if True:
        part = sum(int(a) * int(b) for a, b in zip(_lib.limbs_to_ints(ks), _lib.limbs_to_ints(ss))) % R_MOD
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, part)
            part = sum(parts) % R_MOD
        if rank == 0:
            from oracle import ref_py as o
            G = o.BN.G1 if group == 1 else o.BN.G2
            got = (_unflatten_g1(out) if group == 1 else _unflatten_g2(out))[0]
            parity = G.affine(got) == G.affine(G.mul_scalar(G.G, part))
            if not parity:
                print(json.dumps({"error": "MSM does not match the known-discrete-log expectation"}))
                return 1
    clocks = ClockSampler(c.local)
    if rank == 0:
        clocks.start()
    for _ in range(args.warmup * n_fly):
        step_in_flight()
    torch.cuda.synchronize()
    ms = timed(c, step_in_flight, args.steps, profile=args.profile_region, extra_streams=fly_streams[1:]) / args.steps
    clk = clocks.stop() if rank == 0 else None
    last_msm = None
    if args.dump_outputs:
        k_last = (fly_ctr[0] - 1) % n_fly
        last_msm = np.zeros(words, dtype=np.uint64)
        check((L.b200_g1_sum_partials if group == 1 else L.b200_g2_sum_partials)(
            (d_alls[k_last] if world > 1 else d_parts[k_last]).data_ptr(), world, ptr(last_msm), st))
    # one MSM at a time (its latency), with CUDA events around its accumulation phase for the roofline
    check(L.b200_profile(1))
    prof = (ctypes.c_double * 8)()
    check(L.b200_profile_read(prof))
    ms_one = timed(c, step_device, args.steps) / args.steps
    check(L.b200_profile_read(prof))
    check(L.b200_profile(0))
    for _ in range(2):
        step_e2e()
    e2e_ms = timed(c, step_e2e, args.steps, wall=True) / args.steps
    mode = ctypes.c_int(0)
    check(L.b200_bases_acc_mode(hb.value, ctypes.byref(mode)))
    if world > 1:
        dist.barrier()
        check(L.b200_comm_destroy())
        dist.destroy_process_group()
    if rank != 0:
        return 0
    peak, peak_src = peaks_hbm()
    bpt = 96.0 if group == 1 else 160.0
    k = 0 if group == 1 else 3
    acc_ms, acc_l, acc_terms = prof[k], max(prof[k + 1], 1), prof[k + 2]
    ach = bpt * (acc_terms / acc_l) / (acc_ms / acc_l * 1e-3) / 1e9 if acc_ms > 0 else None
    metric, unit = metric_of(args.workload)
    line = {"metric": metric, "value": n / ms / 1e3, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u256 (mod q)",
            "data": "synthetic", "config": make_config(args, logn, world), "parity_vs_known_dlog": parity,
            "e2e": {"value": n / e2e_ms / 1e3, "unit": unit, "ms_per_step": e2e_ms, "h2d_bytes_per_step": 32 * (hi - lo),
                    "d2h_bytes_per_step": 8 * words,
                    "note": "pinned scalars -> device, b200_msm_device, all-gather of the XYZZ partial records, b200_g*_sum_partials "
                            "to host; the points are the resident CRS"},
            "msms_in_flight": n_fly,
            "one_at_a_time": {"ms_per_step": ms_one, "value": n / ms_one / 1e3, "unit": unit,
                              "note": "the same K steps with ONE MSM in flight: the latency of an MSM; `value` keeps `msms_in_flight` "
                                      "independent MSMs (own base-set objects and streams) in flight"},
            "gpu_launches": int(prof[6]), "clocks": clk, "accumulation_kernel": {1: "batched affine", 2: "xyzz"}[mode.value],
            "whole_msm_hbm_algorithmic_GBps": bpt * n / (ms * 1e-3) / 1e9,
            "roofline": {"bound": "hbm", "kernel": f"G{group} bucket accumulation phase of this rank's shard", "achieved": ach, "peak": peak,
                         "unit": "GB/s", "frac": (ach / peak) if ach else None, "peak_source": peak_src, "traffic": None,
                         "avg_launch_ms": acc_ms / acc_l,
                         "alu": alu_model(acc_terms / acc_l, acc_ms / acc_l, 6 if group == 1 else 6 * 2.6) if acc_ms > 0 else None}}
    if not args.no_extras and world == 1:
        try:
            ref = CpuReference()
            v, cinfo = reference_value(ref, args.workload, n, 5)
            cinfo["value"], cinfo["unit"] = v * n / 1e6, unit
            cinfo["single_thread"] = ref.single_thread()
            line["cpu_baseline"] = cinfo
        except Exception as e:
            line["cpu_baseline"] = {"error": str(e)}
    if last_msm is not None:
        dump_outputs(args.dump_outputs, {"msm": affine_words(G, (_unflatten_g1(last_msm) if group == 1 else _unflatten_g2(last_msm))[0])})
    print(json.dumps(line))
    return 0


def run_verify(args, c):
    """Config 5's verifier side: throughput of bn128.Pairing batches (bn128/bn128.go:179-421) and of groth16.VerifyProof."""
    torch, L = c.torch, c.L
    from gosnark_b200 import _lib
    from gosnark_b200._lib import check, ints_to_limbs, ptr
    from gosnark_b200.bn128 import _flatten_g1, _flatten_g2
    from gosnark_b200.synthetic import CircuitGroth16, rand_limbs
    if c.world > 1:
        raise SystemExit("--workload verify is a single-GPU measurement")
    logn = args.logn if args.logn is not None else default_logn("verify")
    n = 1 << logn
    if args.pairing_kernel is not None:
        check(L.b200_config(_lib.CFG_PAIRING_KERNEL, args.pairing_kernel))
    k1, k2 = rand_limbs(n, 11), rand_limbs(n, 12)
    p1 = np.zeros((n, 12), dtype=np.uint64)
    p2 = np.zeros((n, 24), dtype=np.uint64)
    check(L.b200_g1_mul_batch_bcast(ptr(_flatten_g1([G1_GEN])), ptr(k1), n, ptr(p1)))
    check(L.b200_g2_mul_batch_bcast(ptr(_flatten_g2([G2_GEN])), ptr(k2), n, ptr(p2)))
    out = np.zeros((n, 48), dtype=np.uint64)

    def step():
        check(L.b200_pairing_batch(ptr(p1), ptr(p2), n, ptr(out)))

    step()
    # bilinearity spot check of what we time: e(aG, bH) == e(abG, H)
    from oracle import ref_py as o
    ab = _lib.limbs_to_ints(k1[:1])[0] * _lib.limbs_to_ints(k2[:1])[0] % R_MOD
    q1, q2, o2 = np.zeros((1, 12), dtype=np.uint64), _flatten_g2([G2_GEN]), np.zeros((1, 48), dtype=np.uint64)
    check(L.b200_g1_mul_batch_bcast(ptr(_flatten_g1([G1_GEN])), ptr(ints_to_limbs([ab])), 1, ptr(q1)))
    check(L.b200_pairing_batch(ptr(q1), ptr(q2), 1, ptr(o2)))
    parity = bool((o2[0] == out[0]).all())
    # the two kernels (one thread / one warp per pairing) agree on a sample of this batch, coefficient for coefficient
    ns = min(n, 256)
    outs = []
    for kern in (1, 2):
        check(L.b200_config(_lib.CFG_PAIRING_KERNEL, kern))
        o_k = np.zeros((ns, 48), dtype=np.uint64)
        check(L.b200_pairing_batch(ptr(p1), ptr(p2), ns, ptr(o_k)))
        outs.append(o_k)
    check(L.b200_config(_lib.CFG_PAIRING_KERNEL, args.pairing_kernel if args.pairing_kernel is not None else 0))
    parity = parity and bool((outs[0] == outs[1]).all()) and bool((outs[0] == out[:ns]).all())
    clocks = ClockSampler(c.local)
    clocks.start()
    for _ in range(args.warmup):
        step()
    ms = timed(c, step, args.steps, wall=True) / args.steps
    clk = clocks.stop()
    # groth16.VerifyProof latency on a real instance
    syn = CircuitGroth16(6)
    pk = syn.load_pk()
    pa, pb, pc = np.zeros(12, dtype=np.uint64), np.zeros(24, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
    check(L.b200_groth16_prove(pk, ptr(syn.w), syn.m, ptr(syn.px), syn.px.shape[0], ptr(ints_to_limbs([syn.r])), ptr(ints_to_limbs([syn.s])),
                               ptr(pa), ptr(pb), ptr(pc)))
    ok = syn.verify(pa, pb, pc)
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        ok = ok and syn.verify(pa, pb, pc)
    verify_ms = (time.perf_counter() - t0) * 1e3 / reps
    if args.dump_outputs:
        rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, 4096), replace=False))
        dump_outputs(args.dump_outputs, {"pairing": out[rows].view(np.uint32).reshape(len(rows), 12, 8), "pairing_rows": rows})
    metric, unit = metric_of("verify")
    print(json.dumps({"metric": metric, "value": n / ms * 1e3, "unit": unit, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u256 (mod q), F_q^12",
                      "data": "synthetic", "config": make_config(args, logn, 1), "parity_bilinearity": parity,
                      "e2e": {"value": n / ms * 1e3, "unit": unit, "h2d_bytes_per_step": n * 288, "d2h_bytes_per_step": n * 384,
                              "note": "b200_pairing_batch is a host-pointer call: value and e2e are the same measurement"},
                      "groth16_verify": {"ms_per_call": verify_ms, "accepted": bool(ok)}, "clocks": clk,
                      "gpu_launches": args.steps}))
    return 0 if parity and ok else 1


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    c = setup_dist(args)
    if args.workload == "prove":
        return run_prove(args, c)
    if args.workload in ("g1msm", "g2msm"):
        return run_msm(args, c)
    return run_verify(args, c)


if __name__ == "__main__":
    sys.exit(main())
