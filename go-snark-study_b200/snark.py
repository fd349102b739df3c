"""Host mirror of the reference's root ``snark`` package (Pinocchio) over libb200snark: the prove path
(snark.go:254-289), and — SURVEY §8f rows 1-2 — the trusted setup (snark.go:98-251) and VerifyProof (:292-372).

    pk = {"A","Ap","B","Bp","C","Cp","Kp","G1T","Z"}   (snark.Pk, snark.go:16-26; B is in G2)
    proof = GenerateProofs(circuit, pk, w, px) -> PiA PiAp PiB PiBp PiC PiCp PiH PiKp
"""
import numpy as np

from . import _lib
from ._lib import check, ints_to_limbs, lib, ptr
from .bn128 import R, _flatten_g1, _flatten_g2, _unflatten_g1, _unflatten_g2, reduce_scalar
from .groth16 import KeyCache, _attr, _n_signals, _rand_rho

_ORDER = ("PiA", "PiAp", "PiBp", "PiC", "PiCp", "PiH", "PiKp")


class DeviceProvingKey:
    def __init__(self, pk, n_vars, n_public, window_bits=0):
        m = n_vars
        arr = {k: _flatten_g1(pk[k][:m]) for k in ("A", "Ap", "Bp", "C", "Cp", "Kp")}
        b2 = _flatten_g2(pk["B"][:m])
        g1t = _flatten_g1(pk["G1T"])
        z = ints_to_limbs([int(x) % R for x in pk["Z"]])
        h = _lib._h(0)
        check(lib().b200_pinocchio_pk_load(ptr(arr["A"]), ptr(arr["Ap"]), ptr(b2), ptr(arr["Bp"]), ptr(arr["C"]),
                                           ptr(arr["Cp"]), ptr(arr["Kp"]), m, ptr(g1t), len(pk["G1T"]), ptr(z),
                                           len(pk["Z"]), n_public, window_bits, h))
        self.handle = h.value

    def prove_limbs(self, w_limbs, px_limbs):
        g1 = np.zeros(84, dtype=np.uint64)
        pb = np.zeros(24, dtype=np.uint64)
        check(lib().b200_pinocchio_prove(self.handle, ptr(w_limbs), w_limbs.shape[0], ptr(px_limbs),
                                         px_limbs.shape[0], ptr(g1), ptr(pb)))
        proof = dict(zip(_ORDER, _unflatten_g1(g1)))
        proof["PiB"] = _unflatten_g2(pb)[0]
        return proof

    def free(self):
        if self.handle:
            check(lib().b200_pk_free(self.handle))
            self.handle = 0


_pk_cache = KeyCache(lambda pk, m, npub, c: DeviceProvingKey(pk, m, npub, c))       # see groth16.KeyCache (identity + strong ref)


def LoadProvingKey(circuit, pk, window_bits=0):
    return _pk_cache.get(circuit, pk, window_bits)


def Forget(pk=None):
    _pk_cache.forget(pk)


def GenerateProofs(circuit, pk, w, px):
    """snark.GenerateProofs(circuit, pk, w, px) (snark.go:254). Deterministic."""
    dpk = pk if isinstance(pk, DeviceProvingKey) else LoadProvingKey(circuit, pk)
    wl = ints_to_limbs([reduce_scalar(x) for x in w])
    pl = ints_to_limbs([int(x) % R for x in px])
    return dpk.prove_limbs(wl, pl)


def GenerateTrustedSetup(witnessLength, circuit, alphas, betas, gammas, toxic=None):
    """snark.GenerateTrustedSetup (snark.go:98-251) with the heavy loops on the GPU: Eval(alphas[i], t) as one batched
    evaluation per matrix, every MulScalar as the reference's own double-and-add in batch kernels (so Jacobian X,Y,Z
    equal the reference's for the same toxic values), and the reference's k == a + b + c self-check (:194-199) as
    batched group additions.  ``toxic`` = dict T, Ka, Kb, Kc, Kbeta, Kgamma, RhoA, RhoB (RhoC = RhoA*RhoB, :150);
    drawn like the reference (Fq.Rand) when omitted.  Returns {"Toxic", "Pk", "Vk"} shaped like snark.Setup."""
    from . import bn128
    from ._lib import limbs_to_ints
    from .groth16 import rand_fr
    n_vars, n_public = _attr(circuit, "NVars"), _attr(circuit, "NPublic")
    n_signals = _n_signals(circuit, n_vars)
    tox = {k: rand_fr() for k in ("T", "Ka", "Kb", "Kc", "Kbeta", "Kgamma", "RhoA", "RhoB")} if toxic is None else dict(toxic)
    t, ka, kb, kc, kbeta, kgamma, rho_a, rho_b = (int(tox[k]) % R for k in
                                                  ("T", "Ka", "Kb", "Kc", "Kbeta", "Kgamma", "RhoA", "RhoB"))
    rho_c = rho_a * rho_b % R
    kbg = kbeta * kgamma % R
    nz = len(alphas) - 2                                         # z pol, :210-221
    zl = np.zeros((nz + 1, 4), dtype=np.uint64)
    check(lib().b200_zero_poly(nz, ptr(zl)))
    zpol = limbs_to_ints(zl)
    tl = ints_to_limbs([t])

    def evals(polys):
        n = len(polys[0])
        P = ints_to_limbs([int(x) % R for row in polys for x in row])
        out = np.zeros((len(polys), 4), dtype=np.uint64)
        check(lib().b200_poly_eval_batch(ptr(P), len(polys), n, ptr(tl), ptr(out)))
        return limbs_to_ints(out)

    zt = evals([zpol])[0]
    ra = [rho_a * v % R for v in evals(alphas[:n_signals])]      # rhoAat, :173
    rb = [rho_b * v % R for v in evals(betas[:n_signals])]       # rhoBbt, :181
    rc = [rho_c * v % R for v in evals(gammas[:n_signals])]      # rhoCct, :188
    kt = [(ra[i] + rb[i] + rc[i]) % R for i in range(n_signals)]
    t_pows, t_encr = [], t                                       # G1T = [G, tG, t^2 G, ...], :230-237
    for _ in range(1, len(zpol)):
        t_pows.append(t_encr)
        t_encr = t_encr * t % R
    g1, g2 = bn128.G1(), bn128.G2()
    n = n_signals
    p1 = g1.MulScalarBatch([g1.G], [kb, kbg] + ra + rb + rc + kt + t_pows)
    vkb, g1kbg = p1[0], p1[1]
    A, Bg1, C, K = p1[2:2 + n], p1[2 + n:2 + 2 * n], p1[2 + 2 * n:2 + 3 * n], p1[2 + 3 * n:2 + 4 * n]
    g1t = [g1.G] + p1[2 + 4 * n:]
    p2 = g2.MulScalarBatch([g2.G], [ka, kc, kbg, kgamma, rho_c * zt % R] + rb)
    vka, vkc, g2kbg, g2kg, vkz = p2[:5]
    # the reference's self-check: Affine(G * kt) == Affine(a + bg1 + c), else os.Exit(1)
    ab = _unflatten_g1(g1._op("add", A, Bg1))
    abc = _unflatten_g1(g1._op("add", ab, C))
    if limbs_to_ints(g1._op("affine", abc, out_fe=2)) != limbs_to_ints(g1._op("affine", K, out_fe=2)):
        raise RuntimeError("GenerateTrustedSetup: k != a + b + c (snark.go:194-199)")
    pk = {"G1T": g1t, "A": A, "B": p2[5:], "C": C, "Z": zpol,
          "Ap": g1.MulScalarBatch(A, [ka] * n), "Bp": g1.MulScalarBatch(Bg1, [kb] * n),
          "Cp": g1.MulScalarBatch(C, [kc] * n), "Kp": g1.MulScalarBatch(K, [kbeta] * n)}
    vk = {"Vka": vka, "Vkb": vkb, "Vkc": vkc, "IC": A[:n_public + 1], "G1Kbg": g1kbg, "G2Kbg": g2kbg, "G2Kg": g2kg,
          "Vkz": vkz}
    toxic_out = {"T": t, "Ka": ka, "Kb": kb, "Kc": kc, "Kbeta": kbeta, "Kgamma": kgamma, "RhoA": rho_a, "RhoB": rho_b,
                 "RhoC": rho_c}
    return {"Toxic": toxic_out, "Pk": pk, "Vk": vk}


def VerifyProof(vk, proof, publicSignals, debug=False):
    """snark.VerifyProof(vk, proof, publicSignals, debug) (snark.go:292-372): the twelve pairings of the five checks run
    as ONE batched GPU call (lock-step lanes of a warp), the two F_q^12 products as another; the checks are then
    evaluated in the reference's order, with its ✓/❌ lines when ``debug``."""
    from . import bn128
    bn = bn128.Bn128()
    g1, g2g = bn.G1, bn.G2.G
    vkxpia = vk["IC"][0]
    if len(publicSignals) > len(vk["IC"]) - 1:
        raise IndexError("VerifyProof: len(publicSignals) > len(vk.IC) - 1")     # the reference panics (index out of range)
    if publicSignals:
        terms = g1.MulScalarBatch(list(vk["IC"][1:len(publicSignals) + 1]), list(publicSignals))
        for term in terms:                                                       # :334-337
            vkxpia = g1.Add(vkxpia, term)
    vkx_a = g1.Add(vkxpia, proof["PiA"])
    vkx_a_c = g1.Add(vkx_a, proof["PiC"])
    e = bn.PairingBatch(
        [proof["PiA"], proof["PiAp"], vk["Vkb"], proof["PiBp"], proof["PiC"], proof["PiCp"],
         vkx_a, proof["PiH"], proof["PiC"], vkx_a_c, vk["G1Kbg"], proof["PiKp"]],
        [vk["Vka"], g2g, proof["PiB"], g2g, vk["Vkc"], g2g,
         proof["PiB"], vk["Vkz"], g2g, vk["G2Kbg"], proof["PiB"], vk["G2Kg"]])
    prod = bn.Fq12MulBatch([e[7], e[9]], [e[8], e[10]])
    checks = (
        (e[0] == e[1], "e(piA, Va) == e(piA', g2), valid knowledge commitment for A"),
        (e[2] == e[3], "e(Vb, piB) == e(piB', g2), valid knowledge commitment for B"),
        (e[4] == e[5], "e(piC, Vc) == e(piC', g2), valid knowledge commitment for C"),
        (e[6] == prod[0], "e(Vkx+piA, piB) == e(piH, Vkz) * e(piC, g2), QAP disibility checked"),
        (prod[1] == e[11], "e(Vkx+piA+piC, g2KbetaKgamma) * e(g1KbetaKgamma, piB) == e(piK, g2Kgamma)"),
    )
    for k, (ok, text) in enumerate(checks):
        if debug or (k == 4 and not ok):          # the last failure line is printed unconditionally (snark.go:360-363)
            print(("✓ " if ok else "❌ ") + text)
        if not ok:
            return False
    return True


def _vk_limbs(vk):
    """(IC, Vkb | G1Kbg, Vka | Vkc | Vkz | G2Kbg | G2Kg) in the layout of b200_pinocchio_verify."""
    return (_flatten_g1(vk["IC"]), _flatten_g1([vk["Vkb"], vk["G1Kbg"]]),
            _flatten_g2([vk["Vka"], vk["Vkc"], vk["Vkz"], vk["G2Kbg"], vk["G2Kg"]]))


def VerifyProofBatch(vk, proofs, publicSignals, rho=None, stats=None):
    """VerifyProof for every proofs[i] with publicSignals[i] under one vk, as one random linear combination on the GPU
    (b200_pinocchio_verify_batch): the five checks of every proof raised to random powers and grouped by G2 point, one
    Miller loop per proof and six for the key, one final exponentiation.  rho: per proof, five non-zero 128-bit scalars
    (one per check), secret from whoever made the proofs; drawn here with ``secrets`` when None.  Returns a list of bools,
    False wherever VerifyProof would return False or raise.  ``stats`` (a list) receives the library's counters: proofs in
    the aggregated check, proofs verified one by one, aggregated checks run, Miller loops run."""
    n = len(proofs)
    if len(publicSignals) != n:
        raise ValueError("VerifyProofBatch: one publicSignals list per proof")
    if n == 0:
        return []
    npub = len(publicSignals[0])
    if any(len(p) != npub for p in publicSignals):
        raise ValueError("VerifyProofBatch: every proof needs the same number of public signals")
    if rho is None:
        rho = [[_rand_rho() for _ in range(5)] for _ in range(n)]
    if len(rho) != n or any(len(r) != 5 or any(not 0 < int(x) < (1 << 128) for x in r) for r in rho):
        raise ValueError("VerifyProofBatch: rho must be n lists of five non-zero 128-bit integers")
    ic, vk1, vk2 = _vk_limbs(vk)
    pg1 = _flatten_g1([p[k] for p in proofs for k in _ORDER])
    pb = _flatten_g2([p["PiB"] for p in proofs])
    pub = ints_to_limbs([reduce_scalar(x) for sig in publicSignals for x in sig]) if npub else np.zeros((1, 4), dtype=np.uint64)
    rl = ints_to_limbs([int(x) for r in rho for x in r], 2)
    ok = np.zeros(n, dtype=np.int32)
    st = np.zeros(4, dtype=np.uint64)
    check(lib().b200_pinocchio_verify_batch(ptr(ic), len(vk["IC"]), ptr(vk1), ptr(vk2), n, ptr(pg1), ptr(pb), ptr(pub), npub,
                                            ptr(rl), ptr(ok), ptr(st)))
    if stats is not None:
        stats[:] = [int(x) for x in st]
    return [bool(v == 1) for v in ok]
