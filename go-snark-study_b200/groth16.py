"""Host mirror of the reference's ``groth16`` package prove path
(groth16/groth16.go:225-278) over libb200snark.

    pk  = {"G1": {"Alpha","Beta","Delta","At","BACGamma"}, "G2": {"Beta","Delta","BACGamma"},
           "BACDelta", "PowersTauDelta", "Z"}            (field names of groth16.Pk, groth16.go:15-32)
    proof = GenerateProofs(circuit, pk, w, px)           -> {"PiA","PiB","PiC"} Jacobian tuples

``circuit`` only needs ``NVars`` and ``NPublic`` (all the reference reads from it).
The proving key is uploaded once (``LoadProvingKey``) and cached per pk object.
"""
import secrets

import numpy as np

from . import _lib
from ._lib import check, ints_to_limbs, lib, ptr
from .bn128 import R, _flatten_g1, _flatten_g2, _unflatten_g1, _unflatten_g2, reduce_scalar


def _attr(obj, name):
    return obj[name] if isinstance(obj, dict) else getattr(obj, name)


def _n_signals(circuit, default):
    """len(circuit.Signals) (groth16.go:164, snark.go:171) for dict- and object-style circuits; NVars if absent."""
    if isinstance(circuit, dict):
        sig = circuit.get("Signals")
    else:
        sig = getattr(circuit, "Signals", None)
    return len(sig) if sig is not None else default


def rand_fr():
    """Fq.Rand over r (fields/fq.go:116-132): bitlen/8-1 = 30 random bytes, mod r."""
    return int.from_bytes(secrets.token_bytes(30), "big") % R


class DeviceProvingKey:
    def __init__(self, pk, n_vars, n_public, window_bits=0):
        m = n_vars
        g1, g2 = pk["G1"], pk["G2"]
        assert len(g1["At"]) >= m and len(g1["BACGamma"]) >= m and len(g2["BACGamma"]) >= m and len(pk["BACDelta"]) >= m
        at = _flatten_g1(g1["At"][:m])
        b1 = _flatten_g1(g1["BACGamma"][:m])
        b2 = _flatten_g2(g2["BACGamma"][:m])
        cd = _flatten_g1(pk["BACDelta"][:m])
        ptd = _flatten_g1(pk["PowersTauDelta"])
        z = ints_to_limbs([int(x) % R for x in pk["Z"]])
        a1, be1, d1 = (_flatten_g1([g1[k]]) for k in ("Alpha", "Beta", "Delta"))
        be2, d2 = (_flatten_g2([g2[k]]) for k in ("Beta", "Delta"))
        h = _lib._h(0)
        check(lib().b200_groth16_pk_load(ptr(at), ptr(b1), ptr(b2), ptr(cd), m, ptr(ptd), len(pk["PowersTauDelta"]),
                                         ptr(z), len(pk["Z"]), ptr(a1), ptr(be1), ptr(d1), ptr(be2), ptr(d2),
                                         n_public, window_bits, h))
        self.handle = h.value
        self.m = m

    def prove_limbs(self, w_limbs, px_limbs, r, s):
        pa = np.zeros(12, dtype=np.uint64)
        pb = np.zeros(24, dtype=np.uint64)
        pc = np.zeros(12, dtype=np.uint64)
        rr, ss = ints_to_limbs([r]), ints_to_limbs([s])
        check(lib().b200_groth16_prove(self.handle, ptr(w_limbs), w_limbs.shape[0], ptr(px_limbs), px_limbs.shape[0],
                                       ptr(rr), ptr(ss), ptr(pa), ptr(pb), ptr(pc)))
        return {"PiA": _unflatten_g1(pa)[0], "PiB": _unflatten_g2(pb)[0], "PiC": _unflatten_g1(pc)[0]}

    def free(self):
        if self.handle:
            check(lib().b200_pk_free(self.handle))
            self.handle = 0


class KeyCache:
    """Implicit proving-key cache of the drop-in ``GenerateProofs(circuit, pk, w, px)`` form (the reference takes the key
    by value on every call, groth16.go:225; uploading 384·n bytes and precomputing window tables per call would
    dominate).  An entry holds a STRONG reference to the caller's ``pk`` object and is matched by identity
    (``entry.pk is pk``) plus the shape it was loaded with — never by ``id()`` alone: a freed dict's address can be
    handed to a different key (round-1 bug: a proof under a stale key).  At most ``capacity`` keys stay resident;
    evicting one frees its device tables.  A caller that mutates ``pk`` in place must call ``Forget(pk)``."""

    def __init__(self, factory, capacity=2):
        self.factory, self.capacity, self.entries = factory, capacity, []

    def get(self, circuit, pk, window_bits=0):
        shape = (_attr(circuit, "NVars"), _attr(circuit, "NPublic"), window_bits)
        for k, (epk, eshape, dpk) in enumerate(self.entries):
            if epk is pk and eshape == shape:
                self.entries.append(self.entries.pop(k))          # most recently used last
                return dpk
        dpk = self.factory(pk, shape[0], shape[1], window_bits)
        self.entries.append((pk, shape, dpk))
        while len(self.entries) > self.capacity:
            self.entries.pop(0)[2].free()
        return dpk

    def forget(self, pk=None):
        keep = []
        for e in self.entries:
            if pk is None or e[0] is pk:
                e[2].free()
            else:
                keep.append(e)
        self.entries = keep


_pk_cache = KeyCache(lambda pk, m, npub, c: DeviceProvingKey(pk, m, npub, c))


def LoadProvingKey(circuit, pk, window_bits=0):
    """Explicit handle form: the returned DeviceProvingKey can be passed as ``pk`` to GenerateProofs."""
    return _pk_cache.get(circuit, pk, window_bits)


def Forget(pk=None):
    """Free the device copy of ``pk`` (all cached keys when None)."""
    _pk_cache.forget(pk)


def GenerateProofs(circuit, pk, w, px, r=None, s=None):
    """groth16.GenerateProofs(circuit, pk, w, px) (groth16.go:225).  r, s default
    to fresh randomness like the reference; pass them for reproducible proofs."""
    dpk = pk if isinstance(pk, DeviceProvingKey) else LoadProvingKey(circuit, pk)
    r = rand_fr() if r is None else int(r) % R
    s = rand_fr() if s is None else int(s) % R
    wl = ints_to_limbs([reduce_scalar(x) for x in w])
    pl = ints_to_limbs([int(x) % R for x in px])
    return dpk.prove_limbs(wl, pl, r, s)


def GenerateTrustedSetup(witnessLength, circuit, alphas, betas, gammas, toxic=None):
    """groth16.GenerateTrustedSetup (groth16/groth16.go:94-222) with the heavy loops on the GPU: the
    Eval(alphas[i], tau) evaluations (b200_poly_eval_batch), the z polynomial (b200_zero_poly) and every
    G.MulScalar(generator, k) (b200_g{1,2}_mul_batch_bcast — the reference's own double-and-add, so the
    points are X,Y,Z-identical to the reference's for the same toxic values).  ``toxic`` = dict
    T, Kalpha, Kbeta, Kgamma, Kdelta; drawn like the reference (Fq.Rand) when omitted.  ``witnessLength`` is
    unused, as in the reference.  Returns {"Toxic", "Pk", "Vk"} shaped like groth16.Setup."""
    from . import bn128
    from ._lib import limbs_to_ints
    n_vars, n_public = _attr(circuit, "NVars"), _attr(circuit, "NPublic")
    n_signals = _n_signals(circuit, n_vars)
    tox = {k: rand_fr() for k in ("T", "Kalpha", "Kbeta", "Kgamma", "Kdelta")} if toxic is None else toxic
    t, ka, kb, kg, kd = (int(tox[k]) % R for k in ("T", "Kalpha", "Kbeta", "Kgamma", "Kdelta"))
    if kg == 0 or kd == 0:
        raise ValueError("GenerateTrustedSetup: Kgamma and Kdelta must be invertible mod r (groth16.go:151,201)")
    m = len(alphas)
    nz = m - 2                                                   # z pol: prod_{i=1}^{len(alphas)-2} (x - i), :122-132
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
    inv_delta = pow(kd, -1, R)
    zt_inv_delta = inv_delta * zt % R
    g1, g2 = bn128.G1(), bn128.G2()
    ptd_k, t_encr = [zt_inv_delta], t                            # :139-149
    for _ in range(1, len(zpol)):
        ptd_k.append(t_encr * zt_inv_delta % R)
        t_encr = t_encr * t % R
    at = evals(alphas[:n_signals])
    bt = evals(betas[:n_signals])
    ct = evals(gammas[:n_signals])
    inv_gamma = pow(kg, -1, R)
    c_k = [inv_delta * ((at[i] * kb + bt[i] * ka + ct[i]) % R) % R for i in range(n_public + 1, n_vars)]     # :181-200
    ic_k = [inv_gamma * ((at[i] * kb + bt[i] * ka + ct[i]) % R) % R for i in range(n_public + 1)]            # :202-219
    # one batched scalar multiplication of the G1 generator for every G1 point of the setup
    k1 = ptd_k + [ka, kb, kd] + at + bt + c_k + ic_k
    p1 = g1.MulScalarBatch([g1.G], k1)
    k2 = [kb, kg, kd] + bt
    p2 = g2.MulScalarBatch([g2.G], k2)
    o = 0
    ptd = p1[o:o + len(ptd_k)]; o += len(ptd_k)
    alpha1, beta1, delta1 = p1[o:o + 3]; o += 3
    At = p1[o:o + len(at)]; o += len(at)
    B1 = p1[o:o + len(bt)]; o += len(bt)
    Cd = p1[o:o + len(c_k)]; o += len(c_k)
    IC = p1[o:o + len(ic_k)]
    beta2, gamma2, delta2 = p2[:3]
    pk = {"BACDelta": [(0, 0, 0)] * (n_public + 1) + Cd, "Z": zpol, "PowersTauDelta": ptd,
          "G1": {"Alpha": alpha1, "Beta": beta1, "Delta": delta1, "At": At, "BACGamma": B1},
          "G2": {"Beta": beta2, "Gamma": gamma2, "Delta": delta2, "BACGamma": p2[3:]}}
    vk = {"IC": IC, "G1": {"Alpha": alpha1}, "G2": {"Beta": beta2, "Gamma": gamma2, "Delta": delta2}}
    return {"Toxic": {"T": t, "Kalpha": ka, "Kbeta": kb, "Kgamma": kg, "Kdelta": kd}, "Pk": pk, "Vk": vk}


def VerifyProof(vk, proof, publicSignals, debug=False):
    """groth16.VerifyProof(vk, proof, publicSignals, debug) (groth16/groth16.go:281-305) on the GPU:
    vk = {"IC", "G1": {"Alpha"}, "G2": {"Beta", "Gamma", "Delta"}}, proof = {"PiA", "PiB", "PiC"}."""
    import ctypes
    ic = _flatten_g1(vk["IC"])
    pub = ints_to_limbs([reduce_scalar(x) for x in publicSignals]) if len(publicSignals) else np.zeros((1, 4), dtype=np.uint64)
    ok = ctypes.c_int(0)
    check(lib().b200_groth16_verify(ptr(ic), len(vk["IC"]), ptr(_flatten_g1([vk["G1"]["Alpha"]])),
                                    ptr(_flatten_g2([vk["G2"]["Beta"]])), ptr(_flatten_g2([vk["G2"]["Gamma"]])),
                                    ptr(_flatten_g2([vk["G2"]["Delta"]])), ptr(_flatten_g1([proof["PiA"]])),
                                    ptr(_flatten_g2([proof["PiB"]])), ptr(_flatten_g1([proof["PiC"]])), ptr(pub),
                                    len(publicSignals), ctypes.byref(ok)))
    if debug:
        print("✓ groth16 verification passed" if ok.value else "❌ groth16 verification not passed")
    return bool(ok.value)


def _rand_rho():
    """A uniformly random non-zero 128-bit batching scalar (16 bytes from the OS CSPRNG, 0 rejected)."""
    while True:
        v = int.from_bytes(secrets.token_bytes(16), "little")
        if v:
            return v


def VerifyProofBatch(vk, proofs, publicSignals, rho=None, stats=None):
    """VerifyProof for every proofs[i] with publicSignals[i] under one vk, as one random linear combination on the GPU
    (b200_groth16_verify_batch): one Miller loop per proof, three for the key, one final exponentiation.  rho: one non-zero
    128-bit scalar per proof, secret from whoever made the proofs; drawn here with ``secrets`` when None.  Returns a
    list of bools, False wherever VerifyProof would return False or raise.  ``stats`` (a list) receives the library's
    counters: proofs in the aggregated check, proofs verified one by one, aggregated checks run, Miller loops run."""
    n = len(proofs)
    if len(publicSignals) != n:
        raise ValueError("VerifyProofBatch: one publicSignals list per proof")
    if n == 0:
        return []
    npub = len(publicSignals[0])
    if any(len(p) != npub for p in publicSignals):
        raise ValueError("VerifyProofBatch: every proof needs the same number of public signals")
    if rho is None:
        rho = [_rand_rho() for _ in range(n)]
    if len(rho) != n or any(not 0 < int(r) < (1 << 128) for r in rho):
        raise ValueError("VerifyProofBatch: rho must be n non-zero 128-bit integers")
    pub = ints_to_limbs([reduce_scalar(x) for sig in publicSignals for x in sig]) if npub else np.zeros((1, 4), dtype=np.uint64)
    rl = ints_to_limbs(rho, 2)
    ok = np.zeros(n, dtype=np.int32)
    st = np.zeros(4, dtype=np.uint64)
    check(lib().b200_groth16_verify_batch(ptr(_flatten_g1(vk["IC"])), len(vk["IC"]), ptr(_flatten_g1([vk["G1"]["Alpha"]])),
                                          ptr(_flatten_g2([vk["G2"]["Beta"]])), ptr(_flatten_g2([vk["G2"]["Gamma"]])),
                                          ptr(_flatten_g2([vk["G2"]["Delta"]])), n,
                                          ptr(_flatten_g1([p["PiA"] for p in proofs])), ptr(_flatten_g2([p["PiB"] for p in proofs])),
                                          ptr(_flatten_g1([p["PiC"] for p in proofs])), ptr(pub), npub, ptr(rl), ptr(ok), ptr(st)))
    if stats is not None:
        stats[:] = [int(x) for x in st]
    return [bool(v == 1) for v in ok]
