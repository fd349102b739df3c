"""ctypes binding of libb200snark.so (the C ABI of include/b200snark.h)."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200snark.so")
CFG_ACC_MODE, ACC_AUTO, ACC_AFFINE, ACC_XYZZ = 1, 0, 1, 2
CFG_TMA_STAGING = 2
CFG_SHARD_W_AB, CFG_SHARD_W_G2, CFG_SHARD_AFFINE_MIN_G1, CFG_SHARD_AFFINE_MIN_G2 = 10, 11, 12, 13
CFG_PAIRING_KERNEL = 5  # b200_pairing_batch: 0 default (one warp per pairing), 1 one thread per pairing, 2 one warp
CFG_PK_CONTEXT = 4    # prove context (0 / 1) of proving keys loaded afterwards: two proofs in flight

B200_OK = 0
ERRORS = {-1: "ENODEVICE", -2: "ECUDA", -3: "EINVAL", -4: "ERANGE", -5: "EDIVZERO", -6: "ENOMEM", -7: "ECOMM"}


class B200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libb200snark error {code} ({ERRORS.get(code, '?')}): {msg}")
        self.code = code


_lib = None

_u64p = ctypes.POINTER(ctypes.c_uint64)
_vp = ctypes.c_void_p
_sz = ctypes.c_size_t
_int = ctypes.c_int
_h = ctypes.c_uint64

_SIGNATURES = {
    "b200_init": [_int],
    "b200_shutdown": [],
    "b200_version": [],
    "b200_config": [_int, _int],
    "b200_g1_bases_load": [_vp, _sz, _int, ctypes.POINTER(_h)],
    "b200_g2_bases_load": [_vp, _sz, _int, ctypes.POINTER(_h)],
    "b200_bases_free": [_h],
    "b200_bases_info": [_h, ctypes.POINTER(_sz), ctypes.POINTER(_int), ctypes.POINTER(_int), ctypes.POINTER(_int)],
    "b200_bases_acc_mode": [_h, ctypes.POINTER(_int)],
    "b200_g1_msm": [_h, _vp, _sz, _vp],
    "b200_g2_msm": [_h, _vp, _sz, _vp],
    "b200_msm_device": [_h, _vp, _sz, _int, _vp, _vp],
    "b200_g1_sum_partials": [_vp, _sz, _vp, _vp],
    "b200_g2_sum_partials": [_vp, _sz, _vp, _vp],
    "b200_g1_mul_batch": [_vp, _vp, _sz, _vp],
    "b200_g2_mul_batch": [_vp, _vp, _sz, _vp],
    "b200_g1_mul_batch_bcast": [_vp, _vp, _sz, _vp],
    "b200_g2_mul_batch_bcast": [_vp, _vp, _sz, _vp],
    "b200_poly_mul": [_vp, _sz, _vp, _sz, _vp],
    "b200_poly_div": [_vp, _sz, _vp, _sz, _vp, _vp],
    "b200_groth16_pk_load": [_vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _sz, _int,
                             ctypes.POINTER(_h)],
    "b200_groth16_prove": [_h, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _vp, _vp],
    "b200_pinocchio_pk_load": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _sz, _int,
                               ctypes.POINTER(_h)],
    "b200_pinocchio_prove": [_h, _vp, _sz, _vp, _sz, _vp, _vp],
    "b200_pinocchio_pk_load_shard": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _sz, _int, _int, _int,
                                     ctypes.POINTER(_h)],
    "b200_pinocchio_prove_record_device": [_h, _vp, _sz, _vp, _sz, _vp],
    "b200_pinocchio_finalize_records": [_vp, _int, _vp, _vp],
    "b200_pk_free": [_h],
    "b200_groth16_prove_device": [_h, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _vp],
    "b200_groth16_pk_load_shard": [_vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _sz, _int,
                                   _int, _int, ctypes.POINTER(_h)],
    "b200_groth16_finalize_device": [_h, _vp, _int, _vp, _vp, _vp, _vp],
    "b200_groth16_shard_info": [_h, _vp],
    "b200_comm_unique_id": [_vp],
    "b200_comm_init": [_vp, _int, _int],
    "b200_comm_destroy": [],
    "b200_poly_add": [_vp, _sz, _vp, _sz, _vp],
    "b200_poly_sub": [_vp, _sz, _vp, _sz, _vp],
    "b200_poly_eval": [_vp, _sz, _vp, _vp],
    "b200_poly_eval_batch": [_vp, _sz, _sz, _vp, _vp],
    "b200_zero_poly": [_sz, _vp],
    "b200_pairing_batch": [_vp, _vp, _sz, _vp],
    "b200_fq12_mul_batch": [_vp, _vp, _sz, _vp],
    "b200_groth16_verify": [_vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.POINTER(_int)],
    "b200_groth16_verify_batch": [_vp, _sz, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp],
    "b200_pinocchio_verify": [_vp, _sz, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp],
    "b200_pinocchio_verify_batch": [_vp, _sz, _vp, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp],
    "b200_r1cs_to_qap": [_vp, _vp, _vp, _sz, _sz, _vp, _vp, _vp, _vp],
    "b200_combine_polynomials": [_vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp],
    "b200_g1_add_batch": [_vp, _vp, _sz, _vp], "b200_g2_add_batch": [_vp, _vp, _sz, _vp],
    "b200_g1_double_batch": [_vp, _sz, _vp], "b200_g2_double_batch": [_vp, _sz, _vp],
    "b200_g1_neg_batch": [_vp, _sz, _vp], "b200_g2_neg_batch": [_vp, _sz, _vp],
    "b200_g1_affine_batch": [_vp, _sz, _vp], "b200_g2_affine_batch": [_vp, _sz, _vp],
    "b200_r1cs_load": [_sz, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.POINTER(_h)],
    "b200_r1cs_free": [_h],
    "b200_qap_px": [_h, _vp, _sz, _vp, _vp, _vp, _vp],
    "b200_qap_eval_at": [_h, _vp, _sz, _vp, _vp, _vp, _vp],
    "b200_interpolate": [_vp, _sz, _vp],
    "b200_groth16_prove_witness": [_h, _h, _vp, _sz, _vp, _vp, _vp, _vp, _vp],
    "b200_profile": [_int],
    "b200_profile_read": [ctypes.POINTER(ctypes.c_double)],
}


def lib():
    """Load the CUDA library; fail loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "go-snark-study_b200 has no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        L.b200_last_error.restype = ctypes.c_char_p
        for name, args in _SIGNATURES.items():
            if not hasattr(L, name):
                continue                       # newer header than library: symbol test catches it
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = ctypes.c_int
        _lib = L
    return _lib


def check(rc):
    if rc != B200_OK:
        raise B200Error(rc, lib().b200_last_error().decode())


def init(device=None):
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "-1"))
    check(lib().b200_init(device))


# ---- big-int <-> limb marshalling (what the cgo shim does with big.Int.Bits()) ----
def ints_to_limbs(vals, words_per_val=4):
    """list[int] -> contiguous uint64 array (len, words_per_val), little endian."""
    nbytes = 8 * words_per_val
    buf = bytearray(len(vals) * nbytes)
    for i, v in enumerate(vals):
        buf[i * nbytes:(i + 1) * nbytes] = int(v).to_bytes(nbytes, "little")
    return np.frombuffer(bytes(buf), dtype=np.uint64).reshape(len(vals), words_per_val).copy()


def limbs_to_ints(arr, words_per_val=4):
    raw = np.ascontiguousarray(arr, dtype=np.uint64).tobytes()
    nbytes = 8 * words_per_val
    return [int.from_bytes(raw[i:i + nbytes], "little") for i in range(0, len(raw), nbytes)]


def ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)
