"""ctypes binding of libb200g16.so — the same C-ABI a cgo shim binds (include/b200g16.h).

This module is plumbing for tests / bench / the Python host mirror; it contains no
arithmetic and NO fallback: if the shared library (built by __graft_entry__.build()) is
missing, or no sm_100 device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200g16.so")

DIF, DIT = 0, 1


class B200Error(RuntimeError):
    pass


_lib = None

_u64p = C.POINTER(C.c_uint64)
_vp = C.c_void_p
_sz = C.c_size_t

# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "b200g16_version": (C.c_int, []),
    "b200g16_last_error": (C.c_char_p, []),
    "b200g16_init": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "b200g16_destroy": (None, [_vp]),
    "b200g16_launch_count": (C.c_uint64, [_vp]),
    "b200g16_last_timings": (C.c_int, [_vp, C.POINTER(C.c_float), C.c_int]),
    "b200g16_set_msm_window": (C.c_int, [_vp, C.c_int]),
    "b200g16_set_msm_batch_affine": (C.c_int, [_vp, C.c_int, C.c_int, C.c_uint]),
    "b200g16_bases_upload_g1": (C.c_int, [_vp, _vp, _sz, C.POINTER(_vp)]),
    "b200g16_bases_upload_g2": (C.c_int, [_vp, _vp, _sz, C.POINTER(_vp)]),
    "b200g16_bases_free": (None, [_vp]),
    "b200g16_bases_len": (_sz, [_vp]),
    "b200g16_bases_precompute": (C.c_int, [_vp, _vp, C.c_int]),
    "b200g16_bases_window": (C.c_int, [_vp]),
    "b200g16_msm_plan": (C.c_int, [_vp, _vp, _sz, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "b200g16_bases_download": (C.c_int, [_vp, _sz, _sz, _vp]),
    "b200g16_bases_copy": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "b200g16_fixed_base_mul_g1": (C.c_int, [_vp, _vp, _vp, _sz, _vp]),
    "b200g16_fixed_base_mul_g2": (C.c_int, [_vp, _vp, _vp, _sz, _vp]),
    "b200g16_bases_from_scalars_g1": (C.c_int, [_vp, _vp, _vp, _sz, C.POINTER(_vp)]),
    "b200g16_bases_from_scalars_g2": (C.c_int, [_vp, _vp, _vp, _sz, C.POINTER(_vp)]),
    "b200g16_modmul_probe": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "b200g16_pipe_probe": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "b200g16_fp52_probe": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "b200g16_msm_g1": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "b200g16_msm_g2": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "b200g16_msm_g1_dev": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "b200g16_msm_g1_begin": (C.c_int, [_vp, _vp, _sz, _vp, _sz, C.POINTER(C.c_int)]),
    "b200g16_msm_g1_begin_dev": (C.c_int, [_vp, _vp, _sz, _vp, _sz, C.POINTER(C.c_int)]),
    "b200g16_msm_g1_end": (C.c_int, [_vp, C.c_int, _vp]),
    "b200g16_msm_g2_dev": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "b200g16_msm_g1_batch": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _sz, _vp]),
    "b200g16_msm_g2_batch": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _sz, _vp]),
    "b200g16_msm_g1_batch_dev": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _sz, _vp]),
    "b200g16_msm_g2_batch_dev": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _sz, _vp]),
    "b200g16_ntt": (C.c_int, [_vp, _vp, C.c_uint, C.c_int, C.c_int, C.c_int]),
    "b200g16_ntt_dev": (C.c_int, [_vp, _vp, C.c_uint, C.c_uint, C.c_int, C.c_int, C.c_int]),
    "b200g16_compute_h": (C.c_int, [_vp, _vp, _vp, _vp, _sz, C.c_uint, _vp]),
    "b200g16_compute_h_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint]),
    "b200g16_keccak_f_batch": (C.c_int, [_vp, _vp, _sz]),
    "b200g16_keccak_f_batch_dev": (C.c_int, [_vp, _vp, _sz]),
    "b200g16_keccak_sponge_batch": (C.c_int, [_vp, _vp, _sz, _sz, _vp, _sz]),
    "b200g16_keccak_duplex_batch": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp, _vp]),
    "b200g16_keccak_duplex_batch_dev": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp, _sz, _vp, _vp]),
    "b200g16_keccak_merkle_paths": (C.c_int, [_vp, _vp, _sz, _vp, _vp, _vp, C.c_uint, _sz, _vp, _vp, _vp]),
    "b200g16_keccak_merkle_paths_dev": (C.c_int, [_vp, _vp, _sz, _vp, _vp, _vp, C.c_uint, _sz, _vp, _vp, _vp]),
    "b200g16_pk_upload": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "b200g16_pk_free": (None, [_vp]),
    "b200g16_prove": (C.c_int, [_vp, _vp, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "b200g16_prove_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200g16_prove_batch": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "b200g16_prove_batch_dev": (C.c_int, [_vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200g16_prove_h_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200g16_h_pointwise_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint]),
    "b200g16_prove_begin_dev": (C.c_int, [_vp, _vp, _vp]),
    "b200g16_prove_end_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "b200g16_prove_finish": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200g16_setup": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200g16_setup_wire_polys": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "b200g16_pairing_check": (C.c_int, [_vp, _vp, _vp, _sz, C.POINTER(C.c_int)]),
    "b200g16_pair": (C.c_int, [_vp, _vp, _vp, _sz, _vp]),
    "b200g16_verify": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, C.POINTER(C.c_int)]),
    "b200g16_verify_batch": (C.c_int, [_vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, C.POINTER(C.c_int), _vp]),
    "b200g16_g1_decode": (C.c_int, [_vp, _vp, _sz, C.c_int, _vp, _vp]),
    "b200g16_g2_decode": (C.c_int, [_vp, _vp, _sz, C.c_int, C.c_int, _vp, _vp]),
    "b200g16_g1_encode": (C.c_int, [_vp, _vp, _sz, C.c_int, _vp]),
    "b200g16_g2_encode": (C.c_int, [_vp, _vp, _sz, C.c_int, _vp]),
    "b200g16_group_init": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(_vp)]),
    "b200g16_group_destroy": (None, [_vp]),
    "b200g16_group_size": (C.c_int, [_vp]),
    "b200g16_group_ctx": (_vp, [_vp, C.c_int]),
    "b200g16_host_register": (C.c_int, [_vp, _sz]),
    "b200g16_host_unregister": (C.c_int, [_vp]),
    "b200g16_group_bases_upload_g1": (C.c_int, [_vp, _vp, _sz, C.POINTER(_vp)]),
    "b200g16_group_bases_upload_g2": (C.c_int, [_vp, _vp, _sz, C.POINTER(_vp)]),
    "b200g16_group_bases_precompute": (C.c_int, [_vp, _vp, C.c_int]),
    "b200g16_group_bases_free": (None, [_vp]),
    "b200g16_group_msm_g1": (C.c_int, [_vp, _vp, _vp, _sz, _vp]),
    "b200g16_group_msm_g2": (C.c_int, [_vp, _vp, _vp, _sz, _vp]),
    "b200g16_group_pk_upload": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "b200g16_group_pk_free": (None, [_vp]),
    "b200g16_group_prove": (C.c_int, [_vp, _vp, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "b200g16_group_pk_replicate": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "b200g16_group_prove_batch": (C.c_int, [_vp, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "b200g16_dist_h_init": (C.c_int, [_vp, C.c_uint, C.c_int, C.c_int, _vp]),
    "b200g16_dist_h_open": (C.c_int, [_vp, _vp]),
    "b200g16_dist_h_load": (C.c_int, [_vp, _vp, _vp, _vp]),
    "b200g16_dist_h_slice": (_vp, [_vp, C.c_int]),
    "b200g16_dist_h_phase": (C.c_int, [_vp, C.c_int]),
    "b200g16_dist_h_close": (None, [_vp]),
    "b200g16_g1_add": (C.c_int, [_vp, _vp, _vp]),
    "b200g16_g2_add": (C.c_int, [_vp, _vp, _vp]),
    "b200g16_g1_scalar_mul": (C.c_int, [_vp, _vp, _vp]),
    "b200g16_g2_scalar_mul": (C.c_int, [_vp, _vp, _vp]),
}


def load():
    """dlopen the library (raises if it has not been built — there is no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


# struct b200g16_keccak_digest: keccakSponge.Digest between calls (25 little-endian lanes, then the two positions)
KECCAK_DIGEST = np.dtype([("state", "<u8", (25,)), ("absorb_pos", "<u4"), ("squeeze_pos", "<u4")])
KECCAK_RATE = 136
# sponges up to which b200g16_keccak_duplex_batch runs one warp per sponge (DUPLEX_WARP_MAX in csrc/keccak.cu)
KECCAK_DUPLEX_WARP_MAX = 8192


def keccak_digests(n, tags=None):
    """n fresh digests: NewKeccak, or NewKeccakWithTag(tags[i]) for sponge i (tags: n byte strings of <= 64 bytes, or
    one for all).  Pass them to keccak_duplex_batch with tag=None to start each sponge from its own tag."""
    d = np.zeros(n, dtype=KECCAK_DIGEST)
    d["squeeze_pos"] = KECCAK_RATE
    if tags is not None:
        if isinstance(tags, (bytes, bytearray)):
            tags = [tags] * n
        if len(tags) != n:
            raise B200Error("keccak_digests: one tag per sponge")
        raw = d.view(np.uint8).reshape(n, KECCAK_DIGEST.itemsize)
        for i, t in enumerate(tags):
            if len(t) > 64:
                raise B200Error("keccak_digests: a tag has at most 64 bytes")
            raw[i, KECCAK_RATE:KECCAK_RATE + len(t)] = np.frombuffer(bytes(t), dtype=np.uint8)
    return d


def duplex_script(ops):
    """[("absorb", len) | ("squeeze", len), ...] -> (struct b200g16_duplex_op array, absorbed bytes, squeezed bytes)"""
    kinds = {"absorb": 0, "squeeze": 1}
    arr = np.zeros((len(ops), 2), dtype=np.uint32)
    for k, (kind, n) in enumerate(ops):
        if kind not in kinds or not 0 <= int(n) < 1 << 32:
            raise B200Error(f"duplex op {k}: {kind!r}, {n!r}")
        arr[k] = kinds[kind], int(n)
    return arr, int(arr[arr[:, 0] == 0, 1].sum()), int(arr[arr[:, 0] == 1, 1].sum())


# b200g16_set_msm_batch_affine(mode, levels, min_pairs) as a fresh ctx has it
MSM_BATCH_AFFINE_DEFAULT = (0, 3, 192)


def _check(status):
    if status != 0:
        raise B200Error(f"libb200g16 error {status}: {load().b200g16_last_error().decode()}")


def _dp(dev_ptr):
    """A raw device pointer for the library.  The library works on its OWN (non-blocking) streams and cannot know which
    stream produced the data, so device-side work the caller still has in flight on torch's streams (a clone, a random
    fill) is drained first — the C-ABI's contract for device pointers (include/b200g16.h) is "the memory is ready"."""
    import sys
    torch = sys.modules.get("torch")
    if torch is not None and torch.cuda.is_initialized():
        torch.cuda.current_stream().synchronize()   # the producer's stream only: an open b200g16_msm_g1_begin keeps running
    return _vp(int(dev_ptr))


def _ptr(a):
    return a.ctypes.data_as(_vp)


def _u64(a, cols=None):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    if cols is not None:
        a = a.reshape(-1, cols)
    return a


# ---- host-only helpers (no GPU needed) -----------------------------------------------------
def g1_add(a, b):
    out = np.zeros(8, dtype=np.uint64)
    _check(load().b200g16_g1_add(_ptr(_u64(a)), _ptr(_u64(b)), _ptr(out)))
    return out


def g2_add(a, b):
    out = np.zeros(16, dtype=np.uint64)
    _check(load().b200g16_g2_add(_ptr(_u64(a)), _ptr(_u64(b)), _ptr(out)))
    return out


def g1_scalar_mul(p, k):
    out = np.zeros(8, dtype=np.uint64)
    _check(load().b200g16_g1_scalar_mul(_ptr(_u64(p)), _ptr(_u64(k)), _ptr(out)))
    return out


def g2_scalar_mul(p, k):
    out = np.zeros(16, dtype=np.uint64)
    _check(load().b200g16_g2_scalar_mul(_ptr(_u64(p)), _ptr(_u64(k)), _ptr(out)))
    return out


# bases handles of struct b200g16_setup_out, in field order
SETUP_VECTORS = ("a", "b", "k", "z", "b2", "vk_k", "ped_basis", "ped_basis_exp_sigma")


class PkDesc(C.Structure):
    """struct b200g16_pk_desc (include/b200g16.h)"""
    _fields_ = [
        ("log2_domain", C.c_uint), ("n_wires", _sz),
        ("g1_a", _vp), ("g1_b", _vp), ("g1_k", _vp), ("g1_z", _vp), ("g2_b", _vp),
        ("res_a", _vp), ("res_b", _vp), ("res_k", _vp), ("res_z", _vp), ("res_b2", _vp),
        ("n_a", _sz), ("n_b", _sz), ("n_k", _sz), ("n_z", _sz),
        ("g1_alpha", _vp), ("g1_beta", _vp), ("g1_delta", _vp), ("g2_beta", _vp), ("g2_delta", _vp),
        ("infinity_a", _vp), ("infinity_b", _vp), ("k_skip", _vp),
        ("partial", C.c_int), ("off_a", _sz), ("off_b", _sz), ("off_k", _sz), ("off_z", _sz),
        ("precompute", C.c_int),
    ]


class R1csDesc(C.Structure):
    """struct b200g16_r1cs_desc (include/b200g16.h)"""
    _fields_ = [("n_constraints", _sz), ("n_wires", _sz), ("n_public", _sz), ("coeffs", _vp), ("n_coeffs", _sz),
                ("l_row", _vp), ("l_wire", _vp), ("l_coeff", _vp), ("r_row", _vp), ("r_wire", _vp), ("r_coeff", _vp),
                ("o_row", _vp), ("o_wire", _vp), ("o_coeff", _vp), ("private_committed", _vp),
                ("n_private_committed", _sz), ("commitment_wire", C.c_int64)]


class Toxic(C.Structure):
    """struct b200g16_toxic (include/b200g16.h)"""
    _fields_ = [(n, C.c_uint64 * 4) for n in ("tau", "alpha", "beta", "gamma", "delta", "sigma")]


class SetupOut(C.Structure):
    """struct b200g16_setup_out (include/b200g16.h)"""
    _fields_ = ([("log2_domain", C.c_uint)] + [(n, _vp) for n in SETUP_VECTORS]
                + [(n, C.c_uint64 * 8) for n in ("g1_alpha", "g1_beta", "g1_delta")]
                + [(n, C.c_uint64 * 16) for n in ("g2_beta", "g2_delta", "g2_gamma", "ped_g", "ped_g_sigma_neg")])


def _r1cs_desc(r):
    """struct b200g16_r1cs_desc from a mapping with the fields of groth16.SparseR1CS -> (desc, arrays to keep alive)"""
    keep = {"coeffs": _u64(r["coeffs"], 4), "private_committed": np.ascontiguousarray(r["private_committed"], np.uint32)}
    for p in "lro":
        keep[p + "_row"] = np.ascontiguousarray(r[p + "_row"], dtype=np.uint64)
        keep[p + "_wire"] = np.ascontiguousarray(r[p + "_wire"], dtype=np.uint32)
        keep[p + "_coeff"] = np.ascontiguousarray(r[p + "_coeff"], dtype=np.uint32)
    m = len(keep["l_row"]) - 1
    for p in "lro":    # the library reads row[0 .. m] and the first row[m] terms of every matrix
        row = keep[p + "_row"]
        if m < 0 or len(row) != m + 1:
            raise B200Error(f"r1cs: {p}_row has {len(row)} entries, l_row {m + 1}: one row array per matrix, same length")
        if len(keep[p + "_wire"]) < row[-1] or len(keep[p + "_coeff"]) < row[-1]:
            raise B200Error(f"r1cs: {p}_row ends at {int(row[-1])} but {p}_wire / {p}_coeff hold fewer terms")
    d = R1csDesc()
    d.n_constraints = m
    d.n_wires, d.n_public = int(r["nb_wires"]), int(r["nb_public"])
    d.n_coeffs = keep["coeffs"].shape[0]
    d.n_private_committed = keep["private_committed"].shape[0]
    d.commitment_wire = int(r["commitment_wire"])
    for name, a in keep.items():
        setattr(d, name, _ptr(a) if a.size else None)
    return d, keep


class VkDesc(C.Structure):
    """struct b200g16_vk_desc (include/b200g16.h)"""
    _fields_ = [("g1_alpha", _vp), ("g2_beta", _vp), ("g2_gamma", _vp), ("g2_delta", _vp), ("g1_k", _vp), ("n_k", _sz),
                ("ped_g", _vp), ("ped_g_sigma_neg", _vp)]


def _vk_desc(alpha, beta2, gamma2, delta2, K, ped_g, ped_g_sigma_neg):
    """struct b200g16_vk_desc from numpy points -> (desc, arrays to keep alive during the call)"""
    keep = [_u64(alpha).reshape(8), _u64(beta2).reshape(16), _u64(gamma2).reshape(16), _u64(delta2).reshape(16),
            _u64(K, 8)] + [None if v is None else _u64(v).reshape(16) for v in (ped_g, ped_g_sigma_neg)]
    d = VkDesc()
    d.g1_alpha, d.g2_beta, d.g2_gamma, d.g2_delta, d.g1_k = [_ptr(a) for a in keep[:5]]
    d.n_k = keep[4].shape[0]
    d.ped_g = _ptr(keep[5]) if keep[5] is not None else None
    d.ped_g_sigma_neg = _ptr(keep[6]) if keep[6] is not None else None
    return d, keep


class ProofOut(C.Structure):
    """struct b200g16_proof (include/b200g16.h)"""
    _fields_ = [
        ("ar", C.c_uint64 * 8), ("bs", C.c_uint64 * 16), ("krs", C.c_uint64 * 8),
        ("msm_a", C.c_uint64 * 8), ("msm_b1", C.c_uint64 * 8), ("msm_k", C.c_uint64 * 8),
        ("msm_z", C.c_uint64 * 8), ("msm_b2", C.c_uint64 * 16), ("bs1", C.c_uint64 * 8),
    ]

    def as_dict(self):
        return {name: np.array(getattr(self, name)[:], dtype=np.uint64) for name, _ in self._fields_}


def _pk_desc(log2_domain, n_wires, A, B, K, Z, B2, alpha, beta, delta, beta2, delta2, infinity_a, infinity_b, k_skip,
             partial=False, offsets=(0, 0, 0, 0), precompute=False):
    """struct b200g16_pk_desc from numpy arrays / Bases handles -> (desc, buffers to keep alive during the call)"""
    keep = []

    def vec(v, cols):
        if isinstance(v, Bases):
            return None, v.handle, v.n
        a = _u64(v, cols)
        keep.append(a)
        return _ptr(a), None, a.shape[0]

    d = PkDesc()
    d.log2_domain, d.n_wires = log2_domain, n_wires
    d.partial = int(bool(partial))
    d.precompute = int(bool(precompute))
    d.off_a, d.off_b, d.off_k, d.off_z = [int(x) for x in offsets]
    d.g1_a, d.res_a, d.n_a = vec(A, 8)
    d.g1_b, d.res_b, d.n_b = vec(B, 8)
    d.g1_k, d.res_k, d.n_k = vec(K, 8)
    d.g1_z, d.res_z, d.n_z = vec(Z, 8)
    d.g2_b, d.res_b2, nb2 = vec(B2, 16)
    if nb2 != d.n_b:
        raise B200Error("pk_upload: len(G2.B) != len(G1.B)")
    for name, val, w in (("g1_alpha", alpha, 8), ("g1_beta", beta, 8), ("g1_delta", delta, 8),
                         ("g2_beta", beta2, 16), ("g2_delta", delta2, 16)):
        a = _u64(val).reshape(w)
        keep.append(a)
        setattr(d, name, _ptr(a))
    for name, val in (("infinity_a", infinity_a), ("infinity_b", infinity_b), ("k_skip", k_skip)):
        a = np.ascontiguousarray(val, dtype=np.uint8)
        if a.shape[0] != n_wires:
            raise B200Error(f"pk_upload: {name} must have n_wires entries")
        keep.append(a)
        setattr(d, name, _ptr(a))
    return d, keep


def _batch_rows(what, wires, a, b, c, r, s):
    """The host rows of a batch prove as the library reads them -> (k, wires, a, b, c, r, s); refuses shapes that would
    let it read past a buffer, before any library call."""
    wires, a, b, c = [np.ascontiguousarray(x, dtype=np.uint64) for x in (wires, a, b, c)]
    k = wires.shape[0]
    if wires.ndim != 3 or any(x.ndim != 3 or x.shape[0] != k for x in (a, b, c)) or not a.shape == b.shape == c.shape:
        raise B200Error(f"{what}: wires must be (k, n_wires, 4), a/b/c (k, n_constraints, 4)")
    r, s = _u64(r, 4), _u64(s, 4)
    if r.shape[0] != k or s.shape[0] != k:
        raise B200Error(f"{what}: one r and one s per proof")
    return k, wires, a, b, c, r, s


def host_register(arr):
    """Page-lock a numpy array in place (b200g16_host_register); returns the array."""
    _check(load().b200g16_host_register(_ptr(arr), arr.nbytes))
    return arr


def host_unregister(arr):
    _check(load().b200g16_host_unregister(_ptr(arr)))


class Group:
    """Several GPUs driven from this one process (b200g16_group_*): point-range shards of the proving key, peer
    copies for h, partial points added on the host.  devices may repeat a device (several shards on one GPU)."""

    def __init__(self, devices):
        arr = (C.c_int * len(devices))(*[int(d) for d in devices])
        h = _vp()
        _check(load().b200g16_group_init(arr, len(devices), C.byref(h)))
        self.h, self.devices = h, list(devices)

    def close(self):
        if self.h:
            load().b200g16_group_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __len__(self):
        return int(load().b200g16_group_size(self.h))

    def ctx(self, i):
        """Borrowed Context of the i-th device (do not close it)."""
        c = Context.__new__(Context)
        c.h, c.device = _vp(load().b200g16_group_ctx(self.h, i)), self.devices[i]
        return c

    def upload(self, points, group=1, precompute=False):
        pts = _u64(points, 8 if group == 1 else 16)
        h = _vp()
        fn = load().b200g16_group_bases_upload_g1 if group == 1 else load().b200g16_group_bases_upload_g2
        _check(fn(self.h, _ptr(pts), pts.shape[0], C.byref(h)))
        if precompute:
            _check(load().b200g16_group_bases_precompute(self.h, h, 0))
        return (h, group, pts.shape[0])

    def bases_free(self, gb):
        load().b200g16_group_bases_free(gb[0])

    def msm(self, gb, scalars):
        h, group, n = gb
        sc = _u64(scalars, 4)
        out = np.zeros(8 if group == 1 else 16, dtype=np.uint64)
        fn = load().b200g16_group_msm_g1 if group == 1 else load().b200g16_group_msm_g2
        _check(fn(self.h, h, _ptr(sc), sc.shape[0], _ptr(out)))
        return out

    def pk_upload(self, log2_domain, n_wires, A, B, K, Z, B2, alpha, beta, delta, beta2, delta2, infinity_a, infinity_b,
                  k_skip, precompute=False):
        """The whole key as host arrays; the library cuts and uploads the shards."""
        d, keep = _pk_desc(log2_domain, n_wires, A, B, K, Z, B2, alpha, beta, delta, beta2, delta2, infinity_a, infinity_b,
                           k_skip, False, (0, 0, 0, 0), precompute)
        h = _vp()
        _check(load().b200g16_group_pk_upload(self.h, C.byref(d), C.byref(h)))
        del keep
        return h

    def pk_replicate(self, pk):
        """A whole single-device key (a Context.pk_upload handle, on any device) on every device of the group
        (b200g16_group_pk_replicate): members on the key's device borrow its vectors, every other device gets one
        copy, window tables included.  The source must outlive the returned key; prove with prove_batch."""
        h = _vp()
        _check(load().b200g16_group_pk_replicate(self.h, pk, C.byref(h)))
        return h

    def pk_free(self, pk):
        """Releases a sharded (pk_upload) or a replicated (pk_replicate) key."""
        load().b200g16_group_pk_free(pk)

    def prove(self, pk, wires, a, b, c, r, s, want_h=False, log2_domain=None):
        wires, a, b, c = _u64(wires, 4), _u64(a, 4), _u64(b, 4), _u64(c, 4)
        r, s = _u64(r).reshape(4), _u64(s).reshape(4)
        out = ProofOut()
        h = np.zeros((1 << log2_domain, 4), dtype=np.uint64) if want_h else None
        _check(load().b200g16_group_prove(self.h, pk, _ptr(wires), wires.shape[0], _ptr(a), _ptr(b), _ptr(c), a.shape[0],
                                          _ptr(r), _ptr(s), C.byref(out), _ptr(h) if want_h else None))
        return out.as_dict(), h

    def prove_batch(self, pk, wires, a, b, c, r, s):
        """b200g16_group_prove_batch with a replicated key: Context.prove_batch's arguments and results, the k proofs
        split into contiguous ranges over the members."""
        k, wires, a, b, c, r, s = _batch_rows("group prove_batch", wires, a, b, c, r, s)
        out = (ProofOut * max(k, 1))()
        _check(load().b200g16_group_prove_batch(self.h, pk, k, _ptr(wires), wires.shape[1], _ptr(a), _ptr(b), _ptr(c),
                                                a.shape[1], _ptr(r), _ptr(s), out))
        return [out[j].as_dict() for j in range(k)]


class Bases:
    """Device-resident vector of affine points (one of the proving key's point arrays)."""

    def __init__(self, ctx, handle, group, n):
        self.ctx, self.handle, self.group, self.n = ctx, handle, group, n

    def free(self):
        if self.handle:
            load().b200g16_bases_free(self.handle)
            self.handle = None

    def __len__(self):
        return self.n

    def precompute(self, window_bits=0):
        """Attach a window table (b200g16_bases_precompute); returns the window width used."""
        _check(load().b200g16_bases_precompute(self.ctx.h, self.handle, int(window_bits)))
        return self.window()

    def window(self):
        return int(load().b200g16_bases_window(self.handle))

    def download(self, offset=0, n=None):
        n = self.n - offset if n is None else n
        out = np.zeros((n, 8 if self.group == 1 else 16), dtype=np.uint64)
        _check(load().b200g16_bases_download(self.handle, offset, n, _ptr(out)))
        return out


class Context:
    """One per process per GPU (b200g16_init)."""

    def __init__(self, device=0):
        h = _vp()
        _check(load().b200g16_init(int(device), C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if self.h:
            load().b200g16_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- bookkeeping
    def launch_count(self):
        return int(load().b200g16_launch_count(self.h))

    def last_timings(self):
        buf = (C.c_float * 16)()
        n = load().b200g16_last_timings(self.h, buf, 16)
        return [buf[i] for i in range(n)]

    def set_msm_window(self, c):
        _check(load().b200g16_set_msm_window(self.h, int(c)))

    def set_msm_batch_affine(self, mode, levels=0, min_pairs=0):
        """0 = mixed XYZZ bucket additions, 1 = batched-affine pair tree for large inputs, 2 = always."""
        _check(load().b200g16_set_msm_batch_affine(self.h, int(mode), int(levels), int(min_pairs)))

    # -- bases
    def upload_g1(self, points):
        pts = _u64(points, 8)
        h = _vp()
        _check(load().b200g16_bases_upload_g1(self.h, _ptr(pts), pts.shape[0], C.byref(h)))
        return Bases(self, h, 1, pts.shape[0])

    def upload_g2(self, points):
        pts = _u64(points, 16)
        h = _vp()
        _check(load().b200g16_bases_upload_g2(self.h, _ptr(pts), pts.shape[0], C.byref(h)))
        return Bases(self, h, 2, pts.shape[0])

    def bases_copy(self, bases):
        """A copy of a resident vector (on any device) on this ctx's device, its window table included
        (b200g16_bases_copy, device to device); independent of the source."""
        h = _vp()
        _check(load().b200g16_bases_copy(self.h, bases.handle, C.byref(h)))
        return Bases(self, h, bases.group, bases.n)

    # -- fixed-base batch scalar multiplication (BatchScalarMultiplicationG1/G2)
    def fixed_base_mul(self, base, scalars, group=1, resident=False):
        lib = load()
        words = 8 if group == 1 else 16
        base = _u64(base).reshape(words)
        sc = _u64(scalars, 4)
        n = sc.shape[0]
        if resident:
            h = _vp()
            fn = lib.b200g16_bases_from_scalars_g1 if group == 1 else lib.b200g16_bases_from_scalars_g2
            _check(fn(self.h, _ptr(base), _ptr(sc), n, C.byref(h)))
            return Bases(self, h, group, n)
        out = np.zeros((n, words), dtype=np.uint64)
        fn = lib.b200g16_fixed_base_mul_g1 if group == 1 else lib.b200g16_fixed_base_mul_g2
        _check(fn(self.h, _ptr(base), _ptr(sc), n, _ptr(out)))
        return out

    # -- Groth16 setup (b200g16_setup)
    def setup(self, r1cs, tau, alpha, beta, gamma, delta, sigma):
        """The key of a constraint system (a mapping with groth16.SparseR1CS's fields) for the given toxic waste
        (Montgomery fr.Elements, 4 limbs each) -> dict: log2_domain, the resident vectors as Bases (a, b, k, z, b2,
        vk_k, ped_basis, ped_basis_exp_sigma; the last two None without a commitment), the small points
        (g1_alpha ... ped_g_sigma_neg) and the host flags infinity_a, infinity_b, k_skip."""
        d, keep = _r1cs_desc(r1cs)
        t = Toxic()
        for name, v in zip(("tau", "alpha", "beta", "gamma", "delta", "sigma"), (tau, alpha, beta, gamma, delta, sigma)):
            getattr(t, name)[:] = [int(x) for x in _u64(v).reshape(4)]
        nw = int(d.n_wires)
        flags = [np.zeros(nw, dtype=np.uint8) for _ in range(3)]
        out = SetupOut()
        _check(load().b200g16_setup(self.h, C.byref(d), C.byref(t), *[_ptr(f) for f in flags], C.byref(out)))
        del keep
        res = {"log2_domain": int(out.log2_domain), "infinity_a": flags[0], "infinity_b": flags[1], "k_skip": flags[2]}
        for name in SETUP_VECTORS:
            h = getattr(out, name)
            res[name] = None if not h else Bases(self, _vp(h), 2 if name == "b2" else 1,
                                                 int(load().b200g16_bases_len(_vp(h))))
        for name, _ in SetupOut._fields_[1 + len(SETUP_VECTORS):]:
            res[name] = np.array(getattr(out, name)[:], dtype=np.uint64)
        return res

    def setup_wire_polys(self, r1cs, tau):
        """gnark's setupABC on the GPU: (A, B, C) per wire at tau, each (n_wires, 4) Montgomery."""
        d, keep = _r1cs_desc(r1cs)
        out = [np.zeros((int(d.n_wires), 4), dtype=np.uint64) for _ in range(3)]
        tau = _u64(tau).reshape(4)
        _check(load().b200g16_setup_wire_polys(self.h, C.byref(d), _ptr(tau), *[_ptr(o) for o in out]))
        del keep
        return tuple(out)

    def modmul_probe(self, blocks_per_sm=4, chains=4, iters=2000):
        rate = C.c_double()
        ms = C.c_float()
        _check(load().b200g16_modmul_probe(self.h, blocks_per_sm, chains, iters, C.byref(rate), C.byref(ms)))
        return rate.value, ms.value

    def pipe_probe(self, mode, blocks_per_sm=8, iters=2000):
        rate = C.c_double()
        ms = C.c_float()
        _check(load().b200g16_pipe_probe(self.h, mode, blocks_per_sm, iters, C.byref(rate), C.byref(ms)))
        return rate.value, ms.value

    def fp52_probe(self, variant, blocks_per_sm=4, iters=2000):
        rate = C.c_double()
        ms = C.c_float()
        _check(load().b200g16_fp52_probe(self.h, variant, blocks_per_sm, iters, C.byref(rate), C.byref(ms)))
        return rate.value, ms.value

    # -- NTT / computeH (mirror fft.Domain.FFT / FFTInverse and prove.go computeH)
    def ntt(self, data, inverse=False, coset=False, decimation=DIF):
        """data: (N,4) uint64 Montgomery, N a power of two; returns the transformed copy."""
        a = _u64(data, 4).copy()
        n = a.shape[0]
        if n == 0 or n & (n - 1):
            raise B200Error("ntt: length must be a power of two")
        _check(load().b200g16_ntt(self.h, _ptr(a), n.bit_length() - 1, int(inverse), int(coset), int(decimation)))
        return a

    def ntt_dev(self, d_ptr, log2n, batch=1, inverse=False, coset=False, decimation=DIF):
        _check(load().b200g16_ntt_dev(self.h, _dp(d_ptr), log2n, batch, int(inverse), int(coset), int(decimation)))

    def compute_h(self, a, b, c, log2n):
        a, b, c = _u64(a, 4), _u64(b, 4), _u64(c, 4)
        h = np.zeros((1 << log2n, 4), dtype=np.uint64)
        _check(load().b200g16_compute_h(self.h, _ptr(a), _ptr(b), _ptr(c), a.shape[0], log2n, _ptr(h)))
        return h

    def compute_h_dev(self, d_a, d_b, d_c, log2n):
        _check(load().b200g16_compute_h_dev(self.h, _dp(d_a), _dp(d_b), _dp(d_c), log2n))

    # -- Keccak (mirror keccakf.Permute, keccakSponge.Digest, VerifyMerkleTreeProofs)
    def keccak_f_batch(self, states):
        st = np.ascontiguousarray(states, dtype=np.uint64).reshape(-1, 25).copy()
        _check(load().b200g16_keccak_f_batch(self.h, _ptr(st), st.shape[0]))
        return st

    def keccak_f_batch_dev(self, d_ptr, n):
        _check(load().b200g16_keccak_f_batch_dev(self.h, _dp(d_ptr), n))

    def keccak_sponge_batch(self, inputs, out_len):
        """inputs: (n, in_len) uint8 -> (n, out_len) uint8"""
        a = np.ascontiguousarray(inputs, dtype=np.uint8)
        n, in_len = a.shape
        out = np.zeros((n, out_len), dtype=np.uint8)
        _check(load().b200g16_keccak_sponge_batch(self.h, _ptr(a), in_len, n, _ptr(out), out_len))
        return out

    def keccak_duplex_batch(self, ops, inputs, digests=None, tag=None):
        """keccakSponge.Digest for n sponges running the same op script, state carried across calls.
        ops: [("absorb", len) | ("squeeze", len), ...]; inputs: (n, A) uint8, A = the absorbed bytes of the script;
        digests: (n,) KECCAK_DIGEST to continue from (None: start fresh); tag: bytes of NewKeccakWithTag for every
        sponge (b"" = NewKeccak; ignored digests are not read).  -> (outputs (n, S) uint8, final digests)"""
        script, A, S = duplex_script(ops)
        inp = np.ascontiguousarray(inputs, dtype=np.uint8)
        if inp.ndim != 2 or inp.shape[1] != A:
            raise B200Error(f"keccak_duplex_batch: inputs must be (n, {A})")
        n = inp.shape[0]
        if digests is None:
            dg = np.zeros(n, dtype=KECCAK_DIGEST)
            tag = b"" if tag is None else tag
        else:
            dg = np.ascontiguousarray(digests, dtype=KECCAK_DIGEST).copy()
            if dg.shape != (n,):
                raise B200Error(f"keccak_duplex_batch: {n} digests expected")
        tg = None if tag is None else np.frombuffer(bytes(tag) + b"\0", dtype=np.uint8)
        out = np.zeros((n, S), dtype=np.uint8)
        _check(load().b200g16_keccak_duplex_batch(self.h, _ptr(dg), n, _ptr(tg) if tg is not None else None,
                                                  len(tg) - 1 if tg is not None else 0, _ptr(script), len(ops),
                                                  _ptr(inp), _ptr(out)))
        return out, dg

    def keccak_duplex_batch_dev(self, d_digests, n, ops, d_inputs, d_outputs, tag=None):
        """The same on device pointers: d_digests n x 208 bytes (8-byte aligned), d_inputs n x A and d_outputs n x S
        bytes (any alignment); ops and tag as keccak_duplex_batch (tag None: continue from the digests)."""
        script, _, _ = duplex_script(ops)
        tg = None if tag is None else np.frombuffer(bytes(tag) + b"\0", dtype=np.uint8)
        _check(load().b200g16_keccak_duplex_batch_dev(
            self.h, _dp(d_digests), n, _ptr(tg) if tg is not None else None, len(tg) - 1 if tg is not None else 0,
            _ptr(script), len(ops), _dp(d_inputs) if d_inputs else None, _dp(d_outputs) if d_outputs else None))

    def keccak_merkle_paths(self, leaves, siblings, auth_paths, indexes, expected_root=None):
        """leaves (n, leaf_len) u8; siblings (n, 32) u8; auth_paths (n, height-1, 32) u8;
        indexes (n,) u64 -> (roots (n,32) u8, ok (n,) bool or None)"""
        leaves = np.ascontiguousarray(leaves, dtype=np.uint8)
        siblings = np.ascontiguousarray(siblings, dtype=np.uint8)
        auth_paths = np.ascontiguousarray(auth_paths, dtype=np.uint8)
        indexes = np.ascontiguousarray(indexes, dtype=np.uint64)
        n, leaf_len = leaves.shape
        height = auth_paths.shape[1] + 1
        roots = np.zeros((n, 32), dtype=np.uint8)
        ok = np.zeros(n, dtype=np.uint8) if expected_root is not None else None
        er = np.frombuffer(bytes(expected_root), dtype=np.uint8).copy() if expected_root is not None else None
        _check(load().b200g16_keccak_merkle_paths(
            self.h, _ptr(leaves), leaf_len, _ptr(siblings), _ptr(auth_paths) if auth_paths.size else None,
            _ptr(indexes), height, n, _ptr(er) if er is not None else None, _ptr(roots),
            _ptr(ok) if ok is not None else None))
        return roots, (ok.astype(bool) if ok is not None else None)

    # -- Groth16 prove (pk resident; mirrors groth16_bn254.Prove after Solve)
    def pk_upload(self, log2_domain, n_wires, A, B, K, Z, B2, alpha, beta, delta, beta2, delta2,
                  infinity_a, infinity_b, k_skip, partial=False, offsets=(0, 0, 0, 0), precompute=False):
        """A/B/K/Z/B2: numpy point arrays (host) or Bases (already resident, borrowed).
        partial=True: the vectors are entries [off, off+len) of the full key vectors
        (offsets = (off_a, off_b, off_k, off_z)); prove() then returns partial MSM sums."""
        d, keep = _pk_desc(log2_domain, n_wires, A, B, K, Z, B2, alpha, beta, delta, beta2, delta2, infinity_a, infinity_b,
                           k_skip, partial, offsets, precompute)
        h = _vp()
        _check(load().b200g16_pk_upload(self.h, C.byref(d), C.byref(h)))
        del keep
        return h

    def pk_free(self, pk):
        load().b200g16_pk_free(pk)

    def prove(self, pk, wires, a, b, c, r, s, want_h=False, log2_domain=None):
        wires, a, b, c = _u64(wires, 4), _u64(a, 4), _u64(b, 4), _u64(c, 4)
        r, s = _u64(r).reshape(4), _u64(s).reshape(4)
        out = ProofOut()
        h = np.zeros((1 << log2_domain, 4), dtype=np.uint64) if want_h else None
        _check(load().b200g16_prove(self.h, pk, _ptr(wires), wires.shape[0], _ptr(a), _ptr(b), _ptr(c), a.shape[0],
                                    _ptr(r), _ptr(s), C.byref(out), _ptr(h) if want_h else None))
        return out.as_dict(), h

    def prove_finish(self, pk, msm_a, msm_b1, msm_k, msm_z, msm_b2, r, s):
        """Final assembly from the five complete (summed over shards) MSM results."""
        r, s = _u64(r).reshape(4), _u64(s).reshape(4)
        pts = [_u64(v).reshape(w) for v, w in ((msm_a, 8), (msm_b1, 8), (msm_k, 8), (msm_z, 8), (msm_b2, 16))]
        out = ProofOut()
        _check(load().b200g16_prove_finish(pk, *[_ptr(p) for p in pts], _ptr(r), _ptr(s), C.byref(out)))
        return out.as_dict()

    def prove_dev(self, pk, d_wires, d_a, d_b, d_c, r, s):
        r, s = _u64(r).reshape(4), _u64(s).reshape(4)
        out = ProofOut()
        _check(load().b200g16_prove_dev(self.h, pk, _dp(d_wires), _dp(d_a), _dp(d_b), _dp(d_c),
                                        _ptr(r), _ptr(s), C.byref(out)))
        return out.as_dict()

    def prove_batch(self, pk, wires, a, b, c, r, s):
        """b200g16_prove_batch: k proves of one circuit.  wires (k, n_wires, 4), a/b/c (k, n_constraints, 4), r/s (k, 4),
        all Montgomery -> list of k dicts as prove() returns them."""
        k, wires, a, b, c, r, s = _batch_rows("prove_batch", wires, a, b, c, r, s)
        out = (ProofOut * max(k, 1))()
        _check(load().b200g16_prove_batch(self.h, pk, k, _ptr(wires), wires.shape[1], _ptr(a), _ptr(b), _ptr(c),
                                          a.shape[1], _ptr(r), _ptr(s), out))
        return [out[j].as_dict() for j in range(k)]

    def prove_batch_dev(self, pk, k, d_wires, d_a, d_b, d_c, r, s):
        """b200g16_prove_batch_dev: device pointers to k x n_wires wires and k x N a/b/c rows (zero padded, clobbered;
        h is left in the d_a rows); r/s (k, 4) host -> list of k dicts."""
        r, s = _u64(r, 4), _u64(s, 4)
        out = (ProofOut * max(k, 1))()
        _check(load().b200g16_prove_batch_dev(self.h, pk, k, _dp(d_wires), _dp(d_a), _dp(d_b), _dp(d_c),
                                              _ptr(r), _ptr(s), out))
        return [out[j].as_dict() for j in range(k)]

    # -- pairing / verify (mirror bn254.PairingCheck, bn254.Pair, groth16.Verify)
    def pairing_check(self, g1_points, g2_points):
        p, q = _u64(g1_points, 8), _u64(g2_points, 16)
        if p.shape[0] != q.shape[0]:
            raise B200Error("pairing_check: len(P) != len(Q)")
        ok = C.c_int()
        _check(load().b200g16_pairing_check(self.h, _ptr(p), _ptr(q), p.shape[0], C.byref(ok)))
        return bool(ok.value)

    def pair(self, g1_points, g2_points):
        """-> GT element, (6, 8) uint64: C0.B0, C0.B1, C0.B2, C1.B0, C1.B1, C1.B2 (gnark E12 order)"""
        p, q = _u64(g1_points, 8), _u64(g2_points, 16)
        if p.shape[0] != q.shape[0]:
            raise B200Error("pair: len(P) != len(Q)")
        out = np.zeros((6, 8), dtype=np.uint64)
        _check(load().b200g16_pair(self.h, _ptr(p), _ptr(q), p.shape[0], _ptr(out)))
        return out

    def verify(self, alpha, beta2, gamma2, delta2, K, ar, bs, krs, public_inputs, commitment=None, pok=None,
               ped_g=None, ped_g_sigma_neg=None):
        d, keep = _vk_desc(alpha, beta2, gamma2, delta2, K, ped_g, ped_g_sigma_neg)
        opt = [None if v is None else _u64(v).reshape(w) for v, w in ((commitment, 8), (pok, 8))]
        pts = [_u64(ar).reshape(8), _u64(bs).reshape(16), _u64(krs).reshape(8)]
        pub = _u64(public_inputs, 4)
        ok = C.c_int()
        _check(load().b200g16_verify(self.h, C.byref(d), _ptr(pts[0]), _ptr(pts[1]), _ptr(pts[2]),
                                     _ptr(opt[0]) if opt[0] is not None else None,
                                     _ptr(opt[1]) if opt[1] is not None else None,
                                     _ptr(pub) if pub.shape[0] else None, pub.shape[0], C.byref(ok)))
        return bool(ok.value)

    def verify_batch(self, alpha, beta2, gamma2, delta2, K, ar, bs, krs, public_inputs, coeffs, commitments=None,
                     poks=None, ped_g=None, ped_g_sigma_neg=None, want_each=True):
        """b200g16_verify_batch: k proofs against one vk.  ar (k,8), bs (k,16), krs (k,8), public_inputs (k, n_public, 4)
        Montgomery, coeffs (k or 2k, 2) 128-bit little-endian (rho, then tau with commitments), commitments / poks
        (k,8) or None.  -> (ok_all, ok_each (k,) bool or None)"""
        d, keep = _vk_desc(alpha, beta2, gamma2, delta2, K, ped_g, ped_g_sigma_neg)
        ar, bs, krs = _u64(ar, 8), _u64(bs, 16), _u64(krs, 8)
        k = ar.shape[0]
        if bs.shape[0] != k or krs.shape[0] != k:
            raise B200Error("verify_batch: Ar, Bs, Krs differ in length")
        pub = np.ascontiguousarray(public_inputs, dtype=np.uint64)
        if pub.ndim != 3:
            pub = pub.reshape(k, -1, 4) if pub.size else np.zeros((k, 0, 4), dtype=np.uint64)
        if pub.shape[0] != k:
            raise B200Error("verify_batch: public inputs for %d proofs, %d proofs given" % (pub.shape[0], k))
        co = _u64(coeffs, 2)
        com = None if commitments is None else _u64(commitments, 8)
        pk_ = None if poks is None else _u64(poks, 8)
        if co.shape[0] != (2 * k if com is not None else k) or any(a is not None and a.shape[0] != k for a in (com, pk_)):
            raise B200Error("verify_batch: coefficient / commitment / pok count does not match the proofs")
        ok = C.c_int()
        each = np.zeros(k, dtype=np.uint8) if want_each else None
        _check(load().b200g16_verify_batch(
            self.h, C.byref(d), k, _ptr(ar), _ptr(bs), _ptr(krs), _ptr(com) if com is not None else None,
            _ptr(pk_) if pk_ is not None else None, _ptr(pub) if pub.size else None, pub.shape[1],
            _ptr(co), C.byref(ok), _ptr(each) if want_each and k else None))
        return bool(ok.value), (each.astype(bool) if want_each else None)

    # -- gnark-crypto point encodings (G1Affine.Bytes / RawBytes / SetBytes and the G2 counterparts)
    def encode_points(self, points, group=1, raw=False):
        """points (n, 8|16) uint64 -> (n, record) uint8, record = 32|64 compressed, 64|128 raw"""
        pts = _u64(points, 8 if group == 1 else 16)
        rec = (32 if group == 1 else 64) * (2 if raw else 1)
        out = np.zeros((pts.shape[0], rec), dtype=np.uint8)
        fn = load().b200g16_g1_encode if group == 1 else load().b200g16_g2_encode
        _check(fn(self.h, _ptr(pts), pts.shape[0], int(raw), _ptr(out)))
        return out

    def decode_points(self, data, group=1, raw=False, subgroup_check=True):
        """data: bytes / uint8 array of n fixed-size records -> (points (n, 8|16) uint64, ok (n,) bool)"""
        rec = (32 if group == 1 else 64) * (2 if raw else 1)
        buf = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8) if isinstance(data, (bytes, bytearray))
                                   else data, dtype=np.uint8).reshape(-1, rec)
        n = buf.shape[0]
        out = np.zeros((n, 8 if group == 1 else 16), dtype=np.uint64)
        ok = np.zeros(n, dtype=np.uint8)
        if group == 1:
            _check(load().b200g16_g1_decode(self.h, _ptr(buf), n, int(raw), _ptr(out), _ptr(ok)))
        else:
            _check(load().b200g16_g2_decode(self.h, _ptr(buf), n, int(raw), int(subgroup_check), _ptr(out), _ptr(ok)))
        return out, ok.astype(bool)

    def msm_plan(self, bases, n=None):
        """(window bits c, digits per scalar W) the library uses for an n-point MSM on `bases`."""
        c, w = C.c_int(), C.c_int()
        _check(load().b200g16_msm_plan(self.h, bases.handle, bases.n if n is None else n, C.byref(c), C.byref(w)))
        return c.value, w.value

    def h_pointwise_dev(self, d_a, d_b, d_c, log2n):
        _check(load().b200g16_h_pointwise_dev(self.h, _dp(d_a), _dp(d_b), _dp(d_c), log2n))

    def prove_h_dev(self, pk, d_wires, d_h, r, s):
        """prove_dev with h already computed (d_h: N elements, bit-reversed order)."""
        r, s = _u64(r).reshape(4), _u64(s).reshape(4)
        out = ProofOut()
        _check(load().b200g16_prove_h_dev(self.h, pk, _dp(d_wires), _dp(d_h), _ptr(r), _ptr(s), C.byref(out)))
        return out.as_dict()

    def prove_begin_dev(self, pk, d_wires):
        """First half of a prove: the four witness MSMs are enqueued; returns without waiting."""
        _check(load().b200g16_prove_begin_dev(self.h, pk, _dp(d_wires)))

    def prove_end_dev(self, pk, d_h, r, s):
        """Second half: Z MSM over h (device pointer), wait, assemble."""
        r, s = _u64(r).reshape(4), _u64(s).reshape(4)
        out = ProofOut()
        _check(load().b200g16_prove_end_dev(self.h, pk, _dp(d_h), _ptr(r), _ptr(s), C.byref(out)))
        return out.as_dict()

    # -- computeH split over 2 / 4 / 8 ranks (CUDA IPC peer memory; see sharded.DistributedH)
    def dist_h_init(self, log2n, n_peers, me):
        """-> uint8[192]: the IPC handles of this rank's a / b / c slices"""
        h = np.zeros(192, dtype=np.uint8)
        _check(load().b200g16_dist_h_init(self.h, log2n, n_peers, me, _ptr(h)))
        return h

    def dist_h_open(self, all_handles):
        a = np.ascontiguousarray(all_handles, dtype=np.uint8)
        _check(load().b200g16_dist_h_open(self.h, _ptr(a)))

    def dist_h_load(self, d_a, d_b, d_c):
        _check(load().b200g16_dist_h_load(self.h, _dp(d_a), _dp(d_b), _dp(d_c)))

    def dist_h_slice(self, which):
        p = load().b200g16_dist_h_slice(self.h, which)
        if not p:
            raise B200Error("dist_h_slice: not initialised")
        return int(p)

    def dist_h_phase(self, phase):
        _check(load().b200g16_dist_h_phase(self.h, phase))

    def dist_h_close(self):
        load().b200g16_dist_h_close(self.h)

    # -- MSM (host scalars: numpy (n,4) uint64 Montgomery; or a device pointer + n)
    def msm(self, bases, scalars, offset=0, n=None):
        lib = load()
        words = 8 if bases.group == 1 else 16
        out = np.zeros(words, dtype=np.uint64)
        if isinstance(scalars, np.ndarray):
            sc = _u64(scalars, 4)
            n = sc.shape[0] if n is None else n
            fn = lib.b200g16_msm_g1 if bases.group == 1 else lib.b200g16_msm_g2
            _check(fn(self.h, bases.handle, offset, _ptr(sc), n, _ptr(out)))
        else:  # raw device pointer (e.g. torch tensor .data_ptr())
            fn = lib.b200g16_msm_g1_dev if bases.group == 1 else lib.b200g16_msm_g2_dev
            _check(fn(self.h, bases.handle, offset, _dp(scalars), n, _ptr(out)))
        return out

    def msm_batch(self, bases, scalars, offset=0, n=None, k=None):
        """k MSMs over the same bases (b200g16_msm_g1_batch / _g2_batch): scalars (k, n, 4) uint64 Montgomery, or a device
        pointer to k x n scalars with n and k given.  -> (k, 8) or (k, 16) affine points, row j = msm(bases, scalars[j])"""
        lib = load()
        if isinstance(scalars, np.ndarray):
            sc = np.ascontiguousarray(scalars, dtype=np.uint64)
            if sc.ndim != 3 or sc.shape[2] != 4:
                raise B200Error("msm_batch: scalars must be (k, n, 4)")
            k, n = sc.shape[0], sc.shape[1]
            fn = lib.b200g16_msm_g1_batch if bases.group == 1 else lib.b200g16_msm_g2_batch
            ptr = _ptr(sc)
        else:
            if n is None or k is None:
                raise B200Error("msm_batch: a device pointer needs n and k")
            fn = lib.b200g16_msm_g1_batch_dev if bases.group == 1 else lib.b200g16_msm_g2_batch_dev
            ptr = _dp(scalars)
        out = np.zeros((k, 8 if bases.group == 1 else 16), dtype=np.uint64)
        _check(fn(self.h, bases.handle, offset, ptr, n, k, _ptr(out) if k else None))
        return out

    def msm_begin(self, bases, scalars, offset=0, n=None):
        """Enqueue a G1 MSM (b200g16_msm_g1_begin / _begin_dev) and return its ticket; msm_end(ticket) collects the
        result.  Calls made in between run behind it.  The scalars must stay alive and unchanged until msm_end."""
        lib, ticket = load(), C.c_int(-1)
        if isinstance(scalars, np.ndarray):
            sc = _u64(scalars, 4)
            n = sc.shape[0] if n is None else n
            _check(lib.b200g16_msm_g1_begin(self.h, bases.handle, offset, _ptr(sc), n, C.byref(ticket)))
            self._async_keep = getattr(self, "_async_keep", {})
            self._async_keep[ticket.value] = sc
        else:
            _check(lib.b200g16_msm_g1_begin_dev(self.h, bases.handle, offset, _dp(scalars), n, C.byref(ticket)))
        return ticket.value

    def msm_end(self, ticket):
        out = np.zeros(8, dtype=np.uint64)
        _check(load().b200g16_msm_g1_end(self.h, int(ticket), _ptr(out)))
        getattr(self, "_async_keep", {}).pop(int(ticket), None)
        return out
