"""ctypes binding of libtyplonk_b200.so (include/typlonk_b200.h).

No CPU fallback: if the shared library is missing this module raises at import of the
symbols, and every call needs a CUDA device (tp_ctx_create -> TP_ERR_NO_DEVICE otherwise).
"""
import ctypes as C
import os
from pathlib import Path

_LIB_PATH = Path(os.environ.get("TYPLONK_B200_LIB") or
                 (Path(__file__).resolve().parent / "lib" / "libtyplonk_b200.so"))

G1_BYTES = 97
G2_BYTES = 193
PROOF_FIXED_BYTES = 1472
PROOF_COMPRESSED_FIXED_BYTES = 848
PHASES = ["msm_total", "msm_sort", "msm_accum", "msm_reduce", "ntt", "quotient", "perm", "scan"]

ERRORS = {
    1: "TP_ERR_INVALID_ARG", 2: "TP_ERR_CUDA", 3: "TP_ERR_SRS_TOO_SHORT", 4: "TP_ERR_EMPTY_POLY",
    5: "TP_ERR_ZERO_DENOMINATOR", 6: "TP_ERR_GATE_UNSATISFIED", 7: "TP_ERR_NO_DEVICE",
    8: "TP_ERR_COLLECTIVE", 9: "TP_ERR_BUFFER_TOO_SMALL", 10: "TP_ERR_INVALID_TAG",
    11: "TP_ERR_UNPLACED_VARIABLE", 12: "TP_ERR_MALFORMED",
}

# every symbol include/typlonk_b200.h declares
SYMBOLS = [
    "tp_ctx_create", "tp_ctx_destroy", "tp_last_error", "tp_sync", "tp_comm_unique_id", "tp_ctx_comm_init_rank",
    "tp_ctx_create_multi", "tp_ctx_group_size",
    "tp_prof_enable", "tp_prof_reset", "tp_prof_get", "tp_launch_count",
    "tp_srs_from_secret", "tp_srs_upload", "tp_srs_len", "tp_srs_g1_download", "tp_srs_destroy",
    "tp_commit", "tp_commit_dev", "tp_open", "tp_ntt", "tp_ntt_dev", "tp_perm_prove",
    "tp_circuit_load", "tp_circuit_compile", "tp_circuit_destroy", "tp_circuit_sigma_commitments",
    "tp_prove", "tp_prove_dev", "tp_prove_inputs", "tp_measure_imad_peak", "tp_selftest", "tp_fr_rand_stream", "tp_ctx_set_option", "tp_ctx_get_stat",
    "tp_srs_g2", "tp_srs_set_g2", "tp_kzg_verify", "tp_pairing_check", "tp_verify", "tp_verify_batch", "tp_prove_batch", "tp_verify_prepared", "tp_proof_challenges",
    "tp_trace_create", "tp_trace_destroy", "tp_trace_gate", "tp_trace_gates", "tp_trace_assert_eq", "tp_trace_finish",
    "tp_trace_gate_kinds", "tp_trace_selectors", "tp_trace_permutation", "tp_trace_witness",
    "tp_permutation_builder_create", "tp_permutation_builder_destroy", "tp_permutation_builder_add_row",
    "tp_permutation_builder_add_constrain", "tp_permutation_builder_build",
    "tp_permutation_compile", "tp_fr_from_i64", "tp_fr_from_canonical", "tp_fr_to_canonical",
    "tp_proof_encoded_size", "tp_proof_encode", "tp_proof_decode",
    "tp_srs_serialized_size", "tp_srs_serialize", "tp_srs_deserialize", "tp_build_stamp", "tp_stdrng_words", "tp_circuit_read_poly", "tp_proof_points_in_subgroup",
    "tp_proof_compress", "tp_proof_decompress", "tp_proof_encoded_size_compressed", "tp_proof_encode_compressed",
    "tp_proof_decode_compressed", "tp_proofs_decompress",
    "tp_srs_serialized_size_compressed", "tp_srs_serialize_compressed", "tp_srs_deserialize_compressed",
    "tp_srs_contribute", "tp_srs_verify", "tp_srs_update_check",
    "tp_vk_from_circuit", "tp_vk_destroy", "tp_vk_serialized_size", "tp_vk_serialize", "tp_vk_deserialize",
    "tp_vk_verify", "tp_vk_verify_batch",
]

COMM_ID_BYTES = 128


def comm_unique_id() -> bytes:
    """tp_comm_unique_id: rank 0 makes it, the host language hands it to every rank once (e.g. one
    torch.distributed.broadcast at start-up), every rank passes it to Context.comm_init_rank."""
    out = (C.c_char * COMM_ID_BYTES)()
    rc = lib().tp_comm_unique_id(out)
    if rc != 0:
        raise TyplonkError(rc, "tp_comm_unique_id: libnccl.so.2 could not be loaded")
    return bytes(out)


class DeviceView:
    """`nbytes` of device memory at `ptr` as a __cuda_array_interface__ object (torch.as_tensor aliases it)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


class TyplonkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s (%d): %s" % (ERRORS.get(code, "TP_ERR"), code, msg))
        self.code = code


class GateUnsatisfied(TyplonkError):
    """The reference panics here (`vanishes`, plonk/src/proof.rs:321)."""


_lib = None


def lib():
    """Load the CUDA library (built by `python -m typlonk_b200.build`); loud failure if absent."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise ImportError(
                "typlonk_b200: %s is missing -- build it with `python -m typlonk_b200.build` "
                "(there is no CPU fallback)" % _LIB_PATH)
        _lib = C.CDLL(str(_LIB_PATH))
        _lib.tp_last_error.restype = C.c_char_p
        _lib.tp_last_error.argtypes = [C.c_void_p]
        for name in SYMBOLS:
            getattr(_lib, name)  # AttributeError if the header and the library diverge
    return _lib


def _buf(b):
    """bytes-like -> ctypes pointer (zero copy for bytearray / numpy, copy for bytes)."""
    if isinstance(b, (bytes, bytearray)):
        return (C.c_char * len(b)).from_buffer_copy(b) if isinstance(b, bytes) else (C.c_char * len(b)).from_buffer(b)
    if isinstance(b, int):  # raw host address (e.g. a pinned torch tensor's data_ptr())
        return C.c_void_p(b)
    if hasattr(b, "ctypes"):  # numpy array
        return b.ctypes.data_as(C.c_void_p)
    return b


def fr_rand_stream(seed: int, count: int) -> bytes:
    """count x Fr::rand from StdRng::seed_from_u64(seed), Montgomery bytes (host only)."""
    out = (C.c_char * (32 * count))()
    rc = lib().tp_fr_rand_stream(C.c_uint64(seed), C.c_size_t(count), out)
    if rc != 0:
        raise TyplonkError(rc, "tp_fr_rand_stream")
    return bytes(out)


def stdrng_words(count: int, seed32: bytes = None, seed_u64: int = 0):
    """tp_stdrng_words: `count` raw u32 output words of the library's StdRng (host only)."""
    out = (C.c_uint32 * count)()
    rc = lib().tp_stdrng_words(_buf(seed32) if seed32 is not None else None, C.c_uint64(seed_u64), C.c_size_t(count), out)
    if rc != 0:
        raise TyplonkError(rc, "tp_stdrng_words")
    return list(out)


# ---- host-only entry points (no device, no context) --------------------------------------------
def kzg_verify(g2: bytes, g2s: bytes, commitment: bytes, w: bytes, y_mont: bytes, z_mont: bytes) -> bool:
    """KzgScheme::verify (kzg/src/lib.rs:66-81) on 193-byte G2 / 97-byte G1 ABI records."""
    ok = C.c_int(0)
    rc = lib().tp_kzg_verify(_buf(g2), _buf(g2s), _buf(commitment), _buf(w), _buf(y_mont), _buf(z_mont), C.byref(ok))
    if rc != 0:
        raise TyplonkError(rc, "tp_kzg_verify")
    return bool(ok.value)


def pairing_check(g1s, g2s) -> bool:
    """prod_i e(g1s[i], g2s[i]) == 1."""
    assert len(g1s) == len(g2s)
    ok = C.c_int(0)
    rc = lib().tp_pairing_check(_buf(b"".join(g1s)), _buf(b"".join(g2s)), C.c_size_t(len(g1s)), C.byref(ok))
    if rc != 0:
        raise TyplonkError(rc, "tp_pairing_check")
    return bool(ok.value)


def srs_update_check(prev_tau_g1: bytes, next_tau_g1: bytes, pubkey: bytes) -> bool:
    """tp_srs_update_check: e(next, G2) == e(prev, pubkey) on 97-byte G1 / 193-byte G2 ABI records, with every point in
    its prime-order group and not infinity (host only)."""
    ok = C.c_int(0)
    rc = lib().tp_srs_update_check(_buf(prev_tau_g1), _buf(next_tau_g1), _buf(pubkey), C.byref(ok))
    if rc != 0:
        raise TyplonkError(rc, "tp_srs_update_check")
    return bool(ok.value)


def proof_challenges(proof_fixed: bytes):
    """(alpha, beta, gamma, evaluation point) as Montgomery bytes (plonk/src/proof.rs:235-244)."""
    outs = [(C.c_char * 32)() for _ in range(4)]
    rc = lib().tp_proof_challenges(_buf(proof_fixed), C.c_size_t(len(proof_fixed)), *outs)
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_challenges: malformed proof")
    return tuple(bytes(o) for o in outs)


class Malformed(TyplonkError):
    """A wire encoding that is not canonical / not on the curve / of the wrong length (TP_ERR_MALFORMED)."""


def proof_encode(fixed: bytes, public_inputs_mont: bytes) -> bytes:
    """tp_proof_encode: the 1472-byte block + Vec<Fr> of public inputs (SURVEY.md App. A.6).  Host only."""
    n = len(public_inputs_mont) // 32
    need = C.c_size_t(0)
    lib().tp_proof_encoded_size(C.c_size_t(n), C.byref(need))
    out = (C.c_char * need.value)()
    rc = lib().tp_proof_encode(_buf(fixed), _buf(public_inputs_mont) if n else None, C.c_size_t(n), out,
                               C.c_size_t(need.value), None)
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_encode")
    return bytes(out)


def proof_decode(raw: bytes):
    """tp_proof_decode (checked): -> (fixed block, public inputs as Montgomery bytes).  Raises Malformed."""
    n = C.c_size_t(0)
    rc = lib().tp_proof_decode(_buf(raw), C.c_size_t(len(raw)), None, None, C.c_size_t(0), C.byref(n))
    if rc == 12:
        raise Malformed(rc, "tp_proof_decode: malformed proof encoding")
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_decode")
    fixed = (C.c_char * PROOF_FIXED_BYTES)()
    pis = (C.c_char * (32 * n.value or 1))()
    rc = lib().tp_proof_decode(_buf(raw), C.c_size_t(len(raw)), fixed, pis, C.c_size_t(n.value), C.byref(n))
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_decode")
    return bytes(fixed), bytes(pis)[: 32 * n.value]


def proof_compress(fixed: bytes) -> bytes:
    """tp_proof_compress: 1472-byte block -> 848-byte block with compressed points.  Host only; raises Malformed."""
    out = (C.c_char * PROOF_COMPRESSED_FIXED_BYTES)()
    rc = lib().tp_proof_compress(_buf(fixed), C.c_size_t(len(fixed)), out, C.c_size_t(PROOF_COMPRESSED_FIXED_BYTES))
    if rc == 12:
        raise Malformed(rc, "tp_proof_compress: malformed proof block")
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_compress")
    return bytes(out)


def proof_decompress(block: bytes) -> bytes:
    """tp_proof_decompress (checked): 848-byte block -> 1472-byte block.  Host only; raises Malformed."""
    out = (C.c_char * PROOF_FIXED_BYTES)()
    rc = lib().tp_proof_decompress(_buf(block), C.c_size_t(len(block)), out, C.c_size_t(PROOF_FIXED_BYTES))
    if rc == 12:
        raise Malformed(rc, "tp_proof_decompress: malformed compressed proof block")
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_decompress")
    return bytes(out)


def proof_encode_compressed(fixed: bytes, public_inputs_mont: bytes) -> bytes:
    """tp_proof_encode_compressed: the 848-byte compressed block + Vec<Fr> of public inputs.  Host only."""
    n = len(public_inputs_mont) // 32
    need = C.c_size_t(0)
    lib().tp_proof_encoded_size_compressed(C.c_size_t(n), C.byref(need))
    out = (C.c_char * need.value)()
    rc = lib().tp_proof_encode_compressed(_buf(fixed), _buf(public_inputs_mont) if n else None, C.c_size_t(n), out,
                                          C.c_size_t(need.value), None)
    if rc == 12:
        raise Malformed(rc, "tp_proof_encode_compressed: malformed proof block")
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_encode_compressed")
    return bytes(out)


def proof_decode_compressed(raw: bytes):
    """tp_proof_decode_compressed (checked): -> (uncompressed 1472-byte block, public inputs as Montgomery bytes)."""
    n = C.c_size_t(0)
    rc = lib().tp_proof_decode_compressed(_buf(raw), C.c_size_t(len(raw)), None, None, C.c_size_t(0), C.byref(n))
    if rc == 12:
        raise Malformed(rc, "tp_proof_decode_compressed: malformed proof encoding")
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_decode_compressed")
    fixed = (C.c_char * PROOF_FIXED_BYTES)()
    pis = (C.c_char * (32 * n.value or 1))()
    rc = lib().tp_proof_decode_compressed(_buf(raw), C.c_size_t(len(raw)), fixed, pis, C.c_size_t(n.value), C.byref(n))
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_decode_compressed")
    return bytes(fixed), bytes(pis)[: 32 * n.value]


def proof_points_in_subgroup(fixed: bytes) -> bool:
    """tp_proof_points_in_subgroup: [r]P = 0 for every G1 point of the proof (ark's checked deserialisation)."""
    ok = C.c_int(0)
    rc = lib().tp_proof_points_in_subgroup(_buf(fixed), C.c_size_t(len(fixed)), C.byref(ok))
    if rc == 12:
        raise Malformed(rc, "tp_proof_points_in_subgroup: malformed point")
    if rc != 0:
        raise TyplonkError(rc, "tp_proof_points_in_subgroup")
    return bool(ok.value)


GATE_MUL, GATE_ADD, GATE_DUMMY = 0, 1, 2


class Trace:
    """tp_trace: a circuit recorded once as a flat gate list; padding, selectors, the copy-constraint permutation
    and witnesses come from it natively (plonk/src/builder.rs:119-188, 339-397; permutation/src/lib.rs:62-93;
    plonk/src/proof.rs:33-49).  Host only."""

    def __init__(self, n_inputs: int):
        self._h = C.c_void_p()
        self.n_inputs = n_inputs
        self.rows = None
        self.gate_count = None
        rc = lib().tp_trace_create(C.c_size_t(n_inputs), C.byref(self._h))
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_create")

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.tp_trace_destroy(self._h)
            self._h = None

    def gate(self, kind: int, lhs: int, rhs: int) -> int:
        out = C.c_uint64(0)
        rc = lib().tp_trace_gate(self._h, C.c_int(kind), C.c_uint64(lhs), C.c_uint64(rhs), C.byref(out))
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_gate(%d, %d, %d)" % (kind, lhs, rhs))
        return out.value

    def gates(self, kinds, lhs, rhs):
        """Bulk form over numpy arrays (uint8, uint64, uint64); returns the output ids (uint64)."""
        import numpy as np
        kinds = np.ascontiguousarray(kinds, dtype=np.uint8)
        lhs = np.ascontiguousarray(lhs, dtype=np.uint64)
        rhs = np.ascontiguousarray(rhs, dtype=np.uint64)
        assert len(kinds) == len(lhs) == len(rhs)
        out = np.empty(len(kinds), dtype=np.uint64)
        rc = lib().tp_trace_gates(self._h, C.c_size_t(len(kinds)), _buf(kinds), _buf(lhs), _buf(rhs), _buf(out))
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_gates")
        return out

    def assert_eq(self, a: int, b: int):
        rc = lib().tp_trace_assert_eq(self._h, C.c_uint64(a), C.c_uint64(b))
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_assert_eq(%d, %d)" % (a, b))

    def finish(self):
        rows, gates = C.c_size_t(0), C.c_size_t(0)
        rc = lib().tp_trace_finish(self._h, C.byref(rows), C.byref(gates))
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_finish")
        self.rows, self.gate_count = rows.value, gates.value
        return self.rows, self.gate_count

    def gate_kinds(self) -> bytes:
        out = (C.c_char * self.rows)()
        rc = lib().tp_trace_gate_kinds(self._h, out)
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_gate_kinds")
        return bytes(out)

    def selectors(self) -> bytearray:
        """5 x rows Montgomery Fr, contiguous (q_l | q_r | q_o | q_m | q_c)."""
        out = bytearray(5 * self.rows * 32)
        rc = lib().tp_trace_selectors(self._h, _buf(out))
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_selectors")
        return out

    def permutation(self) -> bytearray:
        """perm[3 * rows] as little-endian u64 (consumes the constraints, like the reference's build)."""
        out = bytearray(3 * self.rows * 8)
        rc = lib().tp_trace_permutation(self._h, _buf(out))
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_permutation")
        return out

    def witness(self, inputs_mont: bytes, blinders_mont: bytes):
        """Three advice columns (rows x 32 B Montgomery each) from n_inputs inputs and nine blinders."""
        assert len(inputs_mont) == 32 * self.n_inputs and len(blinders_mont) == 9 * 32
        cols = [bytearray(self.rows * 32) for _ in range(3)]
        ptrs = (C.c_void_p * 3)(*[C.addressof((C.c_char * len(c)).from_buffer(c)) for c in cols])
        rc = lib().tp_trace_witness(self._h, _buf(inputs_mont), C.c_size_t(self.n_inputs), _buf(blinders_mont), ptrs)
        if rc != 0:
            raise TyplonkError(rc, "tp_trace_witness")
        return cols


class NativePermutationBuilder:
    """tp_permutation_builder: PermutationBuilder<3> (permutation/src/lib.rs:28-93).  Host only."""

    def __init__(self, rows=0):
        self._h = C.c_void_p()
        rc = lib().tp_permutation_builder_create(C.c_size_t(rows), C.byref(self._h))
        if rc != 0:
            raise TyplonkError(rc, "tp_permutation_builder_create")

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.tp_permutation_builder_destroy(self._h)
            self._h = None

    def add_row(self):
        lib().tp_permutation_builder_add_row(self._h)

    def add_constrain(self, left, right) -> bool:
        rc = lib().tp_permutation_builder_add_constrain(self._h, C.c_size_t(left[0]), C.c_size_t(left[1]),
                                                        C.c_size_t(right[0]), C.c_size_t(right[1]))
        if rc == 10:
            return False
        if rc != 0:
            raise TyplonkError(rc, "tp_permutation_builder_add_constrain")
        return True

    def build(self, size: int):
        import struct
        out = bytearray(3 * size * 8)
        rc = lib().tp_permutation_builder_build(self._h, C.c_size_t(size), _buf(out))
        if rc != 0:
            raise TyplonkError(rc, "tp_permutation_builder_build")
        return list(struct.unpack("<%dQ" % (3 * size), out))


class VerifierInputs(C.Structure):
    """tp_verifier_inputs."""
    _fields_ = [("fixed_commitments", C.c_char * (5 * G1_BYTES)), ("sigma_commitments", C.c_char * (3 * G1_BYTES)),
                ("identity", C.c_char * G1_BYTES), ("g2", C.c_char * G2_BYTES), ("g2s", C.c_char * G2_BYTES),
                ("cosets", C.c_uint64 * 12), ("sigma_evals", C.c_uint64 * 8), ("public_eval", C.c_uint64 * 4),
                ("n", C.c_uint64)]


def verify_prepared(fixed, sigma, identity, g2, g2s, cosets_mont, sigma_evals_mont, public_eval_mont, n, proof_fixed) -> bool:
    """tp_verify_prepared: the host half of the verifier from a verification key (ABI records / Montgomery bytes)."""
    v = VerifierInputs()
    C.memmove(C.addressof(v) + VerifierInputs.fixed_commitments.offset, b"".join(fixed), 5 * G1_BYTES)
    C.memmove(C.addressof(v) + VerifierInputs.sigma_commitments.offset, b"".join(sigma), 3 * G1_BYTES)
    C.memmove(C.addressof(v) + VerifierInputs.identity.offset, identity, G1_BYTES)
    C.memmove(C.addressof(v) + VerifierInputs.g2.offset, g2, G2_BYTES)
    C.memmove(C.addressof(v) + VerifierInputs.g2s.offset, g2s, G2_BYTES)
    C.memmove(C.addressof(v) + VerifierInputs.cosets.offset, b"".join(cosets_mont), 96)
    C.memmove(C.addressof(v) + VerifierInputs.sigma_evals.offset, b"".join(sigma_evals_mont), 64)
    C.memmove(C.addressof(v) + VerifierInputs.public_eval.offset, public_eval_mont, 32)
    v.n = n
    ok = C.c_int(0)
    rc = lib().tp_verify_prepared(C.byref(v), _buf(proof_fixed), C.c_size_t(len(proof_fixed)), C.byref(ok))
    if rc != 0:
        raise TyplonkError(rc, "tp_verify_prepared: malformed input")
    return bool(ok.value)


class Context:
    def __init__(self, device=0, stream=None):
        L = lib()
        self._h = C.c_void_p()
        rc = L.tp_ctx_create(C.c_int(device), C.c_void_p(stream or 0), C.byref(self._h))
        if rc != 0:
            raise TyplonkError(rc, "tp_ctx_create failed (no CUDA device? there is no CPU fallback)")
        self._cb = None
        self.device = device

    def _check(self, rc):
        if rc != 0:
            msg = lib().tp_last_error(self._h).decode()
            if rc == 6:
                raise GateUnsatisfied(rc, msg)
            raise TyplonkError(rc, msg)

    def close(self):
        if self._h:
            lib().tp_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def sync(self):
        self._check(lib().tp_sync(self._h))

    def selftest(self):
        f = C.c_int(-1)
        self._check(lib().tp_selftest(self._h, C.byref(f)))
        return f.value

    def measure_imad_peak(self):
        a, b = C.c_double(), C.c_double()
        self._check(lib().tp_measure_imad_peak(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def prof_enable(self, on=True):
        self._check(lib().tp_prof_enable(self._h, C.c_int(1 if on else 0)))

    def prof_reset(self):
        self._check(lib().tp_prof_reset(self._h))

    def prof_get(self):
        ms = (C.c_double * len(PHASES))()
        ln = (C.c_uint64 * len(PHASES))()
        self._check(lib().tp_prof_get(self._h, ms, ln))
        return {p: (ms[i], ln[i]) for i, p in enumerate(PHASES)}

    def launch_count(self):
        v = C.c_uint64()
        self._check(lib().tp_launch_count(self._h, C.byref(v)))
        return v.value

    def set_option(self, name, value):
        """Tunables of the library ("msm_affine_chains": 0/1, "msm_affine_rounds": 0..8, "msm_reduce_l1": 0..2,
        "msm_pipeline": 0..2, "msm_pipe_min_log": 0..27, "msm_acc_staged": 0/1, "msm_fq_lazy": 1 [default] / 0,
        "ntt_radix_log": 2/3, "quotient_all_cosets": 0/1; see the header); results do not depend on them."""
        self._check(lib().tp_ctx_set_option(self._h, name.encode(), C.c_long(int(value))))

    def get_stat(self, name) -> float:
        """Work counters / last MSM plan ("msm_entries", "msm_window_bits", ...), see the header."""
        v = C.c_double()
        self._check(lib().tp_ctx_get_stat(self._h, name.encode(), C.byref(v)))
        return v.value

    def comm_init_rank(self, rank: int, world: int, unique_id: bytes = None):
        """One process per GPU: join the library-owned NCCL communicator as rank `rank` of `world` (before the SRS is
        created).  From here on every MSM is sharded by bucket, the quotient by coset, the witness upload by rows;
        no host-language code runs during a proof."""
        self._check(lib().tp_ctx_comm_init_rank(self._h, C.c_int(rank), C.c_int(world),
                                                _buf(unique_id) if unique_id is not None else None))

    @classmethod
    def multi(cls, devices):
        """tp_ctx_create_multi: ONE context over several GPUs of this process (a device listed twice = two ranks on
        it, exchanging through peer copies instead of NCCL -- how the single-GPU tests run the sharded path)."""
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        self._cb = None
        self.device = devices[0]
        arr = (C.c_int * len(devices))(*devices)
        rc = lib().tp_ctx_create_multi(arr, C.c_int(len(devices)), C.byref(self._h))
        if rc != 0:
            raise TyplonkError(rc, "tp_ctx_create_multi failed (no CUDA device? there is no CPU fallback)")
        return self

    def group_size(self):
        """(ranks behind this context, whether they exchange through NCCL)."""
        n, nc = C.c_int(0), C.c_int(0)
        self._check(lib().tp_ctx_group_size(self._h, C.byref(n), C.byref(nc)))
        return n.value, bool(nc.value)

    # ---- SRS ---------------------------------------------------------------------------
    def srs_from_secret(self, tau_mont: bytes, gates: int):
        h = C.c_void_p()
        self._check(lib().tp_srs_from_secret(self._h, _buf(tau_mont), C.c_size_t(gates), C.byref(h)))
        return SrsHandle(self, h)

    def srs_upload(self, g1_xy: bytes):
        assert len(g1_xy) % 96 == 0
        h = C.c_void_p()
        self._check(lib().tp_srs_upload(self._h, _buf(g1_xy), C.c_size_t(len(g1_xy) // 96), C.byref(h)))
        return SrsHandle(self, h)

    def srs_contribute(self, srs, s_mont: bytes):
        """tp_srs_contribute: (new SRS with g1[i] * s^i and g2s * s, pubkey [s]G2 as a 193-byte ABI record)."""
        h = C.c_void_p()
        pub = (C.c_char * G2_BYTES)()
        self._check(lib().tp_srs_contribute(self._h, srs._h, _buf(s_mont), C.byref(h), pub))
        return SrsHandle(self, h), bytes(pub)

    def srs_verify(self, srs) -> bool:
        """tp_srs_verify: is the SRS the powers of one secret (randomised pairing check, G1 subgroup checks)?"""
        ok = C.c_int(0)
        self._check(lib().tp_srs_verify(self._h, srs._h, C.byref(ok)))
        return bool(ok.value)

    # ---- KZG / NTT / permutation ---------------------------------------------------------
    def commit(self, srs, coeffs_mont: bytes) -> bytes:
        out = (C.c_char * G1_BYTES)()
        self._check(lib().tp_commit(self._h, srs._h, _buf(coeffs_mont), C.c_size_t(len(coeffs_mont) // 32), out))
        return bytes(out)

    def commit_dev(self, srs, dptr: int, length: int) -> bytes:
        out = (C.c_char * G1_BYTES)()
        self._check(lib().tp_commit_dev(self._h, srs._h, C.c_void_p(dptr), C.c_size_t(length), out))
        return bytes(out)

    def open(self, srs, coeffs_mont: bytes, z_mont: bytes):
        w = (C.c_char * G1_BYTES)()
        y = (C.c_char * 32)()
        self._check(lib().tp_open(self._h, srs._h, _buf(coeffs_mont), C.c_size_t(len(coeffs_mont) // 32),
                                  _buf(z_mont), w, y))
        return bytes(w), bytes(y)

    def ntt(self, data_mont, log_n: int, inverse=False, coset_mont: bytes = None) -> bytes:
        buf = bytearray(data_mont)
        assert len(buf) == 32 << log_n
        cos = _buf(coset_mont) if coset_mont is not None else None
        self._check(lib().tp_ntt(self._h, _buf(buf), C.c_uint(log_n), C.c_int(1 if inverse else 0), cos))
        return bytes(buf)

    def ntt_dev(self, dptr: int, log_n: int, inverse=False, coset_mont: bytes = None):
        cos = _buf(coset_mont) if coset_mont is not None else None
        self._check(lib().tp_ntt_dev(self._h, C.c_void_p(dptr), C.c_uint(log_n), C.c_int(1 if inverse else 0), cos))

    def permutation_compile(self, perm_u64: bytes, n: int):
        """tp_permutation_compile: (3 id columns, 3 sigma columns, 3 coset representatives), Montgomery bytes."""
        ids = [bytearray(32 * n) for _ in range(3)]
        sgs = [bytearray(32 * n) for _ in range(3)]
        ip = (C.c_void_p * 3)(*[C.addressof((C.c_char * len(b)).from_buffer(b)) for b in ids])
        sp = (C.c_void_p * 3)(*[C.addressof((C.c_char * len(b)).from_buffer(b)) for b in sgs])
        ks = (C.c_uint64 * 12)()
        self._check(lib().tp_permutation_compile(self._h, _buf(perm_u64), C.c_size_t(n), ip, sp, ks))
        raw = bytes(ks)
        return ids, sgs, [raw[32 * i:32 * i + 32] for i in range(3)]

    def perm_prove(self, values, ids, sigmas, beta_mont: bytes, gamma_mont: bytes) -> bytes:
        n = len(values[0]) // 32
        keep = [_buf(b) for b in list(values) + list(ids) + list(sigmas)]
        arr = lambda xs: (C.c_void_p * 3)(*[C.cast(x, C.c_void_p) for x in xs])  # noqa: E731
        out = (C.c_char * (32 * (n + 1)))()
        self._check(lib().tp_perm_prove(self._h, arr(keep[0:3]), arr(keep[3:6]), arr(keep[6:9]), C.c_size_t(n),
                                        _buf(beta_mont), _buf(gamma_mont), out))
        return bytes(out)

    # ---- circuits ----------------------------------------------------------------------------
    def circuit_load(self, srs, selector_coeffs, ids, sigmas, cosets_mont, n):
        keep = [_buf(b) for b in list(selector_coeffs) + list(ids) + list(sigmas)]
        sel = (C.c_void_p * 5)(*[C.cast(x, C.c_void_p) for x in keep[0:5]])
        idp = (C.c_void_p * 3)(*[C.cast(x, C.c_void_p) for x in keep[5:8]])
        sgp = (C.c_void_p * 3)(*[C.cast(x, C.c_void_p) for x in keep[8:11]])
        cos = _buf(b"".join(cosets_mont))
        h = C.c_void_p()
        self._check(lib().tp_circuit_load(self._h, srs._h, sel, idp, sgp, cos, C.c_size_t(n), C.byref(h)))
        return CircuitHandle(self, h, n, srs)

    def srs_deserialize(self, raw, check=2):
        """tp_srs_deserialize: ark-serialize 0.3 uncompressed Vec<G1> | G2 | tau G2 -> device SRS.
        check: 0 canonical only, 1 + on curve, 2 + prime-order subgroup.  Raises Malformed."""
        h = C.c_void_p()
        rc = lib().tp_srs_deserialize(self._h, _buf(raw), C.c_size_t(len(raw)), C.c_int(check), C.byref(h))
        if rc == 12:
            raise Malformed(rc, lib().tp_last_error(self._h).decode())
        self._check(rc)
        return SrsHandle(self, h)

    def srs_deserialize_compressed(self, raw, check=2):
        """tp_srs_deserialize_compressed: u64 count | count x 48 B G1 | G2 | tau G2 (96 B each) -> device SRS; the
        square roots and checks run on the device.  check: 0 / 1 recover y, 2 + prime-order subgroup.  Raises
        Malformed."""
        h = C.c_void_p()
        rc = lib().tp_srs_deserialize_compressed(self._h, _buf(raw), C.c_size_t(len(raw)), C.c_int(check), C.byref(h))
        if rc == 12:
            raise Malformed(rc, lib().tp_last_error(self._h).decode())
        self._check(rc)
        return SrsHandle(self, h)

    def vk_deserialize(self, raw, check=2):
        """tp_vk_deserialize: a verification key's bytes (1376 + 64n) -> device key.  check: 0 canonical encoding and
        framing, 1 + points on their curves, 2 + prime-order subgroups.  Raises Malformed naming the field."""
        h = C.c_void_p()
        rc = lib().tp_vk_deserialize(self._h, _buf(raw), C.c_size_t(len(raw)), C.c_int(check), C.byref(h))
        if rc == 12:
            raise Malformed(rc, lib().tp_last_error(self._h).decode())
        self._check(rc)
        return VerifyingKeyHandle(self, h)

    def vk_verify_batch(self, keys, key_of, proofs_fixed, public_inputs):
        """tp_vk_verify_batch: proof k (a 1472-byte block) against keys[key_of[k]], public_inputs[k] its Montgomery
        public-input bytes (b"" = none).  Returns (every proof accepted, per-proof verdicts)."""
        count = len(proofs_fixed)
        assert len(public_inputs) == count and len(key_of) == count
        if any(len(p) != PROOF_FIXED_BYTES for p in proofs_fixed):
            raise TyplonkError(1, "vk_verify_batch: every proof must be a %d-byte block" % PROOF_FIXED_BYTES)
        hs = (C.c_void_p * max(len(keys), 1))(*[k._h for k in keys])
        kof = (C.c_uint32 * max(count, 1))(*key_of)
        blob = b"".join(proofs_fixed)
        keep = [(C.c_char * len(b)).from_buffer_copy(b) if b else None for b in public_inputs]
        pis = (C.c_void_p * max(count, 1))(*[C.cast(b, C.c_void_p) if b is not None else None for b in keep])
        npub = (C.c_size_t * max(count, 1))(*[len(b) // 32 for b in public_inputs])
        each = (C.c_int * max(count, 1))()
        all_ok = C.c_int(0)
        self._check(lib().tp_vk_verify_batch(self._h, hs, C.c_size_t(len(keys)), kof, _buf(blob) if count else None,
                                             C.c_size_t(count), pis, npub, C.byref(all_ok), each))
        return bool(all_ok.value), [bool(each[k]) for k in range(count)]

    def proofs_decompress(self, blocks: bytes, count: int):
        """tp_proofs_decompress: `count` contiguous 848-byte blocks -> (count x 1472-byte blocks as one bytes object,
        per-block statuses: 0 = TP_OK, 12 = TP_ERR_MALFORMED with the block zero-filled)."""
        out = (C.c_char * max(count * PROOF_FIXED_BYTES, 1))()
        status = (C.c_int * max(count, 1))()
        self._check(lib().tp_proofs_decompress(self._h, _buf(blocks) if count else None, C.c_size_t(count), out,
                                               C.c_size_t(count * PROOF_FIXED_BYTES), status))
        return bytes(out)[: count * PROOF_FIXED_BYTES], [status[k] for k in range(count)]

    def circuit_compile(self, srs, selector_evals, perm_u64: bytes, n):
        keep = [_buf(b) for b in selector_evals]
        sel = (C.c_void_p * 5)(*[C.cast(x, C.c_void_p) for x in keep])
        fixed = (C.c_char * (5 * G1_BYTES))()
        h = C.c_void_p()
        self._check(lib().tp_circuit_compile(self._h, srs._h, sel, _buf(perm_u64), C.c_size_t(n), C.byref(h), fixed))
        raw = bytes(fixed)
        return CircuitHandle(self, h, n, srs), [raw[i * G1_BYTES:(i + 1) * G1_BYTES] for i in range(5)]


class SrsHandle:
    def __init__(self, ctx, h):
        self.ctx = ctx
        self._h = h

    def __len__(self):
        v = C.c_size_t()
        lib().tp_srs_len(self._h, C.byref(v))
        return v.value

    def serialize(self) -> bytearray:
        """tp_srs_serialize: u64 count | count x 96 B G1 | G2 | tau G2 (ark-serialize 0.3 uncompressed)."""
        need = C.c_size_t(0)
        lib().tp_srs_serialized_size(self._h, C.byref(need))
        out = bytearray(need.value)
        self.ctx._check(lib().tp_srs_serialize(self.ctx._h, self._h, _buf(out), C.c_size_t(len(out)), None))
        return out

    def serialize_compressed(self) -> bytearray:
        """tp_srs_serialize_compressed: u64 count | count x 48 B G1 | G2 | tau G2 (96 B each), compressed points."""
        need = C.c_size_t(0)
        lib().tp_srs_serialized_size_compressed(self._h, C.byref(need))
        out = bytearray(need.value)
        self.ctx._check(lib().tp_srs_serialize_compressed(self.ctx._h, self._h, _buf(out), C.c_size_t(len(out)), None))
        return out

    def download(self, offset=0, count=None) -> bytes:
        count = len(self) - offset if count is None else count
        out = (C.c_char * (96 * count))()
        self.ctx._check(lib().tp_srs_g1_download(self.ctx._h, self._h, C.c_size_t(offset), C.c_size_t(count), out))
        return bytes(out)

    def g2(self):
        """(G2, tau G2) as 193-byte ABI records (srs.rs:46-51)."""
        a, b = (C.c_char * G2_BYTES)(), (C.c_char * G2_BYTES)()
        rc = lib().tp_srs_g2(self._h, a, b)
        if rc != 0:
            raise TyplonkError(rc, "tp_srs_g2: this SRS has no G2 points (set_g2)")
        return bytes(a), bytes(b)

    def set_g2(self, g2: bytes, g2s: bytes):
        rc = lib().tp_srs_set_g2(self._h, _buf(g2), _buf(g2s))
        if rc != 0:
            raise TyplonkError(rc, "tp_srs_set_g2: point not on the twist")

    def destroy(self):
        if self._h:
            lib().tp_srs_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()


class CircuitHandle:
    def __init__(self, ctx, h, n, srs):
        self.ctx = ctx
        self._h = h
        self.n = n
        self.srs = srs

    def prove(self, advice_mont, public_inputs_mont) -> bytes:
        keep = [_buf(b) for b in advice_mont]
        adv = (C.c_void_p * 3)(*[C.cast(x, C.c_void_p) for x in keep])
        out = (C.c_char * PROOF_FIXED_BYTES)()
        self.ctx._check(lib().tp_prove(self.ctx._h, self._h, adv, _buf(public_inputs_mont), out,
                                       C.c_size_t(PROOF_FIXED_BYTES)))
        return bytes(out)

    def prove_inputs(self, advice_mont, public_inputs_mont) -> bytes:
        """tp_prove_inputs: the public-input vector as the caller of prove() gives it (any length <= n)."""
        keep = [_buf(b) for b in advice_mont]
        adv = (C.c_void_p * 3)(*[C.cast(x, C.c_void_p) for x in keep])
        out = (C.c_char * PROOF_FIXED_BYTES)()
        n_public = len(public_inputs_mont) // 32
        self.ctx._check(lib().tp_prove_inputs(self.ctx._h, self._h, adv, _buf(public_inputs_mont) if n_public else None,
                                              C.c_size_t(n_public), out, C.c_size_t(PROOF_FIXED_BYTES)))
        return bytes(out)

    def prove_batch(self, advice_list, public_inputs_list):
        """tp_prove_batch: advice_list[k] is proof k's three witness columns, public_inputs_list[k] its public-input
        vector as prove_inputs takes it (Montgomery bytes, any length <= n; b"" = none).  Returns (proof blocks,
        statuses): status 0 is a proof, 6 (gate unsatisfied) or 5 (zero denominator) a zero-filled block."""
        count = len(advice_list)
        assert len(public_inputs_list) == count
        keep = [(C.c_char * len(b)).from_buffer_copy(b) for cols in advice_list for b in cols]
        adv = (C.c_void_p * max(3 * count, 1))(*[C.cast(b, C.c_void_p) for b in keep])
        pkeep = [(C.c_char * len(b)).from_buffer_copy(b) if b else None for b in public_inputs_list]
        pis = (C.c_void_p * max(count, 1))(*[C.cast(b, C.c_void_p) if b is not None else None for b in pkeep])
        npub = (C.c_size_t * max(count, 1))(*[len(b) // 32 for b in public_inputs_list])
        out = (C.c_char * max(count * PROOF_FIXED_BYTES, 1))()
        status = (C.c_int * max(count, 1))()
        self.ctx._check(lib().tp_prove_batch(self.ctx._h, self._h, C.c_size_t(count), adv, pis, npub, out,
                                             C.c_size_t(count * PROOF_FIXED_BYTES), status))
        raw = bytes(out)
        return ([raw[k * PROOF_FIXED_BYTES:(k + 1) * PROOF_FIXED_BYTES] for k in range(count)],
                [status[k] for k in range(count)])

    def prove_dev(self, advice_dptrs, pi_dptr) -> bytes:
        adv = (C.c_void_p * 3)(*[C.c_void_p(p) for p in advice_dptrs])
        out = (C.c_char * PROOF_FIXED_BYTES)()
        self.ctx._check(lib().tp_prove_dev(self.ctx._h, self._h, adv, C.c_void_p(pi_dptr), out,
                                           C.c_size_t(PROOF_FIXED_BYTES)))
        return bytes(out)

    def verify(self, proof_fixed: bytes, public_inputs_mont: bytes) -> bool:
        ok = C.c_int(0)
        self.ctx._check(lib().tp_verify(self.ctx._h, self._h, _buf(proof_fixed), C.c_size_t(len(proof_fixed)),
                                        _buf(public_inputs_mont) if public_inputs_mont else None,
                                        C.c_size_t(len(public_inputs_mont) // 32), C.byref(ok)))
        return bool(ok.value)

    def verify_batch(self, proofs_fixed, public_inputs):
        """tp_verify_batch: proofs_fixed[k] is proof k's 1472-byte block, public_inputs[k] its public-input vector as
        Montgomery bytes (b"" = none).  Returns (every proof accepted, per-proof verdicts)."""
        count = len(proofs_fixed)
        assert len(public_inputs) == count
        if any(len(p) != PROOF_FIXED_BYTES for p in proofs_fixed):
            raise TyplonkError(1, "verify_batch: every proof must be a %d-byte block" % PROOF_FIXED_BYTES)
        blob = b"".join(proofs_fixed)
        keep = [(C.c_char * len(b)).from_buffer_copy(b) if b else None for b in public_inputs]
        pis = (C.c_void_p * max(count, 1))(*[C.cast(b, C.c_void_p) if b is not None else None for b in keep])
        npub = (C.c_size_t * max(count, 1))(*[len(b) // 32 for b in public_inputs])
        each = (C.c_int * max(count, 1))()
        all_ok = C.c_int(0)
        self.ctx._check(lib().tp_verify_batch(self.ctx._h, self._h, _buf(blob) if count else None, C.c_size_t(count),
                                              pis, npub, C.byref(all_ok), each))
        return bool(all_ok.value), [bool(each[k]) for k in range(count)]

    def verifying_key(self):
        """tp_vk_from_circuit: the circuit's verification key (owns its copies; outlives the circuit)."""
        h = C.c_void_p()
        self.ctx._check(lib().tp_vk_from_circuit(self.ctx._h, self._h, C.byref(h)))
        return VerifyingKeyHandle(self.ctx, h)

    POLY_QUOTIENT, POLY_LINEARISATION, POLY_Z_EVALS, POLY_Z, POLY_A, POLY_B, POLY_C = range(7)

    def read_poly(self, which: int) -> bytes:
        """tp_circuit_read_poly: an intermediate polynomial of the last proof (Montgomery bytes)."""
        cnt = C.c_size_t(0)
        self.ctx._check(lib().tp_circuit_read_poly(self.ctx._h, self._h, C.c_int(which), None, C.c_size_t(0), C.byref(cnt)))
        out = (C.c_char * (32 * cnt.value))()
        self.ctx._check(lib().tp_circuit_read_poly(self.ctx._h, self._h, C.c_int(which), out, C.c_size_t(cnt.value), C.byref(cnt)))
        return bytes(out)

    def sigma_commitments(self):
        out = (C.c_char * (3 * G1_BYTES))()
        self.ctx._check(lib().tp_circuit_sigma_commitments(self.ctx._h, self._h, out))
        raw = bytes(out)
        return [raw[i * G1_BYTES:(i + 1) * G1_BYTES] for i in range(3)]

    def destroy(self):
        if self._h:
            lib().tp_circuit_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()


class VerifyingKeyHandle:
    """A tp_vk: what verify() reads of a compiled circuit (include/typlonk_b200.h, "verification keys")."""

    def __init__(self, ctx, h):
        self.ctx = ctx
        self._h = h

    def serialized_size(self) -> int:
        need = C.c_size_t(0)
        lib().tp_vk_serialized_size(self._h, C.byref(need))
        return need.value

    def serialize(self) -> bytearray:
        """tp_vk_serialize: "TPVK" | u32 1 | u64 n | 3 Fr | 9 G1 | 2 G2 | Vec<Fr> sigma_1 | Vec<Fr> sigma_2."""
        out = bytearray(self.serialized_size())
        self.ctx._check(lib().tp_vk_serialize(self.ctx._h, self._h, _buf(out), C.c_size_t(len(out)), None))
        return out

    def verify(self, proof_fixed: bytes, public_inputs_mont: bytes) -> bool:
        """tp_vk_verify: tp_verify's verdict (and errors) for the circuit the key came from."""
        ok = C.c_int(0)
        self.ctx._check(lib().tp_vk_verify(self.ctx._h, self._h, _buf(proof_fixed), C.c_size_t(len(proof_fixed)),
                                           _buf(public_inputs_mont) if public_inputs_mont else None,
                                           C.c_size_t(len(public_inputs_mont) // 32), C.byref(ok)))
        return bool(ok.value)

    def destroy(self):
        if self._h:
            lib().tp_vk_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                self.destroy()
        except Exception:
            pass
