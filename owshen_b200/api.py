"""ctypes binding of libowshen_b200.so and the host-side mirror of the API BASELINE.json's north_star
names: prove() / verify() / MerkleTree.  The reference (OwshenNetwork/owshen @ c7b1f00) has no such
API (SURVEY.md section 0), so names and error behaviour follow its conventions instead: fallible
calls raise (anyhow::Result -> exception), byte blobs are owned `bytes`, field elements are 32-byte
little-endian (/root/reference/src/blockchain/tx/owshen_airdrop/babyjubjub/mod.rs:7-11).

All hashing, witness generation, NTTs and MSMs run in the CUDA library; nothing here computes.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# OWSHEN_B200_LIB: an alternative build of the same library (e.g. another commit's, for an A/B)
_LIB_PATH = os.environ.get("OWSHEN_B200_LIB") or os.path.join(_HERE, "libowshen_b200.so")
_lib = None

FR_MODULUS = 21888242871839275222246405745257275088548364400416034343698204186575808495617
PROOF_BYTES = 256

OG_OK, OG_E_INVALID, OG_E_VERIFY = 0, -1, -6


class OwshenB200Error(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        msg = lib().og_strerror(code).decode() if _lib is not None else str(code)
        super().__init__(f"owshen_b200 error {code}: {msg}" + (f" ({detail})" if detail else ""))


def build_library(jobs=8):
    """Compile every CUDA source for sm_100a into owshen_b200/libowshen_b200.so (in-tree)."""
    subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), f"-j{jobs}"], check=True, stdout=subprocess.DEVNULL)


_u8p = C.c_char_p
_SIGS = {
    "og_abi_version": (C.c_int32, []),
    "og_strerror": (C.c_char_p, [C.c_int32]),
    "og_last_error": (C.c_char_p, [C.c_void_p]),
    "og_init": (C.c_int32, [C.c_int32, C.POINTER(C.c_void_p)]),
    "og_free": (None, [C.c_void_p]),
    "og_sync": (C.c_int32, [C.c_void_p]),
    "og_stream": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "og_timer_start": (C.c_int32, [C.c_void_p]),
    "og_timer_stop": (C.c_int32, [C.c_void_p, C.POINTER(C.c_float)]),
    "og_launch_count": (C.c_uint64, [C.c_void_p]),
    "og_profile": (C.c_int32, [C.c_void_p, C.c_int32]),
    "og_profile_dump": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_uint64]),
    "og_imad_peak": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "og_int_pipe_peaks": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "og_mul_latency": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "og_hybrid_probe": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double)]),
    "og_fp64_peak": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double)]),
    "og_field_op": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_mimc7_constants": (C.c_int32, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "og_mimc7_hash2": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_mimc7_merkle_paths": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "og_mimc7_merkle_paths_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "og_mimc7_merkle_build": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_mimc7_merkle_append": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "og_bjj_verify_batch": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p]),
    "og_bjj_verify_batch_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p]),
    "og_bjj_sign_batch_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "og_bjj_sign_batch": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "og_msm_g1": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_msm_g2": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_msm_g1_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_msm_g2_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g1_generator_mul": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g2_generator_mul": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g1_generator_mul_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g2_generator_mul_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g1_sum_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g2_sum_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g1_sum": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_g2_sum": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "og_ntt": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32]),
    "og_ntt_dev": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32]),
    "og_withdraw_r1cs_info": (C.c_int32, [C.c_uint32] + [C.POINTER(C.c_uint32)] * 4),
    "og_withdraw_r1cs_export": (C.c_int32, [C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "og_withdraw_witness": (C.c_int32, [C.c_void_p, C.c_uint32] + [C.c_void_p] * 5 + [C.c_uint32, C.c_void_p]),
    "og_groth16_setup_withdraw": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.POINTER(C.c_uint64)]),
    "og_load_pk": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "og_free_pk": (None, [C.c_void_p]),
    "og_pk_info": (C.c_int32, [C.c_void_p] + [C.POINTER(C.c_uint32)] * 4),
    "og_groth16_prove": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "og_groth16_prove_withdraw": (C.c_int32, [C.c_void_p, C.c_void_p] + [C.c_void_p] * 5 + [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "og_groth16_prove_withdraw_dev": (C.c_int32, [C.c_void_p, C.c_void_p] + [C.c_void_p] * 5 + [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "og_groth16_h_evals": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "og_groth16_verify": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p]),
}
ABI_SYMBOLS = tuple(_SIGS)


def lib():
    """Load libowshen_b200.so; raises if the CUDA extension has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise OSError(f"{_LIB_PATH} is missing: build it with owshen_b200.build_library() / "
                          "`make -C owshen_b200/csrc` -- there is no CPU fallback")
        L = C.CDLL(_LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(rc, ctx=None):
    if rc != OG_OK:
        detail = ""
        if ctx is not None and ctx._h:
            detail = lib().og_last_error(ctx._h).decode(errors="replace")
        raise OwshenB200Error(rc, detail)


def _ptr(x):
    """bytes / bytearray / int address / object with .ctypes or data_ptr() -> void*"""
    if x is None:
        return None
    if isinstance(x, int):
        return C.c_void_p(x)
    if isinstance(x, (bytes, bytearray)):
        return C.cast(C.c_char_p(bytes(x)) if isinstance(x, bytearray) else C.c_char_p(x), C.c_void_p)
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    if hasattr(x, "ctypes"):
        return C.c_void_p(x.ctypes.data)
    return C.cast(x, C.c_void_p)


def _need(cond, what):
    """Argument validation at the Python boundary: the C side takes plain pointers and trusts the sizes it is given,
    so every wrapper checks lengths first and raises ValueError (never `assert`, which python -O strips)."""
    if not cond:
        raise ValueError(what)


def _blen(x):
    """Byte length of a bytes-like / array / tensor argument, or None when only an address was passed."""
    if isinstance(x, (bytes, bytearray, memoryview)):
        return len(x)
    if hasattr(x, "nbytes"):
        return int(x.nbytes)
    if hasattr(x, "numel") and hasattr(x, "element_size"):
        return int(x.numel() * x.element_size())
    return None


def _need_len(x, n, name):
    got = _blen(x)
    _need(got is None or got == n, f"{name}: expected {n} bytes, got {got}")


def _bits_array(bits):
    return (C.c_uint32 * len(bits))(*[int(b) & 0xFFFFFFFF for b in bits])


def fr_bytes(x: int) -> bytes:
    return (x % FR_MODULUS).to_bytes(32, "little")


class Context:
    """One CUDA device + one stream (og_ctx)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check(lib().og_init(device, C.byref(self._h)))
        self.device = device

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.og_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:      # interpreter shutdown
            pass

    def sync(self):
        _check(lib().og_sync(self._h), self)

    @property
    def cuda_stream(self) -> int:
        """Address of the cudaStream_t the `_dev` entry points enqueue on (wrap with torch.cuda.ExternalStream)."""
        p = C.c_void_p()
        _check(lib().og_stream(self._h, C.byref(p)), self)
        return p.value or 0

    def timer_start(self):
        _check(lib().og_timer_start(self._h), self)

    def timer_stop(self) -> float:
        ms = C.c_float()
        _check(lib().og_timer_stop(self._h, C.byref(ms)), self)
        return ms.value

    @property
    def launch_count(self) -> int:
        return lib().og_launch_count(self._h)

    def profile(self, enable: bool):
        _check(lib().og_profile(self._h, int(enable)), self)

    def profile_dump(self) -> dict:
        """{kernel: (launches, total_ms)} since the previous dump (synchronises the stream)."""
        buf = C.create_string_buffer(1 << 16)
        _check(lib().og_profile_dump(self._h, buf, len(buf)), self)
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, ms = line.rsplit(",", 2)
            out[name] = (int(n), float(ms))
        return out

    def imad_peak(self):
        a, b = C.c_double(), C.c_double()
        _check(lib().og_imad_peak(self._h, C.byref(a), C.byref(b)), self)
        return a.value, b.value

    def mul_latency(self):
        a, b = C.c_double(), C.c_double()
        _check(lib().og_mul_latency(self._h, C.byref(a), C.byref(b)), self)
        return a.value, b.value

    def hybrid_probe(self) -> dict:
        r = (C.c_double * 4)()
        _check(lib().og_hybrid_probe(self._h, r), self)
        return {"fp64_products_52bit_alone": r[0], "imad_wide_chain_alone": r[1],
                "fp64_products_52bit_mixed": r[2], "imad_wide_chain_mixed": r[3]}

    def fp64_peak(self) -> float:
        v = C.c_double()
        _check(lib().og_fp64_peak(self._h, C.byref(v)), self)
        return v.value

    def int_pipe_peaks(self) -> dict:
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        _check(lib().og_int_pipe_peaks(self._h, C.byref(a), C.byref(b), C.byref(c)), self)
        return {"imad_per_s": a.value, "imad_wide_per_s": b.value, "imad_wide_carry_chain_per_s": c.value}

    # ---- probes / kernels on host buffers -------------------------------------------------------
    def field_op(self, field: str, op: str, a: bytes, b: bytes) -> bytes:
        _need(len(a) % 32 == 0 and len(b) == len(a), "field_op: a and b must be equally long multiples of 32 bytes")
        _need(field in ("fq", "fr") and op in ("mul", "add", "sub"), "field_op: unknown field or op")
        n = len(a) // 32
        out = C.create_string_buffer(32 * n)
        _check(lib().og_field_op(self._h, {"fq": 0, "fr": 1}[field], {"mul": 0, "add": 1, "sub": 2}[op], a, b, n, out), self)
        return out.raw

    def mimc7_hash2(self, left: bytes, right: bytes) -> bytes:
        _need(len(left) % 32 == 0 and len(right) == len(left), "mimc7_hash2: left and right must be equally long multiples of 32 bytes")
        n = len(left) // 32
        out = C.create_string_buffer(32 * n)
        _check(lib().og_mimc7_hash2(self._h, left, right, n, out), self)
        return out.raw

    def merkle_paths(self, leaves: bytes, siblings: bytes, path_bits, depth: int) -> bytes:
        _need(0 <= depth <= 32 and len(leaves) % 32 == 0, "merkle_paths: depth must be <= 32 and leaves a multiple of 32 bytes")
        n = len(leaves) // 32
        _need(len(siblings) == 32 * n * depth and len(path_bits) == n, "merkle_paths: siblings must hold n*depth elements and path_bits n words")
        out = C.create_string_buffer(32 * n * (depth + 1))
        _check(lib().og_mimc7_merkle_paths(self._h, leaves, siblings, _bits_array(path_bits), n, depth, out), self)
        return out.raw

    def merkle_build(self, leaves: bytes) -> bytes:
        _need(len(leaves) % 32 == 0 and len(leaves) >= 32, "merkle_build: leaves must be a non-empty multiple of 32 bytes")
        n = len(leaves) // 32
        _need(n & (n - 1) == 0, "merkle_build: the leaf count must be a power of two (pad with empty leaves)")
        out = C.create_string_buffer(32 * (2 * n - 1))
        _check(lib().og_mimc7_merkle_build(self._h, leaves, n, out), self)
        return out.raw

    def merkle_append(self, depth: int, start: int, leaves: bytes, left_boundary: bytes, zeros: bytes) -> bytes:
        """Nodes of levels 1..depth touched by appending len(leaves)/32 leaves at index `start` (og_mimc7_merkle_append)."""
        _need(1 <= depth <= 32 and len(leaves) % 32 == 0 and len(leaves) > 0, "merkle_append: bad depth or leaves")
        n = len(leaves) // 32
        _need(start >= 0 and start + n <= (1 << depth), "merkle_append: the leaves do not fit the tree")
        _need(len(left_boundary) == 32 * depth and len(zeros) == 32 * depth, "merkle_append: boundary and zeros hold one element per level")
        total = sum(((start + n - 1) >> l) - (start >> l) + 1 for l in range(1, depth + 1))
        out = C.create_string_buffer(32 * total)
        _check(lib().og_mimc7_merkle_append(self._h, depth, start, leaves, n, left_boundary, zeros, out), self)
        return out.raw

    def bjj_verify_batch(self, pk_x: bytes, pk_is_odd: bytes, messages: bytes, signatures: bytes, hash_kind: int = 0) -> bytes:
        """BabyJubJub batch verification; one status byte per signature (1 ok, 0 bad, 2 undecompressible pk)."""
        n = len(pk_is_odd)
        _need(len(pk_x) == 32 * n and len(messages) == 32 * n and len(signatures) == 96 * n, "bjj_verify_batch: inconsistent lengths")
        _need(hash_kind in (0, 1), "bjj_verify_batch: hash_kind must be 0 or 1")
        out = C.create_string_buffer(n)
        _check(lib().og_bjj_verify_batch(self._h, pk_x, pk_is_odd, messages, signatures, n, hash_kind, out), self)
        return out.raw

    def bjj_sign_batch(self, secret_keys: bytes, randomness: bytes, messages: bytes, hash_kind: int = 0):
        """BabyJubJub key derivation + signing, one key per 32 bytes: -> (pk_x, pk_is_odd, signatures, status) with
        status 1 = signed, 2 = the reference's sign() would return Err("Invalid repr")."""
        _need(len(secret_keys) % 32 == 0 and len(randomness) == len(secret_keys) and len(messages) == len(secret_keys),
              "bjj_sign_batch: keys, randomness and messages must be equally long multiples of 32 bytes")
        _need(hash_kind in (0, 1), "bjj_sign_batch: hash_kind must be 0 or 1")
        n = len(secret_keys) // 32
        px, odd = C.create_string_buffer(32 * n), C.create_string_buffer(n)
        sg, st = C.create_string_buffer(96 * n), C.create_string_buffer(n)
        _check(lib().og_bjj_sign_batch(self._h, secret_keys, randomness, messages, n, hash_kind, px, odd, sg, st), self)
        return px.raw, odd.raw[:n], sg.raw, st.raw[:n]

    def msm_g1(self, points: bytes, scalars: bytes) -> bytes:
        _need(len(scalars) % 32 == 0, "msm_g1: scalars must be a multiple of 32 bytes")
        n = len(scalars) // 32
        _need(len(points) == 64 * n, "msm_g1: need one 64-byte point per scalar")
        out = C.create_string_buffer(64)
        _check(lib().og_msm_g1(self._h, points, scalars, n, out), self)
        return out.raw

    def msm_g2(self, points: bytes, scalars: bytes) -> bytes:
        _need(len(scalars) % 32 == 0, "msm_g2: scalars must be a multiple of 32 bytes")
        n = len(scalars) // 32
        _need(len(points) == 128 * n, "msm_g2: need one 128-byte point per scalar")
        out = C.create_string_buffer(128)
        _check(lib().og_msm_g2(self._h, points, scalars, n, out), self)
        return out.raw

    def g1_generator_mul(self, scalars: bytes) -> bytes:
        _need(len(scalars) % 32 == 0, "g1_generator_mul: scalars must be a multiple of 32 bytes")
        n = len(scalars) // 32
        out = C.create_string_buffer(64 * n)
        _check(lib().og_g1_generator_mul(self._h, scalars, n, out), self)
        return out.raw

    def g2_generator_mul(self, scalars: bytes) -> bytes:
        _need(len(scalars) % 32 == 0, "g2_generator_mul: scalars must be a multiple of 32 bytes")
        n = len(scalars) // 32
        out = C.create_string_buffer(128 * n)
        _check(lib().og_g2_generator_mul(self._h, scalars, n, out), self)
        return out.raw

    def g1_sum(self, points: bytes) -> bytes:
        _need(len(points) % 64 == 0, "g1_sum: points must be a multiple of 64 bytes")
        out = C.create_string_buffer(64)
        _check(lib().og_g1_sum(self._h, points, len(points) // 64, out), self)
        return out.raw

    def g2_sum(self, points: bytes) -> bytes:
        _need(len(points) % 128 == 0, "g2_sum: points must be a multiple of 128 bytes")
        out = C.create_string_buffer(128)
        _check(lib().og_g2_sum(self._h, points, len(points) // 128, out), self)
        return out.raw

    def ntt(self, data: bytes, log_n: int, batch: int = 1, inverse=False, coset=False) -> bytes:
        _need(0 <= log_n <= 27 and batch >= 0 and len(data) == (32 * batch) << log_n, "ntt: data must hold batch * 2^log_n elements of 32 bytes")
        buf = C.create_string_buffer(data, len(data))
        _check(lib().og_ntt(self._h, buf, log_n, batch, int(inverse), int(coset)), self)
        return buf.raw

    def withdraw_witness(self, depth, nullifiers: bytes, secrets: bytes, recipients: bytes, siblings: bytes, path_bits) -> bytes:
        _need(len(nullifiers) % 32 == 0 and 1 <= depth <= 32, "withdraw_witness: bad nullifiers length or depth")
        n = len(nullifiers) // 32
        _need(len(secrets) == 32 * n and len(recipients) == 32 * n and len(siblings) == 32 * n * depth and len(path_bits) == n,
              "withdraw_witness: secrets / recipients / siblings / path_bits do not match the batch")
        nv = r1cs_info(depth)["n_vars"]
        out = C.create_string_buffer(32 * n * nv)
        _check(lib().og_withdraw_witness(self._h, depth, nullifiers, secrets, recipients, siblings, _bits_array(path_bits), n, out), self)
        return out.raw


def mimc7_constants():
    out = C.create_string_buffer(32 * 91)
    n = C.c_uint32()
    _check(lib().og_mimc7_constants(out, C.byref(n)))
    return [int.from_bytes(out.raw[32 * i:32 * i + 32], "little") for i in range(n.value)]


def r1cs_info(depth: int) -> dict:
    v = [C.c_uint32() for _ in range(4)]
    _check(lib().og_withdraw_r1cs_info(depth, *[C.byref(x) for x in v]))
    return dict(n_constraints=v[0].value, n_vars=v[1].value, n_pub=v[2].value, log_m=v[3].value)


def r1cs_export(depth: int, which: str):
    """(row_ptr, col_idx, coeffs as ints) of matrix 'A' | 'B' | 'C' of the product's withdraw R1CS."""
    w = "ABC".index(which)
    nnz = C.c_uint64()
    _check(lib().og_withdraw_r1cs_export(depth, w, None, None, None, C.byref(nnz)))
    nc = r1cs_info(depth)["n_constraints"]
    ptr = (C.c_uint32 * (nc + 1))()
    col = (C.c_uint32 * nnz.value)()
    val = C.create_string_buffer(32 * nnz.value)
    _check(lib().og_withdraw_r1cs_export(depth, w, ptr, col, val, C.byref(nnz)))
    return list(ptr), list(col), [int.from_bytes(val.raw[32 * i:32 * i + 32], "little") for i in range(nnz.value)]


def setup_withdraw(ctx: Context, depth: int, tau: int, alpha: int, beta: int, gamma: int, delta: int):
    """Development setup (toxic waste supplied by the caller) -> (pk_bytes, vk_bytes)."""
    toxic = b"".join(fr_bytes(x) for x in (tau, alpha, beta, gamma, delta))
    pl, vl = C.c_uint64(), C.c_uint64()
    _check(lib().og_groth16_setup_withdraw(ctx._h, depth, toxic, None, C.byref(pl), None, C.byref(vl)), ctx)
    pk = C.create_string_buffer(pl.value)
    vk = C.create_string_buffer(vl.value)
    _check(lib().og_groth16_setup_withdraw(ctx._h, depth, toxic, pk, C.byref(pl), vk, C.byref(vl)), ctx)
    return pk.raw[:pl.value], vk.raw[:vl.value]


class ProvingKey:
    """A proving key resident in HBM together with its fixed-base window tables (og_pk)."""

    def __init__(self, ctx: Context, pk_bytes: bytes):
        self.ctx = ctx
        self._h = C.c_void_p()
        _check(lib().og_load_pk(ctx._h, pk_bytes, len(pk_bytes), C.byref(self._h)), ctx)
        v = [C.c_uint32() for _ in range(4)]
        _check(lib().og_pk_info(self._h, *[C.byref(x) for x in v]))
        self.n_vars, self.n_pub, self.log_m, self.depth = (x.value for x in v)

    def close(self):
        # always release the device tables: the key records its device itself and may outlive its Context
        if getattr(self, "_h", None) and _lib is not None:
            _lib.og_free_pk(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def h_evals(self, witness: bytes) -> bytes:
        _need(len(witness) == 32 * self.n_vars, f"h_evals: a witness is {32 * self.n_vars} bytes")
        out = C.create_string_buffer(32 << self.log_m)
        _check(lib().og_groth16_h_evals(self.ctx._h, self._h, witness, out), self.ctx)
        return out.raw

    def prove_witnesses(self, witnesses: bytes, rs: bytes) -> bytes:
        _need(len(rs) % 64 == 0, "prove_witnesses: rs holds 64 bytes (r, s) per proof")
        batch = len(rs) // 64
        _need(len(witnesses) == 32 * batch * self.n_vars, f"prove_witnesses: need {32 * self.n_vars} witness bytes per proof")
        out = C.create_string_buffer(PROOF_BYTES * batch)
        _check(lib().og_groth16_prove(self.ctx._h, self._h, witnesses, batch, rs, out), self.ctx)
        return out.raw

    def prove_withdraw(self, nullifiers, secrets, recipients, siblings, path_bits, rs, want_public=True):
        """Host buffers in, host buffers out (H2D / D2H inside).  Buffers may be bytes or pinned
        tensors / arrays exposing data_ptr() / .ctypes.  Returns (proofs, public_inputs)."""
        batch = len(path_bits)
        _need(self.depth >= 1, "prove_withdraw: this key was not made for the withdraw statement")
        for name, buf, size in (("nullifiers", nullifiers, 32), ("secrets", secrets, 32), ("recipients", recipients, 32),
                                ("siblings", siblings, 32 * self.depth), ("rs", rs, 64)):
            _need_len(buf, size * batch, f"prove_withdraw: {name}")
        bits = path_bits if hasattr(path_bits, "data_ptr") or hasattr(path_bits, "ctypes") else _bits_array(path_bits)
        proofs = C.create_string_buffer(PROOF_BYTES * batch)
        pub = C.create_string_buffer(32 * self.n_pub * batch) if want_public else None
        _check(lib().og_groth16_prove_withdraw(self.ctx._h, self._h, _ptr(nullifiers), _ptr(secrets), _ptr(recipients),
                                               _ptr(siblings), _ptr(bits), batch, _ptr(rs), proofs, pub), self.ctx)
        return proofs.raw, (pub.raw if want_public else None)


def prove(pk: ProvingKey, nullifiers, secrets, recipients, siblings, path_bits, rs):
    """prove(): batch of withdraw proofs from the secret inputs -> (proofs bytes, public inputs bytes)."""
    return pk.prove_withdraw(nullifiers, secrets, recipients, siblings, path_bits, rs)


def verify(vk_bytes: bytes, public_inputs: bytes, proof: bytes) -> bool:
    """verify(): True / False for well-formed input, raises OwshenB200Error on malformed encodings."""
    _need(len(proof) == PROOF_BYTES, f"verify: a proof is {PROOF_BYTES} bytes")
    _need(len(public_inputs) % 32 == 0, "verify: public inputs are 32-byte field elements")
    _need(len(vk_bytes) >= 12, "verify: verifying key too short")
    n_pub = len(public_inputs) // 32
    rc = lib().og_groth16_verify(vk_bytes, len(vk_bytes), public_inputs, n_pub, proof)
    if rc == OG_OK:
        return True
    if rc == OG_E_VERIFY:
        return False
    raise OwshenB200Error(rc)


class MerkleTree:
    """Fixed-depth sparse MiMC7 Merkle tree; every hash runs in the CUDA library, nodes live behind a
    KvStore-shaped interface (owshen_b200/kvstore.py, mirroring /root/reference/src/db/mod.rs:24-52), so a tree
    can be reopened over the same store.

    insert_batch() appends leaves: ONE library call (og_mimc7_merkle_append) hashes every touched ancestor on the
    GPU -- the only stored values it needs are the <= depth left-boundary nodes -- and one batch_put commits the
    nodes together with the undo record of the batch, the way the reference commits a block together with its
    `Key::Delta` (src/blockchain/mod.rs:283-286).  pop_batch() applies the newest undo record like `pop_block`
    (src/blockchain/mod.rs:291-315); rollback(n) pops / re-inserts until exactly n leaves remain.
    path(i) returns (siblings bytes, path_bits int)."""

    def __init__(self, ctx: Context, depth: int, store=None, prefix: bytes = b"mt/"):
        from .kvstore import RamKvStore
        _need(1 <= depth <= 32, "MerkleTree: depth must be in 1..32")
        self.ctx, self.depth = ctx, depth
        self.store = store if store is not None else RamKvStore()
        self.prefix = prefix
        self.zeros = [bytes(32)]
        for _ in range(depth):
            self.zeros.append(ctx.mimc7_hash2(self.zeros[-1], self.zeros[-1]))
        d = self.store.get_raw(prefix + b"depth")
        if d is not None and int.from_bytes(d, "little") != depth:
            raise ValueError("store holds a tree of a different depth")

    # ---- state kept in the store (so that a reopened tree sees it) ----------------------------------------
    @property
    def n_leaves(self) -> int:
        n = self.store.get_raw(self.prefix + b"n")
        return int.from_bytes(n, "little") if n else 0

    @property
    def n_batches(self) -> int:
        n = self.store.get_raw(self.prefix + b"height")
        return int.from_bytes(n, "little") if n else 0

    def _key(self, lvl: int, idx: int) -> bytes:
        return self.prefix + lvl.to_bytes(1, "little") + idx.to_bytes(8, "little")

    def _delta_key(self, height: int) -> bytes:
        return self.prefix + b"delta" + height.to_bytes(8, "little")

    def _get(self, lvl, idx):
        v = self.store.get_raw(self._key(lvl, idx))
        return v if v is not None else self.zeros[lvl]

    @staticmethod
    def _pack_delta(delta) -> bytes:
        out = bytearray()
        for k, v in sorted(delta.items()):
            out += len(k).to_bytes(2, "little") + k
            out += b"\x00" if v is None else b"\x01" + len(v).to_bytes(4, "little") + v
        return bytes(out)

    @staticmethod
    def _unpack_delta(blob: bytes):
        out, o = [], 0
        while o < len(blob):
            kl = int.from_bytes(blob[o:o + 2], "little"); o += 2
            k = blob[o:o + kl]; o += kl
            tag = blob[o]; o += 1
            if tag == 0:
                out.append((k, None))
            else:
                vl = int.from_bytes(blob[o:o + 4], "little"); o += 4
                out.append((k, blob[o:o + vl])); o += vl
        return out

    def insert_batch(self, leaves):
        from .kvstore import MirrorKvStore
        leaves = [bytes(x) if isinstance(x, (bytes, bytearray)) else fr_bytes(x) for x in leaves]
        n, start = len(leaves), self.n_leaves
        if n == 0:
            return []
        _need(all(len(x) == 32 for x in leaves), "insert_batch: a leaf is 32 bytes")
        if start + n > (1 << self.depth):
            raise OverflowError(f"tree of depth {self.depth} holds {1 << self.depth} leaves; {start} present, {n} more requested")
        # the only stored nodes the new hashes depend on: (l, (start >> l) - 1) where (start >> l) is odd
        boundary = b"".join(self._get(l, (start >> l) - 1) if (start >> l) & 1 else bytes(32) for l in range(self.depth))
        counts = [((start + n - 1) >> l) - (start >> l) + 1 for l in range(1, self.depth + 1)]
        nodes = self.ctx.merkle_append(self.depth, start, b"".join(leaves), boundary, b"".join(self.zeros[:self.depth]))
        _need(len(nodes) == 32 * sum(counts), "merkle_append returned the wrong number of nodes")
        overlay = MirrorKvStore(self.store)
        overlay.batch_put_raw((self._key(0, start + k), leaf) for k, leaf in enumerate(leaves))
        o = 0
        for l, cnt in zip(range(1, self.depth + 1), counts):
            first = start >> l
            overlay.batch_put_raw((self._key(l, first + k), nodes[o + 32 * k:o + 32 * k + 32]) for k in range(cnt))
            o += 32 * cnt
        height = self.n_batches
        overlay.batch_put_raw([(self.prefix + b"n", (start + n).to_bytes(8, "little")),
                               (self.prefix + b"depth", self.depth.to_bytes(1, "little")),
                               (self.prefix + b"height", (height + 1).to_bytes(8, "little"))])
        delta = overlay.rollback()                       # old value of every key this batch overwrites
        overlay.batch_put_raw([(self._delta_key(height + 1), self._pack_delta(delta))])
        self.store.batch_put_raw(overlay.buffer().items())
        return list(range(start, start + n))

    def insert(self, leaf) -> int:
        return self.insert_batch([leaf])[0]

    def pop_batch(self) -> int:
        """Undo the newest insert_batch (the tree's `pop_block`); returns how many leaves it removed."""
        height = self.n_batches
        if height == 0:
            return 0
        blob = self.store.get_raw(self._delta_key(height))
        if blob is None:
            raise KeyError("Delta not found!")            # the reference's wording, src/blockchain/mod.rs:305
        before = self.n_leaves
        self.store.batch_put_raw(self._unpack_delta(blob) + [(self._delta_key(height), None)])
        return before - self.n_leaves

    def rollback(self, n_leaves: int) -> None:
        """Shrink the tree to exactly n_leaves leaves: whole batches are popped; when the target falls inside a
        batch, that batch is popped and its surviving prefix re-inserted (one GPU call)."""
        _need(0 <= n_leaves <= self.n_leaves, "rollback: target must not exceed the current leaf count")
        while self.n_leaves > n_leaves:
            have = self.n_leaves
            survivors = None
            # leaves of the newest batch start where the previous batch ended: read that from its undo record
            blob = self.store.get_raw(self._delta_key(self.n_batches))
            if blob is None:
                raise KeyError("Delta not found!")
            old_n = dict(self._unpack_delta(blob)).get(self.prefix + b"n")
            batch_start = int.from_bytes(old_n, "little") if old_n else 0
            if batch_start < n_leaves:
                survivors = [self.store.get_raw(self._key(0, i)) for i in range(batch_start, n_leaves)]
            self.pop_batch()
            assert self.n_leaves == batch_start < have
            if survivors:
                self.insert_batch(survivors)

    def root(self) -> bytes:
        return self._get(self.depth, 0)

    def path(self, idx: int):
        if not 0 <= idx < self.n_leaves:
            raise IndexError(f"leaf {idx} not in the tree ({self.n_leaves} leaves)")
        sibs, bits, i = [], 0, idx
        for lvl in range(self.depth):
            sibs.append(self._get(lvl, i ^ 1))
            bits |= (i & 1) << lvl
            i >>= 1
        return b"".join(sibs), bits

    def paths(self, indices):
        """Authentication paths of many leaves in the layout prove() takes: (siblings, path_bits) with siblings =
        len(indices) x depth x 32 bytes, proof-major, and one path_bits word per leaf."""
        got = [self.path(i) for i in indices]
        return b"".join(s for s, _ in got), [b for _, b in got]
