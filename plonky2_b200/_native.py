"""ctypes binding of libplonky2_b200.so (the C ABI in include/plonky2_b200.h).

The CUDA library is the ONLY compute backend: if it is missing, or no CUDA device is present, the
calls below raise -- there is no CPU fallback."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libplonky2_b200.so")

GL_OK = 0
GL_ERR_BAD_SHAPE, GL_ERR_OOM, GL_ERR_CUDA, GL_ERR_UNSUPPORTED, GL_ERR_BAD_ARG, GL_ERR_POW_FAILED, GL_ERR_DIV_ZERO = 1, 2, 3, 4, 5, 6, 7
MEM_HOST, MEM_DEVICE = 0, 1
COLS_VALUES, COLS_COEFFS, COLS_COEFFS_CANONICAL = 0, 1, 2

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
vp = C.c_void_p

EXPORTS = [
    "gl_ctx_create", "gl_ctx_destroy", "gl_last_error", "gl_ctx_synchronize", "gl_ctx_launch_count",
    "gl_ctx_set_ntt_group", "gl_ctx_set_profiling", "gl_ctx_phase_ms", "gl_ctx_reset_phases", "gl_ctx_stream", "gl_ntt",
    "gl_ntt_bcast", "gl_bcast", "gl_commit_create", "gl_commit_create_sharded", "gl_commit_begin", "gl_commit_add_columns",
    "gl_commit_finish", "gl_commit_shard", "gl_commit_destroy", "gl_commit_num_polys",
    "gl_commit_leaf_width", "gl_commit_degree_log", "gl_commit_rate_bits", "gl_commit_cap_height",
    "gl_commit_cap", "gl_commit_coeffs", "gl_commit_leaves", "gl_commit_digests", "gl_commit_get_lde_values",
    "gl_commit_open", "gl_commit_eval_ext", "gl_openings", "gl_stark_quotient", "gl_stark_quotient_aux", "gl_stark_lookup_helper_columns", "gl_plonk_quotient", "gl_lookup_polys", "gl_commit_dev_lde", "gl_commit_dev_coeffs", "gl_partial_products_and_zs", "gl_poseidon_permute_host",
    "gl_poseidon_permute_many", "gl_poseidon_hash_many", "gl_poseidon_hash_no_pad_many", "gl_poseidon_two_to_one_many", "gl_merkle_build", "gl_merkle_destroy",
    "gl_merkle_cap", "gl_merkle_digests", "gl_merkle_open", "gl_fri_begin", "gl_fri_begin_values", "gl_fri_values_local", "gl_fri_begin_from_coeffs",
    "gl_fri_destroy", "gl_fri_coeffs", "gl_fri_commit_round", "gl_fri_commit_round_sharded", "gl_fri_mix", "gl_fri_fold", "gl_fri_final_poly",
    "gl_fri_open", "gl_fri_num_rounds", "gl_fri_pow",
]


class FriBatch(C.Structure):
    _fields_ = [("point", C.c_uint64 * 2), ("num_polys", C.c_size_t), ("oracle_index", u32p),
                ("poly_index", u32p)]


class ShapeError(ValueError):
    """Mirrors the reference's shape panics (fft.rs:171-177, merkle_tree.rs:195-200, oracle.rs:128)."""


class NativeError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "libplonky2_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
            "plonky2_b200 has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.gl_ctx_create.argtypes = [C.c_int, vp, C.POINTER(vp)]
    L.gl_ctx_destroy.argtypes = [vp]
    L.gl_ctx_destroy.restype = None
    L.gl_last_error.argtypes = [vp]
    L.gl_last_error.restype = C.c_char_p
    L.gl_ctx_synchronize.argtypes = [vp]
    L.gl_ctx_launch_count.argtypes = [vp]
    L.gl_ctx_launch_count.restype = C.c_uint64
    L.gl_ctx_set_ntt_group.argtypes = [vp, C.c_uint32]
    L.gl_ntt.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_size_t, C.c_int, C.c_uint32, C.c_uint64, C.c_int]
    L.gl_ctx_stream.argtypes = [vp]
    L.gl_ctx_stream.restype = vp
    L.gl_ntt_bcast.argtypes = [vp, vp, C.c_size_t, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(vp), C.c_uint32, C.c_size_t]
    L.gl_bcast.argtypes = [vp, vp, C.c_size_t, C.POINTER(vp), C.c_uint32, C.c_uint32]
    L.gl_commit_begin.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_uint32,
                                  vp, C.POINTER(vp)]
    L.gl_commit_add_columns.argtypes = [vp, C.c_uint32, C.c_uint32, vp, C.c_size_t, C.c_int, C.c_int]
    L.gl_commit_finish.argtypes = [vp, vp, C.c_int]
    L.gl_commit_create.argtypes = [vp, vp, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp,
                                   C.c_int, C.c_int, C.POINTER(vp)]
    L.gl_commit_create_sharded.argtypes = [vp, vp, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp,
                                           C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.POINTER(vp)]
    L.gl_commit_shard.argtypes = [vp, u32p, u32p]
    L.gl_ctx_set_profiling.argtypes = [vp, C.c_int]
    L.gl_ctx_phase_ms.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.gl_ctx_reset_phases.argtypes = [vp]
    L.gl_commit_destroy.argtypes = [vp]
    L.gl_commit_destroy.restype = None
    for n in ("gl_commit_num_polys", "gl_commit_leaf_width", "gl_commit_degree_log", "gl_commit_rate_bits",
              "gl_commit_cap_height"):
        getattr(L, n).argtypes = [vp]
        getattr(L, n).restype = C.c_uint32
    L.gl_commit_cap.argtypes = [vp, vp, C.c_int]
    L.gl_commit_coeffs.argtypes = [vp, vp, C.c_int]
    L.gl_commit_leaves.argtypes = [vp, C.c_size_t, C.c_size_t, vp, C.c_int]
    L.gl_commit_digests.argtypes = [vp, vp, C.c_int]
    L.gl_commit_get_lde_values.argtypes = [vp, C.c_size_t, C.c_size_t, vp]
    L.gl_commit_open.argtypes = [vp, vp, C.c_size_t, vp, vp]
    L.gl_commit_eval_ext.argtypes = [vp, vp, vp]
    L.gl_openings.argtypes = [vp, C.POINTER(vp), u32p, C.c_size_t, vp, C.c_size_t, vp, C.c_int]
    L.gl_stark_quotient.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, C.c_uint32, vp]
    L.gl_stark_quotient_aux.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, C.c_uint32, vp]
    L.gl_stark_lookup_helper_columns.argtypes = [vp, vp, C.c_size_t, C.c_uint32, C.c_uint32, vp, vp, C.c_uint32, C.c_uint32,
                                                 vp, C.c_int]
    L.gl_plonk_quotient.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, C.c_uint32,
                                    C.c_uint32, vp]
    L.gl_lookup_polys.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, vp, u32p, C.c_uint32, vp, C.c_int]
    L.gl_commit_dev_lde.argtypes = [vp, C.POINTER(C.c_size_t)]
    L.gl_commit_dev_lde.restype = vp
    L.gl_commit_dev_coeffs.argtypes = [vp]
    L.gl_commit_dev_coeffs.restype = vp
    L.gl_partial_products_and_zs.argtypes = [vp, vp, vp, vp, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64,
                                             C.c_uint32, vp, C.c_int]
    L.gl_poseidon_permute_host.argtypes = [vp]
    L.gl_poseidon_permute_host.restype = None
    L.gl_poseidon_permute_many.argtypes = [vp, vp, C.c_size_t, C.c_int]
    L.gl_poseidon_hash_many.argtypes = [vp, vp, C.c_size_t, C.c_uint32, vp, C.c_int]
    L.gl_poseidon_hash_no_pad_many.argtypes = [vp, vp, C.c_size_t, C.c_uint32, vp, C.c_int]
    L.gl_poseidon_two_to_one_many.argtypes = [vp, vp, C.c_size_t, vp, C.c_int]
    L.gl_merkle_build.argtypes = [vp, vp, C.c_size_t, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(vp)]
    L.gl_merkle_destroy.argtypes = [vp]
    L.gl_merkle_destroy.restype = None
    L.gl_merkle_cap.argtypes = [vp, vp, C.c_int]
    L.gl_merkle_digests.argtypes = [vp, vp, C.c_int]
    L.gl_merkle_open.argtypes = [vp, vp, C.c_size_t, vp, vp]
    L.gl_fri_begin.argtypes = [vp, C.POINTER(vp), C.c_size_t, C.POINTER(FriBatch), C.c_size_t, vp, C.c_uint32,
                               C.c_uint32, C.POINTER(vp)]
    L.gl_fri_begin_values.argtypes = [vp, C.POINTER(vp), C.c_size_t, C.POINTER(FriBatch), C.c_size_t, vp, vp, C.c_uint32,
                                      C.POINTER(vp)]
    L.gl_fri_values_local.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.gl_fri_begin_from_coeffs.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(vp)]
    L.gl_fri_destroy.argtypes = [vp]
    L.gl_fri_destroy.restype = None
    L.gl_fri_coeffs.argtypes = [vp, vp]
    L.gl_fri_commit_round.argtypes = [vp, C.c_uint32, vp]
    L.gl_fri_commit_round_sharded.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32, vp]
    L.gl_fri_mix.argtypes = [vp, vp, vp]
    L.gl_fri_fold.argtypes = [vp, vp]
    L.gl_fri_final_poly.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.gl_fri_open.argtypes = [vp, C.c_uint32, vp, C.c_size_t, vp, vp]
    L.gl_fri_num_rounds.argtypes = [vp]
    L.gl_fri_num_rounds.restype = C.c_uint32
    L.gl_fri_pow.argtypes = [vp, vp, C.c_uint32, C.c_uint32, vp]
    _lib = L
    return L


def check(rc, ctx=None):
    if rc == GL_OK:
        return
    msg = lib().gl_last_error(ctx)
    msg = msg.decode() if msg else "error %d" % rc
    if rc == GL_ERR_BAD_SHAPE:
        raise ShapeError(msg)
    if rc == GL_ERR_OOM:
        raise MemoryError(msg)
    if rc == GL_ERR_DIV_ZERO:
        raise ZeroDivisionError(msg)
    raise NativeError("plonky2_b200 native error %d: %s" % (rc, msg))


def np_ptr(a):
    assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"], "need contiguous uint64"
    return a.ctypes.data_as(vp)


class Context:
    """One gl_ctx per (device, stream) (SURVEY.md section 8b, threading row)."""

    def __init__(self, device=0, stream=None):
        h = vp()
        check(lib().gl_ctx_create(int(device), vp(stream) if stream else None, C.byref(h)))
        self.h = h
        self.device = device

    def synchronize(self):
        check(lib().gl_ctx_synchronize(self.h), self.h)

    @property
    def stream(self):
        """The cudaStream_t (as an int) every call on this context is ordered on."""
        return int(lib().gl_ctx_stream(self.h) or 0)

    @property
    def launch_count(self):
        return int(lib().gl_ctx_launch_count(self.h))

    def set_ntt_group(self, columns):
        check(lib().gl_ctx_set_ntt_group(self.h, int(columns)), self.h)

    PHASES = {"intt": 0, "lde": 1, "leaf_hash": 2, "merkle_levels": 3}

    def set_profiling(self, on):
        check(lib().gl_ctx_set_profiling(self.h, int(bool(on))), self.h)

    def reset_phases(self):
        check(lib().gl_ctx_reset_phases(self.h), self.h)

    def phase_ms(self):
        """{phase: (accumulated ms, scopes)} from CUDA events on this context's stream."""
        out = {}
        for name, pid in self.PHASES.items():
            ms, cnt = C.c_double(), C.c_uint64()
            check(lib().gl_ctx_phase_ms(self.h, pid, C.byref(ms), C.byref(cnt)), self.h)
            out[name] = (ms.value, cnt.value)
        return out

    def close(self):
        if getattr(self, "h", None):
            lib().gl_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device=0):
    """Process-wide default context per device (created on first use; fails loudly without a GPU)."""
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
