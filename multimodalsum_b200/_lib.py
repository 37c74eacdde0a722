"""ctypes binding of libmmsum_b200.so (the C-ABI declared in include/mmsum_b200.h).

The library is the product: if it is missing this module raises — there is no torch/CPU fallback.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MMSUM_LIB_PATH: A/B tooling only (tools/ab_lib.sh builds a second library from another revision of csrc/)
LIB_PATH = os.environ.get("MMSUM_LIB_PATH") or os.path.join(_HERE, "libmmsum_b200.so")

_lib = None


class MmsumError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p), ("D", C.c_void_p),
        ("lda", C.c_int64), ("ldb", C.c_int64), ("ldd", C.c_int64),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("a_mn_major", C.c_int32), ("b_mn_major", C.c_int32),
        ("out_f32", C.c_int32), ("accumulate", C.c_int32), ("splits", C.c_int32),
        ("block_n", C.c_int32), ("raster_m_fast", C.c_int32),
        ("alpha", C.c_float), ("bias", C.c_void_p),
        ("act", C.c_int32), ("aux_mode", C.c_int32), ("aux", C.c_void_p), ("ld_aux", C.c_int64),
        ("A2", C.c_void_p), ("lda2", C.c_int64), ("k_split", C.c_int32),
    ]


class AttnMod(C.Structure):
    _fields_ = [("kv_row_base", C.c_int64), ("o_off", C.c_int64), ("E", C.c_int32), ("Sk", C.c_int32),
                ("loo", C.c_int32), ("ent_base", C.c_int32), ("ent_stride", C.c_int32), ("no_dkv", C.c_int32)]


class AttnArgs(C.Structure):
    _fields_ = [
        ("Q", C.c_void_p), ("ldq", C.c_int64), ("q_col", C.c_int32),
        ("KV", C.c_void_p), ("ldkv", C.c_int64), ("k_col", C.c_int32), ("v_col", C.c_int32),
        ("O", C.c_void_p), ("ldo", C.c_int64),
        ("LSE", C.c_void_p), ("DELTA", C.c_void_p),
        ("key_valid", C.c_void_p), ("ent_valid", C.c_void_p), ("inv_n", C.c_void_p),
        ("dQ", C.c_void_p), ("lddq", C.c_int64), ("dq_col", C.c_int32),
        ("dKV", C.c_void_p), ("lddkv", C.c_int64), ("dk_col", C.c_int32), ("dv_col", C.c_int32),
        ("n_qseq", C.c_int32), ("H", C.c_int32), ("R", C.c_int32), ("causal", C.c_int32),
        ("n_mod", C.c_int32), ("E_total", C.c_int32), ("scale", C.c_float), ("q_rows", C.c_int32),
        ("mods", AttnMod * 3),
    ]


class PrepArgs(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "R", "S", "F", "n_img", "img_keys", "n_mod", "pad_id", "bos_id", "eos_id", "S_enc")] + \
               [(n, C.c_void_p) for n in ("enc_ids", "dec_ids", "labels", "enc_valid", "dec_valid", "mem_valid",
                                          "ent_valid", "pres", "rating_diff", "inv_n")]


class TableArgs(C.Structure):
    _fields_ = [("dataset", C.c_int32), ("B", C.c_int32), ("E", C.c_void_p), ("field", C.c_void_p)] + \
               [("v%d" % i, C.c_void_p) for i in range(6)] + \
               [("W0", C.c_void_p), ("W1", C.c_void_p), ("X", C.c_void_p), ("valid", C.c_void_p)]


def lib():
    """Load (once) and return the shared library; raise loudly when it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MmsumError(
                "libmmsum_b200.so is not built (%s). Run `python -m multimodalsum_b200.build` "
                "(needs nvcc); there is no fallback path." % LIB_PATH)
        if not os.environ.get("MMSUM_LIB_PATH") and os.environ.get("MMSUM_ALLOW_STALE_LIB") != "1":
            from . import build as _build
            if _build.is_current() is False:       # None = no build record next to the library: nothing to compare
                raise MmsumError(
                    "libmmsum_b200.so was built from different sources than the ones in %s (csrc/, include/ or the compiler "
                    "flags changed since). Re-run `python -m multimodalsum_b200.build`." % _HERE)
        _lib = C.CDLL(LIB_PATH)
        for name in EXPORTS:
            fn = getattr(_lib, name)  # AttributeError if the symbol is missing
            fn.restype = C.c_int
    return _lib


# every symbol include/mmsum_b200.h declares (tests/test_host_logic.py cross-checks this list against the header)
EXPORTS = [
    "mmsum_gemm_bf16", "mmsum_attn_fwd", "mmsum_attn_bwd", "mmsum_debug_poison",
    "mmsum_cast_f32_bf16",
    "mmsum_embed_ln_fwd", "mmsum_embed_ln_bwd", "mmsum_add_ln_fwd", "mmsum_add_ln_bwd", "mmsum_colsum",
    "mmsum_gate_fwd", "mmsum_gate_bwd_u", "mmsum_gate_bwd_o", "mmsum_ce_fwd_bwd", "mmsum_prep_step",
    "mmsum_table_fwd", "mmsum_table_bits_bwd", "mmsum_grad_sumsq", "mmsum_adamw_step",
    "mmsum_embed_ln_decode", "mmsum_attn_decode_cross", "mmsum_attn_decode_self", "mmsum_beam_topk", "mmsum_beam_update",
    "mmsum_sample_token",
    "mmsum_gemm_bf16_ordered", "mmsum_gemm_ordered_workspace", "mmsum_add_ln_bwd_ordered", "mmsum_colsum_ordered",
    "mmsum_embed_ln_bwd_ordered", "mmsum_embed_ln_bwd_ordered_subset",
]


def build_info():
    """The record build() wrote next to the library (compiler, flags, source digest) + whether it matches this tree."""
    from . import build as _build
    info = dict(_build.read_build_info() or {})
    info["matches_sources"] = _build.is_current()
    info["path"] = LIB_PATH
    return info


def check(rc, what):
    if rc != 0:
        kind = "invalid argument / driver" if rc < 0 else "cudaError_t"
        raise MmsumError("%s failed: rc=%d (%s)" % (what, rc, kind))
