"""ctypes binding of libb4d.so (the C ABI declared in include/b4d.h).

The library is built in-tree by ``csrc/Makefile`` (``__graft_entry__.build()``)
and loaded from the package directory.  There is no fallback: if the library is
missing, or no CUDA device is present, the product path raises.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# B4D_LIB: developer override (kernel variants built side by side for A/B timing); the default is the in-tree build
LIB_PATH = os.environ.get("B4D_LIB") or os.path.join(_PKG, "libb4d.so")

ABI_VERSION = 1
T_NAMES = ("prep", "match1", "filter1", "norm1", "match2", "filter2", "norm2", "k0")
T_COUNT = 8

# Prototypes of the C ABI, name -> (restype, argtypes), in header order.  load() applies them, so every call converts
# its arguments through ctypes: int64_t / int / float / double take plain Python numbers, and every pointer or array
# parameter is a c_void_p that takes an address (int), None, a ctypes array or byref(struct) -- an ndarray is refused.
_I64, _INT, _F32, _F64, _P = ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_void_p
_CORE = {
    "b4d_version": (_INT, []),
    "b4d_last_error": (ctypes.c_char_p, []),
    "b4d_default_profile": (None, [_P]),
    "b4d_create": (_INT, [_INT, _P, _P]),
    "b4d_destroy": (None, [_P]),
    "b4d_set_profile": (_INT, [_P, _P]),
    "b4d_denoise_u16": (_INT, [_P, _P, _I64, _P, _F32, _P, _INT, _INT]),
    "b4d_denoise_f32": (_INT, [_P, _P, _I64, _P, _F32, _P, _INT, _INT]),
    "b4d_set_pass_voxels": (_INT, [_P, _I64]),
    "b4d_set_pipeline_min_voxels": (_INT, [_P, _I64]),
    "b4d_targets_u16": (_INT, [_P, _P, _I64, _P, _P, _F32, _F32, _P, _P, _INT, _INT]),
    "b4d_denoise_slab_u16": (_INT, [_P, _P, _P, _I64, _I64, _I64, _I64, _F32, _P, _INT, _INT]),
    "b4d_slab_stage1_u16": (_INT, [_P, _P, _P, _I64, _I64, _F32, _INT]),
    "b4d_slab_basic_planes": (_INT, [_P, _I64, _I64, _P, _INT, _INT]),
    "b4d_slab_stage2": (_INT, [_P, _I64, _I64, _P, _INT]),
    "b4d_slab_basic_ptr": (_P, [_P]),
    "b4d_slab_stage2_begin": (_INT, [_P, _I64, _I64]),
    "b4d_slab_stage2_q16": (_INT, [_P, _I64, _I64, _F32, _F32, _F32, _INT, _P, _INT]),
    "b4d_match_stage1": (_INT, [_P, _P, _P, _F32, _P, _P, _P]),
    "b4d_num_refs": (_I64, [_P]),
    "b4d_quantize_u16": (_INT, [_P, _P, _I64, _F32, _F32, _F32, _P, _INT, _INT]),
    "b4d_quantize_trunc_u16": (_INT, [_P, _P, _I64, _F32, _F32, _F32, _P, _INT, _INT]),
    "b4d_denoise_slab_q16_u16": (_INT, [_P, _P, _P, _I64, _I64, _I64, _I64, _F32, _F32, _F32, _F32, _INT, _P, _INT,
                                         _INT]),
    "b4d_denoise_q16_u16": (_INT, [_P, _P, _P, _F32, _F32, _F32, _F32, _INT, _P, _INT, _INT]),
    "b4d_foreground_mask_u16": (_INT, [_P, _P, _I64, _P, _P, _F32, _INT, _P, _INT, _INT]),
    "b4d_chunk_shuffle_u16": (_INT, [_P, _P, _P, _P, _P, _P, _INT, _INT]),
    "b4d_tile_stats": (_INT, [_P, _P, _I64, _F64, _P, _P, _INT]),
    "b4d_stats_from_hist": (_INT, [_P, _F64, _P]),
    "b4d_last_timings": (_INT, [_P, _P, _P]),
    "b4d_stream": (_P, [_P]),
    "b4d_last_match_stats": (_INT, [_P, _P]),
    "b4d_measure_pipe_peaks": (_INT, [_P, _P]),
    "b4d_set_noise_model": (_INT, [_P, _P, _P]),
    "b4d_coherence_gate": (_INT, [_P, _P, _P, _I64, _P, _F64, _F64, _I64, _F64, _INT, _P, _P, _I64, _P, _INT]),
    "b4d_debug_accumulators": (_INT, [_P, _P, _P, _I64]),
}
# include/b4d_noise.h: the noise-level extension (no counterpart in the CPU oracle library)
_NOISE = {
    "b4d_noise_sigma_u16": (_INT, [_P, _P, _I64, _P, _P, _P, _P, _P, _P, _INT]),
    "b4d_noise_sigma_from_hist": (_INT, [_P, _P, _P, _P]),
    "b4d_noise_level_u16": (_INT, [_P, _P, _I64, _P, _P, _INT, _I64, _P, _P, _P, _P, _P, _P, _P, _INT]),
    "b4d_gat_forward_u16": (_INT, [_P, _P, _P, _I64, _P, _INT, _INT]),
    "b4d_gat_inverse_f32": (_INT, [_P, _P, _P, _I64, _P, _INT, _INT]),
    "b4d_denoise_vst_u16": (_INT, [_P, _P, _I64, _P, _P, _F32, _P, _INT, _INT]),
    "b4d_denoise_vst_q16_u16": (_INT, [_P, _P, _I64, _P, _P, _F32, _F32, _F32, _F32, _INT, _P, _INT, _INT]),
}
SIGNATURES = {**_CORE, **_NOISE}
EXPORTS = tuple(_CORE)
NOISE_EXPORTS = tuple(_NOISE)
# include/b4d_vst_slab.h: the z-slab forms of the VST path, a table of their own
VST_SLAB_SIGNATURES = {
    "b4d_denoise_slab_vst_u16": (_INT, [_P, _P, _P, _I64, _I64, _I64, _I64, _P, _F32, _P, _INT, _P, _INT, _INT]),
    "b4d_denoise_slab_vst_q16_u16": (_INT, [_P, _P, _P, _I64, _I64, _I64, _I64, _P, _F32, _P, _INT, _F32, _F32, _F32,
                                             _INT, _P, _INT, _INT]),
    "b4d_slab_stage1_vst_u16": (_INT, [_P, _P, _P, _I64, _I64, _P, _F32, _P, _INT, _INT]),
}
VST_SLAB_EXPORTS = tuple(VST_SLAB_SIGNATURES)
# include/b4d_step_table.h: per-tile quantizer steps, a table of their own
STEP_TABLE_SIGNATURES = {
    "b4d_quantize_tiled_u16": (_INT, [_P, _P, _P, _I64, _P, _P, _P, _F32, _F32, _INT, _P, _INT, _INT]),
    "b4d_dequantize_tiled_f32": (_INT, [_P, _P, _P, _I64, _P, _P, _P, _F32, _F32, _P, _INT, _INT]),
    "b4d_denoise_slab_qt16_u16": (_INT, [_P, _P, _P, _I64, _I64, _I64, _I64, _F32, _F32, _F32, _P, _P, _P, _INT, _P,
                                          _INT, _INT]),
    "b4d_slab_stage2_qt16": (_INT, [_P, _I64, _I64, _F32, _F32, _P, _P, _P, _INT, _P, _INT]),
}
STEP_TABLE_EXPORTS = tuple(STEP_TABLE_SIGNATURES)
NOISE_HIST_BINS = 262141  # B4D_NOISE_HIST_BINS: |d| <= 4 * 65535
NLF_MAX_BINS = 64  # B4D_NLF_MAX_BINS


class Profile(ctypes.Structure):
    """Mirror of ``struct b4d_profile`` (include/b4d.h)."""

    _fields_ = [
        ("abi", ctypes.c_int32),
        ("block", ctypes.c_int32),
        ("step", ctypes.c_int32),
        ("search_ht", ctypes.c_int32),
        ("search_wie", ctypes.c_int32),
        ("k_ht", ctypes.c_int32),
        ("k_wie", ctypes.c_int32),
        ("stages", ctypes.c_int32),
        ("deterministic", ctypes.c_int32),
        ("reserved0", ctypes.c_int32),
        ("tau_ht", ctypes.c_float),
        ("tau_wie", ctypes.c_float),
        ("lambda_ht", ctypes.c_float),
        ("kaiser_beta", ctypes.c_float),
    ]


class Stats(ctypes.Structure):
    """Mirror of ``struct b4d_stats``."""

    _fields_ = [
        ("n", ctypes.c_int64),
        ("n_nonzero", ctypes.c_int64),
        ("offset", ctypes.c_double),
        ("median", ctypes.c_double),
        ("mad", ctypes.c_double),
        ("sigma", ctypes.c_double),
        ("vmin", ctypes.c_double),
        ("vmax", ctypes.c_double),
    ]


_lib = None


class B4DLibraryError(ImportError):
    pass


def load():
    """Load libb4d.so once; raise loudly when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B4DLibraryError(
            "libb4d.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C aind-exaspim-image-compression_b200/csrc`. There is no CPU fallback." % LIB_PATH
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in {**SIGNATURES, **VST_SLAB_SIGNATURES, **STEP_TABLE_SIGNATURES}.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    if lib.b4d_version() != ABI_VERSION:
        raise B4DLibraryError("libb4d.so ABI %d != binding ABI %d" % (lib.b4d_version(), ABI_VERSION))
    _lib = lib
    return lib


class PgModel(ctypes.Structure):
    """Mirror of ``struct b4d_pg_model`` (include/b4d_noise.h)."""

    _fields_ = [("gain", ctypes.c_double), ("offset", ctypes.c_double), ("read_sigma", ctypes.c_double)]


class SegmentScore(ctypes.Structure):
    """Mirror of ``struct b4d_segment_score`` (include/b4d.h)."""

    _fields_ = [("label", ctypes.c_uint64), ("voxels", ctypes.c_int64), ("autocorr", ctypes.c_double),
                ("highfreq", ctypes.c_double)]


def check(rc):
    """Translate a b4d_status into the exception the reference's callers expect."""
    if rc == 0:
        return
    msg = load().b4d_last_error().decode(errors="replace")
    if rc in (-1, -4, -5):  # INVALID, UNSUPPORTED, TOO_LARGE
        if rc == -4:
            raise NotImplementedError(msg)
        raise ValueError(msg)
    if rc == -3:
        raise MemoryError(msg)
    raise RuntimeError("libb4d: %s (status %d)" % (msg, rc))


def default_profile(**overrides):
    p = Profile()
    load().b4d_default_profile(ctypes.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k) or k in ("abi", "reserved0"):
            raise AttributeError("unknown profile field %r" % k)
        setattr(p, k, v)
    return p


def shape3(shape):
    return (ctypes.c_int64 * 3)(*[int(s) for s in shape])
