"""ctypes binding of include/selenite_b200.h. Loading fails loudly: there is no Python or CPU fallback."""
import ctypes as C
import os
import re

from . import build as _build

MAX_STAGES = 4
_lib = None


class Config(C.Structure):
    _fields_ = [("channels", C.c_uint32), ("fs", C.c_uint32), ("device", C.c_int32), ("chain", C.c_uint32)]


class RxF32Params(C.Structure):
    _fields_ = [("fft_len", C.c_uint32), ("hop", C.c_uint32), ("agc_block", C.c_uint32), ("n_stages", C.c_uint32),
                ("biquad", C.c_float * (5 * MAX_STAGES)),
                ("agc_target", C.c_float), ("agc_decay", C.c_float), ("agc_floor", C.c_float), ("agc_gmax", C.c_float)]


class TxF32Params(C.Structure):
    _fields_ = [("fft_len", C.c_uint32), ("hop", C.c_uint32), ("alc_block", C.c_uint32),
                ("alc_target", C.c_float), ("alc_decay", C.c_float), ("alc_floor", C.c_float), ("alc_gmax", C.c_float)]


class TxModParams(C.Structure):
    _fields_ = [("am_carrier", C.c_float), ("am_depth", C.c_float), ("fm_deviation_hz", C.c_float), ("fm_level", C.c_float)]


class RxQ15Params(C.Structure):
    _fields_ = [("ntaps", C.c_uint32), ("agc_block", C.c_uint32), ("agc_window", C.c_uint32),
                ("taps_i", C.c_int16 * 64), ("taps_q", C.c_int16 * 64), ("rel", C.c_int16 * 32),
                ("agc_target", C.c_int16), ("agc_floor", C.c_int16), ("agc_gmax_q15", C.c_uint32),
                ("bq_stages", C.c_uint32), ("bq_postshift", C.c_int32), ("bq_coeffs", C.c_int16 * 24)]


class RxQ15ModeParams(C.Structure):
    _fields_ = [("am_taps", C.c_int16 * 64), ("fm_taps", C.c_int16 * 64), ("fm_floor", C.c_int32)]


class TxQ15ModeParams(C.Structure):
    _fields_ = [("am_taps", C.c_int16 * 64), ("fm_taps", C.c_int16 * 64), ("am_carrier", C.c_int16), ("am_depth", C.c_int16),
                ("fm_target", C.c_int16), ("fm_inc", C.c_int32), ("fm_level", C.c_float)]


class FeederIo(C.Structure):
    _fields_ = [("adc", C.c_void_p), ("usb_in", C.c_void_p), ("usb_out", C.c_void_p), ("dac", C.c_void_p)]


class ChanParams(C.Structure):
    _fields_ = [("bins", C.c_uint32), ("taps_per_branch", C.c_uint32), ("agc_block", C.c_uint32), ("envelope", C.c_uint32),
                ("agc_target", C.c_float), ("agc_decay", C.c_float), ("agc_floor", C.c_float), ("agc_gmax", C.c_float),
                ("proto", C.c_float * 512)]


class ChanQ15Params(C.Structure):
    _fields_ = [("bins", C.c_uint32), ("taps_per_branch", C.c_uint32), ("agc_block", C.c_uint32), ("envelope", C.c_uint32),
                ("proto", C.c_int16 * 512), ("agc_window", C.c_uint32), ("rel", C.c_int16 * 32),
                ("agc_target", C.c_int16), ("agc_floor", C.c_int16), ("agc_gmax_q15", C.c_uint32)]


# every symbol include/selenite_b200.h declares: name -> (restype, argtypes), derived from the header text so the
# binding cannot drift from the ABI
_P = C.c_void_p
_SCALARS = {"int": C.c_int, "int8_t": C.c_int8, "uint8_t": C.c_uint8, "int16_t": C.c_int16, "uint16_t": C.c_uint16,
            "int32_t": C.c_int32, "uint32_t": C.c_uint32, "uint64_t": C.c_uint64, "size_t": C.c_size_t, "float": C.c_float,
            "double": C.c_double}
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "selenite_b200.h")


def _ctype(decl, is_return=False):
    decl = decl.strip()
    if decl in ("void", ""):
        return None
    if "*" in decl or "[" in decl:
        return C.c_char_p if (is_return and "char" in decl) else _P
    base = decl.replace("const", "").split()[0]
    return _SCALARS[base]


def _parse_header():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    out = {}
    for m in re.finditer(r"([A-Za-z_][A-Za-z0-9_ ]*?[ \*]+)([A-Za-z_][A-Za-z0-9_]*)\s*\(([^;{}()]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        if "typedef" in ret:
            continue
        argt = [] if args.strip() in ("void", "") else [_ctype(a) for a in args.split(",")]
        out[name] = (_ctype(ret, True), argt)
    return out


SYMBOLS = _parse_header()


def lib_path():
    # SELENITE_B200_LIB: A/B runs of two builds of the same ABI on one box (profiling aid)
    return os.environ.get("SELENITE_B200_LIB", _build.LIB_PATH)


def load():
    """Load lib/libselenite_b200.so (building it first when nvcc is present and the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if path == _build.LIB_PATH and _build.is_stale():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this box: use the prebuilt library if there is one
            if not os.path.exists(path):
                raise RuntimeError("selenite_lite_b200: CUDA library missing and cannot be built (%s); "
                                   "there is no CPU fallback" % exc)
            # a prebuilt library older than the sources: say so — the argument types below come from the CURRENT header, and a
            # silent ABI drift would be memory corruption rather than an error (set SELENITE_B200_ALLOW_STALE=1 to keep going quietly)
            if not os.environ.get("SELENITE_B200_ALLOW_STALE"):
                import warnings
                warnings.warn("selenite_lite_b200: %s is older than its sources and could not be rebuilt (%s); loading the stale "
                              "library" % (path, exc), RuntimeWarning)
    if not os.path.exists(path):
        raise RuntimeError("selenite_lite_b200: %s not found; run __graft_entry__.build(). There is no CPU fallback." % path)
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
