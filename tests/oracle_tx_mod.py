"""ctypes access to the AM / FM transmit modulators of the oracle (oracle/slo_tx_mod.h; TEST INFRASTRUCTURE ONLY).

The functions take an oracle_lib.Oracle and call its library's `<kind>_tx_mod_f32`, `<kind>_tx_fm_nco` and the three stages the
modulators add. Every call is for ONE channel and takes / returns numpy arrays."""
import ctypes as C

import numpy as np

from oracle_lib import MAX_FFT, f32p, i16p, i32p, u32

u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")


class TxModParams(C.Structure):
    _fields_ = [("fft_len", u32), ("hop", u32), ("alc_block", u32), ("fs", u32),
                ("alc_decay", C.c_float), ("alc_floor", C.c_float), ("alc_gmax", C.c_float),
                ("mask", C.POINTER(C.c_float)), ("modulator", u32),
                ("am_carrier", C.c_float), ("am_depth", C.c_float), ("fm_deviation_hz", C.c_float), ("fm_level", C.c_float)]


class TxModState(C.Structure):
    _fields_ = [("ovl", C.c_int16 * MAX_FFT), ("env", C.c_float), ("phase", C.c_uint32)]


def offset_f32(o, x, k):
    x = np.ascontiguousarray(x, np.float32); d = np.zeros(x.size, np.float32)
    o._f("offset_f32", [f32p, C.c_float, f32p, u32])(x, k, d, x.size); return d


def float_to_q31(o, x):
    x = np.ascontiguousarray(x, np.float32); d = np.zeros(x.size, np.int32)
    o._f("float_to_q31", [f32p, i32p, u32])(x, d, x.size); return d


def q31_to_float(o, x):
    x = np.ascontiguousarray(x, np.int32); d = np.zeros(x.size, np.float32)
    o._f("q31_to_float", [i32p, f32p, u32])(x, d, x.size); return d


def tx_fm_nco(o, phase, level):
    """phase uint32[n] -> int16[n][2] I/Q."""
    ph = np.ascontiguousarray(phase, np.uint32); out = np.zeros(2 * ph.size, np.int16)
    o._f("tx_fm_nco", [u32p, u32, C.c_float, i16p])(ph, ph.size, level, out); return out.reshape(-1, 2)


def tx_mod_f32(o, prm, in_lr, state=None):
    """prm: dsp_if.tx_mod_params_to_dict(...). in_lr int16[frames][2] (L = R mic). Returns out int16[frames][2] I/Q,
    iq f32[frames][2] (pre-ALC baseband), gain f32[frames/alc_block], phase uint32[frames] (FM; zeros for AM), state."""
    p = TxModParams()
    for k in ("fft_len", "hop", "alc_block", "fs", "modulator"):
        setattr(p, k, int(prm[k]))
    for k in ("alc_decay", "alc_floor", "alc_gmax", "am_carrier", "am_depth", "fm_deviation_hz", "fm_level"):
        setattr(p, k, float(prm[k]))
    mask = np.ascontiguousarray(np.asarray(prm["mask"], np.complex64).view(np.float32))
    p.mask = mask.ctypes.data_as(C.POINTER(C.c_float))
    st = state if state is not None else TxModState()
    x = np.ascontiguousarray(in_lr, np.int16).reshape(-1)
    frames = x.size // 2
    out = np.zeros(2 * frames, np.int16); iq = np.zeros(2 * frames, np.float32)
    gain = np.zeros(frames // int(prm["alc_block"]), np.float32); phase = np.zeros(frames, np.uint32)
    fn = o._f("tx_mod_f32", [C.POINTER(TxModParams), C.POINTER(TxModState), i16p, i16p, f32p, f32p, u32p, u32])
    fn(C.byref(p), C.byref(st), x, out, iq, gain, phase, frames)
    return out.reshape(frames, 2), iq.reshape(frames, 2), gain, phase, st


def fm_target(prm):
    """T = 2 fm_deviation_hz / fs (half-turns per sample), evaluated in float32 as the chain does."""
    return np.float32(np.float32(2.0) * np.float32(prm["fm_deviation_hz"])) / np.float32(prm["fs"])


def tone_snr_db(x, fs, f0):
    """SNR of a tone at f0 in x (float): power in +-60 Hz around f0 over the rest of 100 Hz .. 3 kHz (Hann window)."""
    x = np.asarray(x, np.float64); x = x - x.mean()
    X = np.abs(np.fft.rfft(x * np.hanning(x.size))) ** 2
    f = np.fft.rfftfreq(x.size, 1.0 / fs)
    sig = (abs(f - f0) <= 60.0); band = (f >= 100.0) & (f <= 3000.0) & ~sig
    return float(10.0 * np.log10(X[sig].sum() / X[band].sum()))
