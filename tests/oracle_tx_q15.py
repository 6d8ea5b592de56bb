"""ctypes access to the integer SSB modulator of the oracle (oracle/slo_tx_q15.h; TEST INFRASTRUCTURE ONLY).

`tx_ssb_q15` takes an oracle_lib.Oracle (the port: the modulator is composed from stages the port restates) and works on ONE channel.
It takes the parameter dict of RX-SSB-q15 (dsp_if.q15_params_to_dict) and its state structure: both FIR histories hold mic samples."""
import ctypes as C

import numpy as np

from oracle_lib import RxQ15Params, RxQ15State, i16p, u32

u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")


def _params(prm):
    p = RxQ15Params()
    p.ntaps, p.agc_block, p.agc_window, p.lsb = prm["ntaps"], prm["agc_block"], prm["agc_window"], int(prm["lsb"])
    for k in range(64):
        p.taps_i[k] = int(prm["taps_i"][k]); p.taps_q[k] = int(prm["taps_q"][k])
    for k in range(32):
        p.rel[k] = int(prm["rel"][k])
    p.agc_target, p.agc_floor, p.agc_gmax_q15 = int(prm["agc_target"]), int(prm["agc_floor"]), int(prm["agc_gmax_q15"])
    return p


def tx_ssb_q15(o, prm, in_lr, state=None):
    """in_lr int16[frames][2] (L = R mic; L is used). Returns out int16[frames][2] I/Q, iq int16[frames][2] (pre-ALC, after the rail
    order), gain uint32[frames/agc_block] (Q15), state."""
    p = _params(prm)
    st = state if state is not None else RxQ15State()
    x = np.ascontiguousarray(in_lr, np.int16).reshape(-1)
    frames = x.size // 2
    out = np.zeros(2 * frames, np.int16); iq = np.zeros(2 * frames, np.int16)
    gain = np.zeros(frames // int(prm["agc_block"]), np.uint32)
    fn = o._f("tx_ssb_q15", [C.POINTER(RxQ15Params), C.POINTER(RxQ15State), i16p, i16p, i16p, u32p, u32])
    fn(C.byref(p), C.byref(st), x, out, iq, gain, frames)
    return out.reshape(frames, 2), iq.reshape(frames, 2), gain, st


def tx_batch(o, prms, x):
    """x int16 [C][frames][2], prms: one parameter dict per channel (or one for all). Every channel from a zero state.
    Returns out, iq (int16 [C][frames][2]) and gain (uint32 [C][frames/48])."""
    if isinstance(prms, dict):
        prms = [prms] * x.shape[0]
    res = [tx_ssb_q15(o, prms[c], x[c]) for c in range(x.shape[0])]
    return np.stack([r[0] for r in res]), np.stack([r[1] for r in res]), np.stack([r[2] for r in res])


def sideband_db(iq, fs, f0, skip=1000):
    """Power of z = I + jQ at +f0 over its power at -f0 in dB (Hann window, +-60 Hz around each), after `skip` samples of start-up."""
    z = iq[skip:, 0].astype(np.float64) + 1j * iq[skip:, 1].astype(np.float64)
    Z = np.abs(np.fft.fft(z * np.hanning(z.size))) ** 2
    f = np.fft.fftfreq(z.size, 1.0 / fs)
    pos = Z[np.abs(f - f0) <= 60.0].sum(); neg = Z[np.abs(f + f0) <= 60.0].sum()
    return float(10.0 * np.log10(pos / neg))
