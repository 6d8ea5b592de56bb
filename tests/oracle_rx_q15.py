"""ctypes access to the all-mode integer receiver of the oracle (oracle/slo_rx_q15.h; TEST INFRASTRUCTURE ONLY).

`rx_q15` takes an oracle_lib.Oracle (the port: the receiver is composed from stages the port restates) and works on ONE channel. It
takes the parameter dict of DspIf.oracle_params on an RX-Q15 context (dsp_if.q15_mode_params_to_dict: the RX-SSB-q15 dict plus `kind`,
`am_taps`, `fm_taps`, `fm_floor`); the state keeps the last 64 raw frames per rail and the peak window."""
import ctypes as C

import numpy as np

from oracle_lib import RxQ15Params, i16p, u32

u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
KIND_SSB, KIND_AM, KIND_FM = 0, 1, 2


class RxQ15mParams(C.Structure):
    _fields_ = [("q", RxQ15Params), ("kind", u32), ("am_taps", C.c_int16 * 64), ("fm_taps", C.c_int16 * 64), ("fm_floor", C.c_int32)]


class RxQ15mState(C.Structure):
    _fields_ = [("raw_i", C.c_int16 * 64), ("raw_q", C.c_int16 * 64), ("peaks", C.c_int16 * 32)]


def _params(prm):
    p = RxQ15mParams()
    q = p.q
    q.ntaps, q.agc_block, q.agc_window, q.lsb = prm["ntaps"], prm["agc_block"], prm["agc_window"], int(prm["lsb"])
    for k in range(64):
        q.taps_i[k] = int(prm["taps_i"][k]); q.taps_q[k] = int(prm["taps_q"][k])
        p.am_taps[k] = int(prm["am_taps"][k]); p.fm_taps[k] = int(prm["fm_taps"][k])
    for k in range(32):
        q.rel[k] = int(prm["rel"][k])
    q.agc_target, q.agc_floor, q.agc_gmax_q15 = int(prm["agc_target"]), int(prm["agc_floor"]), int(prm["agc_gmax_q15"])
    p.kind, p.fm_floor = int(prm["kind"]), int(prm["fm_floor"])
    return p


def rx_q15(o, prm, in_iq, state=None):
    """in_iq int16[frames][2]. Returns out int16[frames][2] (L = R), audio int16[frames] (pre-AGC detector output),
    gain uint32[frames/agc_block] (Q15), state."""
    p = _params(prm)
    st = state if state is not None else RxQ15mState()
    x = np.ascontiguousarray(in_iq, np.int16).reshape(-1)
    frames = x.size // 2
    out = np.zeros(2 * frames, np.int16); aud = np.zeros(frames, np.int16)
    gain = np.zeros(frames // int(prm["agc_block"]), np.uint32)
    fn = o._f("rx_q15", [C.POINTER(RxQ15mParams), C.POINTER(RxQ15mState), i16p, i16p, i16p, u32p, u32])
    fn(C.byref(p), C.byref(st), x, out, aud, gain, frames)
    return out.reshape(frames, 2), aud, gain, st


def rx_batch(o, prms, x, states=None):
    """x int16 [C][frames][2], prms: one parameter dict per channel (or one for all). Every channel from a zero state unless `states`
    (a list, updated in place) is given. Returns out (int16 [C][frames][2]), audio (int16 [C][frames]) and gain (uint32 [C][frames/48])."""
    if isinstance(prms, dict):
        prms = [prms] * x.shape[0]
    if states is None:
        states = [RxQ15mState() for _ in range(x.shape[0])]
    res = [rx_q15(o, prms[c], x[c], states[c]) for c in range(x.shape[0])]
    return np.stack([r[0] for r in res]), np.stack([r[1] for r in res]), np.stack([r[2] for r in res])


def state_bytes(st):
    return bytes(memoryview(st))
