"""ctypes access to the all-mode integer transmitter of the oracle (oracle/slo_tx_q15_mod.h; TEST INFRASTRUCTURE ONLY).

`tx_q15` takes an oracle_lib.Oracle (the port: the transmitter is composed from stages the port restates) and works on ONE channel. It
takes the parameter dict of DspIf.oracle_params on a TX-Q15 context (dsp_if.tx_q15_mode_params_to_dict: the RX-SSB-q15 dict plus `kind`
and the fields of slb_tx_q15_mode_params); the state keeps the last 64 mic samples, the peak window and the FM phase."""
import ctypes as C

import numpy as np

from oracle_lib import RxQ15Params, i16p, u32

u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
KIND_SSB, KIND_AM, KIND_FM = 0, 1, 2


class TxQ15mParams(C.Structure):
    _fields_ = [("q", RxQ15Params), ("kind", u32), ("am_taps", C.c_int16 * 64), ("fm_taps", C.c_int16 * 64),
                ("am_carrier", C.c_int16), ("am_depth", C.c_int16), ("fm_target", C.c_int16), ("fm_inc", C.c_int32), ("fm_level", C.c_float)]


class TxQ15mState(C.Structure):
    _fields_ = [("raw", C.c_int16 * 64), ("peaks", C.c_int16 * 32), ("phase", C.c_uint32)]


def _params(prm):
    p = TxQ15mParams()
    q = p.q
    q.ntaps, q.agc_block, q.agc_window, q.lsb = prm["ntaps"], prm["agc_block"], prm["agc_window"], int(prm["lsb"])
    for k in range(64):
        q.taps_i[k] = int(prm["taps_i"][k]); q.taps_q[k] = int(prm["taps_q"][k])
        p.am_taps[k] = int(prm["am_taps"][k]); p.fm_taps[k] = int(prm["fm_taps"][k])
    for k in range(32):
        q.rel[k] = int(prm["rel"][k])
    q.agc_target, q.agc_floor, q.agc_gmax_q15 = int(prm["agc_target"]), int(prm["agc_floor"]), int(prm["agc_gmax_q15"])
    p.kind = int(prm["kind"])
    p.am_carrier, p.am_depth, p.fm_target = int(prm["am_carrier"]), int(prm["am_depth"]), int(prm["fm_target"])
    p.fm_inc, p.fm_level = int(prm["fm_inc"]), float(prm["fm_level"])
    return p


def tx_q15(o, prm, in_lr, state=None):
    """in_lr int16[frames][2] (L = R mic; L is used). Returns out int16[frames][2] I/Q, iq int16[frames][2] (the pre-ALC pair),
    gain uint32[frames/agc_block] (Q15), phase uint32[frames], state."""
    p = _params(prm)
    st = state if state is not None else TxQ15mState()
    x = np.ascontiguousarray(in_lr, np.int16).reshape(-1)
    frames = x.size // 2
    out = np.zeros(2 * frames, np.int16); iq = np.zeros(2 * frames, np.int16)
    gain = np.zeros(frames // int(prm["agc_block"]), np.uint32); phase = np.zeros(frames, np.uint32)
    fn = o._f("tx_q15", [C.POINTER(TxQ15mParams), C.POINTER(TxQ15mState), i16p, i16p, i16p, u32p, u32p, u32])
    fn(C.byref(p), C.byref(st), x, out, iq, gain, phase, frames)
    return out.reshape(frames, 2), iq.reshape(frames, 2), gain, phase, st


def tx_batch(o, prms, x, states=None):
    """x int16 [C][frames][2], prms: one parameter dict per channel (or one for all). Every channel from a zero state unless `states`
    (a list, updated in place) is given. Returns out, iq (int16 [C][frames][2]) and gain (uint32 [C][frames/48])."""
    if isinstance(prms, dict):
        prms = [prms] * x.shape[0]
    if states is None:
        states = [TxQ15mState() for _ in range(x.shape[0])]
    res = [tx_q15(o, prms[c], x[c], states[c]) for c in range(x.shape[0])]
    return np.stack([r[0] for r in res]), np.stack([r[1] for r in res]), np.stack([r[2] for r in res])
