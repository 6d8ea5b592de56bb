"""ctypes access to the integer channelizer of the oracle (oracle/slo_chan_q15.h; TEST INFRASTRUCTURE ONLY).

`chan_q15` takes an oracle_lib.Oracle (the port: the chain is composed from stages the port restates) and works on ONE wideband stream. It
takes the parameter dict of DspIf.oracle_params on a CHAN-64-q15 context (dsp_if.chan_q15_params_to_dict); the state keeps each branch's
last 7 inputs per rail and each bin's block peaks."""
import ctypes as C

import numpy as np

from oracle_lib import i16p, u32

u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
BINS, TAPS, WIN = 64, 8, 32


class ChanQ15Params(C.Structure):
    _fields_ = [("bins", u32), ("taps_per_branch", u32), ("agc_block", u32), ("envelope", u32), ("proto", C.c_int16 * (BINS * TAPS)),
                ("agc_window", u32), ("rel", C.c_int16 * WIN), ("agc_target", C.c_int16), ("agc_floor", C.c_int16), ("agc_gmax_q15", u32)]


class ChanQ15State(C.Structure):
    _fields_ = [("fir_i", C.c_int16 * (BINS * TAPS)), ("fir_q", C.c_int16 * (BINS * TAPS)), ("peaks", C.c_int16 * (BINS * WIN))]


def _params(prm):
    p = ChanQ15Params()
    p.bins, p.taps_per_branch, p.agc_block, p.envelope = prm["bins"], prm["taps_per_branch"], prm["agc_block"], int(prm["envelope"])
    for k in range(BINS * TAPS):
        p.proto[k] = int(prm["proto"][k])
    for k in range(WIN):
        p.rel[k] = int(prm["rel"][k])
    p.agc_window, p.agc_target, p.agc_floor, p.agc_gmax_q15 = int(prm["agc_window"]), int(prm["agc_target"]), int(prm["agc_floor"]), int(prm["agc_gmax_q15"])
    return p


def chan_q15(o, prm, in_iq, state=None):
    """in_iq int16[frames][2] one wideband stream. Returns out int16[64][hops][2] (L = R), audio int16[64][hops] (pre-AGC detector output),
    gain uint32[64][hops/3] (Q15), state."""
    p = _params(prm)
    st = state if state is not None else ChanQ15State()
    x = np.ascontiguousarray(in_iq, np.int16).reshape(-1)
    hops = x.size // 2 // BINS
    out = np.zeros(2 * BINS * hops, np.int16); aud = np.zeros(BINS * hops, np.int16)
    gain = np.zeros(BINS * hops // int(prm["agc_block"]), np.uint32)
    fn = o._f("chan_q15", [C.POINTER(ChanQ15Params), C.POINTER(ChanQ15State), i16p, i16p, i16p, u32p, u32])
    fn(C.byref(p), C.byref(st), x, out, aud, gain, x.size // 2)
    return out.reshape(BINS, hops, 2), aud.reshape(BINS, hops), gain.reshape(BINS, -1), st


def chan_batch(o, prm, x, states=None):
    """x int16 [S][frames][2]. Every stream from a zero state unless `states` (a list, updated in place) is given. Returns out
    (int16 [S][64][hops][2]), audio (int16 [S][64][hops]) and gain (uint32 [S][64][hops/3])."""
    if states is None:
        states = [ChanQ15State() for _ in range(x.shape[0])]
    res = [chan_q15(o, prm, x[s], states[s]) for s in range(x.shape[0])]
    return np.stack([r[0] for r in res]), np.stack([r[1] for r in res]), np.stack([r[2] for r in res])
