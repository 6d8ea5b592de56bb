"""ctypes access to the per-channel tuner of the oracle (oracle/slo_tune.h; TEST INFRASTRUCTURE ONLY).

`tune_q15` takes an oracle_lib.Oracle (the port: the tuner is composed from stages the port restates) and works on ONE channel."""
import ctypes as C

import numpy as np

from oracle_lib import i16p, i32, u32


def increment(hz, fs):
    """The NCO increment of an offset (2^-32 turn per sample): llround (hz 2^32 / fs) in double, as slb_set_tune computes it."""
    v = float(hz) * 4294967296.0 / float(fs)
    return int(np.sign(v) * np.floor(abs(v) + 0.5))


def tune_q15(o, x, inc, phase=0, up=False):
    """x int16 [frames][2] I/Q -> (int16 [frames][2], phase after the call). up=False (RX) moves what sits at +inc down to 0."""
    x = np.ascontiguousarray(x, np.int16).reshape(-1)
    out = np.zeros_like(x); ph = C.c_uint32(int(phase) & 0xFFFFFFFF)
    o._f("tune_q15", [i16p, i16p, u32, i32, C.POINTER(C.c_uint32), C.c_int])(x, out, x.size // 2, int(inc), C.byref(ph), int(bool(up)))
    return out.reshape(-1, 2), ph.value


def tune_batch(o, x, incs, up=False):
    """x int16 [C][frames][2], incs [C]: every channel from phase 0."""
    return np.stack([tune_q15(o, x[c], incs[c], 0, up)[0] for c in range(x.shape[0])])
