"""ctypes access to the two oracle libraries (TEST INFRASTRUCTURE ONLY).

`ref`  = oracle/_ref/libslo_ref.so  : the reference's own CMSIS-DSP V1.5.3 sources compiled for this host.
`port` = oracle/_port/libslo_port.so: the plain-C restatement (always buildable, also on the GPU box).
Nothing under selenite_lite_b200/ imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REFERENCE_TREE = "/root/reference"

MAX_STAGES = 4
MAX_FFT = 4096

f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
i16p = np.ctypeslib.ndpointer(np.int16, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
u32 = C.c_uint32
i32 = C.c_int32


class RxF32Params(C.Structure):
    _fields_ = [("fft_len", u32), ("hop", u32), ("agc_block", u32), ("n_stages", u32),
                ("biquad", C.c_float * (5 * MAX_STAGES)),
                ("agc_target", C.c_float), ("agc_decay", C.c_float), ("agc_floor", C.c_float), ("agc_gmax", C.c_float),
                ("mask", C.POINTER(C.c_float)), ("envelope", u32)]


class RxF32State(C.Structure):
    _fields_ = [("ovl", C.c_int16 * (2 * MAX_FFT)), ("bq", C.c_float * (2 * MAX_STAGES)), ("env", C.c_float), ("zlast", C.c_float * 2)]


class TxF32Params(C.Structure):
    _fields_ = [("fft_len", u32), ("hop", u32), ("alc_block", u32),
                ("alc_target", C.c_float), ("alc_decay", C.c_float), ("alc_floor", C.c_float), ("alc_gmax", C.c_float),
                ("mask", C.POINTER(C.c_float))]


class TxF32State(C.Structure):
    _fields_ = [("ovl", C.c_int16 * MAX_FFT), ("env", C.c_float)]


class ChanParams(C.Structure):
    _fields_ = [("bins", u32), ("taps_per_branch", u32), ("agc_block", u32), ("envelope", u32),
                ("agc_target", C.c_float), ("agc_decay", C.c_float), ("agc_floor", C.c_float), ("agc_gmax", C.c_float),
                ("proto", C.POINTER(C.c_float))]


class ChanState(C.Structure):
    _fields_ = [("fir_i", C.c_float * (64 * 8)), ("fir_q", C.c_float * (64 * 8)), ("env", C.c_float * 64)]


class RxQ15Params(C.Structure):
    _fields_ = [("ntaps", u32), ("agc_block", u32), ("agc_window", u32), ("lsb", u32),
                ("taps_i", C.c_int16 * 64), ("taps_q", C.c_int16 * 64), ("rel", C.c_int16 * 32),
                ("agc_target", C.c_int16), ("agc_floor", C.c_int16), ("agc_gmax_q15", u32),
                ("bq_stages", u32), ("bq_postshift", i32), ("bq_coeffs", C.c_int16 * 24)]


class RxQ15State(C.Structure):
    _fields_ = [("fir_i", C.c_int16 * (64 + 192)), ("fir_q", C.c_int16 * (64 + 192)), ("peaks", C.c_int16 * 32), ("bq", C.c_int16 * 16)]


def build_oracles(want_ref=True):
    """Build the port (always) and, when the reference tree is mounted, the reference build."""
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "port"], check=True)
    if want_ref and os.path.isdir(REFERENCE_TREE):
        subprocess.run(["make", "-s", "-j8", "-C", ORACLE_DIR, "ref"], check=True)


class Oracle:
    """One oracle library; every stage takes/returns numpy arrays for ONE channel."""

    def __init__(self, kind):
        assert kind in ("ref", "port")
        self.kind = kind
        path = os.path.join(ORACLE_DIR, "_%s" % kind, "libslo_%s.so" % kind)
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = C.CDLL(path)
        self.p = kind + "_"

    def _f(self, name, argtypes, restype=None):
        fn = getattr(self.lib, self.p + name)
        fn.argtypes = argtypes
        fn.restype = restype
        return fn

    # ---- conversions
    def q15_to_float(self, x):
        x = np.ascontiguousarray(x, np.int16); d = np.empty(x.size, np.float32)
        self._f("q15_to_float", [i16p, f32p, u32])(x.ravel(), d, x.size); return d.reshape(x.shape)

    def float_to_q15(self, x):
        x = np.ascontiguousarray(x, np.float32); d = np.empty(x.size, np.int16)
        self._f("float_to_q15", [f32p, i16p, u32])(x.ravel(), d, x.size); return d.reshape(x.shape)

    # ---- FIR family: returns (out, state)
    def _fir(self, name, dt, ptr, coeffs, state, x, block, extra=(), out_n=None):
        coeffs = np.ascontiguousarray(coeffs, dt); x = np.ascontiguousarray(x, dt)
        state = np.ascontiguousarray(state, dt).copy()
        out = np.zeros(x.size if out_n is None else out_n, dt)
        fn = self._f(name, [ptr, u32] + [u32] * len(extra) + [ptr, ptr, ptr, u32, u32])
        fn(coeffs, coeffs.size, *extra, state, x, out, x.size, block)
        return out, state

    def fir_f32(self, c, st, x, block): return self._fir("fir_f32", np.float32, f32p, c, st, x, block)
    def fir_q15(self, c, st, x, block): return self._fir("fir_q15", np.int16, i16p, c, st, x, block)
    def fir_fast_q15(self, c, st, x, block): return self._fir("fir_fast_q15", np.int16, i16p, c, st, x, block)
    def fir_q31(self, c, st, x, block): return self._fir("fir_q31", np.int32, i32p, c, st, x, block)
    def fir_decimate_f32(self, c, M, st, x, block): return self._fir("fir_decimate_f32", np.float32, f32p, c, st, x, block, (M,), len(x) // M)
    def fir_decimate_q15(self, c, M, st, x, block): return self._fir("fir_decimate_q15", np.int16, i16p, c, st, x, block, (M,), len(x) // M)
    def fir_interpolate_f32(self, c, L, st, x, block): return self._fir("fir_interpolate_f32", np.float32, f32p, c, st, x, block, (L,), len(x) * L)
    def fir_interpolate_q15(self, c, L, st, x, block): return self._fir("fir_interpolate_q15", np.int16, i16p, c, st, x, block, (L,), len(x) * L)
    def fir_decimate_q31(self, c, M, st, x, block): return self._fir("fir_decimate_q31", np.int32, i32p, c, st, x, block, (M,), len(x) // M)
    def fir_interpolate_q31(self, c, L, st, x, block): return self._fir("fir_interpolate_q31", np.int32, i32p, c, st, x, block, (L,), len(x) * L)

    # ---- biquads: returns (out, state)
    def _bq(self, name, dt, ptr, coeffs, nstages, state, x, block, n, extra=()):
        coeffs = np.ascontiguousarray(coeffs, dt); x = np.ascontiguousarray(x, dt)
        state = np.ascontiguousarray(state, dt).copy(); out = np.zeros(x.size, dt)
        fn = self._f(name, [ptr, u32] + [i32] * len(extra) + [ptr, ptr, ptr, u32, u32])
        fn(coeffs, nstages, *extra, state, x, out, n, block)
        return out, state

    def biquad_df2T_f32(self, c, ns, st, x, block): return self._bq("biquad_df2T_f32", np.float32, f32p, c, ns, st, x, block, len(x))
    def biquad_stereo_df2T_f32(self, c, ns, st, x, block): return self._bq("biquad_stereo_df2T_f32", np.float32, f32p, c, ns, st, x, block, len(x) // 2)
    def biquad_df1_f32(self, c, ns, st, x, block): return self._bq("biquad_df1_f32", np.float32, f32p, c, ns, st, x, block, len(x))
    def biquad_df1_q15(self, c, ns, ps, st, x, block): return self._bq("biquad_df1_q15", np.int16, i16p, c, ns, st, x, block, len(x), (ps,))
    def biquad_df1_q31(self, c, ns, ps, st, x, block): return self._bq("biquad_df1_q31", np.int32, i32p, c, ns, st, x, block, len(x), (ps,))

    def sidetone_mix(self, lr, counter, key_down, freq_hz, fs, level):
        """One DAC read's worth of frames int16 [frames][2]; returns (mixed copy, new counter)."""
        d = np.ascontiguousarray(lr, np.int16).copy(); cnt = C.c_uint32(counter)
        self._f("sidetone_mix", [i16p, u32, C.POINTER(C.c_uint32), C.c_int, u32, u32, C.c_float])(d.reshape(-1), d.shape[0], C.byref(cnt), int(key_down), freq_hz, fs, level)
        return d, cnt.value

    def lms_norm_f32(self, coeffs, mu, st, en_x0, x, ref, block):
        """arm_lms_norm_f32: returns (out, err, coeffs, state, en_x0) — copies, the inputs are not modified."""
        c = np.ascontiguousarray(coeffs, np.float32).copy(); s_ = np.ascontiguousarray(st, np.float32).copy()
        ex = np.ascontiguousarray(en_x0, np.float32).copy()
        x = np.ascontiguousarray(x, np.float32); ref = np.ascontiguousarray(ref, np.float32)
        out = np.zeros_like(x); err = np.zeros_like(x)
        self._f("lms_norm_f32", [f32p, u32, C.c_float, f32p, f32p, f32p, f32p, f32p, f32p, u32, u32])(c, c.size, mu, s_, ex, x, ref, out, err, x.size, block)
        return out, err, c, s_, ex

    # ---- transforms (interleaved re/im in, copy out)
    def cfft_f32(self, x, ifft=0, bitrev=1):
        d = np.ascontiguousarray(x, np.float32).copy()
        self._f("cfft_f32", [f32p, u32, C.c_int, C.c_int])(d, d.size // 2, ifft, bitrev); return d

    def cfft_q15_cm4(self, x, ifft=0, bitrev=1):
        """arm_cfft_q15 in the branch the firmware's ARM_MATH_CM4 build compiles (reference build only; the authority for the q15 FFT)."""
        d = np.ascontiguousarray(x, np.int16).copy()
        self._f("cfft_q15_cm4", [i16p, u32, C.c_int, C.c_int])(d, d.size // 2, ifft, bitrev); return d

    def cfft_q15(self, x, ifft=0, bitrev=1):
        d = np.ascontiguousarray(x, np.int16).copy()
        self._f("cfft_q15", [i16p, u32, C.c_int, C.c_int])(d, d.size // 2, ifft, bitrev); return d

    def cfft_q31(self, x, ifft=0, bitrev=1):
        d = np.ascontiguousarray(x, np.int32).copy()
        self._f("cfft_q31", [i32p, u32, C.c_int, C.c_int])(d, d.size // 2, ifft, bitrev); return d

    def rfft_fast_f32(self, x, ifft=0):
        d = np.ascontiguousarray(x, np.float32).copy(); out = np.zeros(d.size, np.float32)
        self._f("rfft_fast_f32", [f32p, f32p, u32, C.c_int])(d, out, d.size, ifft); return out

    # ---- element-wise helpers
    def _ew(self, name, dt, ptr, ins, out_n, pre=(), pre_types=()):
        ins = [np.ascontiguousarray(a, dt) for a in ins]; out = np.zeros(out_n, dt)
        fn = self._f(name, [ptr] + list(pre_types) + [ptr] * (len(ins) - 1) + [ptr, u32])
        return fn, ins, out

    def cmplx_mult_cmplx_f32(self, a, b):
        a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32); d = np.zeros(a.size, np.float32)
        self._f("cmplx_mult_cmplx_f32", [f32p, f32p, f32p, u32])(a, b, d, a.size // 2); return d

    def cmplx_mult_real_f32(self, a, r):
        a = np.ascontiguousarray(a, np.float32); r = np.ascontiguousarray(r, np.float32); d = np.zeros(a.size, np.float32)
        self._f("cmplx_mult_real_f32", [f32p, f32p, f32p, u32])(a, r, d, r.size); return d

    def cmplx_conj_f32(self, a):
        a = np.ascontiguousarray(a, np.float32); d = np.zeros(a.size, np.float32)
        self._f("cmplx_conj_f32", [f32p, f32p, u32])(a, d, a.size // 2); return d

    def cmplx_mag_f32(self, a):
        a = np.ascontiguousarray(a, np.float32); d = np.zeros(a.size // 2, np.float32)
        self._f("cmplx_mag_f32", [f32p, f32p, u32])(a, d, d.size); return d

    def cmplx_mag_squared_f32(self, a):
        a = np.ascontiguousarray(a, np.float32); d = np.zeros(a.size // 2, np.float32)
        self._f("cmplx_mag_squared_f32", [f32p, f32p, u32])(a, d, d.size); return d

    def cmplx_mag_q15(self, a):
        a = np.ascontiguousarray(a, np.int16); d = np.zeros(a.size // 2, np.int16)
        self._f("cmplx_mag_q15", [i16p, i16p, u32])(a, d, d.size); return d

    def max_f32(self, s):
        s = np.ascontiguousarray(s, np.float32); idx = u32(0)
        v = self._f("max_f32", [f32p, u32, C.POINTER(u32)], C.c_float)(s, s.size, C.byref(idx)); return np.float32(v), idx.value

    def rms_f32(self, s): s = np.ascontiguousarray(s, np.float32); return np.float32(self._f("rms_f32", [f32p, u32], C.c_float)(s, s.size))
    def power_f32(self, s): s = np.ascontiguousarray(s, np.float32); return np.float32(self._f("power_f32", [f32p, u32], C.c_float)(s, s.size))
    def mean_f32(self, s): s = np.ascontiguousarray(s, np.float32); return np.float32(self._f("mean_f32", [f32p, u32], C.c_float)(s, s.size))

    def max_q15(self, s):
        s = np.ascontiguousarray(s, np.int16); idx = u32(0)
        v = self._f("max_q15", [i16p, u32, C.POINTER(u32)], C.c_int16)(s, s.size, C.byref(idx)); return int(v), idx.value

    def rms_q15(self, s): s = np.ascontiguousarray(s, np.int16); return int(self._f("rms_q15", [i16p, u32], C.c_int16)(s, s.size))

    def scale_f32(self, s, k):
        s = np.ascontiguousarray(s, np.float32); d = np.zeros(s.size, np.float32)
        self._f("scale_f32", [f32p, C.c_float, f32p, u32])(s, k, d, s.size); return d

    def _bin_f32(self, name, a, b):
        a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32); d = np.zeros(a.size, np.float32)
        self._f(name, [f32p, f32p, f32p, u32])(a, b, d, a.size); return d

    def mult_f32(self, a, b): return self._bin_f32("mult_f32", a, b)
    def add_f32(self, a, b): return self._bin_f32("add_f32", a, b)
    def sub_f32(self, a, b): return self._bin_f32("sub_f32", a, b)

    def abs_f32(self, a):
        a = np.ascontiguousarray(a, np.float32); d = np.zeros(a.size, np.float32)
        self._f("abs_f32", [f32p, f32p, u32])(a, d, a.size); return d

    def scale_q15(self, s, k, shift):
        s = np.ascontiguousarray(s, np.int16); d = np.zeros(s.size, np.int16)
        self._f("scale_q15", [i16p, C.c_int16, i32, i16p, u32])(s, k, shift, d, s.size); return d

    def _bin_q15(self, name, a, b):
        a = np.ascontiguousarray(a, np.int16); b = np.ascontiguousarray(b, np.int16); d = np.zeros(a.size, np.int16)
        self._f(name, [i16p, i16p, i16p, u32])(a, b, d, a.size); return d

    def add_q15(self, a, b): return self._bin_q15("add_q15", a, b)
    def sub_q15(self, a, b): return self._bin_q15("sub_q15", a, b)

    def abs_q15(self, a):
        a = np.ascontiguousarray(a, np.int16); d = np.zeros(a.size, np.int16)
        self._f("abs_q15", [i16p, i16p, u32])(a, d, a.size); return d

    def shift_q15(self, a, sh):
        a = np.ascontiguousarray(a, np.int16); d = np.zeros(a.size, np.int16)
        self._f("shift_q15", [i16p, i32, i16p, u32])(a, sh, d, a.size); return d

    def sin_f32(self, x):
        x = np.ascontiguousarray(x, np.float32); d = np.zeros(x.size, np.float32)
        self._f("sin_f32", [f32p, f32p, u32])(x, d, x.size); return d

    def cos_f32(self, x):
        x = np.ascontiguousarray(x, np.float32); d = np.zeros(x.size, np.float32)
        self._f("cos_f32", [f32p, f32p, u32])(x, d, x.size); return d

    # ---- chains
    def make_rx_params(self, prm):
        """prm: dict with fft_len, hop, agc_block, biquad (n_stages x 5), agc_*, mask (complex64[fft_len])."""
        p = RxF32Params()
        p.fft_len, p.hop, p.agc_block = prm["fft_len"], prm["hop"], prm["agc_block"]
        bq = np.asarray(prm["biquad"], np.float32).reshape(-1, 5)
        p.n_stages = bq.shape[0]
        for i, v in enumerate(bq.ravel()):
            p.biquad[i] = float(v)
        p.agc_target, p.agc_decay = float(prm["agc_target"]), float(prm["agc_decay"])
        p.agc_floor, p.agc_gmax = float(prm["agc_floor"]), float(prm["agc_gmax"])
        mask = np.ascontiguousarray(np.asarray(prm["mask"], np.complex64).view(np.float32))
        p.mask = mask.ctypes.data_as(C.POINTER(C.c_float))
        p._keep = mask
        p.envelope = int(prm.get("envelope", 0))
        return p

    def rx_ssb_f32(self, prm, in_iq, state=None, want_debug=True):
        """in_iq int16[frames][2] one channel. Returns out int16[frames][2], audio f32[frames], gain f32[frames/agc_block], state."""
        p = self.make_rx_params(prm)
        st = state if state is not None else RxF32State()
        x = np.ascontiguousarray(in_iq, np.int16).reshape(-1)
        frames = x.size // 2
        out = np.zeros(2 * frames, np.int16)
        audio = np.zeros(frames, np.float32); gain = np.zeros(frames // prm["agc_block"], np.float32)
        fn = self._f("rx_ssb_f32", [C.POINTER(RxF32Params), C.POINTER(RxF32State), i16p, i16p, C.c_void_p, C.c_void_p, u32])
        fn(C.byref(p), C.byref(st), x, out, audio.ctypes.data if want_debug else None, gain.ctypes.data if want_debug else None, frames)
        return out.reshape(frames, 2), audio, gain, st

    def rx_ssb_f32_batch(self, prm, in_iq, states=None, nthreads=1):
        """in_iq int16[C][frames][2]. Returns out int16[C][frames][2], states."""
        p = self.make_rx_params(prm)
        x = np.ascontiguousarray(in_iq, np.int16)
        Cn, frames = x.shape[0], x.shape[1]
        st = states if states is not None else (RxF32State * Cn)()
        out = np.zeros_like(x)
        fn = self._f("rx_ssb_f32_batch", [C.POINTER(RxF32Params), C.POINTER(RxF32State), i16p, i16p, u32, u32, u32])
        fn(C.byref(p), st, x.reshape(-1), out.reshape(-1), Cn, frames, nthreads)
        return out, st


    def tx_ssb_f32(self, prm, in_lr, state=None):
        """in_lr int16[frames][2] (L = R mic) one channel. Returns out int16[frames][2] I/Q, iq f32[frames][2] (pre-ALC),
        gain f32[frames/alc_block], state."""
        p = TxF32Params()
        p.fft_len, p.hop, p.alc_block = prm["fft_len"], prm["hop"], prm["alc_block"]
        p.alc_target, p.alc_decay = float(prm["alc_target"]), float(prm["alc_decay"])
        p.alc_floor, p.alc_gmax = float(prm["alc_floor"]), float(prm["alc_gmax"])
        mask = np.ascontiguousarray(np.asarray(prm["mask"], np.complex64).view(np.float32))
        p.mask = mask.ctypes.data_as(C.POINTER(C.c_float))
        st = state if state is not None else TxF32State()
        x = np.ascontiguousarray(in_lr, np.int16).reshape(-1)
        frames = x.size // 2
        out = np.zeros(2 * frames, np.int16); iq = np.zeros(2 * frames, np.float32)
        gain = np.zeros(frames // prm["alc_block"], np.float32)
        fn = self._f("tx_ssb_f32", [C.POINTER(TxF32Params), C.POINTER(TxF32State), i16p, i16p, f32p, f32p, u32])
        fn(C.byref(p), C.byref(st), x, out, iq, gain, frames)
        return out.reshape(frames, 2), iq.reshape(frames, 2), gain, st


    def rx_ssb_q15(self, prm, in_iq, state=None):
        """in_iq int16[frames][2] one channel. Returns out int16[frames][2], audio int16[frames] (pre-AGC),
        gain uint32[frames/agc_block] (Q15), state."""
        p = RxQ15Params()
        p.ntaps, p.agc_block, p.agc_window, p.lsb = prm["ntaps"], prm["agc_block"], prm["agc_window"], int(prm["lsb"])
        for k in range(64):
            p.taps_i[k] = int(prm["taps_i"][k]); p.taps_q[k] = int(prm["taps_q"][k])
        for k in range(32):
            p.rel[k] = int(prm["rel"][k])
        p.agc_target, p.agc_floor, p.agc_gmax_q15 = int(prm["agc_target"]), int(prm["agc_floor"]), int(prm["agc_gmax_q15"])
        p.bq_stages, p.bq_postshift = int(prm.get("bq_stages", 0)), int(prm.get("bq_postshift", 0))
        for k in range(6 * p.bq_stages):
            p.bq_coeffs[k] = int(prm["bq_coeffs"][k])
        st = state if state is not None else RxQ15State()
        x = np.ascontiguousarray(in_iq, np.int16).reshape(-1)
        frames = x.size // 2
        out = np.zeros(2 * frames, np.int16); audio = np.zeros(frames, np.int16); gain = np.zeros(frames // prm["agc_block"], np.uint32)
        fn = self._f("rx_ssb_q15", [C.POINTER(RxQ15Params), C.POINTER(RxQ15State), i16p, i16p, i16p, np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS"), u32])
        fn(C.byref(p), C.byref(st), x, out, audio, gain, frames)
        return out.reshape(frames, 2), audio, gain, st

    def chan_f32(self, prm, in_iq, state=None, want_debug=True):
        """One wideband stream int16[frames][2]. Returns out int16[bins][frames/bins][2], audio f32[bins][hops],
        gain f32[bins][hops/agc_block], state."""
        p = ChanParams()
        p.bins, p.taps_per_branch, p.agc_block, p.envelope = prm["bins"], prm["taps_per_branch"], prm["agc_block"], int(prm["envelope"])
        p.agc_target, p.agc_decay = float(prm["agc_target"]), float(prm["agc_decay"])
        p.agc_floor, p.agc_gmax = float(prm["agc_floor"]), float(prm["agc_gmax"])
        proto = np.ascontiguousarray(prm["proto"], np.float32)
        p.proto = proto.ctypes.data_as(C.POINTER(C.c_float))
        st = state if state is not None else ChanState()
        x = np.ascontiguousarray(in_iq, np.int16).reshape(-1)
        frames = x.size // 2; bins = prm["bins"]; hops = frames // bins
        out = np.zeros(2 * bins * hops, np.int16)
        audio = np.zeros(bins * hops, np.float32); gain = np.zeros(bins * hops // prm["agc_block"], np.float32)
        fn = self._f("chan_f32", [C.POINTER(ChanParams), C.POINTER(ChanState), i16p, i16p, C.c_void_p, C.c_void_p, u32])
        fn(C.byref(p), C.byref(st), x, out, audio.ctypes.data if want_debug else None, gain.ctypes.data if want_debug else None, frames)
        return out.reshape(bins, hops, 2), audio.reshape(bins, hops), gain.reshape(bins, -1), st


def _digest(name, args):
    """Stable digest of one oracle call: routine name and every argument (arrays by dtype, shape and bytes)."""
    import hashlib
    h = hashlib.sha256(name.encode())

    def put(a):
        if isinstance(a, dict):
            for k in sorted(a):
                h.update(str(k).encode()); put(a[k])
        elif isinstance(a, (np.ndarray, np.generic)):
            a = np.ascontiguousarray(a); h.update(("%s%s" % (a.dtype.str, a.shape)).encode()); h.update(a.tobytes())
        else:
            h.update(repr(a).encode())
    for a in args:
        put(a)
    return h.hexdigest()


class Recorded:
    """An oracle replayed from stored outputs (tests/golden/pinning.npz, make_golden.py pinning): the i-th call a test makes
    returns what the recorded oracle returned for that test's i-th call, and fails when the arguments differ from the ones
    recorded. With `live` set it records instead: it calls `live` and stores the results in `store`."""

    def __init__(self, store, test_name, live=None):
        self.store, self.test, self.live, self.n = store, test_name, live, 0
        self.kind = "recorded from %s" % (live.kind if live is not None else str(store["source"]))

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def call(*args):
            key = "%s|%d" % (self.test, self.n); self.n += 1
            dig = _digest(name, args)
            if self.live is not None:
                res = getattr(self.live, name)(*args)
                parts = res if isinstance(res, tuple) else (res,)
                self.store[key + "|call"] = np.array("%s %s %d" % (name, dig, len(parts) if isinstance(res, tuple) else -1))
                for j, p in enumerate(parts):
                    if isinstance(p, (np.ndarray, np.generic, int, float)):
                        self.store["%s|%d" % (key, j)] = np.asarray(p)
                return res
            if key + "|call" not in self.store:
                raise AssertionError("no recorded call %s (%s): re-record with tests/golden/make_golden.py pinning" % (key, name))
            rname, rdig, n = str(self.store[key + "|call"]).split()
            assert (rname, rdig) == (name, dig), ("inputs differ from the recorded call", key, name, rname)
            parts = [self.store["%s|%d" % (key, j)][()] if "%s|%d" % (key, j) in self.store else None for j in range(max(int(n), 1))]
            return tuple(parts) if int(n) >= 0 else parts[0]
        return call


class RefRing:
    """The UNMODIFIED reference dsp_if.c built for one sample rate (oracle/_ref/libdspif_<fs>.so)."""

    def __init__(self, fs=48000):
        path = os.path.join(ORACLE_DIR, "_ref", "libdspif_%d.so" % fs)
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        # dsp_if.c keeps its rings in file-scope globals (dsp_if.c:32-35): one loaded image = one channel. Each RefRing
        # therefore loads its own private copy of the library.
        import shutil
        import tempfile
        tmp = tempfile.NamedTemporaryFile(prefix="dspif_", suffix=".so", delete=False)
        tmp.close(); shutil.copyfile(path, tmp.name)
        self.lib = C.CDLL(tmp.name)
        os.unlink(tmp.name)
        L = self.lib
        for n in ("refring_fs", "refring_i2s_buff_size", "refring_i2s_half_size", "refring_dsp_buff_size", "refring_dsp_half_size"):
            getattr(L, n).restype = u32
        self.fs = L.refring_fs(); self.ring = L.refring_dsp_buff_size(); self.half_hw = L.refring_i2s_half_size()
        L.DSP_In_Buff_Write.argtypes = [i16p, C.c_uint16]
        L.DSP_In_Buff_Read.argtypes = [i16p, u32]
        L.DSP_Out_Buff_Write.argtypes = [i16p, u32]
        L.DSP_Out_Buff_Read.argtypes = [i16p, C.c_uint16]
        L.refring_i2s_event.argtypes = [C.c_int, i16p, i16p]
        L.refring_reset()

    def reset(self): self.lib.refring_reset()
    def in_write(self, block_hw): b = np.ascontiguousarray(block_hw, np.int16); self.lib.DSP_In_Buff_Write(b, b.size)
    def in_read(self, nbytes): b = np.zeros(nbytes // 2, np.int16); self.lib.DSP_In_Buff_Read(b, nbytes); return b
    def out_write(self, block_hw): b = np.ascontiguousarray(block_hw, np.int16); self.lib.DSP_Out_Buff_Write(b, b.size * 2)
    def out_read(self, nhw): b = np.zeros(nhw, np.int16); self.lib.DSP_Out_Buff_Read(b, nhw); return b
    def out_mute(self): self.lib.DSP_Out_Buff_Mute()

    def i2s_event(self, half, adc_block):
        a = np.ascontiguousarray(adc_block, np.int16); d = np.zeros(a.size, np.int16)
        self.lib.refring_i2s_event(half, a, d); return d

    def ptrs(self, which):
        o = (u32 * 3)(); self.lib.refring_get_ptrs(which, o); return tuple(o)

    def iq(self, which):
        i = np.zeros(self.ring, np.int16); q = np.zeros(self.ring, np.int16)
        self.lib.refring_get_iq.argtypes = [C.c_int, i16p, i16p]; self.lib.refring_get_iq(which, i, q); return i, q


class PortRing:
    """oracle/port/ring_port.c — restatement of the ring with run-time geometry."""

    def __init__(self, fs=48000, lib=None):
        self.lib = lib or C.CDLL(os.path.join(ORACLE_DIR, "_port", "libslo_port.so"))
        self.lib.port_ring_sizeof.restype = u32
        self.buf = C.create_string_buffer(self.lib.port_ring_sizeof())
        self.lib.port_ring_init(self.buf, u32(fs))
        self.ring = fs // 1000 * 8
        self.lib.port_ring_write.argtypes = [C.c_void_p, C.c_int, i16p, u32]
        self.lib.port_ring_read.argtypes = [C.c_void_p, C.c_int, i16p, u32]

    def in_write(self, b): b = np.ascontiguousarray(b, np.int16); self.lib.port_ring_write(self.buf, 0, b, b.size)
    def out_write(self, b): b = np.ascontiguousarray(b, np.int16); self.lib.port_ring_write(self.buf, 1, b, b.size)
    def in_read(self, nbytes): b = np.zeros(nbytes // 2, np.int16); self.lib.port_ring_read(self.buf, 0, b, b.size); return b
    def out_read(self, nhw): b = np.zeros(nhw, np.int16); self.lib.port_ring_read(self.buf, 1, b, nhw); return b
    def out_mute(self): self.lib.port_ring_mute(self.buf)

    def ptrs(self):
        o = (u32 * 3)(); self.lib.port_ring_get_ptrs(self.buf, o); return tuple(o)

    def iq(self):
        i = np.zeros(self.ring, np.int16); q = np.zeros(self.ring, np.int16)
        self.lib.port_ring_get_iq.argtypes = [C.c_void_p, i16p, i16p]; self.lib.port_ring_get_iq(self.buf, i, q); return i, q
