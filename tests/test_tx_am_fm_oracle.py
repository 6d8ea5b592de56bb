"""The oracle of the AM / FM transmit modulators (oracle/slo_tx_mod.h, DESIGN.md §3.4) on the CPU: the three stages they add
against the CMSIS-DSP V1.5.3 formulas (and against the reference's own routines where that build exists), the modulators'
properties (AM envelope bounds, FM constant envelope and bounded increments, exact continuation across calls), the committed
golden vectors, and the loopback SNR of a 1 kHz mic tone through port TX -> port RX that the GPU loopback test is held to."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_tx_mod as otm
import selenite_lite_b200 as slb
from oracle_lib import f32p, i32p, u32
from selenite_lite_b200.dsp_if import params_to_dict, tx_mod_params_to_dict
from test_golden import GOLD

FS = 48000
ONE_BELOW = np.nextafter(np.float32(1.0), np.float32(0.0))
EDGES = np.array([1.0, -1.0, ONE_BELOW, -ONE_BELOW, 0.5, -0.5, 0.0, 2.0 ** -31, 1.5 * 2.0 ** -31, -1.5 * 2.0 ** -31, 1e-12, -1e-12,
                  0.7071067811865476, -0.3333333333, 2.0, -3.0, 1e9, -1e9], np.float32)   # (|x| 2^31 < 2^63: the C cast is defined)
# the loopback SNR (dB) of a 0.3 FS 1 kHz mic tone, 40 hops, through port tx_mod_f32 -> port rx_ssb_f32 (AM: envelope detector,
# FM: limiter-discriminator), measured on the int16 audio after 8 hops of settling by oracle_tx_mod.tone_snr_db
LOOPBACK_SNR_DB = {slb.MODE_AM: 87.948, slb.MODE_FM: 50.809}


def mod_prm(mode, fs=FS, **over):
    tp = slb.default_tx_f32_params(fs); mp = slb.default_tx_mod_params(fs)
    for k, v in over.items():
        setattr(mp, k, v)
    return tx_mod_params_to_dict(tp, mp, slb.default_mask(fs, tp.fft_len, mode), fs, mode)


def worst_case_mics(T):
    """Rails, a full-scale tone in the pass-band and a rail-to-rail square wave (L = R)."""
    n = np.arange(T)
    pats = [np.full(T, -32768, np.int16), np.full(T, 32767, np.int16),
            np.clip(np.rint(np.sin(2 * np.pi * 1200.0 * n / FS) * 32767), -32768, 32767).astype(np.int16),
            np.where((n // 16) % 2 == 0, 32767, -32768).astype(np.int16)]
    return np.stack([np.stack([p_, p_], axis=1) for p_ in pats])


def loopback_input(T=384 * 40):
    n = np.arange(T)
    m = np.rint(0.3 * 32768 * np.sin(2 * np.pi * 1000.0 * n / FS)).astype(np.int16)
    return np.stack([m, m], axis=1)


def q31_expected(x):
    """CMSIS V1.5.3 arm_float_to_q31, ARM_MATH_ROUNDING not defined: clip_q63_to_q31 ((q63_t) (x * 2147483648.0f))."""
    v = np.trunc(x.astype(np.float64) * 2147483648.0)       # x * 2^31 is exact in float32; the cast truncates
    return np.clip(v, -2147483648.0, 2147483647.0).astype(np.int64).astype(np.int32)


def test_offset_f32(port):
    for k in (1.0, -1.0, 0.25, ONE_BELOW):
        got = otm.offset_f32(port, EDGES, k)
        assert np.array_equal(got.view(np.uint32), (EDGES + np.float32(k)).astype(np.float32).view(np.uint32)), k


def test_float_to_q31(port):
    got = otm.float_to_q31(port, EDGES)
    assert np.array_equal(got, q31_expected(EDGES))
    assert got[0] == 2147483647 and got[1] == -2147483648                   # +1.0 saturates, -1.0 is exact
    assert got[2] == 2147483520 and got[3] == -2147483520                   # just below 1: 2^31 - 2^7, no saturation
    assert got[7] == 1 and got[8] == 1 and got[9] == -1                     # truncation toward zero
    x = np.random.Generator(np.random.PCG64(3)).uniform(-1.2, 1.2, 4096).astype(np.float32)
    assert np.array_equal(otm.float_to_q31(port, x), q31_expected(x))


def test_q31_to_float(port):
    x = np.array([-2 ** 31, 2 ** 31 - 1, 0, 1, -1, 2 ** 24 + 1, -(2 ** 24) - 3, 123456789, -987654321], np.int32)
    got = otm.q31_to_float(port, x)
    assert np.array_equal(got.view(np.uint32), (x.astype(np.float32) / np.float32(2147483648.0)).view(np.uint32))
    assert got[0] == -1.0 and got[1] == 1.0                                 # INT32_MAX rounds to 2^31 before the division
    assert np.all(np.isfinite(got))


def test_port_stages_vs_reference_routines(ref, port):
    """The port's three stages against arm_offset_f32, arm_float_to_q31 and arm_q31_to_float of the reference build, bit for bit."""
    L = ref.lib
    L.arm_offset_f32.argtypes = [f32p, C.c_float, f32p, u32]; L.arm_offset_f32.restype = None
    L.arm_float_to_q31.argtypes = [f32p, i32p, u32]; L.arm_float_to_q31.restype = None
    L.arm_q31_to_float.argtypes = [i32p, f32p, u32]; L.arm_q31_to_float.restype = None
    rng = np.random.Generator(np.random.PCG64(11))
    x = np.concatenate([EDGES, rng.uniform(-1.5, 1.5, 1000).astype(np.float32)])
    d = np.zeros_like(x); L.arm_offset_f32(x, 1.0, d, x.size)
    assert np.array_equal(d.view(np.uint32), otm.offset_f32(port, x, 1.0).view(np.uint32))
    q = np.zeros(x.size, np.int32); L.arm_float_to_q31(x, q, x.size)
    assert np.array_equal(q, otm.float_to_q31(port, x))
    i = rng.integers(-2 ** 31, 2 ** 31, 1000, dtype=np.int64).astype(np.int32)
    f = np.zeros(i.size, np.float32); L.arm_q31_to_float(i, f, i.size)
    assert np.array_equal(f.view(np.uint32), otm.q31_to_float(port, i).view(np.uint32))


@pytest.mark.parametrize("which", ["mic", "worst"])
def test_am_properties(port, which):
    prm = mod_prm(slb.MODE_AM)
    xs = slb.synth_mic(2, 384 * 12) if which == "mic" else worst_case_mics(384 * 12)
    c, d = prm["am_carrier"], prm["am_depth"]
    for x in xs:
        y, iq, gain, _, _ = otm.tx_mod_f32(port, prm, x)
        assert np.all(y[:, 1] == 0)
        lo, hi = int(np.floor(c * (1 - d) * 32768)) - 1, int(np.ceil(c * (1 + d) * 32768)) + 1
        assert y[:, 0].min() >= lo and y[:, 0].max() <= hi, (y[:, 0].min(), y[:, 0].max(), lo, hi)


@pytest.mark.parametrize("which", ["mic", "worst"])
def test_fm_properties(port, which):
    prm = mod_prm(slb.MODE_FM)
    xs = slb.synth_mic(2, 384 * 12) if which == "mic" else worst_case_mics(384 * 12)
    T = float(otm.fm_target(prm))
    for x in xs:
        y, iq, gain, phase, _ = otm.tx_mod_f32(port, prm, x)
        inc = np.diff(np.concatenate([[0], phase]).astype(np.uint32)).view(np.int32).astype(np.int64)
        assert np.max(np.abs(inc)) <= T * 2 ** 31 * (1 + 2 ** -22) + 1, (np.max(np.abs(inc)), T * 2 ** 31)
        # constant envelope: the table's linear interpolation (<= 2e-5 relative) and two truncations to q15
        mag = np.hypot(y[:, 0].astype(np.float64), y[:, 1].astype(np.float64)) / 32768.0
        assert np.max(np.abs(mag - prm["fm_level"])) <= 1e-4 * prm["fm_level"] + 2.0 / 32768.0
        # the output is the NCO of the phase, and nothing else
        assert np.array_equal(otm.tx_fm_nco(port, phase, prm["fm_level"]), y)


@pytest.mark.parametrize("mode", [slb.MODE_AM, slb.MODE_FM])
def test_calls_cut_at_hops_continue_exactly(port, mode):
    """Calls of 384 k frames continue the stream bit for bit (overlap tail, ALC envelope, phase accumulator carried)."""
    prm = mod_prm(mode)
    x = slb.synth_mic(1, 384 * 12)[0]
    whole = otm.tx_mod_f32(port, prm, x)
    st = otm.TxModState(); parts = []
    for a, b in ((0, 384), (384, 384 * 4), (384 * 4, 384 * 5), (384 * 5, 384 * 12)):
        parts.append(otm.tx_mod_f32(port, prm, x[a:b], st))
    for j in range(4):
        assert np.array_equal(np.concatenate([p_[j] for p_ in parts]), whole[j]), j


def test_golden_vectors(port):
    g = np.load(os.path.join(GOLD, "tx_am_fm_f32.npz"))
    for name, mode in (("am", slb.MODE_AM), ("fm", slb.MODE_FM)):
        prm = mod_prm(mode)
        assert np.array_equal(prm["mask"], g["%s_mask" % name])
        y, iq, gain, phase, _ = otm.tx_mod_f32(port, prm, g["%s_in" % name])
        assert np.array_equal(y, g["%s_out" % name]) and np.array_equal(gain, g["%s_gain" % name])
        assert np.allclose(iq, g["%s_iq" % name], rtol=0, atol=1e-6)
        if mode == slb.MODE_FM:
            assert np.array_equal(phase, g["fm_phase"])


@pytest.mark.parametrize("mode", [slb.MODE_AM, slb.MODE_FM])
def test_loopback_snr_through_the_oracle(port, mode):
    """TX-AM -> RX-SSB-f32 in AM and TX-FM -> RX-SSB-f32 in FM, both through the port: the recovered 1 kHz tone's SNR."""
    y = otm.tx_mod_f32(port, mod_prm(mode), loopback_input())[0]
    prm = params_to_dict(slb.default_rx_f32_params(FS), slb.default_mask(FS, 512, mode))
    prm["envelope"] = 1 if mode == slb.MODE_AM else 2
    out = port.rx_ssb_f32(prm, y)[0]
    snr = otm.tone_snr_db(out[384 * 8:, 0], FS, 1000.0)
    assert abs(snr - LOOPBACK_SNR_DB[mode]) < 0.01, snr
