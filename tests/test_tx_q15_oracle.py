"""The oracle of the all-integer SSB modulator TX-SSB-q15 (oracle/slo_tx_q15.h, DESIGN.md §3.7) on the CPU: the sideband convention
(USB puts the mic tone at +f of I + jQ), the loopback through the receive chain of the same family, exact continuation across calls,
the ALC's bounds, the committed golden vectors, and the TX operand planes of the tensor-core kernel against arm_fir_q15 of L."""
import os
import sys

import numpy as np
import pytest

import oracle_tx_q15 as otq
import selenite_lite_b200 as slb
from selenite_lite_b200 import _lib
from selenite_lite_b200.dsp_if import q15_params_to_dict
from test_golden import GOLD

sys.path.insert(0, GOLD)
import make_golden_tx_q15 as mg  # noqa: E402

FS = 48000


def prm(lsb=0, **over):
    p = q15_params_to_dict(slb.default_rx_q15_params(FS), lsb=lsb)
    p.update(over)
    return p


def tone(f0, frames=48 * 200, amp=0.3):
    n = np.arange(frames)
    m = np.rint(amp * 32768 * np.cos(2 * np.pi * f0 * n / FS)).astype(np.int16)
    return np.stack([m, m], axis=1)


@pytest.mark.parametrize("f0", [1000.0, 1500.0, 2500.0])
def test_sideband_is_the_rail_order(port, f0):
    """USB (fq, fi) puts a mic tone at +f0 of I + jQ, LSB (fi, fq) at -f0; the opposite sideband is >= 40 dB down, before and after
    the ALC."""
    x = tone(f0)
    for lsb, sign in ((0, 1.0), (1, -1.0)):
        y, iq, _, _ = otq.tx_ssb_q15(port, prm(lsb), x)
        for z in (iq, y):
            assert sign * otq.sideband_db(z, FS, f0) >= 40.0, (f0, lsb, otq.sideband_db(z, FS, f0))


def test_usb_and_lsb_swap_the_rails(port):
    x = slb.synth_mic(1, 48 * 20)[0]
    _, usb, _, _ = otq.tx_ssb_q15(port, prm(0), x)
    _, lsb, _, _ = otq.tx_ssb_q15(port, prm(1), x)
    assert np.array_equal(usb[:, ::-1], lsb)


def test_loopback_through_the_receive_chain(port):
    """TX-SSB-q15 USB -> RX-SSB-q15: the USB receiver recovers the 1 kHz tone, the LSB receiver rejects it by >= 40 dB. Compared on the
    receivers' pre-AGC audio: the AGC would lift the rejected tone back to its target."""
    y, _, _, _ = otq.tx_ssb_q15(port, prm(0), tone(1000.0))
    _, a_usb, _, _ = port.rx_ssb_q15(prm(0), y)
    _, a_lsb, _, _ = port.rx_ssb_q15(prm(1), y)

    def p1k(a):
        a = a[1000:].astype(np.float64)
        A = np.abs(np.fft.rfft(a * np.hanning(a.size))) ** 2
        f = np.fft.rfftfreq(a.size, 1.0 / FS)
        return A[np.abs(f - 1000.0) <= 60.0].sum()
    assert 10 * np.log10(p1k(a_usb) / p1k(a_lsb)) >= 40.0
    assert np.std(a_usb[1000:].astype(np.float64)) > 1000.0


def test_one_call_equals_two(port):
    x = slb.synth_mic(1, 48 * 60)[0]
    whole = otq.tx_ssb_q15(port, prm(0), x)
    for cut in (48, 48 * 17, 48 * 59):
        st = None
        parts = []
        for a, b in ((0, cut), (cut, x.shape[0])):
            r = otq.tx_ssb_q15(port, prm(0), x[a:b], st); st = r[3]; parts.append(r)
        for j in range(3):
            assert np.array_equal(np.concatenate([p_[j] for p_ in parts]), whole[j]), (cut, j)


def test_alc_bounds(port):
    """The envelope is never below the block's own peak, so no output sample exceeds the target (arm_scale_q15 truncates and the gain
    word rounds down: its saturation cannot be reached). On a quiet channel the gain limit, and with a high limit the floor, set q."""
    p = prm(0)
    x = mg.full_scale_mic(48 * 100)
    y, iq, gain, _ = otq.tx_ssb_q15(port, prm(0, taps_i=mg.hot_taps(p["taps_i"]), taps_q=mg.hot_taps(p["taps_q"])), x)
    assert np.abs(y.astype(np.int32)).max() <= p["agc_target"]
    assert np.sum(iq == -32768) > 0                                        # arm_abs_q15 (-32768) = 32767 is on the path
    x = slb.synth_mic(1, 48 * 100)[0]
    y, _, _, _ = otq.tx_ssb_q15(port, p, x)
    assert np.abs(y.astype(np.int32)).max() <= p["agc_target"]
    quiet = np.zeros((48 * 40, 2), np.int16); quiet[:, 0] = np.arange(48 * 40) % 3 - 1; quiet[:, 1] = 17
    _, _, gain, _ = otq.tx_ssb_q15(port, p, quiet)
    assert np.all(gain == p["agc_gmax_q15"])
    _, _, gain, _ = otq.tx_ssb_q15(port, prm(0, agc_gmax_q15=255 << 15, agc_floor=200), quiet)
    assert np.all(gain == (p["agc_target"] << 15) // 200)


def test_golden_file_regenerates_bit_for_bit(port):
    g = np.load(os.path.join(GOLD, "tx_ssb_q15.npz"))
    v = mg.vectors(port)
    assert sorted(g.files) == sorted(v)
    for k in v:
        assert g[k].dtype == v[k].dtype and np.array_equal(g[k], v[k]), k


def test_golden_vectors_cover_saturation():
    g = np.load(os.path.join(GOLD, "tx_ssb_q15.npz"))
    assert np.sum(np.abs(g["sat_iq"].astype(np.int32)) >= 32767) > 100 and np.sum(g["sat_iq"] == -32768) > 0
    assert np.array_equal(g["usb_iq"][:, ::-1], g["lsb_iq"])


def test_q15_tx_operand_planes_equal_arm_fir_q15_of_l(port, rng):
    """sl_rx_q15_tc.cu, TX planes: both rails take their taps at the L bytes of the window, so slb_design_q15_tc_tx_block gives
    arm_fir_q15 of L with taps_i (rail fi) and taps_q (rail fq) bit for bit — random, rail-to-rail and L != R windows — and R changes
    nothing."""
    lib = _lib.load()

    def tx_block(ti, tq, w):
        out = np.zeros(96, np.int32)
        assert lib.slb_design_q15_tc_tx_block(ti.ctypes.data, tq.ctypes.data, np.ascontiguousarray(w).ctypes.data, out.ctypes.data) == 0
        return out

    def fir64(taps, x):
        # exact int64 arm_fir_q15: acc = sum b[k] x[n-k], (acc >> 15) saturated to 16 bits
        x = x.astype(np.int64); t = taps.astype(np.int64)
        acc = np.array([np.sum(t * x[64 + n - np.arange(64)]) for n in range(48)])
        return np.clip(acc >> 15, -32768, 32767)

    for trial in range(6):
        ti = rng.integers(-32639, 32640, 64).astype(np.int16); tq = rng.integers(-32639, 32640, 64).astype(np.int16)
        if trial == 0:
            p = slb.default_rx_q15_params(FS); ti = np.array(p.taps_i[:64], np.int16); tq = np.array(p.taps_q[:64], np.int16)
        w = rng.integers(-32768, 32768, (112, 2)).astype(np.int16)            # L != R
        if trial == 2:
            w[:, 0] = np.where(np.arange(112) % 2 == 0, 32767, -32768)         # rail to rail
        if trial == 3:
            w[:, 0] = 32767; ti[:] = 32639; tq[:] = -32639                     # both rails saturate
        if trial == 4:
            w[:, 1] = w[:, 0]                                                  # L = R as the codec delivers it
        out = tx_block(ti, tq, w)
        assert np.array_equal(out[:48], fir64(ti, w[:, 0])), trial
        assert np.array_equal(out[48:], fir64(tq, w[:, 0])), trial
        y, _ = port.fir_q15(np.ascontiguousarray(ti[::-1]), np.zeros(64 + 16, np.int16), np.ascontiguousarray(w[:, 0]), 16)
        assert np.array_equal(out[:48], y[64:].astype(np.int32)), trial
        for r in (np.zeros(112, np.int16), np.full(112, -32768, np.int16), rng.integers(-32768, 32768, 112).astype(np.int16)):
            w2 = w.copy(); w2[:, 1] = r
            assert np.array_equal(tx_block(ti, tq, w2), out), trial
    bad = np.zeros(64, np.int16); bad[5] = 32640
    assert lib.slb_design_q15_tc_tx_block(bad.ctypes.data, bad.ctypes.data, np.zeros((112, 2), np.int16).ctypes.data, np.zeros(96, np.int32).ctypes.data) != 0
