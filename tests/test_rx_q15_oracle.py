"""The oracle of the all-mode integer receiver RX-Q15 (oracle/slo_rx_q15.h, DESIGN.md §3.8) and the host halves of its kernel on the CPU:
the FM planes and the AM planes against an int64 arm_fir_q15, the frozen AM / FM low-passes, the quality of both detectors, the
TX-F32 -> RX-Q15 loopback, streaming, and the golden vectors."""
import os
import sys

import numpy as np
import pytest

import oracle_rx_q15 as orq
import oracle_tx_mod as otm
import selenite_lite_b200 as slb
from selenite_lite_b200 import _lib
from selenite_lite_b200.dsp_if import q15_mode_params_to_dict, tx_mod_params_to_dict
from test_golden import GOLD

sys.path.insert(0, GOLD)
import make_golden_rx_q15 as mg  # noqa: E402

FS = 48000
# measured on the port with the frozen defaults (tests below): the FM discriminator's largest distance from 2^15 sin(dphi) over
# tones of -4.8 .. 4.8 kHz at amplitudes 3000 .. 32000; the AM detector's SNR of a 1 kHz tone at 50 % depth with the carrier 1 kHz off;
# the loopback SNR of a 0.3 FS 1 kHz mic tone through port tx_mod_f32 -> port rx_q15, as tests/test_tx_am_fm_oracle.py measures it
FM_BOUND_LSB = 280
AM_OFFSET_SNR_DB = 79.567
LOOPBACK_SNR_DB = {slb.MODE_AM: 78.262, slb.MODE_FM: 44.523}


def prm(mode, **over):
    d = q15_mode_params_to_dict(slb.default_rx_q15_params(FS), slb.default_rx_q15_mode_params(FS), mode)
    d.update(over)
    return d


def iq(z):
    return np.stack([np.rint(z.real), np.rint(z.imag)], 1).clip(-32768, 32767).astype(np.int16)


def fir64(taps, x, n0):
    """exact int64 arm_fir_q15 of window x (112 samples, 64 before the block) at block samples n0 .. 47"""
    x = x.astype(np.int64); t = np.asarray(taps, np.int64)
    acc = np.array([np.sum(t * x[64 + n - np.arange(64)]) for n in range(n0, 48)])
    return np.clip(acc >> 15, -32768, 32767)


def windows(rng):
    yield rng.integers(-32768, 32768, (112, 2)).astype(np.int16)
    yield np.where(rng.random((112, 2)) < 0.5, 32767, -32768).astype(np.int16)
    yield np.full((112, 2), -32768, np.int16)


def test_fm_and_am_planes_equal_int64_fir(rng):
    lib = _lib.load()
    mp = slb.default_rx_q15_mode_params(FS)
    sets = [(np.array(mp.fm_taps[:], np.int16), np.array(mp.am_taps[:], np.int16))]
    sets += [(rng.integers(-32639, 32640, 64).astype(np.int16), rng.integers(-32768, 32640, 64).astype(np.int16)) for _ in range(3)]
    for fm, am in sets:
        for w in windows(rng):
            out = np.zeros(98, np.int32)
            assert lib.slb_design_q15_tc_fm_block(fm.ctypes.data, np.ascontiguousarray(w).ctypes.data, out.ctypes.data) == 0
            assert np.array_equal(out[:49], fir64(fm, w[:, 0], -1)) and np.array_equal(out[49:], fir64(fm, w[:, 1], -1))
            out = np.zeros(96, np.int32)
            assert lib.slb_design_q15_tc_block(am.ctypes.data, am.ctypes.data, np.ascontiguousarray(w).ctypes.data, out.ctypes.data) == 0
            assert np.array_equal(out[:48], fir64(am, w[:, 0], 0)) and np.array_equal(out[48:], fir64(am, w[:, 1], 0))
    bad = np.zeros(64, np.int16); bad[5] = 32640
    assert lib.slb_design_q15_tc_fm_block(bad.ctypes.data, np.zeros((112, 2), np.int16).ctypes.data, np.zeros(98, np.int32).ctypes.data) != 0


def test_default_taps():
    """Both low-passes split into two signed bytes, have DC gain 1 and -6 dB at their cut-off; pass- and stop-band as measured."""
    mp = slb.default_rx_q15_mode_params(FS)
    assert mp.fm_floor == 1 << 18

    def H(t, f):
        return abs(np.sum(np.asarray(t, np.float64) / 32768 * np.exp(-2j * np.pi * f / FS * np.arange(64))))
    for taps, fc, pass_min, stop_db in ((mp.am_taps, 3000.0, 0.8637, -70.42), (mp.fm_taps, 6000.0, 0.9907, -74.83)):
        t = np.array(taps[:], np.int32)
        hl = ((t + 128) & 255) - 128; hh = (t - hl) >> 8
        assert np.all((hh >= -128) & (hh <= 127)) and np.all(t < 32640)
        assert abs(H(t, 0.0) - 1.0) < 2e-4 and abs(20 * np.log10(H(t, fc)) + 6.02) < 0.02
        assert min(H(t, f) for f in np.arange(0, 0.8 * fc, 50)) >= pass_min
        assert 20 * np.log10(max(H(t, f) for f in np.arange(2 * fc, FS / 2, 25))) <= stop_db


def test_fm_discriminator_quality_and_sign(port):
    n = np.arange(48 * 60)
    worst = 0.0
    for f in np.arange(-4800, 4801, 400):
        for A in (3000, 12000, 32000):
            _, a, _, _ = orq.rx_q15(port, prm(slb.MODE_FM), iq(A * np.exp(2j * np.pi * f * n / FS + 0.3j)))
            exp = 32768 * np.sin(2 * np.pi * f / FS)
            worst = max(worst, float(np.max(np.abs(a[200:].astype(np.float64) - exp))))
            if f != 0:
                assert np.all(np.sign(a[200:]) == np.sign(f))          # Im (z[n] conj z[n-1]): a tone above the centre reads positive
    assert worst <= FM_BOUND_LSB, worst
    # below the floor the output is squelched towards zero
    _, a, _, _ = orq.rx_q15(port, prm(slb.MODE_FM), iq(300 * np.exp(2j * np.pi * 2000 * n / FS)))
    assert np.max(np.abs(a[200:])) < 0.2 * 32768 * np.sin(2 * np.pi * 2000 / FS)


def test_am_recovers_a_tone(port):
    """1 kHz at 50 % depth: the tone comes out at |z| / 2 x 0.5 whatever the carrier phase; SNR with the carrier 1 kHz off as measured."""
    n = np.arange(48 * 60)
    amps = []
    for ph in (0.0, 1.0, 2.5):
        _, a, _, _ = orq.rx_q15(port, prm(slb.MODE_AM), iq(9000 * (1 + 0.5 * np.cos(2 * np.pi * 1000 * n / FS)) * np.exp(1j * ph)))
        s = a[480:].astype(np.float64)
        amps.append(2 * abs(np.mean((s - s.mean()) * np.exp(-2j * np.pi * 1000 * n[480:] / FS))))
        assert abs(s.mean() - 4500) < 8                                    # the carrier's DC stays in the audio (2.14: 9000 / 2)
    assert max(amps) - min(amps) < 4 and abs(np.mean(amps) - 2250) < 40, amps
    for off in (1000, -1000):
        _, a, _, _ = orq.rx_q15(port, prm(slb.MODE_AM), iq(9000 * (1 + 0.5 * np.cos(2 * np.pi * 1000 * n / FS)) * np.exp(2j * np.pi * off * n / FS)))
        s = a[480:]
        snr = otm.tone_snr_db((s - int(np.mean(s))).astype(np.int16), FS, 1000.0)
        assert abs(snr - AM_OFFSET_SNR_DB) < 0.01, (off, snr)


@pytest.mark.parametrize("mode", [slb.MODE_AM, slb.MODE_FM])
def test_loopback_from_tx_f32(port, mode):
    tp = slb.default_tx_f32_params(FS); mq = slb.default_tx_mod_params(FS)
    T = 384 * 40
    m = np.rint(0.3 * 32768 * np.cos(2 * np.pi * 1000 * np.arange(T) / FS)).astype(np.int16)
    y = otm.tx_mod_f32(port, tx_mod_params_to_dict(tp, mq, slb.default_mask(FS, tp.fft_len, mode), FS, mode), np.stack([m, m], 1))[0]
    out = orq.rx_q15(port, prm(mode), y)[0]
    snr = otm.tone_snr_db(out[384 * 8:, 0], FS, 1000.0)
    assert abs(snr - LOOPBACK_SNR_DB[mode]) < 0.01, snr


@pytest.mark.parametrize("mode", [slb.MODE_USB, slb.MODE_AM, slb.MODE_FM])
def test_one_call_equals_two(port, mode):
    x = mg.case_input({slb.MODE_USB: "usb", slb.MODE_AM: "am", slb.MODE_FM: "fm"}[mode])
    whole = orq.rx_q15(port, prm(mode), x)
    for cut in (48, 48 * 37):
        st = orq.RxQ15mState()
        a = orq.rx_q15(port, prm(mode), x[:cut], st); b = orq.rx_q15(port, prm(mode), x[cut:], st)
        for j in range(3):
            assert np.array_equal(np.concatenate([a[j], b[j]]), whole[j]), (cut, j)
    assert orq.state_bytes(st) == orq.state_bytes(whole[3])


def test_ssb_kind_is_rx_ssb_q15(port):
    x = mg.case_input("usb")
    for mode in (slb.MODE_USB, slb.MODE_LSB):
        d = prm(mode)
        y, a, g, _ = orq.rx_q15(port, d, x)
        e = port.rx_ssb_q15(d, x)
        assert np.array_equal(y, e[0]) and np.array_equal(a, e[1]) and np.array_equal(g, e[2])


def test_golden_regenerates_bit_for_bit(port):
    g = np.load(os.path.join(GOLD, "rx_q15.npz"))
    v = mg.vectors(port)
    assert sorted(g.files) == sorted(v)
    for k in v:
        assert np.array_equal(g[k], v[k]), k
