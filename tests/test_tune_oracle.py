"""The oracle of the per-channel tuner (oracle/slo_tune.h, DESIGN.md §3.5) on the CPU: the port's tune_q15 against a float64
rotation, exact continuation across calls, the sign convention (a tone at +f lands at 0 Hz after RX tuning by +f, TX tuning moves
0 Hz to +f), the rounding of the offset, and the committed golden vectors."""
import os
import sys

import numpy as np
import pytest

import oracle_tune as otu
import oracle_tx_mod as otm
import selenite_lite_b200 as slb
from selenite_lite_b200.dsp_if import params_to_dict, tx_params_to_dict
from test_golden import GOLD
from test_tx_am_fm_oracle import loopback_input

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden_tune  # noqa: E402

FS = 48000
LOOPBACK_HZ = 7300.0
# the SNR (dB) of a 0.3 FS 1 kHz mic tone, 40 hops, through port tx_ssb_f32 (USB) -> tune_q15 up by LOOPBACK_HZ -> tune_q15 down by
# LOOPBACK_HZ -> port rx_ssb_f32 (USB), measured on the int16 audio after 8 hops of settling by oracle_tx_mod.tone_snr_db
LOOPBACK_SNR_DB = 88.666


def rotate64(x, inc, phase0, up):
    """float64 reference: the same integer phase, an exact exponential, truncation and saturation of arm_float_to_q15."""
    n = np.arange(x.shape[0], dtype=np.uint64)
    phi = ((np.uint64(phase0) + n * np.uint64(inc & 0xFFFFFFFF)) & np.uint64(0xFFFFFFFF)).astype(np.uint32).view(np.int32)
    w = np.exp((1j if up else -1j) * np.pi * phi.astype(np.float64) / 2.0 ** 31)
    z = (x[:, 0].astype(np.float64) + 1j * x[:, 1]) * w
    q = lambda v: np.clip(np.trunc(v), -32768, 32767)
    return np.stack([q(z.real), q(z.imag)], 1)


def full_scale_noise(T, seed=3):
    return np.random.Generator(np.random.PCG64(seed)).integers(-32768, 32768, (T, 2)).astype(np.int16)


@pytest.mark.parametrize("hz", [0.0, 1.0, 37.5, -1234.5, 7300.0, -23999.9, 23999.9])
@pytest.mark.parametrize("up", [False, True])
def test_within_2_lsb_of_a_float64_rotation(port, hz, up):
    x = full_scale_noise(5000)
    inc = otu.increment(hz, FS)
    for phase0 in (0, 0x9E3779B9):
        y, ph = otu.tune_q15(port, x, inc, phase0, up)
        assert np.max(np.abs(y - rotate64(x, inc, phase0, up))) <= 2
        assert ph == (phase0 + x.shape[0] * inc) % 2 ** 32
    if hz == 0.0:
        assert np.array_equal(otu.tune_q15(port, x, 0, 0, up)[0], x)                # w = 1 exactly: the identity


def test_saturates_a_rotated_component_beyond_full_scale(port):
    x = np.tile(np.array([[32767, 32767], [-32768, -32768]], np.int16), (48, 1))   # |z| = sqrt(2) full scale
    y = otu.tune_q15(port, x, otu.increment(6000.0, FS), 0, True)[0]
    assert y.min() == -32768 and y.max() == 32767
    assert np.max(np.abs(y - rotate64(x, otu.increment(6000.0, FS), 0, True))) <= 2


@pytest.mark.parametrize("cut", [1, 383, 1000, 4095])
def test_one_call_equals_two_calls_with_the_phase_carried(port, cut):
    x = full_scale_noise(4096, seed=11)
    for inc, up in ((otu.increment(-1234.5, FS), False), (otu.increment(23999.9, FS), True), (-(2 ** 31 - 1), False)):
        y, ph = otu.tune_q15(port, x, inc, 7, up)
        y1, p1 = otu.tune_q15(port, x[:cut], inc, 7, up)
        y2, p2 = otu.tune_q15(port, x[cut:], inc, p1, up)
        assert np.array_equal(np.concatenate([y1, y2]), y) and p2 == ph


@pytest.mark.parametrize("f", [7300.0, -5100.0, 150.0])
def test_a_tone_at_f_lands_at_0_hz_and_tx_moves_0_hz_to_f(port, f):
    T = 4800
    n = np.arange(T)
    tone = np.stack([np.rint(16000 * np.cos(2 * np.pi * f * n / FS)), np.rint(16000 * np.sin(2 * np.pi * f * n / FS))], 1).astype(np.int16)
    y = otu.tune_q15(port, tone, otu.increment(f, FS), 0, False)[0].astype(np.float64)
    assert np.max(np.abs(y - y.mean(0))) <= 4                                        # DC: the rotation left only rounding
    assert np.max(np.abs(np.hypot(y[:, 0], y[:, 1]) - 16000)) <= 4
    dc = np.tile(np.array([[16000, 0]], np.int16), (T, 1))
    z = otu.tune_q15(port, dc, otu.increment(f, FS), 0, True)[0].astype(np.float64)
    spec = np.abs(np.fft.fft(z[:, 0] + 1j * z[:, 1]))
    assert abs(np.fft.fftfreq(T, 1.0 / FS)[np.argmax(spec)] - f) <= FS / T


def test_offset_rounding():
    assert otu.increment(12000.0, FS) == 2 ** 30 and otu.increment(-12000.0, FS) == -(2 ** 30)
    assert otu.increment(0.0, FS) == 0
    inc = otu.increment(7300.3, FS)
    assert abs(inc * FS / 2 ** 32 - 7300.3) <= 0.5 * FS / 2 ** 32


def test_golden_vectors_regenerate_exactly(port):
    g = np.load(os.path.join(GOLD, "tune_f32.npz"))
    fresh = make_golden_tune.compute(port)
    assert sorted(g.files) == sorted(fresh)
    for k in g.files:
        assert g[k].dtype == fresh[k].dtype and g[k].shape == fresh[k].shape and g[k].tobytes() == fresh[k].tobytes(), k


def oracle_loopback_audio(port, hz=LOOPBACK_HZ):
    inc = otu.increment(hz, FS)
    y = port.tx_ssb_f32(tx_params_to_dict(slb.default_tx_f32_params(FS), slb.default_mask(FS, 512, slb.MODE_USB)), loopback_input())[0]
    z = otu.tune_q15(port, otu.tune_q15(port, y, inc, 0, True)[0], inc, 0, False)[0]
    return port.rx_ssb_f32(params_to_dict(slb.default_rx_f32_params(FS), slb.default_mask(FS, 512, slb.MODE_USB)), z)[0]


def test_loopback_snr_through_the_oracle(port):
    snr = otm.tone_snr_db(oracle_loopback_audio(port)[384 * 8:, 0], FS, 1000.0)
    assert abs(snr - LOOPBACK_SNR_DB) < 0.01, snr
