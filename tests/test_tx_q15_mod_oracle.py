"""The oracle of the all-mode integer transmitter TX-Q15 (oracle/slo_tx_q15_mod.h, DESIGN.md §3.9) on the CPU: the SSB-style modes are
TX-SSB-q15, the AM envelope and the FM phase and envelope stay in their bounds, streaming and mode changes, the TX-Q15 -> RX-Q15
loopback, and the golden vectors."""
import ctypes
import os
import sys

import numpy as np
import pytest

import oracle_rx_q15 as orq
import oracle_tx_mod as otm
import oracle_tx_q15 as otx
import oracle_tx_q15_mod as otq
import selenite_lite_b200 as slb
from selenite_lite_b200.dsp_if import q15_mode_params_to_dict, tx_q15_mode_params_to_dict
from test_golden import GOLD

sys.path.insert(0, GOLD)
import make_golden_tx_q15_mod as mg  # noqa: E402

FS = 48000
SSB_MODES = (slb.MODE_LSB, slb.MODE_USB, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG, slb.MODE_PKT)
# measured on the port with the frozen defaults: the SNR of a 0.3 FS 1 kHz mic tone through port tx_q15 -> port rx_q15 in the same mode,
# as tests/test_rx_q15_oracle.py measures the TX-F32 -> RX-Q15 loopback
LOOPBACK_SNR_DB = {slb.MODE_AM: 72.780, slb.MODE_FM: 44.439}


def prm(mode, **over):
    d = tx_q15_mode_params_to_dict(slb.default_rx_q15_params(FS), slb.default_tx_q15_mode_params(FS), mode)
    d.update(over)
    return d


def mic(m):
    m = np.asarray(m, np.int16)
    return np.stack([m, m], 1)


def tone(T, amp=0.3, f=1000.0):
    return np.rint(amp * 32768 * np.cos(2 * np.pi * f * np.arange(T) / FS)).astype(np.int16)


def test_defaults():
    mp = slb.default_tx_q15_mode_params(FS)
    rx = slb.default_rx_q15_mode_params(FS)
    assert list(mp.am_taps) == list(rx.am_taps) and list(mp.fm_taps) == list(rx.am_taps)
    assert (mp.am_carrier, mp.am_depth, mp.fm_target, mp.fm_inc) == (16384, 26214, 8192, round(2500 * 2 ** 32 / 48000 / 8192))
    assert np.float32(mp.fm_level) == np.float32(0.5)


@pytest.mark.parametrize("mode", SSB_MODES)
def test_ssb_modes_are_tx_ssb_q15(port, mode):
    x = mic(np.concatenate([slb.synth_mic(1, 48 * 60)[0][:, 0], mg.case_input("sat")[:48 * 40, 0]]))
    d = prm(mode)
    y, iq, g, ph, _ = otq.tx_q15(port, d, x)
    e = otx.tx_ssb_q15(port, d, x)
    assert np.array_equal(y, e[0]) and np.array_equal(iq, e[1]) and np.array_equal(g, e[2])
    assert not ph.any()


def test_am_envelope_in_bounds(port):
    d = prm(slb.MODE_AM); c, dep = d["am_carrier"], d["am_depth"]
    n = 48 * 80
    rng = np.random.default_rng(3)
    for m in (tone(n), rng.integers(-32768, 32768, n), np.where(np.arange(n) % 24 < 12, 32767, -32768), np.full(n, -32768),
              np.where(np.arange(n) % 96 < 48, 32767, -32768)):
        y, iq, _, _, _ = otq.tx_q15(port, d, mic(m))
        assert not y[:, 1].any() and not iq[:, 1].any()
        I = y[:, 0].astype(np.int64)
        lo, hi = c - (c * dep >> 15) - 2, c + (c * dep >> 15) + 2                  # (two truncation LSBs: arm_scale_q15 twice)
        assert I.min() >= lo and I.max() <= hi, (I.min(), I.max(), lo, hi)
        assert I.max() < 32767 and I.min() > -32768                               # no saturation at the defaults


def test_fm_phase_and_envelope(port):
    d = prm(slb.MODE_FM)
    n = 48 * 80
    rng = np.random.default_rng(4)
    for m in (tone(n), rng.integers(-32768, 32768, n), np.where(np.arange(n) % 24 < 12, 32767, -32768)):
        y, iq, _, ph, st = otq.tx_q15(port, d, mic(m))
        inc = np.diff(np.concatenate([[0], ph]).astype(np.uint32)).view(np.int32).astype(np.int64)
        assert np.abs(inc).max() <= d["fm_target"] * abs(d["fm_inc"])
        assert np.array_equal(otm.tx_fm_nco(port, ph, d["fm_level"]), y)
        assert st.phase == ph[-1]
        r = np.hypot(y[:, 0].astype(np.float64), y[:, 1].astype(np.float64))
        assert np.abs(r - d["fm_level"] * 32768).max() < 4                        # the table NCO's interpolation and truncation
    # a positive mic step moves the carrier up: the phase advances
    _, _, _, ph, _ = otq.tx_q15(port, d, mic(np.full(48 * 4, 8000)))
    assert np.all(np.diff(ph).astype(np.uint32).view(np.int32)[100:] > 0)


@pytest.mark.parametrize("mode", [slb.MODE_AM, slb.MODE_FM, slb.MODE_USB])
def test_one_call_equals_any_cut(port, mode):
    x = mg.case_input({slb.MODE_USB: "usb", slb.MODE_AM: "am", slb.MODE_FM: "fm"}[mode])
    whole = otq.tx_q15(port, prm(mode), x)
    for cuts in ((48,), (48 * 37,), (48, 48 * 16, 48 * 17, 48 * 64)):
        st = otq.TxQ15mState(); parts = []
        for a, b in zip((0,) + cuts, cuts + (len(x),)):
            parts.append(otq.tx_q15(port, prm(mode), x[a:b], st))
        for j in range(4):
            assert np.array_equal(np.concatenate([p[j] for p in parts]), whole[j]), (cuts, j)
        assert bytes(memoryview(st)) == bytes(memoryview(whole[4]))


def restore(dst, raw):
    ctypes.memmove(ctypes.addressof(dst), raw, len(raw))


def test_mode_changes_hold_the_phase_through_am(port):
    x = mg.case_input("fm")
    st = otq.TxQ15mState(); seg = 48 * 20; ph_end = None
    for i, mode in enumerate((slb.MODE_USB, slb.MODE_FM, slb.MODE_AM, slb.MODE_FM)):
        before = bytes(memoryview(st))
        y, _, _, ph, _ = otq.tx_q15(port, prm(mode), x[i * seg:(i + 1) * seg], st)
        if mode == slb.MODE_USB:
            assert st.phase == 0
        if mode == slb.MODE_AM:
            assert st.phase == ph_end and np.all(ph == ph_end) and not y[:, 1].any()
        if mode == slb.MODE_FM and ph_end is not None:
            # the second FM stretch continues from the held phase: the same stretch from the same state with the phase at zero, offset
            s0 = otq.TxQ15mState(); restore(s0, before); s0.phase = 0
            ref = otq.tx_q15(port, prm(mode), x[i * seg:(i + 1) * seg], s0)[3]
            assert np.array_equal((ref.astype(np.uint64) + ph_end) % 2 ** 32, ph.astype(np.uint64))
        ph_end = int(st.phase)
    assert ph_end != 0


@pytest.mark.parametrize("mode", [slb.MODE_AM, slb.MODE_FM])
def test_loopback_to_rx_q15(port, mode):
    T = 48 * 320
    y = otq.tx_q15(port, prm(mode), mic(tone(T)))[0]
    rp = q15_mode_params_to_dict(slb.default_rx_q15_params(FS), slb.default_rx_q15_mode_params(FS), mode)
    out = orq.rx_q15(port, rp, y)[0]
    snr = otm.tone_snr_db(out[48 * 64:, 0], FS, 1000.0)
    assert abs(snr - LOOPBACK_SNR_DB[mode]) < 0.01, snr


def test_golden_regenerates_bit_for_bit(port):
    g = np.load(os.path.join(GOLD, "tx_q15.npz"))
    v = mg.vectors(port)
    assert sorted(g.files) == sorted(v)
    for k in v:
        assert np.array_equal(g[k], v[k]), k
