"""Writes tests/golden/tx_q15.npz: the all-mode integer transmitter TX-Q15 (DESIGN.md §3.9) on one channel, 100 firmware blocks each,
with the default parameters: AM and FM on a 1 kHz mic tone at 0.3 full scale with speech-like bursts, an SSB channel (USB, the SSB test
mic) and a saturating case (FM with am_taps / fm_taps at their largest splittable value, fm_inc = 65535 and rail-to-rail squares, so the
FIR, the ALC and the phase accumulator all hit their limits). Output, the pre-ALC pair, the gain words and the phase after each sample.
    python tests/golden/make_golden_tx_q15_mod.py
Written by the port (oracle/port): every stage it calls is pinned bit-exact to the reference (tests/test_oracle_pinning.py); the gain
law and the phase accumulator are ours. Needs no reference tree; the other golden files are left untouched."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib  # noqa: E402
import oracle_tx_q15_mod as otq  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402
from selenite_lite_b200.dsp_if import tx_q15_mode_params_to_dict  # noqa: E402

FRAMES = 48 * 100
CASES = (("am", slb.MODE_AM), ("fm", slb.MODE_FM), ("usb", slb.MODE_USB), ("sat", slb.MODE_FM))


def case_input(name):
    """L = R mic frames int16 [FRAMES][2]"""
    n = np.arange(FRAMES)
    rng = np.random.Generator(np.random.PCG64(0x7A15))
    if name in ("am", "fm"):
        env = np.where((n // 1200) % 2 == 0, 1.0, 0.25)
        m = np.rint(0.3 * 32768 * env * np.cos(2 * np.pi * 1000 * n / 48000) + rng.normal(0, 100, FRAMES)).clip(-32768, 32767).astype(np.int16)
    elif name == "usb":
        return slb.synth_mic(1, FRAMES)[0]
    else:
        m = np.where(n % 24 < 12, 32767, -32768).astype(np.int16)
        m[2400:2880] = -32768; m[3000:3400] = 0
    return np.stack([m, m], 1)


def case_params(name, mode):
    prm = tx_q15_mode_params_to_dict(slb.default_rx_q15_params(48000), slb.default_tx_q15_mode_params(48000), mode)
    if name == "sat":
        prm["fm_taps"] = np.full(64, 32639, np.int16); prm["fm_inc"] = 65535; prm["fm_target"] = 32767
    return prm


def vectors(port):
    mp = slb.default_tx_q15_mode_params(48000)
    out = {"am_taps": np.array(mp.am_taps[:], np.int16), "fm_taps": np.array(mp.fm_taps[:], np.int16),
           "consts": np.array([mp.am_carrier, mp.am_depth, mp.fm_target, mp.fm_inc], np.int64), "fm_level": np.array(mp.fm_level, np.float32)}
    for name, mode in CASES:
        x = case_input(name)
        y, iq, gain, phase, _ = otq.tx_q15(port, case_params(name, mode), x)
        out["%s_in" % name] = x; out["%s_out" % name] = y; out["%s_iq" % name] = iq; out["%s_gain" % name] = gain; out["%s_phase" % name] = phase
    return out


def main():
    oracle_lib.build_oracles(want_ref=False)
    path = os.path.join(HERE, "tx_q15.npz")
    np.savez_compressed(path, **vectors(oracle_lib.Oracle("port")))
    print("tx_q15.npz", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
