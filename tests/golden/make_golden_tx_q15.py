"""Writes tests/golden/tx_ssb_q15.npz: the all-integer SSB modulator TX-SSB-q15 (DESIGN.md §3.7) on one mic channel (L = R), 100
firmware blocks each: USB and LSB with the default parameters on a two-tone + noise mic, and a saturating case (the default taps x 4,
clipped to the split range |tap| < 32640, on a full-scale mic). Output, pre-ALC (I, Q) after the rail order, and the gain words.
    python tests/golden/make_golden_tx_q15.py
Written by the port (oracle/port): the reference firmware has no modulator, and the port's fir_q15, abs_q15, max_q15 and scale_q15
are pinned bit-exact to the reference (tests/test_oracle_pinning.py). Needs no reference tree; the other golden files are left untouched."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib  # noqa: E402
import oracle_tx_q15 as otq  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402
from selenite_lite_b200.dsp_if import q15_params_to_dict  # noqa: E402

FRAMES = 48 * 100
CASES = (("usb", 0), ("lsb", 1), ("sat", 0))


def hot_taps(taps):
    return np.clip(4 * np.asarray(taps, np.int32), -32639, 32639).astype(np.int16)


def full_scale_mic(frames):
    rng = np.random.Generator(np.random.PCG64(0x7815))
    m = rng.integers(-32768, 32768, frames).astype(np.int16)
    m[480:960] = -32768; m[1440:1920] = 32767
    m[2400:2880] = np.where((np.arange(480) // 12) % 2 == 0, 32767, -32768)
    return np.stack([m, m], axis=1)


def case_params(name, lsb):
    prm = q15_params_to_dict(slb.default_rx_q15_params(48000), lsb=lsb)
    if name == "sat":
        prm["taps_i"] = hot_taps(prm["taps_i"]); prm["taps_q"] = hot_taps(prm["taps_q"])
    return prm


def vectors(port):
    p = slb.default_rx_q15_params(48000)
    out = {"taps_i": np.array(p.taps_i[:], np.int16), "taps_q": np.array(p.taps_q[:], np.int16), "rel": np.array(p.rel[:], np.int16),
           "agc": np.array([p.agc_window, p.agc_target, p.agc_floor, p.agc_gmax_q15], np.int64)}
    for name, lsb in CASES:
        x = full_scale_mic(FRAMES) if name == "sat" else slb.synth_mic(1, FRAMES)[0]
        y, iq, gain, _ = otq.tx_ssb_q15(port, case_params(name, lsb), x)
        out["%s_in" % name] = x; out["%s_out" % name] = y; out["%s_iq" % name] = iq; out["%s_gain" % name] = gain
    return out


def main():
    oracle_lib.build_oracles(want_ref=False)
    path = os.path.join(HERE, "tx_ssb_q15.npz")
    np.savez_compressed(path, **vectors(oracle_lib.Oracle("port")))
    print("tx_ssb_q15.npz", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
