"""Writes tests/golden/tx_am_fm_f32.npz: the AM and FM transmit modulators of the all-mode TX chain (DESIGN.md §3.4) with the
default modulator constants on one mic channel (L = R), two-tone + noise, 20 hops.  python tests/golden/make_golden_tx_am_fm.py
Written by the port (oracle/port): the reference firmware has no modulator, and the three stages the port adds for it are checked
against the reference's own CMSIS-DSP routines where that build exists (tests/test_tx_am_fm_oracle.py). Needs no reference tree;
the other golden files (make_golden.py) are left untouched."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib  # noqa: E402
import oracle_tx_mod as otm  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402


def main():
    oracle_lib.build_oracles(want_ref=False)
    port = oracle_lib.Oracle("port")
    tp = slb.default_tx_f32_params(48000); mp = slb.default_tx_mod_params(48000)
    out = {"alc": np.array([tp.alc_decay, tp.alc_floor, tp.alc_gmax], np.float32),
           "mod": np.array([mp.am_carrier, mp.am_depth, mp.fm_deviation_hz, mp.fm_level], np.float32)}
    for name, mode in (("am", slb.MODE_AM), ("fm", slb.MODE_FM)):
        mask = slb.default_mask(48000, tp.fft_len, mode)
        x = slb.synth_mic(1, 20 * 384)[0]
        y, iq, gain, phase, _ = otm.tx_mod_f32(port, slb.dsp_if.tx_mod_params_to_dict(tp, mp, mask, 48000, mode), x)
        out["%s_in" % name] = x; out["%s_out" % name] = y; out["%s_iq" % name] = iq; out["%s_gain" % name] = gain; out["%s_mask" % name] = mask
        if mode == slb.MODE_FM:
            out["fm_phase"] = phase
    path = os.path.join(HERE, "tx_am_fm_f32.npz")
    np.savez_compressed(path, **out)
    print("tx_am_fm_f32.npz", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
