"""Writes tests/golden/chan64_q15.npz: the integer channelizer CHAN-64-q15 (DESIGN.md §3.10) on one 192 kHz wideband stream of 32 ms
(6144 frames = 96 hops) with the default parameters, three cases: `product` (the config-4 test stream, product detector), `envelope`
(the same stream, envelope detector) and `rail` (rail-to-rail squares of different periods on the two rails, product detector: the
branch FIRs and the FFT at their limits). Output, pre-AGC detector output and the gain words.
    python tests/golden/make_golden_chan64_q15.py
Written by the port (oracle/port): every stage it calls is restated there and pinned bit-exact (the q15 FFT to the Cortex-M4 branch,
tests/test_chan64_q15_oracle.py); the gain law is ours. Needs no reference tree; the other golden files are left untouched."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_chan_q15 as ocq  # noqa: E402
import oracle_lib  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402
from selenite_lite_b200.dsp_if import chan_q15_params_to_dict  # noqa: E402

FRAMES = 6144
CASES = (("product", 0), ("envelope", 1), ("rail", 0))


def case_input(name):
    if name != "rail":
        return slb.synth_wideband(1, FRAMES)[0]
    n = np.arange(FRAMES)
    return np.stack([np.where(n % 128 < 64, 32767, -32768), np.where(n % 40 < 20, -32768, 32767)], 1).astype(np.int16)


def case_params(envelope):
    prm = chan_q15_params_to_dict(slb.default_chan_q15_params(192000))
    prm["envelope"] = envelope
    return prm


def vectors(port):
    out = {"proto": case_params(0)["proto"]}
    for name, env in CASES:
        x = case_input(name)
        y, a, gain, _ = ocq.chan_q15(port, case_params(env), x)
        out["%s_in" % name] = x; out["%s_out" % name] = y; out["%s_audio" % name] = a; out["%s_gain" % name] = gain
    return out


def main():
    oracle_lib.build_oracles(want_ref=False)
    path = os.path.join(HERE, "chan64_q15.npz")
    np.savez_compressed(path, **vectors(oracle_lib.Oracle("port")))
    print("chan64_q15.npz", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
