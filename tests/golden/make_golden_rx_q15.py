"""Writes tests/golden/rx_q15.npz: the all-mode integer receiver RX-Q15 (DESIGN.md §3.8) on one channel, 100 firmware blocks each, with
the default parameters: AM (a 1 kHz tone at 50 % depth on a carrier 300 Hz off the channel centre), FM (a 1 kHz tone at 2.5 kHz
deviation), an SSB channel (USB, the SSB test signal) and a saturating case (FM with fm_floor = 1 on rail-to-rail squares and a
full-scale carrier stepping a quarter turn per sample, so the FIRs, the magnitude and the discriminator all hit their limits). Output,
pre-AGC detector output and the gain words.
    python tests/golden/make_golden_rx_q15.py
Written by the port (oracle/port): every stage it calls is pinned bit-exact to the reference (tests/test_oracle_pinning.py); the
discriminator and the gain law are ours. Needs no reference tree; the other golden files are left untouched."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib  # noqa: E402
import oracle_rx_q15 as orq  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402
from selenite_lite_b200.dsp_if import q15_mode_params_to_dict  # noqa: E402

FRAMES = 48 * 100
CASES = (("am", slb.MODE_AM), ("fm", slb.MODE_FM), ("usb", slb.MODE_USB), ("sat", slb.MODE_FM))


def iq(z):
    return np.stack([np.rint(z.real), np.rint(z.imag)], 1).clip(-32768, 32767).astype(np.int16)


def case_input(name):
    n = np.arange(FRAMES)
    rng = np.random.Generator(np.random.PCG64(0x1A0F))
    noise = rng.normal(0, 200, FRAMES) + 1j * rng.normal(0, 200, FRAMES)
    if name == "am":
        return iq(9000.0 * (1 + 0.5 * np.cos(2 * np.pi * 1000 * n / 48000)) * np.exp(2j * np.pi * 300 * n / 48000) + noise)
    if name == "fm":
        return iq(12000.0 * np.exp(2.5j * np.sin(2 * np.pi * 1000 * n / 48000)) + noise)
    if name == "usb":
        return slb.synth_iq(1, FRAMES)[0]
    x = iq(32767.0 * np.exp(0.5j * np.pi * (n % 4)))
    sq = np.where(np.arange(FRAMES) % 24 < 12, 32767, -32768).astype(np.int16)
    x[960:1920, 0] = sq[960:1920]; x[960:1920, 1] = np.roll(sq, 6)[960:1920]
    x[2400:2880] = -32768; x[3000:3400] = 0
    return x


def case_params(name, mode):
    prm = q15_mode_params_to_dict(slb.default_rx_q15_params(48000), slb.default_rx_q15_mode_params(48000), mode)
    if name == "sat":
        prm["fm_floor"] = 1
    return prm


def vectors(port):
    mp = slb.default_rx_q15_mode_params(48000)
    out = {"am_taps": np.array(mp.am_taps[:], np.int16), "fm_taps": np.array(mp.fm_taps[:], np.int16), "fm_floor": np.array(mp.fm_floor, np.int64)}
    for name, mode in CASES:
        x = case_input(name)
        y, a, gain, _ = orq.rx_q15(port, case_params(name, mode), x)
        out["%s_in" % name] = x; out["%s_out" % name] = y; out["%s_audio" % name] = a; out["%s_gain" % name] = gain
    return out


def main():
    oracle_lib.build_oracles(want_ref=False)
    path = os.path.join(HERE, "rx_q15.npz")
    np.savez_compressed(path, **vectors(oracle_lib.Oracle("port")))
    print("rx_q15.npz", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
