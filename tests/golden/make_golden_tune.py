"""Writes tests/golden/tune_f32.npz: the per-channel tuner (DESIGN.md §3.5) of the f32 RX and TX chains on one I/Q channel.
python tests/golden/make_golden_tune.py
Written by the port (oracle/port): the reference firmware has no tuner, and every stage the tuner is composed of is one the port
already restates and the other tests hold to the reference. Needs no reference tree; the other golden files are left untouched.

Contents: the tuner alone (RX and TX direction) at offsets 0, +-small, negative and near +-fs/2; two calls with a retune between
them, the phase carried; an RX-SSB-f32 chain (USB) behind the RX tuner and a TX-SSB-f32 chain (USB) in front of the TX tuner."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib  # noqa: E402
import oracle_tune as otu  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402
from selenite_lite_b200.dsp_if import params_to_dict, tx_params_to_dict  # noqa: E402

FS = 48000
OFFSETS_HZ = np.array([0.0, 37.5, -1234.5, 7300.0, -23999.9, 23999.9], np.float64)
RETUNE_HZ = (1500.0, -2750.25)
T = 4 * 384


def compute(port):
    x = slb.synth_iq(1, T, f0=7300.0 + 1000.0, amp=0.45)[0]
    out = {"fs": np.array([FS], np.uint32), "offsets_hz": OFFSETS_HZ, "x": x}
    incs = np.array([otu.increment(f, FS) for f in OFFSETS_HZ], np.int32)
    out["incs"] = incs
    out["rx"] = np.stack([otu.tune_q15(port, x, int(i), 0, False)[0] for i in incs])
    out["tx"] = np.stack([otu.tune_q15(port, x, int(i), 0, True)[0] for i in incs])
    # two calls, retuned between them: the second call starts from the phase the first left
    a, b = (otu.increment(f, FS) for f in RETUNE_HZ)
    y1, ph = otu.tune_q15(port, x[:1000], a, 0, False)
    y2, ph = otu.tune_q15(port, x[1000:], b, ph, False)
    out["retune_incs"] = np.array([a, b], np.int32); out["retune_rx"] = np.concatenate([y1, y2]); out["retune_phase"] = np.array([ph], np.uint32)
    # chains: RX-SSB-f32 (USB) on the RX-tuned input, TX-SSB-f32 (USB) then the TX tuner
    inc = otu.increment(7300.0, FS)
    rx_prm = params_to_dict(slb.default_rx_f32_params(FS), slb.default_mask(FS, 512, slb.MODE_USB))
    out["rx_ssb_out"] = port.rx_ssb_f32(rx_prm, otu.tune_q15(port, x, inc, 0, False)[0])[0]
    mic = slb.synth_mic(1, T)[0]
    tx_prm = tx_params_to_dict(slb.default_tx_f32_params(FS), slb.default_mask(FS, 512, slb.MODE_USB))
    out["mic"] = mic
    out["tx_ssb_out"] = otu.tune_q15(port, port.tx_ssb_f32(tx_prm, mic)[0], inc, 0, True)[0]
    out["chain_inc"] = np.array([inc], np.int32)
    return out


def main():
    oracle_lib.build_oracles(want_ref=False)
    out = compute(oracle_lib.Oracle("port"))
    path = os.path.join(HERE, "tune_f32.npz")
    np.savez_compressed(path, **out)
    print("tune_f32.npz", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
