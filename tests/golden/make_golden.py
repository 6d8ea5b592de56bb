"""Generates tests/golden/*.npz by RUNNING THE REFERENCE here (oracle/_ref = /root/reference's CMSIS-DSP V1.5.3 and
dsp_if.c compiled for x86). The reference owns no golden vectors (SURVEY.md §4), so these are its outputs on frozen
seeded inputs. Re-run only in a container where /root/reference is mounted:  python tests/golden/make_golden.py
Chain parameters come from the product's frozen default design (pure data: slb_default_*), inputs from
selenite_lite_b200.signals (SURVEY.md §8d)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402
from selenite_lite_b200.dsp_if import params_to_dict  # noqa: E402


def golden_q15(ref):
    """RX-SSB-q15 (all-integer chain): tone + noise on the wanted sideband, USB and LSB, and a full-scale random input
    that drives every saturation point (FIR __SSAT, arm_add_q15, arm_abs_q15 of -32768, arm_scale_q15)."""
    qp = slb.default_rx_q15_params(48000)
    q = {"q15_taps_i": np.array(qp.taps_i[:], np.int16), "q15_taps_q": np.array(qp.taps_q[:], np.int16), "q15_rel": np.array(qp.rel[:], np.int16),
         "q15_agc": np.array([qp.agc_window, qp.agc_target, qp.agc_floor, qp.agc_gmax_q15], np.int64)}
    rng = np.random.Generator(np.random.PCG64(slb.signals.SEED + 15))
    for name, lsb, f0, sb in (("usb", 0, 1000.0, +1), ("lsb", 1, 1700.0, -1)):
        x = slb.synth_iq(1, 20 * 384, f0=f0, sideband=sb)[0]
        y, audio, gain, _ = ref.rx_ssb_q15(slb.dsp_if.q15_params_to_dict(qp, lsb), x)
        q["q15_%s_in" % name] = x; q["q15_%s_out" % name] = y; q["q15_%s_audio" % name] = audio; q["q15_%s_gain" % name] = gain
    x = rng.integers(-32768, 32768, (10 * 384, 2)).astype(np.int16)
    x[100:164] = -32768; x[500:564, 0] = 32767; x[500:564, 1] = -32768
    y, audio, gain, _ = ref.rx_ssb_q15(slb.dsp_if.q15_params_to_dict(qp, 0), x)
    q["q15_sat_in"] = x; q["q15_sat_out"] = y; q["q15_sat_audio"] = audio; q["q15_sat_gain"] = gain
    np.savez_compressed(os.path.join(HERE, "rx_ssb_q15.npz"), **q)
    print("rx_ssb_q15.npz", os.path.getsize(os.path.join(HERE, "rx_ssb_q15.npz")), "bytes")


def golden_fm(ref):
    """RX-SSB-f32 chain with the FM detector (mode byte 0x08): a carrier frequency-modulated by a 1 kHz tone, +-2.5 kHz deviation,
    once centred and once 1.5 kHz off the channel centre (a constant offset in the discriminator output), 20 hops each."""
    p = slb.default_rx_f32_params(48000)
    mask = slb.default_mask(48000, p.fft_len, slb.MODE_FM)
    out = {"fm_mask": mask, "fm_biquad": np.array(p.biquad[:10], np.float32), "fm_agc": np.array([p.agc_target, p.agc_decay, p.agc_floor, p.agc_gmax], np.float32)}
    for name, fc in (("centre", 0.0), ("offset", 1500.0)):
        x = slb.synth_fm(1, 20 * 384, carrier_hz=fc)[0]
        prm = params_to_dict(p, mask); prm["envelope"] = 2
        y, audio, gain, _ = ref.rx_ssb_f32(prm, x)
        out["fm_%s_in" % name] = x; out["fm_%s_out" % name] = y; out["fm_%s_audio" % name] = audio; out["fm_%s_gain" % name] = gain
    np.savez_compressed(os.path.join(HERE, "rx_fm_f32.npz"), **out)
    print("rx_fm_f32.npz", os.path.getsize(os.path.join(HERE, "rx_fm_f32.npz")), "bytes")


def golden_fft_fixed(ref):
    """arm_cfft_q15 (in the ARM_MATH_DSP branch of the firmware's ARM_MATH_CM4 build: oracle/ref_glue/cm4_fft_q15.c) and arm_cfft_q31
    of the reference build on frozen inputs: N = 64 (4^3), 128 (2 * 4^3), 1024, 2048; forward and inverse; moderate and full-scale."""
    rng = np.random.Generator(np.random.PCG64(slb.signals.SEED + 0xFF7))
    out = {}
    for N in (16, 64, 128, 1024, 2048):
        for amp, tag in ((6000, "m"), (32767, "f")):
            x15 = rng.integers(-amp, amp + 1, 2 * N).astype(np.int16)
            x31 = rng.integers(-(amp << 16), (amp << 16) + 1, 2 * N).astype(np.int32)
            out["q15_%d_%s_in" % (N, tag)] = x15; out["q31_%d_%s_in" % (N, tag)] = x31
            for ifft in (0, 1):
                out["q15_%d_%s_%d" % (N, tag, ifft)] = ref.cfft_q15_cm4(x15, ifft)
                out["q31_%d_%s_%d" % (N, tag, ifft)] = ref.cfft_q31(x31, ifft)
    np.savez_compressed(os.path.join(HERE, "cfft_fixed.npz"), **out)
    print("cfft_fixed.npz", os.path.getsize(os.path.join(HERE, "cfft_fixed.npz")), "bytes")


def golden_pinning():
    """pinning.npz: what the oracle returns on the fixed inputs of the tests that compare the port with the reference
    (test_oracle_pinning.py, test_golden.py::test_am_chain_port_vs_ref), recorded by running those tests; the ref_or_recorded
    fixture replays it where the reference build is absent. Recorded from the reference build when it exists, else from the
    port (the file's `source` says which), whose agreement with the reference is what those same tests check."""
    import pytest
    tests = os.path.dirname(HERE)
    os.environ["SLB_RECORD_PINNING"] = os.path.join(HERE, "pinning.npz")
    rc = pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(tests, "test_oracle_pinning.py"),
                      os.path.join(tests, "test_golden.py") + "::test_am_chain_port_vs_ref"])
    print("pinning.npz", os.path.getsize(os.path.join(HERE, "pinning.npz")), "bytes, pytest rc", int(rc))


def main():
    oracle_lib.build_oracles()
    if len(sys.argv) > 1 and sys.argv[1] == "pinning":
        return golden_pinning()
    ref = oracle_lib.Oracle("ref")
    if len(sys.argv) > 1 and sys.argv[1] == "fft_fixed":
        return golden_fft_fixed(ref)
    if len(sys.argv) > 1 and sys.argv[1] == "q15":      # later additions regenerate alone: the older fixtures stay untouched
        return golden_q15(ref)
    if len(sys.argv) > 1 and sys.argv[1] == "fm":
        return golden_fm(ref)
    rng = np.random.Generator(np.random.PCG64(slb.signals.SEED))

    # ---- RX-SSB-f32, config-1 style: one channel, tone +1000 Hz + noise, 20 hops; and an LSB tone at -1700 Hz
    p = slb.default_rx_f32_params(48000)
    out = {}
    for name, mode, f0, sb in (("usb", slb.MODE_USB, 1000.0, +1), ("lsb", slb.MODE_LSB, 1700.0, -1)):
        mask = slb.default_mask(48000, p.fft_len, mode)
        x = slb.synth_iq(1, 20 * 384, f0=f0, sideband=sb)[0]
        y, audio, gain, _ = ref.rx_ssb_f32(params_to_dict(p, mask), x)
        out["rx_%s_in" % name] = x; out["rx_%s_out" % name] = y; out["rx_%s_audio" % name] = audio; out["rx_%s_gain" % name] = gain
        out["rx_%s_mask" % name] = mask
    out["rx_biquad"] = np.array(p.biquad[:10], np.float32)
    out["rx_agc"] = np.array([p.agc_target, p.agc_decay, p.agc_floor, p.agc_gmax], np.float32)
    np.savez_compressed(os.path.join(HERE, "rx_ssb_f32.npz"), **out)

    # ---- TX-SSB-f32, config-3 style: one mic channel (L = R), two-tone + noise, 20 hops, USB and LSB
    tp = slb.default_tx_f32_params(48000)
    tx = {}
    for name, mode in (("usb", slb.MODE_USB), ("lsb", slb.MODE_LSB)):
        mask = slb.default_mask(48000, tp.fft_len, mode)
        x = slb.synth_mic(1, 20 * 384)[0]
        y, iq, gain, _ = ref.tx_ssb_f32(slb.dsp_if.tx_params_to_dict(tp, mask), x)
        tx["tx_%s_in" % name] = x; tx["tx_%s_out" % name] = y; tx["tx_%s_iq" % name] = iq; tx["tx_%s_gain" % name] = gain
        tx["tx_%s_mask" % name] = mask
    tx["tx_alc"] = np.array([tp.alc_target, tp.alc_decay, tp.alc_floor, tp.alc_gmax], np.float32)
    np.savez_compressed(os.path.join(HERE, "tx_ssb_f32.npz"), **tx)

    # ---- CHAN-64-f32, config-4 style: one 192 kHz wideband stream, tones in a random half of the bins, 36 hops;
    #      product detector and envelope detector
    cp = slb.default_chan_params(192000)
    ch = {}
    xw = slb.synth_wideband(1, 768 * 3)[0]
    ch["chan_in"] = xw; ch["chan_proto"] = np.array(cp.proto[:512], np.float32)
    ch["chan_agc"] = np.array([cp.agc_target, cp.agc_decay, cp.agc_floor, cp.agc_gmax], np.float32)
    for name, envl in (("prod", 0), ("env", 1)):
        prm = slb.dsp_if.chan_params_to_dict(cp); prm["envelope"] = envl
        y, audio, gain, _ = ref.chan_f32(prm, xw)
        ch["chan_%s_out" % name] = y; ch["chan_%s_audio" % name] = audio; ch["chan_%s_gain" % name] = gain
    np.savez_compressed(os.path.join(HERE, "chan64_f32.npz"), **ch)

    # ---- the firmware ring (unmodified dsp_if.c): ramp through In_Buff_Write/In_Buff_Read and Out_Buff_Write/Out_Buff_Read
    ring = {}
    for fs in (48000, 96000):
        r = oracle_lib.RefRing(fs)
        nb = 40; hw = r.half_hw
        ramp = (np.arange(nb * hw // 2, dtype=np.int64) % 30000).astype(np.int16)
        blocks = np.stack([ramp, -ramp], 1).reshape(nb, hw)            # I = n, Q = -n
        rx_out, tx_out, ptrs = [], [], []
        for b in range(nb):
            r.in_write(blocks[b]); rx_out.append(r.in_read(hw * 2))
            r.out_write(blocks[b]); tx_out.append(r.out_read(hw))
            ptrs.append(r.ptrs(0) + r.ptrs(1))
        ring["in_%d" % fs] = blocks; ring["rx_%d" % fs] = np.stack(rx_out); ring["tx_%d" % fs] = np.stack(tx_out)
        ring["ptrs_%d" % fs] = np.array(ptrs, np.uint32)
    np.savez_compressed(os.path.join(HERE, "ring.npz"), **ring)

    # ---- stage known-answer vectors (integer stages: bit-exact pins)
    st = {}
    x15 = rng.integers(-32768, 32768, 48 * 6).astype(np.int16)
    c15 = rng.integers(-6000, 6000, 64).astype(np.int16)
    st["q15_x"] = x15; st["q15_c"] = c15
    st["fir_q15"] = ref.fir_q15(c15, np.zeros(64 + 48, np.int16), x15, 48)[0]
    st["fir_fast_q15"] = ref.fir_fast_q15(c15, np.zeros(64 + 48, np.int16), x15, 48)[0]
    bq15 = np.array([8000, 0, -16000, 8000, 15000, -7000, 4000, 0, 8000, 4000, 9000, -3000], np.int16)
    st["bq15_c"] = bq15
    st["biquad_df1_q15"] = ref.biquad_df1_q15(bq15, 2, 1, np.zeros(8, np.int16), x15, 48)[0]
    st["scale_q15"] = ref.scale_q15(x15, 23170, 1)
    st["cmplx_mag_q15"] = ref.cmplx_mag_q15(x15)
    xf = (rng.standard_normal(48 * 6) * 0.4).astype(np.float32)
    st["f32_x"] = xf
    st["float_to_q15"] = ref.float_to_q15(xf * 3)
    st["cfft_f32_512"] = ref.cfft_f32(rng.standard_normal(1024).astype(np.float32))
    st["cfft_in_512"] = np.random.Generator(np.random.PCG64(slb.signals.SEED)).standard_normal(1)  # placeholder, replaced below
    z = np.random.Generator(np.random.PCG64(7)).standard_normal(1024).astype(np.float32)
    st["cfft_in_512"] = z; st["cfft_f32_512"] = ref.cfft_f32(z); st["icfft_f32_512"] = ref.cfft_f32(z, 1, 1)
    cbq = np.array(p.biquad[:10], np.float32)
    st["biquad_df2T_f32"] = ref.biquad_df2T_f32(cbq, 2, np.zeros(4, np.float32), xf, 48)[0]
    np.savez_compressed(os.path.join(HERE, "stages.npz"), **st)
    golden_q15(ref)
    for f in ("rx_ssb_f32.npz", "tx_ssb_f32.npz", "chan64_f32.npz", "ring.npz", "stages.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")


if __name__ == "__main__":
    main()
