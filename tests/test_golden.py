"""Oracle vs the committed golden vectors (outputs of the reference itself, tests/golden/make_golden.py).
Runs on the CPU; on a box without /root/reference this is what pins the port."""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rx_params(g, name):
    return dict(fft_len=512, hop=384, agc_block=48, biquad=g["rx_biquad"].reshape(2, 5), agc_target=g["rx_agc"][0],
                agc_decay=g["rx_agc"][1], agc_floor=g["rx_agc"][2], agc_gmax=g["rx_agc"][3], mask=g["rx_%s_mask" % name])


def audio_tolerance(ref_audio, block=int(os.environ.get("SLB_TOL_BLOCK", "384"))):
    """1e-5 relative per sample, made well-defined at zero crossings (SURVEY.md §7): 1e-5 * max(|ref[n]|, rms of ref over
    the 384-frame super-block holding n). The super-block is one overlap-save frame: float32 FFT rounding noise scales
    with the energy of the whole frame, so a quieter stretch inside a loud frame (filter start-up) cannot be held to
    1e-5 of its own local level by ANY float32 implementation — the reference against its own restatement included."""
    r = ref_audio.astype(np.float64).reshape(-1, block)
    rms = np.sqrt(np.mean(r ** 2, axis=1, keepdims=True))
    return (1e-5 * np.maximum(np.abs(r), rms)).reshape(-1)


@pytest.mark.parametrize("name", ["usb", "lsb"])
def test_port_chain_vs_golden(port, name):
    g = np.load(os.path.join(GOLD, "rx_ssb_f32.npz"))
    out, audio, gain, _ = port.rx_ssb_f32(rx_params(g, name), g["rx_%s_in" % name])
    assert np.all(np.abs(audio - g["rx_%s_audio" % name]) <= audio_tolerance(g["rx_%s_audio" % name]) + 1e-9)
    assert np.allclose(gain, g["rx_%s_gain" % name], rtol=1e-5)
    d = np.abs(out.astype(np.int32) - g["rx_%s_out" % name].astype(np.int32))
    assert d.max() <= 1 and np.mean(d > 0) < 0.02           # a 1e-7 float difference can flip the truncating pack by one LSB


@pytest.mark.parametrize("name", ["usb", "lsb"])
def test_ref_chain_reproduces_golden(ref, name):
    g = np.load(os.path.join(GOLD, "rx_ssb_f32.npz"))
    out, audio, gain, _ = ref.rx_ssb_f32(rx_params(g, name), g["rx_%s_in" % name])
    assert np.array_equal(out, g["rx_%s_out" % name]) and np.array_equal(audio, g["rx_%s_audio" % name])


def tx_params(g, name):
    return dict(fft_len=512, hop=384, alc_block=48, alc_target=g["tx_alc"][0], alc_decay=g["tx_alc"][1],
                alc_floor=g["tx_alc"][2], alc_gmax=g["tx_alc"][3], mask=g["tx_%s_mask" % name])


def iq_tolerance(ref_iq, block=384):
    """audio_tolerance for a complex stream [frames][2]: 1e-5 * max(|z[n]|, rms of |z| over the super-block)."""
    z = ref_iq.astype(np.float64); mag = np.hypot(z[:, 0], z[:, 1]).reshape(-1, block)
    rms = np.sqrt(np.mean(mag ** 2, axis=1, keepdims=True))
    return np.repeat((1e-5 * np.maximum(mag, rms)).reshape(-1, 1), 2, axis=1)


@pytest.mark.parametrize("name", ["usb", "lsb"])
def test_port_tx_chain_vs_golden(port, name):
    g = np.load(os.path.join(GOLD, "tx_ssb_f32.npz"))
    out, iq, gain, _ = port.tx_ssb_f32(tx_params(g, name), g["tx_%s_in" % name])
    assert np.all(np.abs(iq - g["tx_%s_iq" % name]) <= iq_tolerance(g["tx_%s_iq" % name]) + 1e-9)
    assert np.allclose(gain, g["tx_%s_gain" % name], rtol=1e-5)
    d = np.abs(out.astype(np.int32) - g["tx_%s_out" % name].astype(np.int32))
    assert d.max() <= 1 and np.mean(d > 0) < 0.02


@pytest.mark.parametrize("name", ["usb", "lsb"])
def test_ref_tx_chain_reproduces_golden(ref, name):
    g = np.load(os.path.join(GOLD, "tx_ssb_f32.npz"))
    out, iq, gain, _ = ref.tx_ssb_f32(tx_params(g, name), g["tx_%s_in" % name])
    assert np.array_equal(out, g["tx_%s_out" % name]) and np.array_equal(iq, g["tx_%s_iq" % name])


def test_tx_chain_is_a_single_sideband_modulator(port):
    """Domain property, independent of any implementation: a real two-tone through the USB chain comes out with its
    energy on the positive-frequency side only (opposite sideband suppressed by the mask's stop band), and LSB mirrors."""
    g = np.load(os.path.join(GOLD, "tx_ssb_f32.npz"))
    for name, sign in (("usb", +1), ("lsb", -1)):
        z = g["tx_%s_iq" % name].astype(np.float64); z = (z[:, 0] + 1j * z[:, 1])[1536:]
        spec = np.abs(np.fft.fft(z * np.hanning(z.size))) ** 2
        f = np.fft.fftfreq(z.size, 1 / 48000.0)
        wanted = spec[(sign * f > 250) & (sign * f < 2800)].sum(); other = spec[(sign * f < -250) & (sign * f > -2800)].sum()
        assert 10 * np.log10(wanted / other) > 60.0


def chan_params(g, envelope=0):
    return dict(bins=64, taps_per_branch=8, agc_block=3, envelope=envelope, agc_target=g["chan_agc"][0], agc_decay=g["chan_agc"][1],
                agc_floor=g["chan_agc"][2], agc_gmax=g["chan_agc"][3], proto=g["chan_proto"])


def chan_tolerance(ref_audio, window=12):
    """Channelizer audio [bins][hops]: 1e-5 * max(|ref|, rms over ALL bins of the same 12-hop (4 ms) window) - the
    64-point FFT mixes every branch into every bin, so its float32 rounding noise scales with the whole spectrum frame."""
    r = ref_audio.astype(np.float64)
    bins, hops = r.shape
    w = r.reshape(bins, hops // window, window)
    rms = np.sqrt(np.mean(w ** 2, axis=(0, 2), keepdims=True))
    return (1e-5 * np.maximum(np.abs(w), rms)).reshape(bins, hops)


@pytest.mark.parametrize("name,envelope", [("prod", 0), ("env", 1)])
def test_port_chan_chain_vs_golden(port, name, envelope):
    g = np.load(os.path.join(GOLD, "chan64_f32.npz"))
    out, audio, gain, _ = port.chan_f32(chan_params(g, envelope), g["chan_in"])
    assert np.all(np.abs(audio - g["chan_%s_audio" % name]) <= chan_tolerance(g["chan_%s_audio" % name]) + 1e-9)
    assert np.allclose(gain, g["chan_%s_gain" % name], rtol=2e-5)
    d = np.abs(out.astype(np.int32) - g["chan_%s_out" % name].astype(np.int32))
    assert d.max() <= 1 and np.mean(d > 0) < 0.02


@pytest.mark.parametrize("name,envelope", [("prod", 0), ("env", 1)])
def test_ref_chan_chain_reproduces_golden(ref, name, envelope):
    g = np.load(os.path.join(GOLD, "chan64_f32.npz"))
    out, audio, gain, _ = ref.chan_f32(chan_params(g, envelope), g["chan_in"])
    assert np.array_equal(out, g["chan_%s_out" % name]) and np.array_equal(audio, g["chan_%s_audio" % name])


def test_chan_chain_is_a_channelizer(port):
    """Domain property: a tone at bin-centre + 500 Hz appears in its own bin as a 500 Hz tone at the 3 kHz narrowband
    rate, and empty bins stay at the noise floor (> 20 dB below)."""
    import selenite_lite_b200 as slb
    g = np.load(os.path.join(GOLD, "chan64_f32.npz"))
    occ = slb.signals.wideband_occupancy(0)
    a = g["chan_prod_audio"].astype(np.float64)[:, 12:]
    rms = np.sqrt(np.mean(a ** 2, axis=1))
    assert 20 * np.log10(rms[occ].min() / rms[~occ].max()) > 15.0
    k = int(np.nonzero(occ)[0][0]); n = np.arange(a.shape[1])
    basis = np.stack([np.cos(2 * np.pi * 500 * n / 3000.0), np.sin(2 * np.pi * 500 * n / 3000.0)], 1)
    coef, *_ = np.linalg.lstsq(basis, a[k], rcond=None)
    assert np.sum((a[k] - basis @ coef) ** 2) < 0.05 * np.sum(a[k] ** 2)


def test_chan_blocking_independence(port):
    """Carried state (branch FIR histories, per-bin envelope): 3 calls of 768 frames == one call of 2304."""
    g = np.load(os.path.join(GOLD, "chan64_f32.npz"))
    prm = chan_params(g); x = g["chan_in"]
    whole, _, _, _ = port.chan_f32(prm, x)
    st = None; parts = []
    for h in range(3):
        o, _, _, st = port.chan_f32(prm, x[768 * h:768 * (h + 1)], st)
        parts.append(o)
    assert np.array_equal(np.concatenate(parts, 1), whole)


def test_chain_blocking_independence(port):
    """Carried state: 20 hops in one call == 20 calls of one hop (the firmware cadence accumulates 8 x 48 frames)."""
    g = np.load(os.path.join(GOLD, "rx_ssb_f32.npz"))
    prm = rx_params(g, "usb"); x = g["rx_usb_in"]
    whole, _, _, _ = port.rx_ssb_f32(prm, x)
    st = None; parts = []
    for h in range(20):
        o, _, _, st = port.rx_ssb_f32(prm, x[384 * h:384 * (h + 1)], st)
        parts.append(o)
    assert np.array_equal(np.concatenate(parts), whole)


def test_port_stages_vs_golden(port):
    s = np.load(os.path.join(GOLD, "stages.npz"))
    x, c = s["q15_x"], s["q15_c"]
    assert np.array_equal(port.fir_q15(c, np.zeros(112, np.int16), x, 48)[0], s["fir_q15"])
    assert np.array_equal(port.fir_fast_q15(c, np.zeros(112, np.int16), x, 48)[0], s["fir_fast_q15"])
    assert np.array_equal(port.biquad_df1_q15(s["bq15_c"], 2, 1, np.zeros(8, np.int16), x, 48)[0], s["biquad_df1_q15"])
    assert np.array_equal(port.scale_q15(x, 23170, 1), s["scale_q15"])
    assert np.array_equal(port.cmplx_mag_q15(x), s["cmplx_mag_q15"])
    assert np.array_equal(port.float_to_q15(s["f32_x"] * 3), s["float_to_q15"])
    rms = np.sqrt(np.mean(s["cfft_f32_512"].astype(np.float64) ** 2))
    assert np.max(np.abs(port.cfft_f32(s["cfft_in_512"]) - s["cfft_f32_512"])) < 2e-6 * rms
    assert np.max(np.abs(port.cfft_f32(s["cfft_in_512"], 1, 1) - s["icfft_f32_512"])) < 2e-6 * rms / 512 * 30
    bq = np.load(os.path.join(GOLD, "rx_ssb_f32.npz"))["rx_biquad"]
    assert np.array_equal(port.biquad_df2T_f32(bq, 2, np.zeros(4, np.float32), s["f32_x"], 48)[0], s["biquad_df2T_f32"])


# ---- RX-SSB-q15 (all-integer chain): every comparison is bit-exact ----
def q15_params(g, lsb=0):
    w, target, floor, gmax = [int(v) for v in g["q15_agc"]]
    return dict(ntaps=64, agc_block=48, agc_window=w, lsb=lsb, taps_i=g["q15_taps_i"], taps_q=g["q15_taps_q"], rel=g["q15_rel"],
                agc_target=target, agc_floor=floor, agc_gmax_q15=gmax)


@pytest.mark.parametrize("name,lsb", [("usb", 0), ("lsb", 1), ("sat", 0)])
def test_port_q15_chain_vs_golden(port, name, lsb):
    g = np.load(os.path.join(GOLD, "rx_ssb_q15.npz"))
    y, audio, gain, _ = port.rx_ssb_q15(q15_params(g, lsb), g["q15_%s_in" % name])
    assert np.array_equal(audio, g["q15_%s_audio" % name])
    assert np.array_equal(gain, g["q15_%s_gain" % name])
    assert np.array_equal(y, g["q15_%s_out" % name])


@pytest.mark.parametrize("name,lsb", [("usb", 0), ("lsb", 1), ("sat", 0)])
def test_ref_q15_chain_reproduces_golden(ref, name, lsb):
    g = np.load(os.path.join(GOLD, "rx_ssb_q15.npz"))
    y, audio, gain, _ = ref.rx_ssb_q15(q15_params(g, lsb), g["q15_%s_in" % name])
    assert np.array_equal(y, g["q15_%s_out" % name]) and np.array_equal(audio, g["q15_%s_audio" % name]) and np.array_equal(gain, g["q15_%s_gain" % name])


def test_q15_chain_is_a_single_sideband_demodulator(port):
    """Mid-band, the wanted sideband comes through at about unity and the other is suppressed by the Hilbert pair by
    > 40 dB. (64 taps at 48 kHz make a wide transition: the band edges 300 / 2700 Hz sit at -6 dB.)"""
    g = np.load(os.path.join(GOLD, "rx_ssb_q15.npz"))
    n = np.arange(4800)
    for f0 in (1000.0, 1500.0, 2000.0):
        ph = 2 * np.pi * f0 * n / 48000.0
        up = np.stack([np.round(8000 * np.cos(ph)), np.round(8000 * np.sin(ph))], 1).astype(np.int16)     # +f0: upper sideband
        lo = np.stack([np.round(8000 * np.cos(ph)), np.round(-8000 * np.sin(ph))], 1).astype(np.int16)    # -f0
        a_uu = port.rx_ssb_q15(q15_params(g, 0), up)[1][200:].astype(np.float64)
        a_ul = port.rx_ssb_q15(q15_params(g, 0), lo)[1][200:].astype(np.float64)
        a_ll = port.rx_ssb_q15(q15_params(g, 1), lo)[1][200:].astype(np.float64)
        assert 0.9 * 8000 / np.sqrt(2) < a_uu.std() < 1.02 * 8000 / np.sqrt(2)
        assert abs(a_ll.std() - a_uu.std()) < 0.02 * a_uu.std()
        assert 20 * np.log10(a_uu.std() / max(a_ul.std(), 1e-9)) > 40.0


def test_q15_chain_blocking_independence(port):
    """One call over the stream == the same stream fed in pieces (the carried FIR state and peak window are the whole state)."""
    g = np.load(os.path.join(GOLD, "rx_ssb_q15.npz"))
    x = g["q15_usb_in"]; prm = q15_params(g, 0)
    whole = port.rx_ssb_q15(prm, x)[0]
    st, parts = None, []
    for a, b in ((0, 48), (48, 480), (480, 4800), (4800, 7680)):
        y, _, _, st = port.rx_ssb_q15(prm, x[a:b], st)
        parts.append(y)
    assert np.array_equal(np.concatenate(parts), whole)


def test_am_chain_port_vs_ref(port, ref_or_recorded):
    """RX chain with the envelope detector (mode AM): the restatement against the reference build on the same input."""
    ref = ref_or_recorded
    g = np.load(os.path.join(GOLD, "rx_ssb_f32.npz"))
    prm = rx_params(g, "usb"); prm["envelope"] = 1
    x = g["rx_usb_in"]
    y_r, a_r, g_r, _ = ref.rx_ssb_f32(prm, x)
    y_p, a_p, g_p, _ = port.rx_ssb_f32(prm, x)
    assert np.all(a_r >= 0) and np.all(np.abs(a_p - a_r) <= audio_tolerance(a_r) + 1e-12)
    d = np.abs(y_p.astype(np.int32) - y_r.astype(np.int32))
    assert d.max() <= 1 and np.mean(d > 0) < 0.02


def fm_params(g):
    return dict(fft_len=512, hop=384, agc_block=48, biquad=g["fm_biquad"].reshape(2, 5), agc_target=g["fm_agc"][0], agc_decay=g["fm_agc"][1],
                agc_floor=g["fm_agc"][2], agc_gmax=g["fm_agc"][3], mask=g["fm_mask"], envelope=2)


def fm_audio_ok(audio, ref_audio):
    """FM discriminator output: the same 1e-5 bar as every float chain, the first super-block (filter fill-up) included. The
    limiter's floor (SLO_FM_FLOOR = 2^-10 on |z[n] conj z[n-1]|, i.e. -30 dBFS of baseband amplitude) keeps the division from
    magnifying the float32 rounding of the channel filter while the baseband is still near zero."""
    return bool(np.all(np.abs(audio - ref_audio) <= audio_tolerance(ref_audio) + 1e-9))


def fm_int16_ok(out, ref_out):
    """int16 result of the FM chain: the bar of the other float chains — single-LSB flips of the truncating pack
    (arm_float_to_q15.c:147) on < 2 % of the samples."""
    d = np.abs(out.astype(np.int32) - ref_out.astype(np.int32))
    return bool(d.max() <= 1 and np.mean(d > 0) < 0.02)


@pytest.mark.parametrize("name", ["centre", "offset"])
def test_port_fm_chain_vs_golden(port, name):
    """The FM detector of the chain (limiter-discriminator composed from arm_cmplx_conj_f32, arm_cmplx_mult_cmplx_f32,
    arm_cmplx_mag_f32; oracle/chains.inc.c): port vs the outputs of the reference build."""
    g = np.load(os.path.join(GOLD, "rx_fm_f32.npz"))
    out, audio, gain, _ = port.rx_ssb_f32(fm_params(g), g["fm_%s_in" % name])
    assert fm_audio_ok(audio, g["fm_%s_audio" % name])
    assert np.allclose(gain, g["fm_%s_gain" % name], rtol=2e-5)
    assert fm_int16_ok(out, g["fm_%s_out" % name])
    # what the discriminator is: the sine of the carrier's phase step — a 1 kHz tone of amplitude sin (2 pi 2500 / 48000), offset by
    # sin (2 pi fc / 48000) when the carrier sits fc off the channel centre (the biquad passes both)
    a = g["fm_%s_audio" % name][3000:7000].astype(np.float64); n = np.arange(3000, 7000)
    basis = np.stack([np.cos(2 * np.pi * 1000.0 * n / 48000.0), np.sin(2 * np.pi * 1000.0 * n / 48000.0), np.ones(n.size)], 1)
    c, *_ = np.linalg.lstsq(basis, a, rcond=None)
    assert abs(np.hypot(c[0], c[1]) - np.sin(2 * np.pi * 2500.0 / 48000.0)) < 0.02
    assert abs(c[2] - (np.sin(2 * np.pi * 1500.0 / 48000.0) if name == "offset" else 0.0)) < 0.02


@pytest.mark.parametrize("name", ["centre", "offset"])
def test_ref_fm_chain_reproduces_golden(ref, name):
    g = np.load(os.path.join(GOLD, "rx_fm_f32.npz"))
    out, audio, gain, _ = ref.rx_ssb_f32(fm_params(g), g["fm_%s_in" % name])
    assert np.array_equal(out, g["fm_%s_out" % name]) and np.array_equal(audio, g["fm_%s_audio" % name])


def test_ref_fixed_point_ffts_reproduce_golden(ref):
    """tests/golden/cfft_fixed.npz = arm_cfft_q15 (ARM_MATH_DSP branch, oracle/ref_glue/cm4_fft_q15.c) and arm_cfft_q31 of the reference build."""
    g = np.load(os.path.join(GOLD, "cfft_fixed.npz"))
    n = 0
    for key in g.files:
        if key.endswith("_in"):
            kind, N, tag, _ = key.split("_")
            for ifft in (0, 1):
                fn = ref.cfft_q15_cm4 if kind == "q15" else ref.cfft_q31
                assert np.array_equal(fn(g[key], ifft), g["%s_%s_%s_%d" % (kind, N, tag, ifft)]); n += 1
    assert n == 40
    # and the reason the CM4-path build exists: the C branch of the same routine is NOT the firmware's arithmetic (SURVEY.md §8c.3)
    x = g["q15_1024_m_in"]
    assert not np.array_equal(ref.cfft_q15(x, 0), ref.cfft_q15_cm4(x, 0))
    assert np.max(np.abs(ref.cfft_q15(x, 0).astype(np.int32) - ref.cfft_q15_cm4(x, 0))) <= 8
