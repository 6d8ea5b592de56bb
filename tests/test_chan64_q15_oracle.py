"""The oracle of the integer channelizer CHAN-64-q15 (oracle/slo_chan_q15.h, DESIGN.md §3.10) on the CPU: the port's arm_cfft_q15 against
the reference vectors and the NumPy model, the chain against a NumPy restatement, the default prototype's headroom, the measured quality
of the integer arithmetic, streaming, and the golden vectors."""
import sys

import numpy as np
import pytest

import fft_fixed_model as ffm
import oracle_chan_q15 as ocq
import selenite_lite_b200 as slb
from selenite_lite_b200.dsp_if import chan_q15_params_to_dict
from test_golden import GOLD

sys.path.insert(0, GOLD)
import make_golden_chan64_q15 as mg  # noqa: E402

FS, M, P, BLK = 192000, 64, 8, 3
# measured on the port with the default parameters (tests below): the SNR of the tone's bin (integer chain against the same FIR and DFT
# in float64) for an in-bin tone at these levels, and the power of that tone in the neighbouring bins relative to its own bin
SNR_DB = {-1: 76.703, -20: 56.888, -40: 36.999, -60: 17.111}
ADJ_REJECTION_DB = 76.297


def prm(**over):
    d = chan_q15_params_to_dict(slb.default_chan_q15_params(FS))
    d.update(over)
    return d


def branch_taps(proto):
    """e[r][p] = h[64 p + 63 - r]"""
    return np.asarray(proto, np.int64).reshape(P, M)[:, ::-1].T


def np_branches(proto, x, hist=None):
    """int64 arm_fir_q15 of every branch and rail before the >> 15: [hops][64] per rail (hist: the 7 previous hops, [7][64][2])"""
    e = branch_taps(proto)
    hops = x.shape[0] // M
    w = np.asarray(x, np.int64).reshape(hops, M, 2)
    w = np.concatenate([np.zeros((P - 1, M, 2), np.int64) if hist is None else hist, w])
    acc = sum(e[:, p][None, :, None] * w[P - 1 - p:P - 1 - p + hops] for p in range(P))
    return acc[..., 0], acc[..., 1]


def np_spectrum(proto, x):
    """the integer spectrum per hop, int16 [hops][64][2]: branch FIRs (>> 15, saturated) and fft_fixed_model.cfft_q15"""
    ai, aq = np_branches(proto, x)
    v = np.stack([np.clip(ai >> 15, -32768, 32767), np.clip(aq >> 15, -32768, 32767)], -1).astype(np.int16)
    return ffm.cfft_q15(v.reshape(v.shape[0], 2 * M)).reshape(-1, M, 2)


def np_agc(p, audio):
    """the gain law of rx_ssb_q15 per bin over audio int16 [64][hops] from an empty window: (out, gain)"""
    a = audio.astype(np.int64)
    peaks = np.abs(a).clip(max=32767).reshape(M, -1, BLK).max(-1)
    nb = peaks.shape[1]
    hist = np.concatenate([np.zeros((M, 32), np.int64), peaks], 1)
    env = peaks.copy()
    rel = np.asarray(p["rel"], np.int64)
    for j in range(1, p["agc_window"]):
        env = np.maximum(env, (hist[:, 32 - j:32 - j + nb] * rel[j]) >> 15)
    q = np.minimum((int(p["agc_target"]) << 15) // np.maximum(env, int(p["agc_floor"])), int(p["agc_gmax_q15"]))
    s = np.zeros_like(q)
    while np.any((q >> s) > 32767):
        s += (q >> s) > 32767
    g = np.repeat(q >> s, BLK, 1); sh = np.repeat(s, BLK, 1)
    y = np.clip((a * g) >> (15 - sh), -32768, 32767).astype(np.int16)
    return np.stack([y, y], -1), q.astype(np.uint32)


def tone(dbfs, f, frames, phase=0.3):
    n = np.arange(frames)
    z = 10 ** (dbfs / 20) * 32767 * np.exp(1j * (2 * np.pi * f * n / FS + phase))
    return np.stack([np.rint(z.real), np.rint(z.imag)], 1).clip(-32768, 32767).astype(np.int16)


def snr_db(proto, x, k, skip=8):
    """SNR of bin k: the integer spectrum against the same FIR and DFT (/ 64) in float64"""
    xi = np_spectrum(proto, x)[skip:, k]
    zi = xi[:, 0].astype(np.float64) + 1j * xi[:, 1]
    ai, aq = np_branches(proto, x)
    v = (ai + 1j * aq)[skip:] / 32768.0
    zr = np.fft.fft(v, axis=1)[:, k] / M
    return 10 * np.log10(np.sum(np.abs(zr) ** 2) / np.sum(np.abs(zi - zr) ** 2))


# ---------------------------------------------------------------------------------------------------------------------- the q15 FFT
def test_port_cfft_q15_equals_reference_vectors_and_model(port, rng):
    g = np.load(GOLD + "/cfft_fixed.npz")
    n = 0
    for key in g.files:
        if key.startswith("q15_") and key.endswith("_in"):
            _, N, tag, _ = key.split("_")
            for ifft in (0, 1):
                assert np.array_equal(port.cfft_q15(g[key], ifft), g["q15_%s_%s_%d" % (N, tag, ifft)]), (key, ifft); n += 1
    assert n == 20
    for N in (16, 64, 128):
        x = np.concatenate([rng.integers(-32768, 32768, (6, 2 * N)), np.full((1, 2 * N), -32768), np.full((1, 2 * N), 32767)]).astype(np.int16)
        for ifft in (0, 1):
            want = ffm.cfft_q15(x, ifft)
            for i in range(x.shape[0]):
                assert np.array_equal(port.cfft_q15(x[i], ifft), want[i]), (N, ifft, i)


# ---------------------------------------------------------------------------------------------------------------------- the chain
@pytest.mark.parametrize("envelope", [0, 1])
def test_chan_q15_equals_numpy_restatement(port, rng, envelope):
    p = prm(envelope=envelope)
    x = np.concatenate([slb.synth_wideband(1, 3072)[0], rng.integers(-32768, 32768, (3072, 2)).astype(np.int16)])
    y, audio, gain, _ = ocq.chan_q15(port, p, x)
    spec = np_spectrum(p["proto"], x)                                        # [hops][64][2]
    if envelope:
        want = np.stack([port.cmplx_mag_q15(spec[h].reshape(-1)) for h in range(spec.shape[0])], 1)
    else:
        want = spec[:, :, 0].T
    assert np.array_equal(audio, want)
    wy, wg = np_agc(p, want)
    assert np.array_equal(gain, wg) and np.array_equal(y, wy)


def test_default_prototype_never_saturates_a_branch():
    p = prm()
    e = branch_taps(p["proto"])
    assert abs(int(np.sum(p["proto"])) - 32 * 32768) <= 256                   # DC gain 32
    worst = np.abs(e).sum(1).max()
    assert worst <= 0.76 * 32768, worst / 32768
    # the input that drives each branch to its largest sum: every tap's sample at the rail of the tap's sign, both rails
    for r in range(M):
        x = np.zeros((P * M, 2), np.int16)
        for q in range(P):                                                   # x_r[m - q] sits at frame 64 (7 - q) + r for m = 7
            x[M * (P - 1 - q) + r] = 32767 if e[r, q] >= 0 else -32768
        ai, aq = np_branches(p["proto"], x)
        assert np.abs(ai >> 15).max() < 32768 and np.abs(aq >> 15).max() < 32768


def test_in_bin_tone_snr_is_pinned():
    p = prm()
    got = {lvl: snr_db(p["proto"], tone(lvl, 5 * FS / M + 500.0, 64 * 200), 5) for lvl in SNR_DB}
    for lvl, want in SNR_DB.items():
        assert abs(got[lvl] - want) < 0.01, (lvl, got[lvl], want)


def test_adjacent_bin_rejection_is_pinned():
    p = prm()
    s = np_spectrum(p["proto"], tone(-1, 9 * FS / M, 64 * 200))[8:].astype(np.float64)
    pw = (s ** 2).sum(-1).sum(0)
    rej = 10 * np.log10(pw[9] / max(pw[8], pw[10]))
    assert abs(rej - ADJ_REJECTION_DB) < 0.01, rej


def test_calls_cut_at_768_frames_equal_one_call(port, rng):
    for envelope in (0, 1):
        p = prm(envelope=envelope, agc_window=17)
        x = np.concatenate([slb.synth_wideband(1, 768 * 5)[0], rng.integers(-3000, 3000, (768 * 3, 2)).astype(np.int16)])
        y, a, g, _ = ocq.chan_q15(port, p, x)
        st = ocq.ChanQ15State(); parts = []
        for c0 in range(0, x.shape[0], 768):
            parts.append(ocq.chan_q15(port, p, x[c0:c0 + 768], st))
        assert np.array_equal(np.concatenate([q[0] for q in parts], 1), y)
        assert np.array_equal(np.concatenate([q[1] for q in parts], 1), a)
        assert np.array_equal(np.concatenate([q[2] for q in parts], 1), g)


def test_golden_regenerates_bit_for_bit(port):
    g = np.load(GOLD + "/chan64_q15.npz")
    v = mg.vectors(port)
    assert sorted(v) == sorted(g.files)
    for k in g.files:
        assert np.array_equal(v[k], g[k]), k
