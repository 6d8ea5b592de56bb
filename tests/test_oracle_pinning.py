"""Pin the plain-C restatement (oracle/port) against the reference itself run here (oracle/_ref = the vendored
CMSIS-DSP V1.5.3 sources compiled for x86, SURVEY.md §8c). The reference ships no golden vectors (SURVEY.md §4), so
execution of its own code is the pin. Integer routines must agree bit for bit; float routines to a stated tolerance.
Where the reference build is absent, `ref` replays the outputs recorded on these same inputs (tests/golden/pinning.npz)."""
import numpy as np
import pytest

BLOCK = 48


@pytest.fixture
def ref(ref_or_recorded):
    return ref_or_recorded


def q15(rng, n, amp=32767):
    return rng.integers(-amp, amp + 1, n).astype(np.int16)


def f32(rng, n, amp=1.0):
    return (rng.standard_normal(n) * amp).astype(np.float32)


def test_conversions(ref, port, rng):
    x = np.concatenate([q15(rng, 4096), np.array([-32768, 32767, 0, -1, 1], np.int16)])
    assert np.array_equal(ref.q15_to_float(x), port.q15_to_float(x))
    f = np.concatenate([f32(rng, 4096, 0.5), np.array([1.5, -1.5, 0.99999, -1.0, 1.0, 3.05e-5, -3.05e-5, 0.0], np.float32)])
    assert np.array_equal(ref.float_to_q15(f), port.float_to_q15(f))
    # q15 -> f32 -> q15 is the identity (SURVEY Appendix A)
    assert np.array_equal(port.float_to_q15(port.q15_to_float(x)), x)


@pytest.mark.parametrize("ntaps", [4, 16, 64, 130])
def test_fir_q15_family_bit_exact(ref, port, rng, ntaps):
    c = q15(rng, ntaps, 8000); x = q15(rng, BLOCK * 20)
    st = np.zeros(ntaps + BLOCK, np.int16)
    for name in ("fir_q15", "fir_fast_q15"):
        o_r, s_r = getattr(ref, name)(c, st, x, BLOCK); o_p, s_p = getattr(port, name)(c, st, x, BLOCK)
        assert np.array_equal(o_r, o_p), name
        assert np.array_equal(s_r[:ntaps - 1], s_p[:ntaps - 1]), name
    # saturating case: full-scale coefficients
    c2 = np.full(ntaps, 32767, np.int16); x2 = np.full(BLOCK * 2, 32767, np.int16)
    assert np.array_equal(ref.fir_q15(c2, st, x2, BLOCK)[0], port.fir_q15(c2, st, x2, BLOCK)[0])


def test_fir_q31_bit_exact(ref, port, rng):
    c = rng.integers(-2**28, 2**28, 32).astype(np.int32); x = rng.integers(-2**31, 2**31 - 1, BLOCK * 8).astype(np.int32)
    st = np.zeros(32 + BLOCK, np.int32)
    assert np.array_equal(ref.fir_q31(c, st, x, BLOCK)[0], port.fir_q31(c, st, x, BLOCK)[0])


@pytest.mark.parametrize("ntaps", [5, 64, 129])
def test_fir_f32(ref, port, rng, ntaps):
    c = f32(rng, ntaps, 0.1); x = f32(rng, BLOCK * 20)
    st = np.zeros(ntaps + BLOCK, np.float32)
    o_r, s_r = ref.fir_f32(c, st, x, BLOCK); o_p, s_p = port.fir_f32(c, st, x, BLOCK)
    # same products, same sequential order, no contraction on either side -> identical
    assert np.array_equal(o_r, o_p)
    assert np.array_equal(s_r[:ntaps - 1], s_p[:ntaps - 1])


def test_fir_decimate_interpolate(ref, port, rng):
    c = f32(rng, 64, 0.1); x = f32(rng, BLOCK * 8)
    st = np.zeros(64 + BLOCK, np.float32)
    assert np.array_equal(ref.fir_decimate_f32(c, 4, st, x, BLOCK)[0], port.fir_decimate_f32(c, 4, st, x, BLOCK)[0])
    assert np.array_equal(ref.fir_interpolate_f32(c, 4, st, x, BLOCK)[0], port.fir_interpolate_f32(c, 4, st, x, BLOCK)[0])
    cq = q15(rng, 64, 4000); xq = q15(rng, BLOCK * 8); sq = np.zeros(64 + BLOCK, np.int16)
    assert np.array_equal(ref.fir_decimate_q15(cq, 4, sq, xq, BLOCK)[0], port.fir_decimate_q15(cq, 4, sq, xq, BLOCK)[0])
    assert np.array_equal(ref.fir_interpolate_q15(cq, 4, sq, xq, BLOCK)[0], port.fir_interpolate_q15(cq, 4, sq, xq, BLOCK)[0])
    # q31 (arm_fir_decimate_q31.c:60, arm_fir_interpolate_q31.c:62): full-range samples, q63 accumulator >> 31, no saturation
    c31 = rng.integers(-2**27, 2**27, 64).astype(np.int32); x31 = rng.integers(-2**31, 2**31 - 1, BLOCK * 8).astype(np.int32)
    s31 = np.zeros(64 + BLOCK, np.int32)
    for M in (2, 4):
        assert np.array_equal(ref.fir_decimate_q31(c31, M, s31, x31, BLOCK)[0], port.fir_decimate_q31(c31, M, s31, x31, BLOCK)[0])
        assert np.array_equal(ref.fir_interpolate_q31(c31, M, s31, x31, BLOCK)[0], port.fir_interpolate_q31(c31, M, s31, x31, BLOCK)[0])


@pytest.mark.parametrize("ntaps", [8, 32])
def test_lms_norm_f32_bit_exact(ref, port, rng, ntaps):
    """arm_lms_norm_f32.c:161: output, error, adapted coefficients, state buffer head, energy and x0 — reference vs port, with the
    instance carried over two calls."""
    n = BLOCK * 40
    t = np.arange(n)
    d = (0.3 * np.sin(2 * np.pi * 1000.0 * t / 48000.0) + 0.05 * rng.standard_normal(n)).astype(np.float32)
    x = np.concatenate([np.zeros(3, np.float32), d[:-3]])                        # the decorrelation delay of a line enhancer
    c0 = np.zeros(ntaps, np.float32); st0 = np.zeros(ntaps + BLOCK, np.float32); ex0 = np.zeros(2, np.float32)
    h = n // 2
    for orc_a, orc_b in ((ref, port),):
        ra = orc_a.lms_norm_f32(c0, 0.05, st0, ex0, x[:h], d[:h], BLOCK); rb = orc_b.lms_norm_f32(c0, 0.05, st0, ex0, x[:h], d[:h], BLOCK)
        for u, v in zip(ra, rb):
            assert np.array_equal(u[:ntaps - 1] if u.size == ntaps + BLOCK else u, v[:ntaps - 1] if v.size == ntaps + BLOCK else v)
        ra2 = orc_a.lms_norm_f32(ra[2], 0.05, ra[3], ra[4], x[h:], d[h:], BLOCK); rb2 = orc_b.lms_norm_f32(rb[2], 0.05, rb[3], rb[4], x[h:], d[h:], BLOCK)
        assert np.array_equal(ra2[0], rb2[0]) and np.array_equal(ra2[1], rb2[1]) and np.array_equal(ra2[2], rb2[2]) and np.array_equal(ra2[4], rb2[4])
    # what it is for: the error output is the audio with the tone notched out (auto-notch), the filter output is the tone (noise reduction)
    tail = slice(n // 2 - 2000, n // 2)
    assert np.std(ra[1][tail]) < 0.5 * np.std(d[tail]) and np.std(ra[0][tail]) > 0.6 * np.std(d[tail])


def _sos_cmsis(order=4, fc=300.0, fs=48000.0):
    from scipy import signal
    sos = signal.butter(order, fc, "highpass", fs=fs, output="sos")
    return np.stack([np.r_[s[0:3], -s[4], -s[5]] for s in sos]).astype(np.float32)


def test_biquads_f32(ref, port, rng):
    c = _sos_cmsis(); ns = c.shape[0]; x = f32(rng, BLOCK * 50, 0.3)
    for name, nst in (("biquad_df2T_f32", 2), ("biquad_df1_f32", 4)):
        st = np.zeros(nst * ns, np.float32)
        o_r, s_r = getattr(ref, name)(c, ns, st, x, BLOCK); o_p, s_p = getattr(port, name)(c, ns, st, x, BLOCK)
        assert np.array_equal(o_r, o_p), name
        assert np.array_equal(s_r, s_p), name
    st = np.zeros(4 * ns, np.float32)
    o_r, s_r = ref.biquad_stereo_df2T_f32(c, ns, st, x, BLOCK); o_p, s_p = port.biquad_stereo_df2T_f32(c, ns, st, x, BLOCK)
    assert np.array_equal(o_r, o_p) and np.array_equal(s_r, s_p)


def test_biquads_fixed_bit_exact(ref, port, rng):
    cf = _sos_cmsis(2, 1000.0)[0]
    c15 = np.round(cf / 2 * 32768).astype(np.int16)               # postShift = 1
    c15 = np.array([c15[0], 0, c15[1], c15[2], c15[3], c15[4]] * 2, np.int16)
    x = q15(rng, BLOCK * 40, 20000); st = np.zeros(8, np.int16)
    o_r, s_r = ref.biquad_df1_q15(c15, 2, 1, st, x, BLOCK); o_p, s_p = port.biquad_df1_q15(c15, 2, 1, st, x, BLOCK)
    assert np.array_equal(o_r, o_p) and np.array_equal(s_r, s_p)
    c31 = np.tile(np.round(cf / 2 * 2**31).astype(np.int64).clip(-2**31, 2**31 - 1).astype(np.int32), 2)
    x31 = rng.integers(-2**30, 2**30, BLOCK * 40).astype(np.int32); st31 = np.zeros(8, np.int32)
    o_r, s_r = ref.biquad_df1_q31(c31, 2, 1, st31, x31, BLOCK); o_p, s_p = port.biquad_df1_q31(c31, 2, 1, st31, x31, BLOCK)
    assert np.array_equal(o_r, o_p) and np.array_equal(s_r, s_p)


@pytest.mark.parametrize("N", [16, 32, 64, 128, 256, 512, 1024, 2048, 4096])
def test_cfft_f32(ref, port, rng, N):
    x = f32(rng, 2 * N)
    for ifft in (0, 1):
        a = ref.cfft_f32(x, ifft, 1); b = port.cfft_f32(x, ifft, 1)
        rms = np.sqrt(np.mean(a.astype(np.float64) ** 2))
        assert np.max(np.abs(a - b)) <= 2e-6 * rms, (N, ifft)
    # and against numpy, to pin the sign/scale conventions of both
    z = np.fft.fft(x.view(np.complex64).astype(np.complex128))
    assert np.max(np.abs(port.cfft_f32(x).view(np.complex64) - z)) <= 1e-6 * np.sqrt(np.mean(np.abs(z) ** 2))


@pytest.mark.parametrize("N", [32, 256, 1024])
def test_rfft_fast_f32(ref, port, rng, N):
    x = f32(rng, N)
    a = ref.rfft_fast_f32(x, 0); b = port.rfft_fast_f32(x, 0)
    rms = np.sqrt(np.mean(a.astype(np.float64) ** 2))
    assert np.max(np.abs(a - b)) <= 2e-6 * rms
    assert np.max(np.abs(ref.rfft_fast_f32(a, 1) - port.rfft_fast_f32(a, 1))) <= 2e-6


def test_complex_and_stats(ref, port, rng):
    a = f32(rng, 1024); b = f32(rng, 1024)
    for name in ("cmplx_mult_cmplx_f32",):
        assert np.array_equal(getattr(ref, name)(a, b), getattr(port, name)(a, b))
    assert np.array_equal(ref.cmplx_mult_real_f32(a, b[:512]), port.cmplx_mult_real_f32(a, b[:512]))
    for name in ("cmplx_conj_f32", "cmplx_mag_f32", "cmplx_mag_squared_f32", "abs_f32"):
        assert np.array_equal(getattr(ref, name)(a), getattr(port, name)(a)), name
    for name in ("mult_f32", "add_f32", "sub_f32"):
        assert np.array_equal(getattr(ref, name)(a, b), getattr(port, name)(a, b)), name
    assert np.array_equal(ref.scale_f32(a, 0.37), port.scale_f32(a, 0.37))
    for n in (1, 3, 48, 1024):
        assert ref.max_f32(a[:n]) == port.max_f32(a[:n])
        for name in ("rms_f32", "power_f32", "mean_f32"):
            assert getattr(ref, name)(a[:n]) == getattr(port, name)(a[:n]), (name, n)
    q = q15(rng, 2048); r = q15(rng, 2048)
    assert np.array_equal(ref.cmplx_mag_q15(q), port.cmplx_mag_q15(q))
    for n in (1, 48, 2048):
        assert ref.max_q15(q[:n]) == port.max_q15(q[:n])
        assert ref.rms_q15(q[:n]) == port.rms_q15(q[:n])
    assert np.array_equal(ref.add_q15(q, r), port.add_q15(q, r))
    assert np.array_equal(ref.sub_q15(q, r), port.sub_q15(q, r))
    edge = np.array([-32768, 32767, 0, -1], np.int16)
    assert np.array_equal(ref.abs_q15(np.r_[q, edge]), port.abs_q15(np.r_[q, edge]))
    for k, sh in ((12345, 0), (-32768, 1), (32767, 3), (700, -2)):
        assert np.array_equal(ref.scale_q15(q, k, sh), port.scale_q15(q, k, sh)), (k, sh)
    for sh in (-3, 0, 2):
        assert np.array_equal(ref.shift_q15(q, sh), port.shift_q15(q, sh)), sh


def test_sin_cos_table(ref, port, rng):
    x = np.concatenate([(rng.random(5000) * 40 - 20).astype(np.float32), np.array([0, -1e-7, 6.2831855, -6.2831855], np.float32)])
    assert np.array_equal(ref.sin_f32(x), port.sin_f32(x))
    assert np.array_equal(ref.cos_f32(x), port.cos_f32(x))
    # arm_sin_f32 is NOT libm sinf (SURVEY Appendix A): table error up to ~2e-5
    # (the last element also pins a quirk: x = -2*pi maps to table index 512 & 0x1ff = 0 with fract = 512 -> 6.283)
    assert ref.sin_f32(x)[-1] > 6.0
    assert 1e-6 < np.max(np.abs(ref.sin_f32(x[:-1]) - np.sin(x[:-1].astype(np.float64)))) < 4e-5


def test_q15_chain_with_the_optional_biquad_bit_exact(ref, port, rng):
    """oracle/chains.inc.c rx_ssb_q15 with arm_biquad_cascade_df1_q15 between mixer and AGC: reference build vs port."""
    import selenite_lite_b200 as slb
    from test_golden import GOLD, q15_params
    import os
    g = np.load(os.path.join(GOLD, "rx_ssb_q15.npz"))
    prm = q15_params(g, 0)
    from scipy import signal
    b, a = signal.butter(2, 2600.0, "lowpass", fs=48000)
    c = np.round(np.array([b[0], b[1], b[2], -a[1], -a[2]]) / 2 * 32768).astype(np.int16)
    prm.update(bq_stages=1, bq_postshift=1, bq_coeffs=np.array([c[0], 0, c[1], c[2], c[3], c[4]], np.int16))
    x = slb.synth_iq(1, 48 * 60)[0]
    o_r, a_r, g_r, _ = ref.rx_ssb_q15(prm, x); o_p, a_p, g_p, _ = port.rx_ssb_q15(prm, x)
    assert np.array_equal(o_r, o_p) and np.array_equal(a_r, a_p) and np.array_equal(g_r, g_p)
    prm0 = q15_params(g, 0)
    assert not np.array_equal(ref.rx_ssb_q15(prm0, x)[1], a_r)
