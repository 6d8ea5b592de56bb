"""The NumPy model of arm_cfft_q15 / arm_cfft_q31 (fft_fixed_model.py), pinned three ways without a GPU:

- bit for bit to every vector committed from the reference build (tests/golden/cfft_fixed.npz: N = 16, 64, 1024 pure radix-4 and
  N = 128, 2048 radix-4-by-2, moderate and rail-to-rail inputs, both directions, q15 and q31);
- to the float64 DFT at all nine sizes, scaled by the routines' documented output format, within a few LSB;
- to the twiddle tables the library regenerates, and to the reference build itself where that build exists.

Pinned like this, the model is the authority the GPU tests (test_gpu_fft_fixed.py) compare with at N = 32, 256, 512 and 4096,
where no reference vectors exist."""
import os

import numpy as np
import pytest

import fft_fixed_model as model

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfft_fixed.npz")

# Output format (integer.fraction bits) of arm_cfft_q15 / arm_cfft_q31 by size, for a q15 / q31 input: the tables of
# arm_cfft_radix4_q15.c:94-104, arm_cfft_radix4_q31.c and arm_cfft_q15.c / arm_cfft_q31.c. Forward and inverse share them: every
# stage scales the same way in both directions, so the inverse is the unnormalised inverse DFT scaled the same as the forward one.
OUTPUT_FORMAT = {
    ("q15", 0): {16: "5.11", 32: "6.10", 64: "7.9", 128: "8.8", 256: "9.7", 512: "10.6", 1024: "11.5", 2048: "12.4", 4096: "13.3"},
    ("q15", 1): {16: "5.11", 32: "6.10", 64: "7.9", 128: "8.8", 256: "9.7", 512: "10.6", 1024: "11.5", 2048: "12.4", 4096: "13.3"},
    ("q31", 0): {16: "5.27", 32: "6.26", 64: "7.25", 128: "8.24", 256: "9.23", 512: "10.22", 1024: "11.21", 2048: "12.20", 4096: "13.19"},
    ("q31", 1): {16: "5.27", 32: "6.26", 64: "7.25", 128: "8.24", 256: "9.23", 512: "10.22", 1024: "11.21", 2048: "12.20", 4096: "13.19"},
}

# Largest difference from the scaled float64 DFT, in output LSB, per type. Measured once on the model over the inputs of
# test_model_matches_the_float64_dft (seeded) at all nine sizes and both directions: q15 11.7 LSB, q31 32.0 LSB, both at
# radix-4-by-2 sizes (the pure radix-4 sizes stay near half of that). Bounds: those maxima with a margin of about half.
DFT_BOUND_LSB = {"q15": 16.0, "q31": 48.0}

FULL = {"q15": 32767, "q31": 2**31 - 1}
DTYPE = {"q15": np.int16, "q31": np.int32}


def output_shift(kind, N, ifft):
    """Bits the output is scaled down by relative to the unnormalised DFT of the integer input: integer bits - 1."""
    ibits, fbits = (int(v) for v in OUTPUT_FORMAT[(kind, ifft)][N].split("."))
    assert ibits + fbits == (16 if kind == "q15" else 32)
    return ibits - 1


def test_output_format_table_is_one_over_n():
    """The header's description (include/selenite_b200.h: the reference's scaling, 1/N for N = 4^m): the table says 1/N at every
    size, the radix-4-by-2 ones included, in both directions."""
    for kind in ("q15", "q31"):
        for ifft in (0, 1):
            assert sorted(OUTPUT_FORMAT[(kind, ifft)]) == list(model.SIZES)
            for N in model.SIZES:
                assert 1 << output_shift(kind, N, ifft) == N, (kind, ifft, N)


def test_model_equals_every_reference_vector():
    g = np.load(GOLD)
    checked = 0
    for key in g.files:
        if not key.endswith("_in"):
            continue
        kind, N, tag, _ = key.split("_")
        x = g[key]
        assert x.dtype == DTYPE[kind] and x.shape == (2 * int(N),)
        for ifft in (0, 1):
            exp = g["%s_%s_%s_%d" % (kind, N, tag, ifft)]
            got = model.cfft(kind, x, ifft)
            assert got.dtype == exp.dtype and np.array_equal(got, exp), (key, ifft, int(np.max(np.abs(got.astype(np.int64) - exp))))
            checked += 1
    # 5 sizes x 2 amplitudes x 2 directions x 2 types
    assert checked == 40


def dft_inputs(kind, N, rng):
    """[transforms][2 N]: moderate random, single-bin tones, impulses, DC. (Inputs that drive the q15 lane sums into saturation
    are not linear any more; test_q15_lane_operations_at_their_limits and the GPU tests cover them.)"""
    full = FULL[kind]
    n = np.arange(N)
    rows = []
    mod = (full + 1) // 4
    rows += list(rng.integers(-mod, mod + 1, (6, 2 * N)))
    # single-bin tones: a random bin and phase, and bins 0, 1, N / 2 and N - 1 with the peak on an axis, at 1 - 2^-6 of full scale.
    # At exactly full scale such a peak overflows in the reference itself (test_full_scale_peak_wraps_as_in_the_reference).
    amp = full * (1 - 2.0 ** -6)
    for k, ph0 in ((int(rng.integers(N)), rng.random() * 2 * np.pi), (0, 0.0), (1, np.pi / 2), (N // 2, np.pi), (N - 1, np.pi / 4)):
        ph = 2 * np.pi * k * n / N + ph0
        rows.append(np.stack([np.round(amp * np.cos(ph)), np.round(amp * np.sin(ph))], 1).reshape(-1))
    for i in (0, 1, N - 1, int(rng.integers(N))):
        z = np.zeros((N, 2)); z[i] = rng.integers(-full - 1, full + 1, 2); rows.append(z.reshape(-1))
    for v in ((-full - 1, -full - 1), (full, full), tuple(rng.integers(-full - 1, full + 1, 2))):
        z = np.zeros((N, 2)); z[:] = v; rows.append(z.reshape(-1))
    return np.array(rows).astype(DTYPE[kind])


@pytest.mark.parametrize("kind", ["q15", "q31"])
@pytest.mark.parametrize("N", model.SIZES)
@pytest.mark.parametrize("ifft", [0, 1])
def test_model_matches_the_float64_dft(kind, N, ifft):
    rng = np.random.Generator(np.random.PCG64(1000 * N + 10 * ifft + (kind == "q31")))
    x = dft_inputs(kind, N, rng)
    got = model.cfft(kind, x, ifft).astype(np.float64).reshape(len(x), N, 2)
    xf = x.astype(np.float64).reshape(len(x), N, 2)
    z = xf[..., 0] + 1j * xf[..., 1]
    X = np.fft.ifft(z, axis=-1) * N if ifft else np.fft.fft(z, axis=-1)
    X = X / 2.0 ** output_shift(kind, N, ifft)
    err = np.maximum(np.abs(got[..., 0] - X.real), np.abs(got[..., 1] - X.imag)).max(axis=-1)
    assert np.all(err <= DFT_BOUND_LSB[kind]), (kind, N, ifft, int(np.argmax(err)), float(err.max()))


def test_q15_lane_operations_at_their_limits():
    """The dual 16-bit instructions the model restates, at the values where a slip shows (ARM v7E-M: the Q forms saturate each
    half-word, the SH forms halve without saturating and round toward minus infinity, ASX / SAX cross the high half-word of the
    second operand into the low result, SMUAD and friends wrap at 32 bits). The committed vectors never saturate a lane sum, so
    this is what holds the saturation without the reference build."""
    for op, a, b, exp in (
        (model.qadd16, (32767, -32768), (1, -1), (32767, -32768)),
        (model.qadd16, (30000, -30000), (-30000, 30000), (0, 0)),
        (model.qsub16, (-32768, 32767), (1, -1), (-32768, 32767)),
        (model.qsub16, (16384, -16384), (-16384, 16384), (32767, -32768)),
        (model.shadd16, (32767, -32768), (32767, -32768), (32767, -32768)),
        (model.shadd16, (-3, 3), (0, 0), (-2, 1)),
        (model.shsub16, (-32768, 32767), (32767, -32768), (-32768, 32767)),
        (model.qasx, (-32768, 0), (7, 1), (-32768, 7)),
        (model.qsax, (32767, 0), (7, 1), (32767, -7)),
        (model.shasx, (-32768, 0), (7, 1), (-16385, 3)),
        (model.shsax, (32767, 0), (7, 1), (16384, -4)),
    ):
        assert tuple(int(v) for v in op(a, b)) == exp, (op.__name__, a, b)
    assert model.smuad((-32768, -32768), (-32768, -32768)) == -2**31          # 2^31 wraps
    assert (model.smuad((3, 5), (7, 11)), model.smusd((3, 5), (7, 11))) == (76, -34)
    assert (model.smuadx((3, 5), (7, 11)), model.smusdx((3, 5), (7, 11))) == (68, -2)


def full_scale_tone(kind, N, k, ph0):
    n = np.arange(N)
    ph = 2 * np.pi * k * n / N + ph0
    return np.stack([np.round(FULL[kind] * np.cos(ph)), np.round(FULL[kind] * np.sin(ph))], 1).reshape(-1).astype(DTYPE[kind])


def test_full_scale_peak_wraps_as_in_the_reference():
    """The routines have no headroom for a full-scale tone whose peak lands on an axis. q15 at N = 2 * 4^m: the peak is 16384 before
    the final doubling (p <<= 1 in a q31_t, stored back into a q15_t, arm_cfft_q15.c), which wraps it to -32768. q31: the radix-4
    stages after the first sum four quarter-scale values with 32-bit wrapping adds. The model wraps where the reference does; the
    GPU tests use these tones to tell a wrapping kernel from a saturating one."""
    y = model.cfft_q15(full_scale_tone("q15", 128, 1, np.pi / 2), 1).reshape(-1, 2)
    assert y[127, 1] == -32768                                   # the inverse puts +j 32767 at bin N - 1: wrapped
    y = model.cfft_q15(full_scale_tone("q15", 64, 1, np.pi / 2), 1).reshape(-1, 2)
    assert y[63, 1] > 32760                                      # N = 4^m: no doubling, no wrap
    y = model.cfft_q31(full_scale_tone("q31", 64, 1, np.pi / 2), 0).reshape(-1, 2)
    assert abs(int(y[1, 1]) - (2**31 - 1)) > 2**29               # +j (2^31 - 1) at bin 1, wrapped on the way
    y = model.cfft_q31(full_scale_tone("q31", 32, 1, np.pi / 2), 0).reshape(-1, 2)
    assert y[1, 1] > 2**31 - 64                                  # the same tone at N = 32 stays within range


@pytest.mark.parametrize("N", model.SIZES)
def test_model_twiddles_equal_the_library_tables(N):
    """slb_design_twiddle_q15 / _q31 (what the kernels are given) equal the model's tables, and every entry is within 1 LSB of
    float64 cos and sin."""
    from selenite_lite_b200 import _lib
    lib = _lib.load()
    n = 3 * N // 4 * 2
    t15 = np.zeros(n, np.int16); t31 = np.zeros(n, np.int32)
    assert lib.slb_design_twiddle_q15(N, t15.ctypes.data) == 0 and lib.slb_design_twiddle_q31(N, t31.ctypes.data) == 0
    m15, m31 = model.twiddle_q15(N), model.twiddle_q31(N)
    assert np.array_equal(t15, m15) and np.array_equal(t31, m31)
    a = 2 * np.pi * np.arange(3 * N // 4) / N
    exact = np.stack([np.cos(a), np.sin(a)], 1).reshape(-1)
    assert np.max(np.abs(m15 / 32768.0 - exact)) <= 1.0 / 32768
    assert np.max(np.abs(m31 / 2.0**31 - exact)) <= 1.0 / 2.0**31
    assert m15[0] == 32767 and m31[0] == 2**31 - 1                   # cos 0 = +1.0, clipped


@pytest.mark.parametrize("N", model.SIZES)
def test_model_equals_the_reference_build(ref, N):
    rng = np.random.Generator(np.random.PCG64(N))
    for amp in (5000, 32767):
        x15 = rng.integers(-amp, amp + 1, (4, 2 * N)).astype(np.int16)
        x31 = rng.integers(-(amp << 16), (amp << 16) + 1, (4, 2 * N)).astype(np.int32)
        for ifft in (0, 1):
            for i in range(len(x15)):
                assert np.array_equal(model.cfft_q15(x15[i], ifft), ref.cfft_q15_cm4(x15[i], ifft)), ("q15", N, amp, ifft, i)
                assert np.array_equal(model.cfft_q31(x31[i], ifft), ref.cfft_q31(x31[i], ifft)), ("q31", N, amp, ifft, i)
