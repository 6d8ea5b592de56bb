"""GPU parity of the batched stage library (slb_st_*) against the oracle, routine by routine, through the C ABI.
Integer routines and the sequential float routines: bit-exact. FFT: 2e-6 of output RMS."""
import numpy as np
import pytest

import oracle_lib
import selenite_lite_b200 as slb

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

C, B, NB = 3, 48, 7
N = B * NB


@pytest.fixture(scope="module")
def ctx():
    return slb.DspIf(C, chain=slb.CHAIN_PASS)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def q15(rng, *shape, amp=32767):
    return rng.integers(-amp, amp + 1, shape).astype(np.int16)


def f32(rng, *shape, amp=1.0):
    return (rng.standard_normal(shape) * amp).astype(np.float32)


def test_elementwise_float(ctx, best_oracle, rng):
    a, b = f32(rng, C, N), f32(rng, C, N)
    o = best_oracle
    for name, args, exp in (
        ("scale_f32", (dev(a), 0.37), lambda: np.stack([o.scale_f32(a[c], 0.37) for c in range(C)])),
        ("mult_f32", (dev(a), dev(b)), lambda: np.stack([o.mult_f32(a[c], b[c]) for c in range(C)])),
        ("add_f32", (dev(a), dev(b)), lambda: np.stack([o.add_f32(a[c], b[c]) for c in range(C)])),
        ("sub_f32", (dev(a), dev(b)), lambda: np.stack([o.sub_f32(a[c], b[c]) for c in range(C)])),
        ("abs_f32", (dev(a),), lambda: np.stack([o.abs_f32(a[c]) for c in range(C)])),
    ):
        d = torch.zeros((C, N), dtype=torch.float32, device="cuda")
        ctx.st(name, *args, d, N)
        assert np.array_equal(d.cpu().numpy(), exp()), name


def test_conversions(ctx, best_oracle, rng):
    x = q15(rng, C, N); x[0, :4] = [-32768, 32767, 0, -1]
    d = torch.zeros((C, N), dtype=torch.float32, device="cuda")
    ctx.st("q15_to_float", dev(x), d, N)
    assert np.array_equal(d.cpu().numpy(), best_oracle.q15_to_float(x))
    f = f32(rng, C, N, amp=0.6); f[1, :6] = [1.5, -1.5, 0.99999, -1.0, 3.05e-5, -3.05e-5]
    q = torch.zeros((C, N), dtype=torch.int16, device="cuda")
    ctx.st("float_to_q15", dev(f), q, N)
    assert np.array_equal(q.cpu().numpy(), best_oracle.float_to_q15(f))


def test_elementwise_q15(ctx, best_oracle, rng):
    a, b = q15(rng, C, N), q15(rng, C, N); a[0, :4] = [-32768, 32767, 0, -1]
    o = best_oracle
    d = torch.zeros((C, N), dtype=torch.int16, device="cuda")
    for k, sh in ((12345, 0), (-32768, 1), (32767, 3), (700, -2)):
        ctx.st("scale_q15", dev(a), k, sh, d, N)
        assert np.array_equal(d.cpu().numpy(), np.stack([o.scale_q15(a[c], k, sh) for c in range(C)])), (k, sh)
    for name in ("add_q15", "sub_q15"):
        ctx.st(name, dev(a), dev(b), d, N)
        assert np.array_equal(d.cpu().numpy(), np.stack([getattr(o, name)(a[c], b[c]) for c in range(C)])), name
    ctx.st("abs_q15", dev(a), d, N)
    assert np.array_equal(d.cpu().numpy(), np.stack([o.abs_q15(a[c]) for c in range(C)]))
    for sh in (-3, 0, 2):
        ctx.st("shift_q15", dev(a), sh, d, N)
        assert np.array_equal(d.cpu().numpy(), np.stack([o.shift_q15(a[c], sh) for c in range(C)])), sh


def test_complex_math(ctx, best_oracle, rng):
    a, b = f32(rng, C, 2 * N), f32(rng, C, 2 * N); r = f32(rng, C, N)
    o = best_oracle
    d2 = torch.zeros((C, 2 * N), dtype=torch.float32, device="cuda"); d1 = torch.zeros((C, N), dtype=torch.float32, device="cuda")
    ctx.st("cmplx_mult_cmplx_f32", dev(a), dev(b), d2, N)
    assert np.array_equal(d2.cpu().numpy(), np.stack([o.cmplx_mult_cmplx_f32(a[c], b[c]) for c in range(C)]))
    ctx.st("cmplx_mult_real_f32", dev(a), dev(r), d2, N)
    assert np.array_equal(d2.cpu().numpy(), np.stack([o.cmplx_mult_real_f32(a[c], r[c]) for c in range(C)]))
    ctx.st("cmplx_conj_f32", dev(a), d2, N)
    assert np.array_equal(d2.cpu().numpy(), np.stack([o.cmplx_conj_f32(a[c]) for c in range(C)]))
    for name in ("cmplx_mag_f32", "cmplx_mag_squared_f32"):
        ctx.st(name, dev(a), d1, N)
        assert np.array_equal(d1.cpu().numpy(), np.stack([getattr(o, name)(a[c]) for c in range(C)])), name
    q = q15(rng, C, 2 * N); dq = torch.zeros((C, N), dtype=torch.int16, device="cuda")
    ctx.st("cmplx_mag_q15", dev(q), dq, N)
    assert np.array_equal(dq.cpu().numpy(), np.stack([o.cmplx_mag_q15(q[c]) for c in range(C)]))


def test_sin_cos_table(ctx, best_oracle, rng):
    x = (rng.random((C, N)) * 40 - 20).astype(np.float32); x[0, :3] = [0, -1e-7, 6.2831855]
    d = torch.zeros((C, N), dtype=torch.float32, device="cuda")
    ctx.st("sin_f32", dev(x), d, N)
    assert np.array_equal(d.cpu().numpy(), best_oracle.sin_f32(x.reshape(-1)).reshape(C, N))
    ctx.st("cos_f32", dev(x), d, N)
    assert np.array_equal(d.cpu().numpy(), best_oracle.cos_f32(x.reshape(-1)).reshape(C, N))


@pytest.mark.parametrize("name,dt,ntaps", [("fir_f32", np.float32, 64), ("fir_f32", np.float32, 129), ("fir_q15", np.int16, 64),
                                           ("fir_fast_q15", np.int16, 64), ("fir_q31", np.int32, 32)])
def test_fir_family_bit_exact_with_carried_state(ctx, best_oracle, rng, name, dt, ntaps):
    if dt == np.float32:
        c, x = f32(rng, ntaps, amp=0.1), f32(rng, C, 2 * N)
    elif dt == np.int16:
        c, x = q15(rng, ntaps, amp=6000), q15(rng, C, 2 * N)
    else:
        c = rng.integers(-2**28, 2**28, ntaps).astype(np.int32); x = rng.integers(-2**31, 2**31 - 1, (C, 2 * N)).astype(np.int32)
    tdt = {np.float32: torch.float32, np.int16: torch.int16, np.int32: torch.int32}[dt]
    hist = torch.zeros((C, ntaps - 1), dtype=tdt, device="cuda")
    outs = []
    for part in (x[:, :N], x[:, N:]):                       # two calls: the history must carry
        d = torch.zeros((C, N), dtype=tdt, device="cuda")
        ctx.st(name, c, ntaps, hist, dev(part), d, N)
        outs.append(d.cpu().numpy())
    got = np.concatenate(outs, 1)
    for ch in range(C):
        exp, _ = getattr(best_oracle, name)(c, np.zeros(ntaps + B, dt), x[ch], B)
        assert np.array_equal(got[ch], exp), (name, ch)


def run_fir_calls(ctx, name, c, x, lengths, tdt):
    """One FIR call per entry of `lengths`, over consecutive pieces of x [C][sum(lengths)], the history carried between calls."""
    hist = torch.zeros((C, len(c) - 1), dtype=tdt, device="cuda")
    outs, a = [], 0
    for n in lengths:
        d = torch.zeros((C, n), dtype=tdt, device="cuda")
        ctx.st(name, c, len(c), hist, dev(x[:, a:a + n]), d, n)
        outs.append(d.cpu().numpy()); a += n
    return np.concatenate(outs, 1), hist.cpu().numpy()


@pytest.mark.parametrize("name", ["fir_f32", "fir_q31"])
def test_fir_grid_stride_and_short_calls_with_carried_state(ctx, best_oracle, rng, name):
    """fir_common caps the grid at 1024 x 256 threads: only a call of more than 262 144 outputs per channel runs the grid-stride
    loop of fir_kernel (two calls of 300 000 here). A call shorter than the history (n < ntaps - 1) leaves a new history that is
    partly the old one; the call after it shows whether that history was right."""
    if name == "fir_f32":
        dt, tdt, c = np.float32, torch.float32, f32(rng, 129, amp=0.1)
        x = f32(rng, C, 600000)
    else:
        dt, tdt, c = np.int32, torch.int32, rng.integers(-2**28, 2**28, 64).astype(np.int32)
        x = rng.integers(-2**31, 2**31 - 1, (C, 600000)).astype(np.int32)
    ntaps = len(c)
    short = 96 if ntaps == 129 else 48                        # a whole number of oracle blocks, shorter than the history
    for lengths in ((300000, 300000), (480, short, 480)):
        xs = x[:, :sum(lengths)]
        got, hist = run_fir_calls(ctx, name, c, xs, lengths, tdt)
        for ch in range(C):
            exp, _ = getattr(best_oracle, name)(c, np.zeros(ntaps + B, dt), xs[ch], B)
            assert np.array_equal(got[ch], exp), (name, lengths, ch, int(np.argmax(got[ch] != exp)))
            assert np.array_equal(hist[ch], xs[ch, -(ntaps - 1):]), (name, lengths, "history", ch)


def test_stage_calls_on_two_streams_do_not_share_staged_coefficients(ctx, best_oracle, rng):
    """The stage library stages a call's coefficients in the context's scratch buffer and consumes them on the caller's stream.
    Calls of one context on DIFFERENT streams are ordered through that buffer (ctx_scratch_on), so a second filter's
    coefficients cannot replace the first's before its kernel has read them: 40 alternating calls with two tap sets on two
    streams, every result bit-exact."""
    ca, cb = f32(rng, 64, amp=0.1), f32(rng, 64, amp=0.1)
    x = f32(rng, C, 16 * N)
    xd = dev(x)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    outs = []
    for i in range(40):
        c, s = (ca, sa) if i % 2 == 0 else (cb, sb)
        hist = torch.zeros((C, 63), dtype=torch.float32, device="cuda"); d = torch.zeros((C, 16 * N), dtype=torch.float32, device="cuda")
        ctx.st("fir_f32", c, 64, hist, xd, d, 16 * N, stream=s.cuda_stream)
        outs.append(d)
    torch.cuda.synchronize()
    exp = [np.stack([best_oracle.fir_f32(c, np.zeros(64 + B, np.float32), x[ch], B)[0] for ch in range(C)]) for c in (ca, cb)]
    for i, d in enumerate(outs):
        assert np.array_equal(d.cpu().numpy(), exp[i % 2]), i


def test_fir_decimate_interpolate(ctx, best_oracle, rng):
    c, x = f32(rng, 64, amp=0.1), f32(rng, C, 2 * N)
    cq, xq = q15(rng, 64, amp=4000), q15(rng, C, 2 * N)
    for name, cc, xx, tdt, dt in (("f32", c, x, torch.float32, np.float32), ("q15", cq, xq, torch.int16, np.int16)):
        hist = torch.zeros((C, 63), dtype=tdt, device="cuda"); outs = []
        for part in (xx[:, :N], xx[:, N:]):
            d = torch.zeros((C, N // 4), dtype=tdt, device="cuda")
            ctx.st("fir_decimate_" + name, cc, 64, 4, hist, dev(part), d, N); outs.append(d.cpu().numpy())
        got = np.concatenate(outs, 1)
        for ch in range(C):
            assert np.array_equal(got[ch], getattr(best_oracle, "fir_decimate_" + name)(cc, 4, np.zeros(64 + B, dt), xx[ch], B)[0]), ("dec", name, ch)
        hist = torch.zeros((C, 15), dtype=tdt, device="cuda"); outs = []
        for part in (xx[:, :N], xx[:, N:]):
            d = torch.zeros((C, N * 4), dtype=tdt, device="cuda")
            ctx.st("fir_interpolate_" + name, cc, 64, 4, hist, dev(part), d, N); outs.append(d.cpu().numpy())
        got = np.concatenate(outs, 1)
        for ch in range(C):
            assert np.array_equal(got[ch], getattr(best_oracle, "fir_interpolate_" + name)(cc, 4, np.zeros(64 + B, dt), xx[ch], B)[0]), ("int", name, ch)


def test_fir_decimate_interpolate_q31(ctx, best_oracle, rng):
    """arm_fir_decimate_q31.c:60 / arm_fir_interpolate_q31.c:62, bit-exact with the history carried across two calls."""
    c31 = rng.integers(-2**27, 2**27, 64).astype(np.int32); xx = rng.integers(-2**31, 2**31 - 1, (C, 2 * N)).astype(np.int32)
    for M in (2, 4):
        hist = torch.zeros((C, 63), dtype=torch.int32, device="cuda"); outs = []
        for part in (xx[:, :N], xx[:, N:]):
            d = torch.zeros((C, N // M), dtype=torch.int32, device="cuda")
            ctx.st("fir_decimate_q31", c31, 64, M, hist, dev(part), d, N); outs.append(d.cpu().numpy())
        got = np.concatenate(outs, 1)
        for ch in range(C):
            assert np.array_equal(got[ch], best_oracle.fir_decimate_q31(c31, M, np.zeros(64 + B, np.int32), xx[ch], B)[0]), ("dec", M, ch)
        hist = torch.zeros((C, 64 // M - 1), dtype=torch.int32, device="cuda"); outs = []
        for part in (xx[:, :N], xx[:, N:]):
            d = torch.zeros((C, N * M), dtype=torch.int32, device="cuda")
            ctx.st("fir_interpolate_q31", c31, 64, M, hist, dev(part), d, N); outs.append(d.cpu().numpy())
        got = np.concatenate(outs, 1)
        for ch in range(C):
            assert np.array_equal(got[ch], best_oracle.fir_interpolate_q31(c31, M, np.zeros(64 + B, np.int32), xx[ch], B)[0]), ("int", M, ch)


@pytest.mark.parametrize("N", [16, 32, 64, 128, 256, 512, 1024, 2048, 4096])
@pytest.mark.parametrize("ifft", [0, 1])
def test_cfft_q15_q31_bit_exact(ctx, rng, N, ifft):
    """arm_cfft_q15 (arm_cfft_q15.c:77, the ARM_MATH_DSP branch of the firmware's Cortex-M4 build) and arm_cfft_q31 (arm_cfft_q31.c:77),
    batched [channels][count][2 N] in place: bit for bit against the reference build (every size: both the pure radix-4 and the
    radix-4-by-2 decompositions), moderate and rail-to-rail inputs (the q15 lane sums saturate)."""
    try:
        ref = oracle_lib.Oracle("ref")
    except (FileNotFoundError, OSError):
        pytest.skip("reference build absent: the committed vectors (test_cfft_fixed_golden_vectors) are the check")
    count = 3
    for amp in (5000, 32767):
        x15 = rng.integers(-amp, amp + 1, (C, count, 2 * N)).astype(np.int16)
        x31 = rng.integers(-(amp << 16), (amp << 16) + 1, (C, count, 2 * N)).astype(np.int32)
        d15 = dev(x15); d31 = dev(x31)
        ctx.st("cfft_q15", d15, N, count, ifft); ctx.st("cfft_q31", d31, N, count, ifft)
        g15, g31 = d15.cpu().numpy(), d31.cpu().numpy()
        for ch in range(C):
            for k in range(count):
                assert np.array_equal(g15[ch, k], ref.cfft_q15_cm4(x15[ch, k], ifft)), ("q15", N, amp, ch, k)
                assert np.array_equal(g31[ch, k], ref.cfft_q31(x31[ch, k], ifft)), ("q31", N, amp, ch, k)


def test_cfft_fixed_golden_vectors(ctx):
    """The same transforms against vectors committed from the reference build (tests/golden/make_golden.py fft_fixed)."""
    import os
    from test_golden import GOLD
    g = np.load(os.path.join(GOLD, "cfft_fixed.npz"))
    for key in g.files:
        if not key.endswith("_in"):
            continue
        kind, N, tag, _ = key.split("_"); N = int(N)
        x = np.tile(g[key], (C, 1, 1))
        for ifft in (0, 1):
            d = dev(x)
            ctx.st("cfft_" + kind, d, N, 1, ifft)
            got = d.cpu().numpy()
            for ch in range(C):
                assert np.array_equal(got[ch, 0], g["%s_%d_%s_%d" % (kind, N, tag, ifft)]), (key, ifft, ch)


@pytest.mark.parametrize("ntaps", [8, 32, 64])
def test_lms_norm_f32_bit_exact_with_carried_state(ctx, best_oracle, rng, ntaps):
    """arm_lms_norm_f32.c:161 per channel (every channel adapts its own coefficients): output, error, coefficients and the carried
    instance (history, energy, x0) bit for bit, over two calls of ragged length; and the auto-notch it is for."""
    n1, n2 = 48 * 30 + 17, 48 * 20
    t = np.arange(n1 + n2)
    d = np.stack([(0.3 * np.sin(2 * np.pi * (700.0 + 90.0 * ch) * t / 48000.0) + 0.05 * rng.standard_normal(t.size)) for ch in range(C)]).astype(np.float32)
    x = np.concatenate([np.zeros((C, 3), np.float32), d[:, :-3]], 1)
    coeffs = torch.zeros((C, ntaps), dtype=torch.float32, device="cuda"); state = torch.zeros((C, ntaps + 1), dtype=torch.float32, device="cuda")
    outs, errs = [], []
    for a, b in ((0, n1), (n1, n1 + n2)):
        o = torch.zeros((C, b - a), dtype=torch.float32, device="cuda"); e = torch.zeros_like(o)
        ctx.st("lms_norm_f32", coeffs, ntaps, 0.05, state, dev(x[:, a:b]), dev(d[:, a:b]), o, e, b - a)
        outs.append(o.cpu().numpy()); errs.append(e.cpu().numpy())
    got_o, got_e = np.concatenate(outs, 1), np.concatenate(errs, 1)
    cf, stt = coeffs.cpu().numpy(), state.cpu().numpy()
    for ch in range(C):
        eo, ee, ec, es, ex = best_oracle.lms_norm_f32(np.zeros(ntaps, np.float32), 0.05, np.zeros(ntaps + 1, np.float32), np.zeros(2, np.float32), x[ch], d[ch], 1)
        assert np.array_equal(got_o[ch], eo) and np.array_equal(got_e[ch], ee), ch
        assert np.array_equal(cf[ch], ec) and np.array_equal(stt[ch, :ntaps - 1], es[:ntaps - 1]) and np.array_equal(stt[ch, ntaps - 1:], ex), ch
    if ntaps >= 32:
        assert np.std(got_e[:, -2000:]) < 0.5 * np.std(d[:, -2000:])


@pytest.mark.parametrize("ntaps", [96, 128])
def test_lms_norm_f32_large_taps_partial_warp(best_oracle, rng, ntaps):
    """Above 84 taps the kernel's dynamic shared memory exceeds 48 KB (the opt-in attribute path), and 70 channels make three
    warps of channels, the last one partial (6 of 32 lanes): every channel bit for bit, over two calls of ragged length."""
    Cl = 70
    lctx = slb.DspIf(Cl, chain=slb.CHAIN_PASS)
    n1, n2 = 48 * 6 + 17, 48 * 4
    t = np.arange(n1 + n2)
    d = np.stack([(0.3 * np.sin(2 * np.pi * (500.0 + 37.0 * ch) * t / 48000.0) + 0.05 * rng.standard_normal(t.size)) for ch in range(Cl)]).astype(np.float32)
    x = np.concatenate([np.zeros((Cl, 3), np.float32), d[:, :-3]], 1)
    coeffs = torch.zeros((Cl, ntaps), dtype=torch.float32, device="cuda"); state = torch.zeros((Cl, ntaps + 1), dtype=torch.float32, device="cuda")
    outs, errs = [], []
    for a, b in ((0, n1), (n1, n1 + n2)):
        o = torch.zeros((Cl, b - a), dtype=torch.float32, device="cuda"); e = torch.zeros_like(o)
        lctx.st("lms_norm_f32", coeffs, ntaps, 0.05, state, dev(x[:, a:b]), dev(d[:, a:b]), o, e, b - a)
        outs.append(o.cpu().numpy()); errs.append(e.cpu().numpy())
    got_o, got_e = np.concatenate(outs, 1), np.concatenate(errs, 1)
    cf, stt = coeffs.cpu().numpy(), state.cpu().numpy()
    for ch in range(Cl):
        eo, ee, ec, es, ex = best_oracle.lms_norm_f32(np.zeros(ntaps, np.float32), 0.05, np.zeros(ntaps + 1, np.float32), np.zeros(2, np.float32), x[ch], d[ch], 1)
        assert np.array_equal(got_o[ch], eo) and np.array_equal(got_e[ch], ee), (ntaps, ch)
        assert np.array_equal(cf[ch], ec) and np.array_equal(stt[ch, :ntaps - 1], es[:ntaps - 1]) and np.array_equal(stt[ch, ntaps - 1:], ex), (ntaps, ch)


def test_biquads_at_the_stage_limit_and_q15_postshifts(ctx, best_oracle, rng):
    """SLB_MAX_STAGES = 4 stages for every biquad form (the existing test runs 2), and biquad_df1_q15 with postshift 0 and 2 beside
    the 1 tested elsewhere; state carried across two calls."""
    ns = slb._lib.MAX_STAGES
    cf = np.tile(np.array(slb.default_rx_f32_params(48000).biquad[:10], np.float32), 2)
    x = f32(rng, C, 2 * N, amp=0.3)
    for name, per_stage in (("biquad_df2T_f32", 2), ("biquad_df1_f32", 4)):
        st = torch.zeros((C, per_stage * ns), dtype=torch.float32, device="cuda"); outs = []
        for part in (x[:, :N], x[:, N:]):
            d = torch.zeros((C, N), dtype=torch.float32, device="cuda")
            ctx.st(name, cf, ns, st, dev(part), d, N); outs.append(d.cpu().numpy())
        got = np.concatenate(outs, 1)
        for ch in range(C):
            exp, est = getattr(best_oracle, name)(cf, ns, np.zeros(per_stage * ns, np.float32), x[ch], B)
            assert np.array_equal(got[ch], exp) and np.array_equal(st[ch].cpu().numpy(), est), (name, ch)
    xs = f32(rng, C, 2 * N, amp=0.3)
    st = torch.zeros((C, 4 * ns), dtype=torch.float32, device="cuda"); d = torch.zeros((C, 2 * N), dtype=torch.float32, device="cuda")
    ctx.st("biquad_stereo_df2T_f32", cf, ns, st, dev(xs), d, N)
    for ch in range(C):
        exp, est = best_oracle.biquad_stereo_df2T_f32(cf, ns, np.zeros(4 * ns, np.float32), xs[ch], B)
        assert np.array_equal(d[ch].cpu().numpy(), exp) and np.array_equal(st[ch].cpu().numpy(), est), ("stereo", ch)
    c15 = np.tile(np.array([8000, 0, -16000, 8000, 15000, -7000, 4000, 0, 8000, 4000, 9000, -3000], np.int16), 2)
    xq = q15(rng, C, 2 * N, amp=20000)
    for ps in (0, 2):
        st = torch.zeros((C, 4 * ns), dtype=torch.int16, device="cuda"); outs = []
        for part in (xq[:, :N], xq[:, N:]):
            d = torch.zeros((C, N), dtype=torch.int16, device="cuda")
            ctx.st("biquad_df1_q15", c15, ns, ps, st, dev(part), d, N); outs.append(d.cpu().numpy())
        got = np.concatenate(outs, 1)
        for ch in range(C):
            exp, est = best_oracle.biquad_df1_q15(c15, ns, ps, np.zeros(4 * ns, np.int16), xq[ch], B)
            assert np.array_equal(got[ch], exp) and np.array_equal(st[ch].cpu().numpy(), est), ("df1_q15", ps, ch)
    c31 = np.tile((np.array([0.25, -0.5, 0.25, 0.45, -0.2, 0.12, 0.24, 0.12, 0.27, -0.09]) * 2**31).astype(np.int64).astype(np.int32), 2)
    x31 = rng.integers(-2**30, 2**30, (C, 2 * N)).astype(np.int32)
    st = torch.zeros((C, 4 * ns), dtype=torch.int32, device="cuda"); outs = []
    for part in (x31[:, :N], x31[:, N:]):
        d = torch.zeros((C, N), dtype=torch.int32, device="cuda")
        ctx.st("biquad_df1_q31", c31, ns, 1, st, dev(part), d, N); outs.append(d.cpu().numpy())
    got = np.concatenate(outs, 1)
    for ch in range(C):
        exp, est = best_oracle.biquad_df1_q31(c31, ns, 1, np.zeros(4 * ns, np.int32), x31[ch], B)
        assert np.array_equal(got[ch], exp) and np.array_equal(st[ch].cpu().numpy(), est), ("df1_q31", ch)


def test_biquads_bit_exact_with_carried_state(ctx, best_oracle, rng):
    p = slb.default_rx_f32_params(48000)
    cf = np.array(p.biquad[:10], np.float32)
    x = f32(rng, C, 2 * N, amp=0.3)
    for name, per_stage in (("biquad_df2T_f32", 2), ("biquad_df1_f32", 4)):
        st = torch.zeros((C, per_stage * 2), dtype=torch.float32, device="cuda"); outs = []
        for part in (x[:, :N], x[:, N:]):
            d = torch.zeros((C, N), dtype=torch.float32, device="cuda")
            ctx.st(name, cf, 2, st, dev(part), d, N); outs.append(d.cpu().numpy())
        got = np.concatenate(outs, 1)
        for ch in range(C):
            exp, est = getattr(best_oracle, name)(cf, 2, np.zeros(per_stage * 2, np.float32), x[ch], B)
            assert np.array_equal(got[ch], exp), (name, ch)
            assert np.array_equal(st[ch].cpu().numpy(), est), (name, "state", ch)
    xs = f32(rng, C, 2 * N, amp=0.3)                         # N stereo frames
    st = torch.zeros((C, 8), dtype=torch.float32, device="cuda"); d = torch.zeros((C, 2 * N), dtype=torch.float32, device="cuda")
    ctx.st("biquad_stereo_df2T_f32", cf, 2, st, dev(xs), d, N)
    for ch in range(C):
        exp, est = best_oracle.biquad_stereo_df2T_f32(cf, 2, np.zeros(8, np.float32), xs[ch], B)
        assert np.array_equal(d[ch].cpu().numpy(), exp) and np.array_equal(st[ch].cpu().numpy(), est)
    c15 = np.array([8000, 0, -16000, 8000, 15000, -7000, 4000, 0, 8000, 4000, 9000, -3000], np.int16)
    xq = q15(rng, C, N, amp=20000)
    st = torch.zeros((C, 8), dtype=torch.int16, device="cuda"); d = torch.zeros((C, N), dtype=torch.int16, device="cuda")
    ctx.st("biquad_df1_q15", c15, 2, 1, st, dev(xq), d, N)
    for ch in range(C):
        exp, est = best_oracle.biquad_df1_q15(c15, 2, 1, np.zeros(8, np.int16), xq[ch], B)
        assert np.array_equal(d[ch].cpu().numpy(), exp) and np.array_equal(st[ch].cpu().numpy(), est)
    c31 = (np.array([0.25, -0.5, 0.25, 0.45, -0.2, 0.12, 0.24, 0.12, 0.27, -0.09]) * 2**31).astype(np.int64).astype(np.int32)
    x31 = rng.integers(-2**30, 2**30, (C, N)).astype(np.int32)
    st = torch.zeros((C, 8), dtype=torch.int32, device="cuda"); d = torch.zeros((C, N), dtype=torch.int32, device="cuda")
    ctx.st("biquad_df1_q31", c31, 2, 1, st, dev(x31), d, N)
    for ch in range(C):
        exp, est = best_oracle.biquad_df1_q31(c31, 2, 1, np.zeros(8, np.int32), x31[ch], B)
        assert np.array_equal(d[ch].cpu().numpy(), exp) and np.array_equal(st[ch].cpu().numpy(), est)


def test_block_statistics(ctx, best_oracle, rng):
    x = f32(rng, C, N); o = best_oracle
    out = torch.zeros((C, NB), dtype=torch.float32, device="cuda"); idx = torch.zeros((C, NB), dtype=torch.int32, device="cuda")
    ctx.st("max_f32", dev(x), N, B, out, idx)
    for c in range(C):
        for b in range(NB):
            v, i = o.max_f32(x[c, b * B:(b + 1) * B])
            assert out[c, b].item() == v and idx[c, b].item() == i
    for name in ("rms_f32", "power_f32", "mean_f32"):
        ctx.st(name, dev(x), N, B, out)
        exp = np.array([[getattr(o, name)(x[c, b * B:(b + 1) * B]) for b in range(NB)] for c in range(C)], np.float32)
        assert np.array_equal(out.cpu().numpy(), exp), name
    q = q15(rng, C, N)
    outq = torch.zeros((C, NB), dtype=torch.int16, device="cuda")
    ctx.st("max_q15", dev(q), N, B, outq, idx)
    assert np.array_equal(outq.cpu().numpy(), np.array([[o.max_q15(q[c, b * B:(b + 1) * B])[0] for b in range(NB)] for c in range(C)]))
    ctx.st("rms_q15", dev(q), N, B, outq)
    assert np.array_equal(outq.cpu().numpy(), np.array([[o.rms_q15(q[c, b * B:(b + 1) * B]) for b in range(NB)] for c in range(C)]))


@pytest.mark.parametrize("nfft", [16, 64, 256, 512, 1024, 4096])
def test_batched_cfft(ctx, best_oracle, rng, nfft):
    cnt = 2
    x = f32(rng, C, cnt, 2 * nfft)
    for ifft in (0, 1):
        d = dev(x)
        ctx.st("cfft_f32", d, nfft, cnt, ifft)
        got = d.cpu().numpy()
        for c in range(C):
            for k in range(cnt):
                exp = best_oracle.cfft_f32(x[c, k], ifft, 1)
                rms = np.sqrt(np.mean(exp.astype(np.float64) ** 2))
                assert np.max(np.abs(got[c, k] - exp)) <= 3e-6 * rms, (nfft, ifft)


@pytest.mark.parametrize("nfft", [32, 128, 512, 2048, 4096])
def test_batched_rfft_fast(ctx, best_oracle, rng, nfft):
    """arm_rfft_fast_f32: forward packing (X[0], X[N/2], then Re/Im pairs) and the inverse, tolerance class of the float FFTs."""
    cnt = 2
    x = f32(rng, C, cnt, nfft)
    out = torch.zeros((C, cnt, nfft), dtype=torch.float32, device="cuda")
    ctx.st("rfft_fast_f32", dev(x), out, nfft, cnt, 0)
    spec = out.cpu().numpy()
    back = torch.zeros_like(out)
    ctx.st("rfft_fast_f32", out, back, nfft, cnt, 1)
    back = back.cpu().numpy()
    for c in range(C):
        for k in range(cnt):
            exp = best_oracle.rfft_fast_f32(x[c, k], 0)
            rms = np.sqrt(np.mean(exp.astype(np.float64) ** 2))
            assert np.max(np.abs(spec[c, k] - exp)) <= 3e-6 * rms, nfft
            exp_b = best_oracle.rfft_fast_f32(exp, 1)
            assert np.max(np.abs(back[c, k] - exp_b)) <= 3e-6 * np.sqrt(np.mean(exp_b.astype(np.float64) ** 2)), nfft


@pytest.mark.parametrize("nfft", [64, 1024])
def test_spectrum_export(best_oracle, rng, nfft):
    """slb_rx_spectrum_device = arm_q15_to_float -> arm_cfft_f32 -> arm_cmplx_mag_squared_f32 per channel."""
    Cs = 5
    x = slb.synth_iq(Cs, nfft)
    d = slb.DspIf(Cs, chain=slb.CHAIN_RX_SSB_F32)
    got = d.spectrum(torch.from_numpy(x).cuda()).cpu().numpy()
    o = best_oracle
    for c in range(Cs):
        f = o.q15_to_float(x[c].reshape(-1))
        exp = o.cmplx_mag_squared_f32(o.cfft_f32(f, 0, 1))
        assert np.max(np.abs(got[c] - exp)) <= 1e-5 * np.max(exp), (nfft, c)
    assert int(np.argmax(got[0])) == int(round(slb.channel_tone_hz(0) * nfft / 48000.0))     # the tone sits in its bin
