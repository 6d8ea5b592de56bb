"""slb_st_cfft_q15 / slb_st_cfft_q31 on the GPU against the bit-exact NumPy model of arm_cfft_q15 (DSP branch) / arm_cfft_q31
(fft_fixed_model.py, pinned by test_fft_fixed_model.py to the reference vectors and to the float64 DFT): bit for bit, at every
size 16 .. 4096, both directions, every transform of the batch, with inputs that drive the saturating lanes, the wrapping
doublings and the largest intermediate sums."""
import numpy as np
import pytest

import fft_fixed_model as model
import selenite_lite_b200 as slb

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

C, COUNT = 5, 3
FULL = {"q15": 32767, "q31": 2**31 - 1}
DTYPE = {"q15": np.int16, "q31": np.int32}
CLASSES = ("moderate", "rails_random", "rails_held", "tone", "impulse")
SLB_ERR_ARG = -1


@pytest.fixture(scope="module")
def ctx():
    return slb.DspIf(C, chain=slb.CHAIN_PASS)


def make_inputs(kind, N, cls, rng, count=COUNT):
    """[C][count][2 N], different data in every transform."""
    T, full = C * count, FULL[kind]
    lo, hi = -full - 1, full
    n = np.arange(N)
    if cls == "moderate":
        x = rng.integers(-(full + 1) // 8, (full + 1) // 8, (T, 2 * N))
    elif cls == "rails_random":
        x = rng.integers(lo, hi, (T, 2 * N), endpoint=True)
    elif cls == "rails_held":
        # every lane at one of the two rails (the q15 lane sums saturate), the first transform held at the negative rail throughout
        x = np.where(rng.random((T, 2 * N)) < 0.5, lo, hi)
        x[0] = lo
    elif cls == "tone":
        # full-scale single-bin tones (amplitude 2^15 / 2^31, clipped to the rails). The odd transforms take a random bin and phase;
        # the even ones bins N/16, 2 N/16, ... with the peak on an axis, where the q15 radix-4-by-2 doubling and the q31 sums wrap
        # in the reference (test_fft_fixed_model.py::test_full_scale_peak_wraps_as_in_the_reference): at every radix-4-by-2 size
        # and direction, some of them tell a wrapping doubling from a saturating one.
        t = np.arange(T)
        bins = np.where(t % 2 == 0, (N // 16) * (t // 2 + 1) % N, rng.integers(0, N, T))
        ph0 = np.where(t % 2 == 0, (t // 2 % 4) * np.pi / 2, rng.random(T) * 2 * np.pi)
        ph = 2 * np.pi * bins[:, None] * n[None] / N + ph0[:, None]
        x = np.stack([np.round((full + 1.0) * np.cos(ph)), np.round((full + 1.0) * np.sin(ph))], -1).reshape(T, 2 * N)
    else:
        # impulses at index 0 and N - 1, alternately, of random complex value up to the rails
        x = np.zeros((T, N, 2), np.int64)
        at = np.where(np.arange(T) % 2 == 0, 0, N - 1)
        x[np.arange(T), at] = rng.integers(lo, hi, (T, 2), endpoint=True)
        x = x.reshape(T, 2 * N)
    return np.clip(x, lo, hi).astype(DTYPE[kind]).reshape(C, count, 2 * N)


def gpu_cfft(ctx, kind, x, N, ifft, stream=None):
    d = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    ctx.st("cfft_" + kind, d, N, x.shape[1], ifft, stream=stream)
    return d


def assert_bit_exact(got, x, kind, ifft, what):
    """Every transform of the batch against the model; on a mismatch, name the first differing (channel, transform, sample)."""
    exp = model.cfft(kind, x, ifft)
    if not np.array_equal(got, exp):
        bad = np.argwhere(got != exp)[0]
        raise AssertionError("%s: first difference at (channel, transform, word) = %s: got %d, model %d; %d words differ"
                             % (what, tuple(bad), got[tuple(bad)], exp[tuple(bad)], int(np.count_nonzero(got != exp))))


@pytest.mark.parametrize("kind", ["q15", "q31"])
@pytest.mark.parametrize("N", model.SIZES)
@pytest.mark.parametrize("ifft", [0, 1])
def test_cfft_fixed_every_size_bit_exact(ctx, kind, N, ifft):
    rng = np.random.Generator(np.random.PCG64(7919 * N + 2 * ifft + (kind == "q31")))
    for cls in CLASSES:
        x = make_inputs(kind, N, cls, rng)
        got = gpu_cfft(ctx, kind, x, N, ifft).cpu().numpy()
        assert_bit_exact(got, x, kind, ifft, "%s N=%d ifft=%d %s" % (kind, N, ifft, cls))


@pytest.mark.parametrize("kind,N,ifft,count", [("q15", 4096, 0, 820), ("q31", 4096, 1, 820), ("q15", 32, 1, 8192), ("q31", 32, 0, 8192)])
def test_cfft_fixed_wide_batch(ctx, kind, N, ifft, count):
    """C x count = 4100 transforms of 4096 points or 40960 of 32 points: many waves of CTAs, the last rows of the batch checked
    like the first."""
    rng = np.random.Generator(np.random.PCG64(N + count))
    x = np.concatenate([make_inputs(kind, N, cls, rng, count // 4) for cls in ("moderate", "rails_random", "rails_held", "tone")], 1)
    got = gpu_cfft(ctx, kind, x, N, ifft).cpu().numpy()
    assert got.shape == (C, count, 2 * N)
    assert_bit_exact(got, x, kind, ifft, "%s N=%d ifft=%d wide" % (kind, N, ifft))


@pytest.mark.parametrize("kind", ["q15", "q31"])
def test_cfft_fixed_staged_twiddles_on_two_streams(ctx, kind):
    """Each call stages its twiddle table in the context's scratch buffer and consumes it on the caller's stream; calls on
    different streams are ordered through that buffer (ctx_scratch_on). 20 calls of N = 4096 on one stream alternate with 20 of
    N = 32 on another, on one context: every result is bit-exact, so no call ran with the other size's table."""
    rng = np.random.Generator(np.random.PCG64(4096 + (kind == "q31")))
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    jobs = []
    for i in range(40):
        N, count, s = (4096, 16, sa) if i % 2 == 0 else (32, 64, sb)
        x = make_inputs(kind, N, "rails_random" if i % 4 < 2 else "moderate", rng, count)
        jobs.append((N, x, torch.from_numpy(x).cuda()))
    torch.cuda.synchronize()
    for i, (N, x, d) in enumerate(jobs):
        ctx.st("cfft_" + kind, d, N, x.shape[1], i % 4 >= 2, stream=(sa if i % 2 == 0 else sb).cuda_stream)
    torch.cuda.synchronize()
    for N in (4096, 32):
        for ifft in (0, 1):
            sel = [j for j in range(40) if jobs[j][0] == N and (j % 4 >= 2) == ifft]
            got = np.stack([jobs[j][2].cpu().numpy() for j in sel])
            exp = model.cfft(kind, np.stack([jobs[j][1] for j in sel]), ifft)
            assert np.array_equal(got, exp), (kind, N, ifft, [sel[k] for k in range(len(sel)) if not np.array_equal(got[k], exp[k])])


@pytest.mark.parametrize("kind", ["q15", "q31"])
def test_cfft_fixed_refusals_launch_nothing(ctx, kind):
    """N = 8, 48, 8192 and count = 0 are refused with SLB_ERR_ARG before anything is staged or launched; the data is untouched."""
    x = make_inputs(kind, 4096, "moderate", np.random.Generator(np.random.PCG64(5)), 1)
    d = torch.from_numpy(x).cuda()
    fn = getattr(ctx.lib, "slb_st_cfft_" + kind)
    for N, count in ((8, 1), (48, 1), (8192, 1), (64, 0), (16, 0)):
        before = ctx.kernel_launches()
        assert fn(ctx.h, d.data_ptr(), N, count, 0, None) == SLB_ERR_ARG, (N, count)
        assert ctx.kernel_launches() == before, (N, count)
    torch.cuda.synchronize()
    assert np.array_equal(d.cpu().numpy(), x)
    before = ctx.kernel_launches()
    assert fn(ctx.h, d.data_ptr(), 16, 1, 0, None) == 0                    # and the context still works
    assert ctx.kernel_launches() == before + 1
