"""GPU parity of the integer channelizer CHAN-64-q15 (DESIGN.md §3.10), called through the C ABI, against the oracle (the port's chan_q15,
oracle/slo_chan_q15.h) and the golden vectors: output, pre-AGC detector output and gain words byte for byte."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_chan_q15 as ocq
import selenite_lite_b200 as slb
from selenite_lite_b200 import build as _build
from test_golden import GOLD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CH, FS = slb.CHAIN_CHAN64_Q15, 192000


def ctx(streams, mode=None, **over):
    d = slb.DspIf(streams, fs=FS, chain=CH)
    if mode is not None:
        d.DSP_Set_Mode(mode)
    if over:
        p = d.chan_q15_params()
        for k, v in over.items():
            setattr(p, k, v)
        d.set_chan_q15_params(p)
    return d


def run_gpu(d, x, want_dbg=True):
    S, T = x.shape[0], x.shape[1]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    audio = torch.zeros((S, 64, T // 64), dtype=torch.int16, device="cuda") if want_dbg else None
    gain = torch.zeros((S, 64, T // 192), dtype=torch.int32, device="cuda") if want_dbg else None
    d.set_q15_debug_taps(audio, gain)
    y = d.chan_process(xd)
    torch.cuda.synchronize()
    d.set_q15_debug_taps(None, None)
    return y.cpu().numpy(), (audio.cpu().numpy() if want_dbg else None), (gain.cpu().numpy().view(np.uint32) if want_dbg else None)


def check(port, d, x, y, audio, gain, states=None):
    exp, ea, eg = ocq.chan_batch(port, d.oracle_params(), x, states)
    for s in range(x.shape[0]):
        assert np.array_equal(y[s], exp[s]), (s, np.argwhere(np.any(y[s] != exp[s], -1))[:4])
        if audio is not None:
            assert np.array_equal(audio[s], ea[s]), s
            assert np.array_equal(gain[s], eg[s]), s


def rails(T):
    n = np.arange(T)
    tone = np.exp(2j * np.pi * (5 * 3000.0) * n / FS)
    full = np.stack([np.clip(np.rint(tone.real * 32767), -32768, 32767), np.clip(np.rint(tone.imag * 32767), -32768, 32767)], 1)
    sq = np.stack([np.where(n % 128 < 64, 32767, -32768), np.where(n % 40 < 20, -32768, 32767)], 1)
    return np.stack([np.full((T, 2), -32768), np.full((T, 2), 32767), sq, full]).astype(np.int16)


@pytest.mark.parametrize("name,mode", [("product", slb.MODE_USB), ("envelope", slb.MODE_AM), ("rail", slb.MODE_LSB)])
def test_golden_vectors(name, mode):
    g = np.load(os.path.join(GOLD, "chan64_q15.npz"))
    d = ctx(1, mode)
    assert np.array_equal(np.array(d.chan_q15_params().proto[:], np.int16), g["proto"])
    y, audio, gain = run_gpu(d, g["%s_in" % name][None])
    assert np.array_equal(y[0], g["%s_out" % name]) and np.array_equal(audio[0], g["%s_audio" % name]) and np.array_equal(gain[0], g["%s_gain" % name])


@pytest.mark.parametrize("streams,frames,mode", [(1, 768, slb.MODE_USB), (2, 6144, slb.MODE_AM), (3, 6144 + 768, slb.MODE_USB),
                                                 (5, 6144 * 3, slb.MODE_AM), (9, 6144 * 2 + 768 * 5, slb.MODE_USB)])
def test_vs_oracle_ragged_shapes(port, streams, frames, mode):
    """A single partial tile, exactly one tile, ragged last tiles, several tiles chained by the published block peaks."""
    x = slb.synth_wideband(streams, frames)
    d = ctx(streams, mode)
    check(port, d, x, *run_gpu(d, x))


@pytest.mark.parametrize("mode", [slb.MODE_USB, slb.MODE_AM])
def test_rail_to_rail_and_full_scale_tones(port, mode):
    """Both rails held at -32768 and at +32767 (DC in bin 0), rail-to-rail squares, a full-scale complex tone at the centre of bin 5."""
    x = rails(6144 * 2 + 768)
    d = ctx(4, mode)
    check(port, d, x, *run_gpu(d, x))


@pytest.mark.parametrize("window", [1, 16, 17])
def test_loud_tile_then_quiet_ones(port, rng, window):
    """A loud first tile, then quiet ones: the gains of the first blocks of each later tile look back across the tile boundary."""
    T = 3072 * 5
    x = (rng.integers(-40, 40, (3, T, 2))).astype(np.int16)
    x[:, :3072] = rails(3072)[[3, 2, 0]]
    x[1, 3072 * 2 + 1000:3072 * 2 + 1300] = 25000                           # a burst in the middle of a later tile
    d = ctx(3, slb.MODE_USB, agc_window=window)
    check(port, d, x, *run_gpu(d, x))


def test_window_18_and_bad_geometry_are_refused():
    d = ctx(1)
    before = bytes(memoryview(d.chan_q15_params()))
    for field, value in (("agc_window", 18), ("bins", 32), ("taps_per_branch", 16), ("agc_block", 6)):
        p = d.chan_q15_params(); setattr(p, field, value)
        with pytest.raises(slb.SeleniteError, match="-4"):
            d.set_chan_q15_params(p)
        assert bytes(memoryview(d.chan_q15_params())) == before, field


def test_calls_cut_at_768_frames_and_checkpoint(port, rng):
    S, T = 3, 768 * 12
    x = np.concatenate([slb.synth_wideband(S, 768 * 8), rng.integers(-2000, 2000, (S, 768 * 4, 2)).astype(np.int16)], 1)
    whole = ctx(S, slb.MODE_AM, agc_window=17)
    yw, aw, gw = run_gpu(whole, x)
    check(port, whole, x, yw, aw, gw)
    d = ctx(S, slb.MODE_AM, agc_window=17)
    parts = []
    for c0 in range(0, 768 * 7, 768):
        parts.append(run_gpu(d, x[:, c0:c0 + 768]))
    snap = d.state_save()
    rest = run_gpu(d, x[:, 768 * 7:])
    e = ctx(S, slb.MODE_AM, agc_window=17)
    e.state_load(snap)
    again = run_gpu(e, x[:, 768 * 7:])
    for k in range(3):
        assert np.array_equal(np.concatenate([p[k] for p in parts] + [rest[k]], 2), (yw, aw, gw)[k]), k
        assert np.array_equal(again[k], rest[k]), k
    # SLB_DSP_Init clears the FIR history and the peaks: the next call equals a fresh context
    d.DSP_Init()
    assert np.array_equal(run_gpu(d, x[:, :768 * 2])[0], run_gpu(ctx(S, slb.MODE_AM, agc_window=17), x[:, :768 * 2])[0])


def test_64_streams_shards_and_host_path():
    """Config 4's width: shards of 2 and 8 ranks equal the whole, and the host path equals the device path, bit for bit."""
    S, T = 64, 6144 * 2
    x = slb.synth_wideband(S, T)
    whole, _, _ = run_gpu(ctx(S), x, want_dbg=False)
    for world in (2, 8):
        for rank in range(world):
            lo, hi = slb.shard.shard_range(S, rank, world)
            y, _, _ = run_gpu(ctx(hi - lo), x[lo:hi], want_dbg=False)
            assert np.array_equal(y, whole[lo:hi]), (world, rank)
    h = ctx(S)
    assert np.array_equal(h.chan_process(x), whole)
    assert np.array_equal(h.chan_process(x), run_gpu(ctx(S), np.concatenate([x, x], 1), want_dbg=False)[0][:, :, T // 64:])


def test_refusals():
    for fs in (48000, 96000):
        with pytest.raises(slb.SeleniteError, match="-1"):
            slb.DspIf(2, fs=fs, chain=CH)
    d = ctx(2)
    with pytest.raises(slb.SeleniteError, match="-4"):
        d.DSP_Set_Mode(slb.MODE_FM)
    assert d.chan_q15_params().envelope == 0
    blk = np.zeros((2, 384), np.int16)
    for call in (lambda: d.DSP_In_Buff_Write(blk), lambda: d.DSP_In_Buff_Read(768), lambda: d.DSP_Out_Buff_Write(blk),
                 lambda: d.DSP_Out_Buff_Read(384), lambda: d.DSP_In_Buff_Write_Ch(blk), lambda: d.DSP_Set_Sidetone(700, 0.1),
                 lambda: d.feeder_run(adc=np.zeros((2, 192 * 8, 2), np.int16)), lambda: d.live_open(8)):
        with pytest.raises(slb.SeleniteError, match="-4"):
            call()
    with pytest.raises(slb.SeleniteError, match="-3"):
        d.rx_process(torch.zeros((2, 768, 2), dtype=torch.int16, device="cuda"))
    with pytest.raises(slb.SeleniteError, match="-1"):
        d.chan_process(torch.zeros((2, 768 + 64, 2), dtype=torch.int16, device="cuda"))
    with pytest.raises(slb.SeleniteError, match="-3"):
        d.set_chan_params(slb.default_chan_params())
    for other in (slb.DspIf(2, fs=FS, chain=slb.CHAIN_CHAN64_F32), slb.DspIf(2, chain=slb.CHAIN_RX_SSB_Q15)):
        with pytest.raises(slb.SeleniteError, match="-3"):
            other.chan_q15_params()
        with pytest.raises(slb.SeleniteError, match="-3"):
            other.set_chan_q15_params(slb.default_chan_q15_params())


@pytest.mark.timeout(900, method="thread")
def test_scale_1024_streams_2s(port):
    """1024 wideband streams x 2 s: sampled streams against the oracle."""
    S, T = 1024, 384000
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    x = torch.randint(-9000, 9000, (S, T, 2), dtype=torch.int16, device="cuda", generator=g)
    d = ctx(S)
    y = d.chan_process(x)
    torch.cuda.synchronize()
    for s in (0, 1, 147, 511, 512, 1023):
        exp = ocq.chan_q15(port, d.oracle_params(), x[s].cpu().numpy())[0]
        assert np.array_equal(y[s].cpu().numpy(), exp), s


@pytest.mark.timeout(1500, method="thread")
def test_parity_on_the_stress_build():
    """This file's parity tests on the stress build (random delays at every flag publication and poll), like
    tests/test_gpu_stress_build.py does for the other chains."""
    if not os.path.exists(_build.STRESS_LIB_PATH):
        pytest.skip("stress build not present (python __graft_entry__.py builds it)")
    env = dict(os.environ, SELENITE_B200_LIB=_build.STRESS_LIB_PATH)
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "900",
                        os.path.abspath(__file__), "-k", "not stress_build and not scale"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1400)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
