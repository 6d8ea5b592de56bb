"""GPU parity of the all-mode integer receiver RX-Q15 (SLB_CHAIN_RX_Q15, DESIGN.md §3.8: the SSB-style modes exactly as RX-SSB-q15, AM by
arm_cmplx_mag_q15, FM by the integer limiter-discriminator, all on the integer tensor cores), called through the C ABI, against the oracle
(oracle/slo_rx_q15.h through tests/oracle_rx_q15.py), RX-SSB-q15 itself and the committed golden vectors. Every stage is integer
arithmetic, so every comparison is BIT-EXACT: pre-AGC detector output, per-block gain word, output and carried state."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_rx_q15 as orq
import selenite_lite_b200 as slb
import test_gpu_ring as ring
from selenite_lite_b200 import build as _build
from test_golden import GOLD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CH = slb.CHAIN_RX_Q15
MODES = [slb.MODE_USB, slb.MODE_AM, slb.MODE_LSB, slb.MODE_FM, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG, slb.MODE_PKT]
ERR_STATE, ERR_UNSUPPORTED = -3, -4


def synth(Cn, T, seed=1):
    """Per channel: an AM carrier (50 % depth, 1 kHz), an FM signal (2.5 kHz deviation, 1 kHz) or the SSB test signal, by channel."""
    x = slb.synth_iq(Cn, T)
    n = np.arange(T)
    rng = np.random.Generator(np.random.PCG64(seed))
    for c in range(Cn):
        if MODES[c % len(MODES)] == slb.MODE_AM:
            z = 9000.0 * (1 + 0.5 * np.cos(2 * np.pi * 1000 * n / 48000)) * np.exp(1j * (2 * np.pi * 300 * n / 48000 + c))
        elif MODES[c % len(MODES)] == slb.MODE_FM:
            z = 12000.0 * np.exp(1j * (2.5 * np.sin(2 * np.pi * (700 + 50 * c) * n / 48000) + c))
        else:
            continue
        z = z + rng.normal(0, 300, T) + 1j * rng.normal(0, 300, T)
        x[c] = np.stack([np.rint(z.real), np.rint(z.imag)], 1).clip(-32768, 32767).astype(np.int16)
    return x


def run_gpu(d, x, want_dbg=True):
    """Returns out int16 [C][T][2] (L = R), pre-AGC detector output int16 [C][T], gain words uint32 [C][T/48]."""
    Cn, T = x.shape[0], x.shape[1]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    aud = torch.zeros((Cn, T), dtype=torch.int16, device="cuda") if want_dbg else None
    gain = torch.zeros((Cn, T // 48), dtype=torch.int32, device="cuda") if want_dbg else None
    d.set_q15_debug_taps(aud, gain)
    y = d.rx_process(xd)
    torch.cuda.synchronize()
    d.set_q15_debug_taps(None, None)
    return y.cpu().numpy(), (aud.cpu().numpy() if want_dbg else None), (gain.cpu().numpy().view(np.uint32) if want_dbg else None)


def set_modes(d, n, shift=0):
    for c in range(n):
        d.DSP_Set_Mode(MODES[(c + shift) % len(MODES)], channel=c)


def check_vs_oracle(o, d, x, y, aud, gain, channels, shift=0):
    for c in channels:
        exp, e_a, e_g, _ = orq.rx_q15(o, d.oracle_params(MODES[(c + shift) % len(MODES)]), x[c])
        if aud is not None:
            assert np.array_equal(aud[c], e_a), (c, int(np.argmax(aud[c] != e_a)))
            assert np.array_equal(gain[c], e_g), c
        assert np.array_equal(y[c], exp), (c, int(np.argmax(np.any(y[c] != exp, axis=1))))


@pytest.mark.parametrize("name,mode", [("am", slb.MODE_AM), ("fm", slb.MODE_FM), ("usb", slb.MODE_USB), ("sat", slb.MODE_FM)])
def test_golden_vectors(name, mode):
    g = np.load(os.path.join(GOLD, "rx_q15.npz"))
    d = slb.DspIf(1, chain=CH)
    d.DSP_Set_Mode(mode)
    mp = d.rx_q15_mode_params()
    assert np.array_equal(np.array(mp.am_taps[:], np.int16), g["am_taps"]) and np.array_equal(np.array(mp.fm_taps[:], np.int16), g["fm_taps"])
    assert mp.fm_floor == int(g["fm_floor"])
    if name == "sat":
        mp.fm_floor = 1; d.set_rx_q15_mode_params(mp)
    y, aud, gain = run_gpu(d, g["%s_in" % name][None])
    assert np.array_equal(aud[0], g["%s_audio" % name])
    assert np.array_equal(gain[0], g["%s_gain" % name])
    assert np.array_equal(y[0], g["%s_out" % name])


def test_ssb_channels_equal_rx_ssb_q15():
    """An RX-Q15 context of SSB-style channels is RX-SSB-q15, byte for byte, state included."""
    Cn, T = 24, 48 * 100
    modes = [slb.MODE_USB, slb.MODE_LSB, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG, slb.MODE_PKT]
    x = slb.synth_iq(Cn, T)
    a = slb.DspIf(Cn, chain=CH); b = slb.DspIf(Cn, chain=slb.CHAIN_RX_SSB_Q15)
    for c in range(Cn):
        a.DSP_Set_Mode(modes[c % 6], channel=c); b.DSP_Set_Mode(modes[c % 6], channel=c)
    ra = run_gpu(a, x); rb = run_gpu(b, x)
    for u, v in zip(ra, rb):
        assert np.array_equal(u, v)
    sa = np.frombuffer(bytes(a.state_save()), np.uint8); sb = np.frombuffer(bytes(b.state_save()), np.uint8)
    assert sa.size == sb.size and np.count_nonzero(sa != sb) <= 8          # the header's chain id differs, nothing else
    # in a mixed context the SSB channels (a listed launch) still equal RX-SSB-q15's
    m = slb.DspIf(Cn, chain=CH)
    for c in range(Cn):
        m.DSP_Set_Mode(modes[c % 6] if c % 4 else (slb.MODE_AM if c % 8 else slb.MODE_FM), channel=c)
    ym, am, gm = run_gpu(m, x)
    ssb = [c for c in range(Cn) if c % 4]
    assert np.array_equal(ym[ssb], rb[0][ssb]) and np.array_equal(am[ssb], rb[1][ssb]) and np.array_equal(gm[ssb], rb[2][ssb])


@pytest.mark.parametrize("channels,frames", [(1, 48), (7, 1488), (8, 4800), (9, 96), (150, 3072 + 480), (300, 48 * 33)])
def test_mixed_batches_vs_oracle(port, channels, frames):
    x = synth(channels, frames, seed=channels)
    d = slb.DspIf(channels, chain=CH); set_modes(d, channels)
    y, aud, gain = run_gpu(d, x)
    check_vs_oracle(port, d, x, y, aud, gain, range(channels) if channels <= 150 else range(0, channels, 7))


def test_streaming_cuts(port):
    Cn, T = 16, 48 * 400
    x = synth(Cn, T)
    whole = slb.DspIf(Cn, chain=CH); set_modes(whole, Cn)
    w = run_gpu(whole, x)
    for cut in (768 * 3, 48 * 37, 48):
        d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
        parts = [run_gpu(d, np.ascontiguousarray(x[:, a:b])) for a, b in ((0, cut), (cut, T))]
        for j in range(3):
            assert np.array_equal(np.concatenate([p_[j] for p_ in parts], 1), w[j]), (cut, j)
    check_vs_oracle(port, whole, x, *w, range(Cn))


def test_mode_changes_between_calls(port):
    """SSB -> AM -> FM -> SSB on every channel (each channel starts at a different point of the cycle), against the oracle run with the
    same schedule on one carried state per channel: the FIRs restart from the raw history with the new taps, the peak window carries."""
    Cn, seg = 12, 48 * 45
    x = synth(Cn, 4 * seg)
    cycle = [slb.MODE_USB, slb.MODE_AM, slb.MODE_FM, slb.MODE_LSB]
    d = slb.DspIf(Cn, chain=CH)
    states = [orq.RxQ15mState() for _ in range(Cn)]
    for s in range(4):
        for c in range(Cn):
            d.DSP_Set_Mode(cycle[(s + c) % 4], channel=c)
        xs = np.ascontiguousarray(x[:, s * seg:(s + 1) * seg])
        y, aud, gain = run_gpu(d, xs)
        for c in range(Cn):
            e, e_a, e_g, _ = orq.rx_q15(port, d.oracle_params(cycle[(s + c) % 4]), xs[c], states[c])
            assert np.array_equal(aud[c], e_a) and np.array_equal(gain[c], e_g) and np.array_equal(y[c], e), (s, c)


def test_every_saturation_point(port, rng):
    """Rail-to-rail squares on both rails, a full-scale carrier, FM at the floor with the largest x (d saturates) and zero input."""
    Cn, T = 16, 4800
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    mp = d.rx_q15_mode_params(); mp.fm_floor = 1; d.set_rx_q15_mode_params(mp)
    x = rng.integers(-32768, 32768, (Cn, T, 2)).astype(np.int16)
    sq = np.where(np.arange(T) % 24 < 12, 32767, -32768).astype(np.int16)
    for c in range(0, 4):
        x[c, :, 0] = sq; x[c, :, 1] = np.roll(sq, 6 * c)
    n = np.arange(T)
    for c in (4, 5):                                                       # full-scale carrier
        x[c, :, 0] = np.rint(32767 * np.cos(2 * np.pi * 2000 * n / 48000)); x[c, :, 1] = np.rint(32767 * np.sin(2 * np.pi * 2000 * n / 48000))
    for c in (3, 11):                                                      # FM: quarter-turn steps at full scale, floor 1
        ph = (np.pi / 2) * (n % 4)
        x[c, :, 0] = np.rint(32767 * np.cos(ph)).clip(-32768, 32767); x[c, :, 1] = np.rint(32767 * np.sin(ph))
    x[6] = 0; x[7, 1000:3000] = 0
    y, aud, gain = run_gpu(d, x)
    check_vs_oracle(port, d, x, y, aud, gain, range(Cn))
    assert int(np.sum(np.abs(aud[[3, 11]].astype(np.int32)) >= 32767)) > 0 or int(np.sum(aud[[3, 11]] == -32768)) > 0
    assert not np.any(y[6])


def test_host_path_equals_device_path_when_sliced():
    Cn, T = 13, 1536 * 6 + 48 * 5
    x = synth(Cn, T)
    d_dev = slb.DspIf(Cn, chain=CH); set_modes(d_dev, Cn)
    y_dev = d_dev.rx_process(torch.from_numpy(x).cuda()).cpu().numpy()
    os.environ["SELENITE_B200_SLICE_BYTES"] = str(5 * 4 * 1536); os.environ["SELENITE_B200_SLICE_CHANNELS"] = "5"
    try:
        d_host = slb.DspIf(Cn, chain=CH); set_modes(d_host, Cn)
        y_host = d_host.rx_process(x)                                          # numpy -> slb_rx_process_host, 3 channel blocks x 7 slices
    finally:
        del os.environ["SELENITE_B200_SLICE_BYTES"]; del os.environ["SELENITE_B200_SLICE_CHANNELS"]
    assert np.array_equal(y_host, y_dev)
    assert bytes(d_host.state_save()) == bytes(d_dev.state_save())


def test_refusals():
    d = slb.DspIf(2, chain=CH)
    lib, h = d.lib, d.h
    before, mbefore = bytes(d.rx_q15_params()), bytes(d.rx_q15_mode_params())

    def refused(edit, mode_params=False):
        if mode_params:
            p = d.rx_q15_mode_params(); edit(p)
            assert lib.slb_set_rx_q15_mode_params(h, C.byref(p)) == ERR_UNSUPPORTED
        else:
            p = d.rx_q15_params(); edit(p)
            assert lib.slb_set_rx_q15_params(h, C.byref(p)) == ERR_UNSUPPORTED
        assert bytes(d.rx_q15_params()) == before and bytes(d.rx_q15_mode_params()) == mbefore
    refused(lambda p: setattr(p, "bq_stages", 1))
    refused(lambda p: p.taps_i.__setitem__(7, 32640))
    refused(lambda p: p.taps_q.__setitem__(60, 32767))
    refused(lambda p: setattr(p, "agc_window", 18))
    refused(lambda p: p.am_taps.__setitem__(3, 32640), True)
    refused(lambda p: p.fm_taps.__setitem__(40, 32767), True)
    refused(lambda p: setattr(p, "fm_floor", 0), True)
    refused(lambda p: setattr(p, "fm_floor", -5), True)
    assert lib.slb_set_tune(h, None) == ERR_UNSUPPORTED
    assert lib.slb_set_tune_channel(h, 0, 100.0) == ERR_UNSUPPORTED
    x = torch.zeros((2, 96, 2), dtype=torch.int16, device="cuda"); y = torch.empty_like(x)
    assert lib.slb_tx_process_device(h, x.data_ptr(), y.data_ptr(), 96, None) == ERR_STATE
    xh = np.zeros((2, 96, 2), np.int16); yh = np.empty_like(xh)
    assert lib.slb_tx_process_host(h, xh.ctypes.data, yh.ctypes.data, 96) == ERR_STATE
    mp = _mode_params(d)
    for other in (slb.CHAIN_RX_SSB_Q15, slb.CHAIN_TX_SSB_Q15, slb.CHAIN_RX_SSB_F32):
        o = slb.DspIf(2, chain=other)
        assert o.lib.slb_set_rx_q15_mode_params(o.h, C.byref(mp)) == ERR_STATE
    with pytest.raises(slb.SeleniteError):
        slb.DspIf(2, fs=96000, chain=CH)


def _mode_params(d):
    return d.rx_q15_mode_params()


def test_1ms_api_equals_bulk(port):
    """Behind the firmware's 1 ms cadence with every mode byte: each block is demodulated in the call that delivers it (no added
    latency), then rides the ring — the same ring fed with the bulk output."""
    Cn, nblk = 9, 40
    x = synth(Cn, 48 * nblk)
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    bulk = slb.DspIf(Cn, chain=CH); set_modes(bulk, Cn)
    y, _, _ = run_gpu(bulk, x, want_dbg=False)
    check_vs_oracle(port, bulk, x, y, None, None, range(Cn))
    p = slb.DspIf(Cn, chain=slb.CHAIN_PASS)
    for b in range(nblk):
        d.DSP_In_Buff_Write(x[:, 48 * b:48 * (b + 1)].reshape(Cn, -1))
        p.DSP_In_Buff_Write(y[:, 48 * b:48 * (b + 1)].reshape(Cn, -1))
        assert np.array_equal(d.DSP_In_Buff_Read(192), p.DSP_In_Buff_Read(192)), b


def test_per_channel_cadence_equals_one_channel_contexts():
    ring.test_chain_behind_the_ring_under_per_channel_cadence(CH)


def test_feeder_equals_the_per_tick_calls(rng):
    ring.test_stream_feeder_equals_the_per_tick_calls(CH, 50, rng)


def test_live_feeder_equals_the_per_tick_calls(rng):
    ring.test_live_feeder_pipeline_equals_the_per_tick_calls(CH, 10, rng)


def test_direction_switch_flushes_chain_state():
    ring.test_rx_tx_switch_flushes_rings_and_chain_state(CH)


def test_checkpoint_round_trip_mid_stream():
    """Same layout and size as RX-SSB-q15 (64 raw frames, the peak window, sidebands; the mode bytes decide the kinds); a restored context
    continues bit for bit."""
    Cn, T = 11, 48 * 60
    x = synth(Cn, T)
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    assert d.state_save().size == slb.DspIf(Cn, chain=slb.CHAIN_RX_SSB_Q15).state_save().size
    y1, _, _ = run_gpu(d, np.ascontiguousarray(x[:, :48 * 23]), want_dbg=False)
    snap = d.state_save()
    y2, a2, g2 = run_gpu(d, np.ascontiguousarray(x[:, 48 * 23:]))
    e = slb.DspIf(Cn, chain=CH)                                               # modes come back with the checkpoint
    e.state_load(snap)
    z2, za2, zg2 = run_gpu(e, np.ascontiguousarray(x[:, 48 * 23:]))
    assert np.array_equal(z2, y2) and np.array_equal(za2, a2) and np.array_equal(zg2, g2)
    whole = slb.DspIf(Cn, chain=CH); set_modes(whole, Cn)
    yw, _, _ = run_gpu(whole, x, want_dbg=False)
    assert np.array_equal(np.concatenate([y1, y2], 1), yw)


_DROPIN = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import oracle_lib, oracle_rx_q15 as orq, selenite_lite_b200 as slb
from selenite_lite_b200 import _lib
lib = _lib.load()
lib.DSP_Init(); lib.DSP_Set_Mode(slb.MODE_FM)
n = np.arange(48 * 30)
z = 12000.0 * np.exp(1j * 2.5 * np.sin(2 * np.pi * 900 * n / 48000))
x = np.stack([np.rint(z.real), np.rint(z.imag)], 1).astype(np.int16)
prm = slb.dsp_if.q15_mode_params_to_dict(slb.default_rx_q15_params(48000), slb.default_rx_q15_mode_params(48000), slb.MODE_FM)
exp = orq.rx_q15(oracle_lib.Oracle("port"), prm, x)[0]
p = slb.DspIf(1, chain=slb.CHAIN_PASS)
for b in range(30):
    blk = np.ascontiguousarray(x[48 * b:48 * b + 48]).reshape(-1)
    lib.DSP_In_Buff_Write(blk.ctypes.data, 96)
    got = np.zeros(96, np.int16); lib.DSP_In_Buff_Read(got.ctypes.data, 192)
    p.DSP_In_Buff_Write(exp[48 * b:48 * b + 48].reshape(1, -1))
    assert np.array_equal(got, p.DSP_In_Buff_Read(192)[0]), b
assert lib.slb_dropin_status() == 0
print("dropin ok")
"""


def test_dropin_with_the_chain_env():
    env = dict(os.environ, SELENITE_B200_CHAIN="rx_q15")
    r = subprocess.run([sys.executable, "-c", _DROPIN, ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "dropin ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.timeout(900, method="thread")
def test_scale_1024_channels_10s(port):
    """1024 channels x 10 s, mixed modes: whole streams against the oracle on channels spread over the batch."""
    Cn, T = 1024, 480000
    x = np.ascontiguousarray(np.tile(synth(16, T), (Cn // 16, 1, 1)))
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    y, _, _ = run_gpu(d, x, want_dbg=False)
    for c in (0, 1, 3, 147, 511, 514, 777, 1019, 1022, 1023):
        exp = orq.rx_q15(port, d.oracle_params(MODES[c % len(MODES)]), x[c])[0]
        assert np.array_equal(y[c], exp), (c, int(np.argmax(np.any(y[c] != exp, axis=1))))


@pytest.mark.timeout(900, method="thread")
def test_scale_8192_channels_2s(port):
    """8192 channels x 2 s, mixed modes: every SSB-style channel equals RX-SSB-q15 on the same input; sampled AM and FM channels equal
    the oracle."""
    Cn, T = 8192, 96000
    g = torch.Generator(device="cuda"); g.manual_seed(11)
    x = torch.randint(-12000, 12000, (Cn, T, 2), dtype=torch.int16, device="cuda", generator=g)
    d = slb.DspIf(Cn, chain=CH); r = slb.DspIf(Cn, chain=slb.CHAIN_RX_SSB_Q15)
    kinds = np.array([MODES[(c * 5) % len(MODES)] for c in range(Cn)])
    for c in range(Cn):
        d.DSP_Set_Mode(int(kinds[c]), channel=c)
        if kinds[c] not in (slb.MODE_AM, slb.MODE_FM):
            r.DSP_Set_Mode(int(kinds[c]), channel=c)
    y = d.rx_process(x); yr = r.rx_process(x)
    torch.cuda.synchronize()
    ssb = torch.from_numpy(np.nonzero((kinds != slb.MODE_AM) & (kinds != slb.MODE_FM))[0]).cuda()
    assert torch.equal(y[ssb], yr[ssb])
    del yr
    for c in [c for c in range(Cn) if kinds[c] in (slb.MODE_AM, slb.MODE_FM)][::900] + [8191 if kinds[8191] in (slb.MODE_AM, slb.MODE_FM) else 8190]:
        exp = orq.rx_q15(port, d.oracle_params(int(kinds[c])), x[c].cpu().numpy())[0]
        assert np.array_equal(y[c].cpu().numpy(), exp), c


@pytest.mark.timeout(1500, method="thread")
def test_parity_on_the_stress_build():
    """This file's parity tests on the stress build (random delays at every hand-over), like tests/test_gpu_stress_build.py does for the others."""
    if not os.path.exists(_build.STRESS_LIB_PATH):
        pytest.skip("stress build not present (python __graft_entry__.py builds it)")
    env = dict(os.environ, SELENITE_B200_LIB=_build.STRESS_LIB_PATH)
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "900",
                        os.path.abspath(__file__), "-k", "not stress_build and not scale"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1400)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
