"""GPU parity of the all-mode integer transmitter TX-Q15 (SLB_CHAIN_TX_Q15, DESIGN.md §3.9: the SSB-style modes exactly as TX-SSB-q15,
AM as carrier plus scaled audio, FM as an integer phase accumulator through the table NCO, all on the integer tensor cores), called
through the C ABI, against the oracle (oracle/slo_tx_q15_mod.h through tests/oracle_tx_q15_mod.py), TX-SSB-q15 itself and the committed
golden vectors. Every comparison is BIT-EXACT: the pre-ALC pair, the per-block gain word, the output and the carried state."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_tx_q15_mod as otq
import selenite_lite_b200 as slb
import test_gpu_ring as ring
from selenite_lite_b200 import build as _build
from test_golden import GOLD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CH = slb.CHAIN_TX_Q15
MODES = [slb.MODE_USB, slb.MODE_AM, slb.MODE_LSB, slb.MODE_FM, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG, slb.MODE_PKT]
ERR_STATE, ERR_UNSUPPORTED = -3, -4


def synth(Cn, T, seed=1):
    """Per channel a mic (L = R) of two tones with bursts and noise; channel c detunes and rescales it. L != R on odd channels (R is
    ignored by every mode)."""
    x = slb.synth_mic(Cn, T, first_channel=seed)
    rng = np.random.Generator(np.random.PCG64(seed))
    n = np.arange(T)
    for c in range(Cn):
        env = np.where((n // (480 + 48 * c)) % 3 == 0, 1.5, 0.3 + 0.05 * (c % 5))
        x[c, :, 0] = np.rint(x[c, :, 0] * env).clip(-32768, 32767)
        x[c, :, 1] = x[c, :, 0] if c % 2 == 0 else rng.integers(-32768, 32768, T)
    return x


def run_gpu(d, x, want_dbg=True):
    """Returns out int16 [C][T][2] I/Q, the pre-ALC pair int16 [C][T][2], gain words uint32 [C][T/48]."""
    Cn, T = x.shape[0], x.shape[1]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    iq = torch.zeros((Cn, T, 2), dtype=torch.int16, device="cuda") if want_dbg else None
    gain = torch.zeros((Cn, T // 48), dtype=torch.int32, device="cuda") if want_dbg else None
    d.set_q15_debug_taps(iq, gain)
    y = d.tx_process(xd)
    torch.cuda.synchronize()
    d.set_q15_debug_taps(None, None)
    return y.cpu().numpy(), (iq.cpu().numpy() if want_dbg else None), (gain.cpu().numpy().view(np.uint32) if want_dbg else None)


def set_modes(d, n, shift=0):
    for c in range(n):
        d.DSP_Set_Mode(MODES[(c + shift) % len(MODES)], channel=c)


def phases(d):
    """The phase words of a TX-Q15 checkpoint: after the chain state, before the 2 x 4 per-channel ring pointers."""
    blob = np.frombuffer(bytes(d.state_save()), np.uint8); Cn = d.channels
    end = blob.size - 2 * Cn * 16
    return blob[end - 4 * Cn:end].view(np.uint32).copy()


def check_vs_oracle(o, d, x, y, iq, gain, channels, shift=0, states=None):
    for c in channels:
        exp, e_iq, e_g, _, _ = otq.tx_q15(o, d.oracle_params(MODES[(c + shift) % len(MODES)]), x[c], None if states is None else states[c])
        if iq is not None:
            assert np.array_equal(iq[c], e_iq), (c, int(np.argmax(np.any(iq[c] != e_iq, axis=1))))
            assert np.array_equal(gain[c], e_g), c
        assert np.array_equal(y[c], exp), (c, int(np.argmax(np.any(y[c] != exp, axis=1))))


@pytest.mark.parametrize("name,mode", [("am", slb.MODE_AM), ("fm", slb.MODE_FM), ("usb", slb.MODE_USB), ("sat", slb.MODE_FM)])
def test_golden_vectors(name, mode):
    g = np.load(os.path.join(GOLD, "tx_q15.npz"))
    d = slb.DspIf(1, chain=CH)
    d.DSP_Set_Mode(mode)
    mp = d.tx_q15_mode_params()
    assert np.array_equal(np.array(mp.am_taps[:], np.int16), g["am_taps"]) and np.array_equal(np.array(mp.fm_taps[:], np.int16), g["fm_taps"])
    assert [mp.am_carrier, mp.am_depth, mp.fm_target, mp.fm_inc] == list(g["consts"]) and np.float32(mp.fm_level) == g["fm_level"]
    if name == "sat":
        for k in range(64):
            mp.fm_taps[k] = 32639
        mp.fm_inc = 65535; mp.fm_target = 32767; d.set_tx_q15_mode_params(mp)
    y, iq, gain = run_gpu(d, g["%s_in" % name][None])
    assert np.array_equal(iq[0], g["%s_iq" % name])
    assert np.array_equal(gain[0], g["%s_gain" % name])
    assert np.array_equal(y[0], g["%s_out" % name])
    if mode == slb.MODE_FM:
        assert phases(d)[0] == g["%s_phase" % name][-1]


def test_ssb_channels_equal_tx_ssb_q15():
    """A TX-Q15 context of SSB-style channels is TX-SSB-q15, byte for byte; in a mixed context the SSB channels (a listed launch) too."""
    Cn, T = 24, 48 * 100
    modes = [slb.MODE_USB, slb.MODE_LSB, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG, slb.MODE_PKT]
    x = synth(Cn, T)
    a = slb.DspIf(Cn, chain=CH); b = slb.DspIf(Cn, chain=slb.CHAIN_TX_SSB_Q15)
    for c in range(Cn):
        a.DSP_Set_Mode(modes[c % 6], channel=c); b.DSP_Set_Mode(modes[c % 6], channel=c)
    ra = run_gpu(a, x); rb = run_gpu(b, x)
    for u, v in zip(ra, rb):
        assert np.array_equal(u, v)
    m = slb.DspIf(Cn, chain=CH)
    for c in range(Cn):
        m.DSP_Set_Mode(modes[c % 6] if c % 4 else (slb.MODE_AM if c % 8 else slb.MODE_FM), channel=c)
    ym, qm, gm = run_gpu(m, x)
    ssb = [c for c in range(Cn) if c % 4]
    assert np.array_equal(ym[ssb], rb[0][ssb]) and np.array_equal(qm[ssb], rb[1][ssb]) and np.array_equal(gm[ssb], rb[2][ssb])


@pytest.mark.parametrize("channels,frames", [(1, 48), (7, 1488), (9, 96), (13, 768 * 2 + 48 * 5), (150, 3072 + 480), (300, 48 * 33)])
def test_mixed_batches_vs_oracle(port, channels, frames):
    x = synth(channels, frames, seed=channels)
    d = slb.DspIf(channels, chain=CH); set_modes(d, channels)
    y, iq, gain = run_gpu(d, x)
    check_vs_oracle(port, d, x, y, iq, gain, range(channels) if channels <= 150 else range(0, channels, 7))


def test_streaming_cuts_and_phase(port):
    """Cuts in mid-supertile, on a supertile boundary and one block in; the phase words at the end are the oracle's."""
    Cn, T = 16, 48 * 400
    x = synth(Cn, T)
    whole = slb.DspIf(Cn, chain=CH); set_modes(whole, Cn)
    w = run_gpu(whole, x)
    for cuts in ((768 * 3,), (48 * 37,), (48,), (48 * 5, 768 * 4, 768 * 4 + 48 * 20)):
        d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
        parts = [run_gpu(d, np.ascontiguousarray(x[:, a:b])) for a, b in zip((0,) + cuts, cuts + (T,))]
        for j in range(3):
            assert np.array_equal(np.concatenate([p_[j] for p_ in parts], 1), w[j]), (cuts, j)
        assert np.array_equal(phases(d), phases(whole))
    check_vs_oracle(port, whole, x, *w, range(Cn))
    ph = phases(whole)
    for c in range(Cn):
        st = otq.tx_q15(port, whole.oracle_params(MODES[c % len(MODES)]), x[c])[4]
        assert ph[c] == st.phase, c
    assert np.count_nonzero(ph) >= 2


def test_several_groups_per_cta_and_odd_supertiles(port):
    """Two CTAs per launch (SELENITE_B200_TC_GRID), so every CTA walks several channel groups of each kind, on streams of an odd
    number of supertiles (the set that starts a group alternates) and cut into calls of one to five supertiles: output and final
    phase words equal the oracle's."""
    Cn, T = 48, 768 * 6 + 48 * 7
    x = synth(Cn, T, seed=3)
    os.environ["SELENITE_B200_TC_GRID"] = "2"
    try:
        whole = slb.DspIf(Cn, chain=CH); set_modes(whole, Cn)
        w = run_gpu(whole, x)
        for cuts in ((768 * 2 + 48 * 3,), (48, 768 + 48 * 2, 768 * 3 + 48 * 5)):
            d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
            parts = [run_gpu(d, np.ascontiguousarray(x[:, a:b])) for a, b in zip((0,) + cuts, cuts + (T,))]
            for j in range(3):
                assert np.array_equal(np.concatenate([p_[j] for p_ in parts], 1), w[j]), (cuts, j)
            assert np.array_equal(phases(d), phases(whole))
    finally:
        del os.environ["SELENITE_B200_TC_GRID"]
    check_vs_oracle(port, whole, x, *w, range(Cn))
    ph = phases(whole)
    for c in range(Cn):
        assert ph[c] == otq.tx_q15(port, whole.oracle_params(MODES[c % len(MODES)]), x[c])[4].phase, c


def test_mode_changes_between_calls(port):
    """SSB -> FM -> AM -> FM on every channel (each channel starts at a different point of the cycle), against the oracle run with the
    same schedule on one carried state per channel: the phase is held through the other modes."""
    Cn, seg = 12, 48 * 45
    x = synth(Cn, 4 * seg)
    cycle = [slb.MODE_USB, slb.MODE_FM, slb.MODE_AM, slb.MODE_FM]
    d = slb.DspIf(Cn, chain=CH)
    states = [otq.TxQ15mState() for _ in range(Cn)]
    for s in range(4):
        for c in range(Cn):
            d.DSP_Set_Mode(cycle[(s + c) % 4], channel=c)
        xs = np.ascontiguousarray(x[:, s * seg:(s + 1) * seg])
        y, iq, gain = run_gpu(d, xs)
        for c in range(Cn):
            e, e_iq, e_g, _, _ = otq.tx_q15(port, d.oracle_params(cycle[(s + c) % 4]), xs[c], states[c])
            assert np.array_equal(iq[c], e_iq) and np.array_equal(gain[c], e_g) and np.array_equal(y[c], e), (s, c)
        assert list(phases(d)) == [st.phase for st in states], s


def test_every_saturation_point(port, rng):
    """Rail-to-rail squares, full-scale noise and silence with the largest splittable taps, the largest increment and targets."""
    Cn, T = 16, 4800
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    mp = d.tx_q15_mode_params()
    for k in range(64):
        mp.am_taps[k] = 32639 if k % 2 else -32640 + 1; mp.fm_taps[k] = 32639
    mp.fm_inc = -65535; mp.fm_target = 32767; mp.am_depth = 32767; mp.am_carrier = 32767
    d.set_tx_q15_mode_params(mp)
    x = rng.integers(-32768, 32768, (Cn, T, 2)).astype(np.int16)
    sq = np.where(np.arange(T) % 24 < 12, 32767, -32768).astype(np.int16)
    for c in range(0, 8):
        x[c, :, 0] = np.roll(sq, 3 * c)
    x[9] = 0; x[11, 1000:3000] = -32768
    y, iq, gain = run_gpu(d, x)
    check_vs_oracle(port, d, x, y, iq, gain, range(Cn))
    assert np.any(y[1, :, 0] == 32767)                                       # AM at full carrier and depth saturates the add


def test_host_path_equals_device_path_when_sliced():
    Cn, T = 13, 1536 * 6 + 48 * 5
    x = synth(Cn, T)
    d_dev = slb.DspIf(Cn, chain=CH); set_modes(d_dev, Cn)
    y_dev = d_dev.tx_process(torch.from_numpy(x).cuda()).cpu().numpy()
    os.environ["SELENITE_B200_SLICE_BYTES"] = str(5 * 4 * 1536); os.environ["SELENITE_B200_SLICE_CHANNELS"] = "5"
    try:
        d_host = slb.DspIf(Cn, chain=CH); set_modes(d_host, Cn)
        y_host = d_host.tx_process(x)                                          # numpy -> slb_tx_process_host, 3 channel blocks x 7 slices
    finally:
        del os.environ["SELENITE_B200_SLICE_BYTES"]; del os.environ["SELENITE_B200_SLICE_CHANNELS"]
    assert np.array_equal(y_host, y_dev)
    assert bytes(d_host.state_save()) == bytes(d_dev.state_save())


def test_refusals():
    d = slb.DspIf(2, chain=CH)
    lib, h = d.lib, d.h
    before, mbefore = bytes(d.rx_q15_params()), bytes(d.tx_q15_mode_params())

    def refused(edit, mode_params=False):
        if mode_params:
            p = d.tx_q15_mode_params(); edit(p)
            assert lib.slb_set_tx_q15_mode_params(h, C.byref(p)) == ERR_UNSUPPORTED
        else:
            p = d.rx_q15_params(); edit(p)
            assert lib.slb_set_rx_q15_params(h, C.byref(p)) == ERR_UNSUPPORTED
        assert bytes(d.rx_q15_params()) == before and bytes(d.tx_q15_mode_params()) == mbefore
    refused(lambda p: setattr(p, "bq_stages", 1))
    refused(lambda p: p.taps_i.__setitem__(7, 32640))
    refused(lambda p: p.taps_q.__setitem__(60, 32767))
    refused(lambda p: setattr(p, "agc_window", 18))
    refused(lambda p: p.am_taps.__setitem__(3, 32640), True)
    refused(lambda p: p.fm_taps.__setitem__(40, 32767), True)
    refused(lambda p: setattr(p, "am_carrier", -1), True)
    refused(lambda p: setattr(p, "am_depth", 0), True)
    refused(lambda p: setattr(p, "fm_target", 0), True)
    refused(lambda p: setattr(p, "fm_inc", 65536), True)
    refused(lambda p: setattr(p, "fm_inc", -65536), True)
    assert lib.slb_set_tune(h, None) == ERR_UNSUPPORTED
    assert lib.slb_set_tune_channel(h, 0, 100.0) == ERR_UNSUPPORTED
    x = torch.zeros((2, 96, 2), dtype=torch.int16, device="cuda"); y = torch.empty_like(x)
    assert lib.slb_rx_process_device(h, x.data_ptr(), y.data_ptr(), 96, None) == ERR_STATE
    xh = np.zeros((2, 96, 2), np.int16); yh = np.empty_like(xh)
    assert lib.slb_rx_process_host(h, xh.ctypes.data, yh.ctypes.data, 96) == ERR_STATE
    mp = d.tx_q15_mode_params()
    for other in (slb.CHAIN_RX_SSB_Q15, slb.CHAIN_TX_SSB_Q15, slb.CHAIN_RX_Q15, slb.CHAIN_TX_F32):
        o = slb.DspIf(2, chain=other)
        assert o.lib.slb_set_tx_q15_mode_params(o.h, C.byref(mp)) == ERR_STATE
        assert o.lib.slb_get_tx_q15_mode_params(o.h, C.byref(mp)) == ERR_STATE
    rmp = slb.default_rx_q15_mode_params()
    assert lib.slb_set_rx_q15_mode_params(h, C.byref(rmp)) == ERR_STATE and lib.slb_get_rx_q15_mode_params(h, C.byref(rmp)) == ERR_STATE
    t = slb.DspIf(2, chain=slb.CHAIN_TX_SSB_Q15)                             # TX-SSB-q15 keeps refusing AM and FM
    assert t.lib.SLB_DSP_Set_Mode(t.h, slb.MODE_AM) == ERR_UNSUPPORTED and t.lib.SLB_DSP_Set_Mode(t.h, slb.MODE_FM) == ERR_UNSUPPORTED
    with pytest.raises(slb.SeleniteError):
        slb.DspIf(2, fs=96000, chain=CH)


def test_1ms_api_equals_bulk(port):
    """Behind the firmware's 1 ms cadence with every mode byte: each block is modulated in the call that delivers it (no added latency),
    then rides the ring — the same ring fed with the bulk output."""
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
    assert np.array_equal(phases(d), phases(bulk))


def test_per_channel_cadence_with_every_mode():
    """Per-channel cadence (dsp_if.c:252-300 per channel) with AM and FM channels beside SSB ones: every channel of the batched context
    equals a one-channel context that sees only that channel's events, across a checkpoint taken in mid-stream."""
    Cn, ticks, B = 8, 120, 48
    x = synth(Cn, ticks * B)
    d = slb.DspIf(Cn, chain=CH); single = [slb.DspIf(1, chain=CH) for _ in range(Cn)]
    for c in range(Cn):
        d.DSP_Set_Mode(MODES[c], channel=c); single[c].DSP_Set_Mode(MODES[c])
    rng = np.random.Generator(np.random.PCG64(5))
    pos = [0] * Cn
    for t in range(ticks):
        if t == 60:
            snap = d.state_save(); d = slb.DspIf(Cn, chain=CH); d.state_load(snap)
        act = np.array([(not ((c == 1 and t % 13 == 12) or (c == 3 and t % 5 == 4) or (c == 5 and rng.random() < 0.1)),
                         not ((c == 2 and t % 17 == 16) or (c == 3 and t % 7 == 6) or (c == 6 and rng.random() < 0.1))) for c in range(Cn)])
        blk = np.zeros((Cn, 2 * B), np.int16)
        for c in range(Cn):
            if act[c, 0]:
                blk[c] = x[c, pos[c]:pos[c] + B].reshape(-1); pos[c] += B
        d.DSP_In_Buff_Write_Ch(blk, act[:, 0].astype(np.uint8))
        got = d.DSP_In_Buff_Read_Ch(4 * B, act[:, 1].astype(np.uint8))
        for c in range(Cn):
            if act[c, 0]: single[c].DSP_In_Buff_Write(blk[c:c + 1])
            exp = single[c].DSP_In_Buff_Read(4 * B)[0] if act[c, 1] else np.zeros(2 * B, np.int16)
            assert np.array_equal(got[c], exp), (t, c)
    assert list(phases(d)) == [phases(s)[0] for s in single]


@pytest.fixture
def mixed_contexts(monkeypatch):
    """slb.DspIf for the ring helpers of test_gpu_ring.py: TX-Q15 contexts come with every mode byte, AM and FM included."""
    orig = slb.DspIf

    def make(n, *a, **k):
        d = orig(n, *a, **k)
        if k.get("chain") == CH:
            set_modes(d, n, shift=1)
        return d
    monkeypatch.setattr(slb, "DspIf", make)


def test_feeder_equals_the_per_tick_calls(rng, mixed_contexts):
    ring.test_stream_feeder_equals_the_per_tick_calls(CH, 50, rng)


def test_live_feeder_equals_the_per_tick_calls(rng, mixed_contexts):
    ring.test_live_feeder_pipeline_equals_the_per_tick_calls(CH, 10, rng)


def test_direction_switch_flushes_chain_state(mixed_contexts):
    ring.test_rx_tx_switch_flushes_rings_and_chain_state(CH)


def test_direction_switch_and_init_zero_the_phase():
    Cn = 4
    x = synth(Cn, 48 * 40)
    d = slb.DspIf(Cn, chain=CH); d.DSP_Set_Mode(slb.MODE_FM)
    run_gpu(d, x, want_dbg=False)
    assert np.count_nonzero(phases(d)) == Cn
    d.DSP_Set_TX()
    assert not phases(d).any()
    run_gpu(d, x, want_dbg=False)
    assert np.count_nonzero(phases(d)) == Cn
    d.DSP_Init()
    assert not phases(d).any()


def test_checkpoint_round_trip_mid_fm():
    """TX-SSB-q15's layout plus the phase words (4 bytes per channel); a context restored in the middle of FM continues bit for bit."""
    Cn, T = 11, 48 * 60
    x = synth(Cn, T)
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    assert d.state_save().size == slb.DspIf(Cn, chain=slb.CHAIN_TX_SSB_Q15).state_save().size + 4 * Cn
    y1, _, _ = run_gpu(d, np.ascontiguousarray(x[:, :48 * 23]), want_dbg=False)
    snap = d.state_save()
    assert phases(d)[3] != 0
    y2, q2, g2 = run_gpu(d, np.ascontiguousarray(x[:, 48 * 23:]))
    e = slb.DspIf(Cn, chain=CH)                                               # modes come back with the checkpoint
    e.state_load(snap)
    z2, zq2, zg2 = run_gpu(e, np.ascontiguousarray(x[:, 48 * 23:]))
    assert np.array_equal(z2, y2) and np.array_equal(zq2, q2) and np.array_equal(zg2, g2)
    assert np.array_equal(phases(e), phases(d))
    whole = slb.DspIf(Cn, chain=CH); set_modes(whole, Cn)
    yw, _, _ = run_gpu(whole, x, want_dbg=False)
    assert np.array_equal(np.concatenate([y1, y2], 1), yw)


_DROPIN = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import oracle_lib, oracle_tx_q15_mod as otq, selenite_lite_b200 as slb
from selenite_lite_b200 import _lib
lib = _lib.load()
lib.DSP_Init(); lib.DSP_Set_Mode(slb.MODE_FM)
x = slb.synth_mic(1, 48 * 30)[0]
prm = slb.dsp_if.tx_q15_mode_params_to_dict(slb.default_rx_q15_params(48000), slb.default_tx_q15_mode_params(48000), slb.MODE_FM)
exp = otq.tx_q15(oracle_lib.Oracle("port"), prm, x)[0]
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
    env = dict(os.environ, SELENITE_B200_CHAIN="tx_q15")
    r = subprocess.run([sys.executable, "-c", _DROPIN, ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "dropin ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.timeout(900, method="thread")
def test_scale_1024_channels_10s(port):
    """1024 channels x 10 s, mixed modes: whole streams against the oracle on channels spread over the batch."""
    Cn, T = 1024, 480000
    x = np.ascontiguousarray(np.tile(synth(16, T), (Cn // 16, 1, 1)))
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    y, _, _ = run_gpu(d, x, want_dbg=False)
    ph = phases(d)
    for c in (0, 1, 3, 147, 511, 514, 777, 1019, 1022, 1023):
        exp, _, _, _, st = otq.tx_q15(port, d.oracle_params(MODES[c % len(MODES)]), x[c])
        assert np.array_equal(y[c], exp), (c, int(np.argmax(np.any(y[c] != exp, axis=1))))
        assert ph[c] == st.phase, c


@pytest.mark.timeout(900, method="thread")
def test_scale_8192_channels_2s(port):
    """8192 channels x 2 s, mixed modes: every SSB-style channel equals TX-SSB-q15 on the same input; sampled AM and FM channels equal
    the oracle."""
    Cn, T = 8192, 96000
    g = torch.Generator(device="cuda"); g.manual_seed(11)
    x = torch.randint(-12000, 12000, (Cn, T, 2), dtype=torch.int16, device="cuda", generator=g)
    d = slb.DspIf(Cn, chain=CH); r = slb.DspIf(Cn, chain=slb.CHAIN_TX_SSB_Q15)
    kinds = np.array([MODES[(c * 5) % len(MODES)] for c in range(Cn)])
    for c in range(Cn):
        d.DSP_Set_Mode(int(kinds[c]), channel=c)
        if kinds[c] not in (slb.MODE_AM, slb.MODE_FM):
            r.DSP_Set_Mode(int(kinds[c]), channel=c)
    y = d.tx_process(x); yr = r.tx_process(x)
    torch.cuda.synchronize()
    ssb = torch.from_numpy(np.nonzero((kinds != slb.MODE_AM) & (kinds != slb.MODE_FM))[0]).cuda()
    assert torch.equal(y[ssb], yr[ssb])
    del yr
    for c in [c for c in range(Cn) if kinds[c] in (slb.MODE_AM, slb.MODE_FM)][::900] + [8191 if kinds[8191] in (slb.MODE_AM, slb.MODE_FM) else 8190]:
        exp = otq.tx_q15(port, d.oracle_params(int(kinds[c])), x[c].cpu().numpy())[0]
        assert np.array_equal(y[c].cpu().numpy(), exp), c


@pytest.mark.timeout(1500, method="thread")
def test_parity_on_the_stress_build():
    """This file's parity tests on the stress build (random delays at every hand-over, the two-set phase hand-over included), like
    tests/test_gpu_stress_build.py does for the others."""
    if not os.path.exists(_build.STRESS_LIB_PATH):
        pytest.skip("stress build not present (python __graft_entry__.py builds it)")
    env = dict(os.environ, SELENITE_B200_LIB=_build.STRESS_LIB_PATH)
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "900",
                        os.path.abspath(__file__), "-k", "not stress_build and not scale"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1400)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
