"""GPU tests of per-channel tuning (slb_set_tune, DESIGN.md §3.5) on the f32 RX and TX chains, against the oracle tuner
(oracle/slo_tune.h through tests/oracle_tune.py).

The tuner is a q15 -> q15 stage that is bit-exact to the oracle, so most checks are byte-for-byte: a tuned RX context on x equals an
untuned one on the oracle-tuned x (output and debug taps), and a tuned TX context's output equals the oracle tuner applied to an
untuned context's output, for every call pattern (cuts, paths, host slices, checkpoints, ring paths, shards, retunes)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_tune as otu
import oracle_tx_mod as otm
import selenite_lite_b200 as slb
from selenite_lite_b200 import build as _build
from test_golden import GOLD, audio_tolerance
from test_gpu_rx_ssb_f32 import check_int16
from test_tune_oracle import LOOPBACK_HZ, LOOPBACK_SNR_DB
from test_tx_am_fm_oracle import loopback_input

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL8 = [slb.MODE_USB, slb.MODE_LSB, slb.MODE_CW, slb.MODE_CWR, slb.MODE_AM, slb.MODE_FM, slb.MODE_DIG, slb.MODE_PKT]
TX_MODES = [slb.MODE_USB, slb.MODE_LSB, slb.MODE_AM, slb.MODE_FM, slb.MODE_CW]


def offsets(C, fs=48000, seed=1, zero_every=3):
    """Random offsets within +-0.45 fs; every `zero_every`-th channel untuned."""
    hz = np.random.Generator(np.random.PCG64(seed)).uniform(-0.45 * fs, 0.45 * fs, C)
    hz[::zero_every] = 0.0
    return hz


def incs_of(d):
    return np.array([d.tune(c)[0] for c in range(d.channels)], np.int64)


def make(C, modes, chain=slb.CHAIN_RX_SSB_F32, hz=None, fs=48000, path=slb.RX_PATH_AUTO):
    d = slb.DspIf(C, fs=fs, chain=chain); d.set_rx_path(path)
    for c in range(C):
        d.DSP_Set_Mode(modes[c % len(modes)], channel=c)
    if hz is not None:
        d.set_tune(hz)
    return d


def rx_dev(d, x, taps=False):
    C, T = x.shape[0], x.shape[1]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    audio = torch.zeros((C, T), dtype=torch.float32, device="cuda") if taps else None
    gain = torch.zeros((C, T // 48), dtype=torch.float32, device="cuda") if taps else None
    d.set_debug_taps(audio, gain)
    y = d.rx_process(xd); torch.cuda.synchronize()
    d.set_debug_taps(None, None)
    return (y.cpu().numpy(), audio.cpu().numpy(), gain.cpu().numpy()) if taps else y.cpu().numpy()


def tx_dev(d, x):
    y = d.tx_process(torch.from_numpy(np.ascontiguousarray(x)).cuda()); torch.cuda.synchronize()
    return y.cpu().numpy()


def tune_cuts(port, x, incs, up, cuts=None, retune=None):
    """The oracle tuner per channel over the stream, the phase carried across `cuts`; retune = (cut index, new incs). A segment with
    inc = 0 passes unchanged and keeps the phase, as the library skips untuned channels (tune_q15 would rotate it by the carried phase)."""
    out = np.empty_like(x)
    cuts = [0, x.shape[1]] if cuts is None else cuts
    for c in range(x.shape[0]):
        ph, inc = 0, int(incs[c])
        for i in range(len(cuts) - 1):
            if retune is not None and i == retune[0]:
                inc = int(retune[1][c])
            if inc == 0:
                out[c, cuts[i]:cuts[i + 1]] = x[c, cuts[i]:cuts[i + 1]]
            else:
                out[c, cuts[i]:cuts[i + 1]], ph = otu.tune_q15(port, x[c, cuts[i]:cuts[i + 1]], inc, ph, up)
    return out


@pytest.mark.parametrize("path", [slb.RX_PATH_AUTO, slb.RX_PATH_FFT])
def test_rx_all_modes_byte_identical_to_the_oracle_tuned_input(port, best_oracle, path):
    C, T = 16, 1536 * 2 + 384
    hz = offsets(C, seed=2)
    d = make(C, ALL8, hz=hz, path=path)
    x = tune_cuts(port, slb.synth_iq(C, T, amp=0.3), incs_of(d), up=True)    # each station sits at its channel's offset
    y, a, g = rx_dev(d, x, taps=True)
    xt = tune_cuts(port, x, incs_of(d), up=False)
    y0, a0, g0 = rx_dev(make(C, ALL8, path=path), xt, taps=True)
    assert np.array_equal(y, y0) and np.array_equal(a.view(np.uint32), a0.view(np.uint32)) and np.array_equal(g.view(np.uint32), g0.view(np.uint32))
    for c in range(C):                                                        # the composition rx_ssb_f32 (tune_q15 (x, down))
        if ALL8[c % 8] in (slb.MODE_USB, slb.MODE_LSB, slb.MODE_DIG, slb.MODE_PKT):
            exp, ao, _, _ = best_oracle.rx_ssb_f32(d.oracle_params(ALL8[c % 8]), xt[c])
            assert np.all(np.abs(a[c] - ao) <= audio_tolerance(ao) + 1e-9), c
            check_int16(y[c], exp)


@pytest.mark.parametrize("chain,modes", [(slb.CHAIN_TX_SSB_F32, [slb.MODE_USB, slb.MODE_LSB, slb.MODE_CW]), (slb.CHAIN_TX_F32, TX_MODES)])
def test_tx_output_is_the_oracle_tuner_of_the_untuned_output(port, chain, modes):
    C, T = 10, 1536 * 2 + 768
    x = slb.synth_mic(C, T)
    d = make(C, modes, chain, hz=offsets(C, seed=3))
    y = tx_dev(d, x)
    y0 = tx_dev(make(C, modes, chain), x)
    assert np.array_equal(y, tune_cuts(port, y0, incs_of(d), up=True))


def drive(factory, x, cuts, paths, ckpt_at, tx):
    d = factory(); parts = []
    for i in range(len(cuts) - 1):
        d.set_rx_path(paths[i % len(paths)])
        if i == ckpt_at:
            snap = d.state_save(); d = factory(); d.state_load(snap)         # the restored context re-applies its offsets (factory)
        xi = np.ascontiguousarray(x[:, cuts[i]:cuts[i + 1]])
        parts.append(tx_dev(d, xi) if tx else rx_dev(d, xi))
    return np.concatenate(parts, 1)


@pytest.mark.parametrize("tx", [False, True])
def test_continuity_across_cuts_paths_slices_checkpoints(port, tx):
    C, T = 11, 1536 * 4
    modes = TX_MODES if tx else ALL8
    chain = slb.CHAIN_TX_F32 if tx else slb.CHAIN_RX_SSB_F32
    hz = offsets(C, seed=4)
    x = slb.synth_mic(C, T) if tx else slb.synth_iq(C, T)
    incs = incs_of(make(C, modes, chain, hz=hz))
    cuts = [0, 384, 1536, 1536 + 768, 1536 * 3, T]
    paths = [slb.RX_PATH_AUTO, slb.RX_PATH_FFT]
    got = drive(lambda: make(C, modes, chain, hz=hz), x, cuts, paths, 3, tx)
    if tx:
        ref = tune_cuts(port, drive(lambda: make(C, modes, chain), x, cuts, paths, 3, tx), incs, up=True)
    else:
        ref = drive(lambda: make(C, modes, chain), tune_cuts(port, x, incs, up=False), cuts, paths, 3, tx)
    assert np.array_equal(got, ref)
    whole = tx_dev(make(C, modes, chain, hz=hz), x) if tx else rx_dev(make(C, modes, chain, hz=hz), x)
    for env in ({"SELENITE_B200_SLICE_BYTES": str(C * 4 * 1536)}, {"SELENITE_B200_SLICE_BYTES": str(4 * 4 * 1536), "SELENITE_B200_SLICE_CHANNELS": "4"}):
        os.environ.update(env)
        try:
            d = make(C, modes, chain, hz=hz)
            y_host = d.tx_process(x) if tx else d.rx_process(x)
        finally:
            for k in env:
                del os.environ[k]
        assert np.array_equal(y_host, whole)


def test_ring_paths_feeder_live_and_per_channel_cadence(port):
    """Behind the firmware ring the tuned context equals an untuned one fed the oracle-tuned stream (1 ms API, slb_feeder_run, live
    feeder), and under per-channel cadence every channel equals a tuned one-channel context that sees only its own events."""
    C, B, ticks = 5, 48, 32
    hz = offsets(C, seed=5, zero_every=4)
    modes = [slb.MODE_USB, slb.MODE_LSB, slb.MODE_AM, slb.MODE_FM, slb.MODE_CW]
    x = slb.synth_iq(C, 2 * ticks * B)
    incs = incs_of(make(C, modes, hz=hz))
    xt = tune_cuts(port, x, incs, up=False)
    a = make(C, modes, hz=hz); a0 = make(C, modes)
    got, exp = [], []
    for t in range(2 * ticks):
        a.DSP_In_Buff_Write(x[:, t * B:(t + 1) * B].reshape(C, -1)); got.append(a.DSP_In_Buff_Read(4 * B))
        a0.DSP_In_Buff_Write(xt[:, t * B:(t + 1) * B].reshape(C, -1)); exp.append(a0.DSP_In_Buff_Read(4 * B))
    exp = np.stack(exp, 1).reshape(C, -1, 2)
    assert np.array_equal(np.stack(got, 1).reshape(C, -1, 2), exp)
    n = ticks * B
    b = make(C, modes, hz=hz)
    assert np.array_equal(np.concatenate([b.feeder_run(x[:, :n])[0], b.feeder_run(x[:, n:2 * n])[0]], 1), exp)
    e = make(C, modes, hz=hz); lv = e.live_open(8, 3, rx=True, tx=False); out = []
    for k in range(2 * ticks // 8):
        if lv.in_flight() == 3:
            out.append(lv.pop()[0])
        lv.push(x[:, k * 8 * B:(k + 1) * 8 * B])
    while lv.in_flight():
        out.append(lv.pop()[0])
    lv.close()
    assert np.array_equal(np.concatenate(out, 1), exp)
    d = make(C, modes, hz=hz); single = [make(1, [modes[c]], hz=hz[c:c + 1]) for c in range(C)]
    pos = [0] * C
    for t in range(60):
        w = np.array([not (c == 1 and t % 7 == 6) and not (c == 3 and t % 5 == 4) for c in range(C)])
        r = np.array([not (c == 0 and t % 11 == 10) and not (c == 4 and t % 3 == 2) for c in range(C)])
        blk = np.zeros((C, 2 * B), np.int16)
        for c in range(C):
            if w[c]:
                blk[c] = x[c, pos[c] % x.shape[1]:pos[c] % x.shape[1] + B].reshape(-1); pos[c] += B
        d.DSP_In_Buff_Write_Ch(blk, w.astype(np.uint8)); got = d.DSP_In_Buff_Read_Ch(4 * B, r.astype(np.uint8))
        for c in range(C):
            if w[c]:
                single[c].DSP_In_Buff_Write(blk[c:c + 1])
            ex = single[c].DSP_In_Buff_Read(4 * B)[0] if r[c] else np.zeros(2 * B, np.int16)
            assert np.array_equal(got[c], ex), (t, c)


def test_stream_shards_hold_their_slice_of_the_offsets():
    C, T = 12, 1536 * 2
    hz = offsets(C, seed=6)
    x = slb.synth_iq(C, T)
    whole = rx_dev(make(C, ALL8, hz=hz), x)
    parts = [rx_dev(make(6, ALL8[s:] + ALL8[:s], hz=hz[s:s + 6]), x[s:s + 6]) for s in (0, 6)]
    assert np.array_equal(np.concatenate(parts, 0), whole)


def test_retune_mid_stream_is_phase_continuous(port):
    C, T = 6, 1536 * 3
    hz_a, hz_b = offsets(C, seed=7), offsets(C, seed=8, zero_every=2)
    x = slb.synth_iq(C, T)
    cuts = [0, 1536, T]
    d = make(C, ALL8, hz=hz_a); inc_a = incs_of(d)
    y1 = rx_dev(d, x[:, :1536]); d.set_tune(hz_b); inc_b = incs_of(d); y2 = rx_dev(d, x[:, 1536:])
    xt = tune_cuts(port, x, inc_a, False, cuts, retune=(1, inc_b))
    d0 = make(C, ALL8)
    assert np.array_equal(np.concatenate([y1, y2], 1), np.concatenate([rx_dev(d0, xt[:, :1536]), rx_dev(d0, xt[:, 1536:])], 1))
    # single channels retuned one by one (slb_set_tune_channel) behave the same
    d = make(C, ALL8, hz=hz_a); y1 = rx_dev(d, x[:, :1536])
    for c in range(C):
        d.set_tune_channel(c, hz_b[c])
    assert np.array_equal(np.concatenate([y1, rx_dev(d, x[:, 1536:])], 1), np.concatenate([y1, y2], 1))
    # around a retune issued between live-feeder pushes, each chunk uses the offsets in force when it was pushed
    B, chunk = 48, 8
    e = make(C, ALL8, hz=hz_a); lv = e.live_open(chunk, 3, rx=True, tx=False)
    n = chunk * B; out = []
    for k in range(T // n):
        if k == 5:
            e.set_tune(hz_b)
        if lv.in_flight() == 3:
            out.append(lv.pop()[0])
        lv.push(x[:, k * n:(k + 1) * n])
    while lv.in_flight():
        out.append(lv.pop()[0])
    lv.close()
    xr = tune_cuts(port, x, inc_a, False, [0, 5 * n, T], retune=(1, inc_b))
    assert np.array_equal(np.concatenate(out, 1), make(C, ALL8).feeder_run(xr)[0])


def test_zero_offsets_change_nothing():
    C, T = 9, 1536 * 2
    x = slb.synth_iq(C, T)
    never = make(C, ALL8); zero = make(C, ALL8, hz=0.0); reset = make(C, ALL8, hz=offsets(C)); reset.set_tune(None)
    again = make(C, ALL8, hz=offsets(C))
    for c in range(C):
        again.set_tune_channel(c, 0.0)
    ys = []
    for d in (never, zero, reset, again):
        n0 = d.kernel_launches(); ys.append(rx_dev(d, x)); ys.append(d.kernel_launches() - n0)
    assert all(np.array_equal(ys[0], ys[2 * k]) for k in range(4)) and len(set(ys[1::2])) == 1
    # the caller's input is never written, also when it is mixed
    d = make(C, ALL8, hz=offsets(C)); xd = torch.from_numpy(x).cuda(); keep = xd.clone()
    d.rx_process(xd); torch.cuda.synchronize()
    assert torch.equal(xd, keep)
    t = make(C, TX_MODES, slb.CHAIN_TX_F32); t0 = make(C, TX_MODES, slb.CHAIN_TX_F32, hz=np.zeros(C))
    m = slb.synth_mic(C, T)
    n0, n1 = t.kernel_launches(), t0.kernel_launches()
    assert np.array_equal(tx_dev(t, m), tx_dev(t0, m)) and t.kernel_launches() - n0 == t0.kernel_launches() - n1


def test_refusals_rounding_and_96k(port):
    for chain in (slb.CHAIN_PASS, slb.CHAIN_RX_SSB_Q15, slb.CHAIN_CHAN64_F32):
        d = slb.DspIf(4, fs=192000 if chain == slb.CHAIN_CHAN64_F32 else 48000, chain=chain)
        for call in (lambda: d.set_tune(100.0), lambda: d.set_tune_channel(0, 100.0), lambda: d.tune(0)):
            with pytest.raises(slb.SeleniteError, match=r"-4"):
                call()
    d = make(3, [slb.MODE_USB])
    for bad in (24000.0, -24000.0, 1e12, float("nan"), float("inf")):
        with pytest.raises(slb.SeleniteError, match=r"-1"):
            d.set_tune_channel(1, bad)
        with pytest.raises(slb.SeleniteError, match=r"-1"):
            d.set_tune([0.0, bad, 0.0])
    assert d.tune(1) == (0, 0.0)                                                 # a refused call changed nothing
    with pytest.raises(slb.SeleniteError, match=r"-1"):
        d.set_tune_channel(3, 10.0)
    with pytest.raises(slb.SeleniteError, match=r"-1"):
        d.tune(3)
    for hz in (7300.3, -23999.9, 23999.99, 0.001, 12000.0):
        d.set_tune_channel(2, hz)
        inc, real = d.tune(2)
        assert inc == otu.increment(hz, 48000) and real == inc * 48000 / 2.0 ** 32
    # 96 kHz: the same contract at the other shipped rate
    C, T = 4, 1536 * 2
    hz = [0.0, 30000.0, -47000.0, 1234.5]
    d = make(C, [slb.MODE_USB, slb.MODE_LSB], fs=96000, hz=hz)
    assert d.tune(2)[0] == otu.increment(-47000.0, 96000)
    x = slb.synth_iq(C, T, fs=96000)
    assert np.array_equal(rx_dev(d, x), rx_dev(make(C, [slb.MODE_USB, slb.MODE_LSB], fs=96000), tune_cuts(port, x, incs_of(d), False)))
    t = make(C, [slb.MODE_USB], slb.CHAIN_TX_SSB_F32, fs=96000, hz=hz); m = slb.synth_mic(C, T, fs=96000)
    assert np.array_equal(tx_dev(t, m), tune_cuts(port, tx_dev(make(C, [slb.MODE_USB], slb.CHAIN_TX_SSB_F32, fs=96000), m), incs_of(t), True))


def test_misaligned_caller_input_is_refused_before_the_mixer():
    """slb_rx_process_device on a tuned context with a caller row that is not 16-byte aligned (a contiguous view at a frame offset)
    returns SLB_ERR_CUDA (misaligned address) without launching anything; the context goes on as if the call had not been made."""
    C, T = 3, 1536
    x = slb.synth_iq(C, T)
    d = make(C, [slb.MODE_USB, slb.MODE_LSB], hz=[1000.0, -2500.0, 0.0])
    buf = torch.zeros(C * T * 2 + 2, dtype=torch.int16, device="cuda")
    xm = buf[2:].view(C, T, 2)                                                    # 4 bytes past a 16-byte boundary
    xm.copy_(torch.from_numpy(x).cuda())
    assert xm.is_contiguous() and xm.data_ptr() % 16 == 4
    n0 = d.kernel_launches()
    with pytest.raises(slb.SeleniteError, match=r"-2"):
        d.rx_process(xm)
    torch.cuda.synchronize()
    assert d.kernel_launches() == n0
    assert np.array_equal(rx_dev(d, x), rx_dev(make(C, [slb.MODE_USB, slb.MODE_LSB], hz=[1000.0, -2500.0, 0.0]), x))


def test_loopback_and_rejection():
    """TX-USB at +f into RX-USB at +f on the GPU: the 1 kHz tone's SNR is within 0.1 dB of the oracle loop (test_tune_oracle.py); a
    station at 0 Hz is rejected by an RX context tuned 10 kHz away."""
    y = tx_dev(make(1, [slb.MODE_USB], slb.CHAIN_TX_SSB_F32, hz=[LOOPBACK_HZ]), loopback_input()[None])
    a = rx_dev(make(1, [slb.MODE_USB], hz=[LOOPBACK_HZ]), y)
    snr = otm.tone_snr_db(a[0, 384 * 8:, 0], 48000, 1000.0)
    assert abs(snr - LOOPBACK_SNR_DB) <= 0.1, snr
    x = slb.synth_iq(1, 384 * 40, f0=1000.0)
    on = otm.tone_snr_db(rx_dev(make(1, [slb.MODE_USB]), x)[0, 384 * 8:, 0], 48000, 1000.0)
    off = otm.tone_snr_db(rx_dev(make(1, [slb.MODE_USB], hz=[10000.0]), x)[0, 384 * 8:, 0], 48000, 1000.0)
    assert on > 20.0 and off < 0.0, (on, off)


@pytest.mark.timeout(900, method="thread")
def test_scale_1024_channels_and_one_long_channel(port, best_oracle):
    C, T = 1024, 96000
    base = slb.synth_iq(16, T)
    rng = np.random.Generator(np.random.PCG64(10))
    x = np.ascontiguousarray(base[rng.integers(0, 16, C)])
    hz = rng.uniform(-23000.0, 23000.0, C); hz[::5] = 0.0
    d = make(C, ALL8, hz=hz)
    y = rx_dev(d, x)
    for c in sorted(set(rng.integers(0, C, 6).tolist()) | {0, 1, C - 1}):
        xt = tune_cuts(port, x[c:c + 1], [d.tune(c)[0]], False)
        assert np.array_equal(y[c:c + 1], rx_dev(make(1, [ALL8[c % 8]]), xt)), c
        if ALL8[c % 8] in (slb.MODE_USB, slb.MODE_LSB, slb.MODE_DIG, slb.MODE_PKT):
            check_int16(y[c], best_oracle.rx_ssb_f32(d.oracle_params(ALL8[c % 8]), xt[0])[0])
    # one channel x 10 s: many CTAs of the mixer share the channel, and the phase advances once per call
    T1 = 480000
    x1 = slb.synth_iq(1, T1)
    d = make(1, [slb.MODE_USB], hz=[7300.3]); inc = d.tune(0)[0]
    y1 = rx_dev(d, x1); y2 = rx_dev(d, x1[:, :1536])
    xt, ph = otu.tune_q15(port, x1[0], inc, 0, False)
    xt2, _ = otu.tune_q15(port, x1[0, :1536], inc, ph, False)
    d0 = make(1, [slb.MODE_USB])
    assert np.array_equal(y1, rx_dev(d0, xt[None])) and np.array_equal(y2, rx_dev(d0, xt2[None]))


@pytest.mark.timeout(1500, method="thread")
def test_parity_on_the_stress_build():
    """This file's parity tests on the stress build (random delays at every hand-over), like tests/test_gpu_stress_build.py does for the others."""
    if not os.path.exists(_build.STRESS_LIB_PATH):
        pytest.skip("stress build not present (python __graft_entry__.py builds it)")
    env = dict(os.environ, SELENITE_B200_LIB=_build.STRESS_LIB_PATH)
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "900",
                        os.path.abspath(__file__), "-k", "not stress_build"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1400)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
