"""GPU parity of the all-integer SSB modulator TX-SSB-q15 (SLB_CHAIN_TX_SSB_Q15, DESIGN.md §3.7: the mic through the fir_q15 Hilbert
pair of RX-SSB-q15 on the integer tensor cores, the rail order by sideband, the q15 ALC), called through the C ABI, against the oracle
(oracle/slo_tx_q15.h through tests/oracle_tx_q15.py) and the committed golden vectors. Every stage is integer arithmetic, so every
comparison is BIT-EXACT: pre-ALC (I, Q), per-block gain word and output."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_tx_q15 as otq
import selenite_lite_b200 as slb
import test_gpu_ring as ring
from selenite_lite_b200 import build as _build
from test_golden import GOLD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CH = slb.CHAIN_TX_SSB_Q15
MODES = [slb.MODE_USB, slb.MODE_LSB, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG, slb.MODE_PKT]
ERR_STATE, ERR_UNSUPPORTED = -3, -4


def run_gpu(d, x, want_dbg=True):
    """Returns out int16 [C][T][2] I/Q, pre-ALC (I, Q) int16 [C][T][2], gain words uint32 [C][T/48]."""
    Cn, T = x.shape[0], x.shape[1]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    iq = torch.zeros((Cn, T, 2), dtype=torch.int16, device="cuda") if want_dbg else None
    gain = torch.zeros((Cn, T // 48), dtype=torch.int32, device="cuda") if want_dbg else None
    d.set_q15_debug_taps(iq, gain)
    y = d.tx_process(xd)
    torch.cuda.synchronize()
    d.set_q15_debug_taps(None, None)
    return y.cpu().numpy(), (iq.cpu().numpy() if want_dbg else None), (gain.cpu().numpy().view(np.uint32) if want_dbg else None)


def set_modes(d, n):
    for c in range(n):
        d.DSP_Set_Mode(MODES[c % len(MODES)], channel=c)


def hot(d):
    """The context's taps x 4 clipped to the split range (taps < 32640): the FIRs saturate on a loud mic."""
    p = d.rx_q15_params()
    for k in range(64):
        p.taps_i[k] = int(np.clip(4 * p.taps_i[k], -32639, 32639)); p.taps_q[k] = int(np.clip(4 * p.taps_q[k], -32639, 32639))
    d.set_rx_q15_params(p)


def check_vs_oracle(o, d, x, y, iq, gain, channels):
    for c in channels:
        exp, e_iq, e_g, _ = otq.tx_ssb_q15(o, d.oracle_params(MODES[c % len(MODES)]), x[c])
        if iq is not None:
            assert np.array_equal(iq[c], e_iq), (c, int(np.argmax(np.any(iq[c] != e_iq, axis=1))))
            assert np.array_equal(gain[c], e_g), c
        assert np.array_equal(y[c], exp), (c, int(np.argmax(np.any(y[c] != exp, axis=1))))


@pytest.mark.parametrize("name,mode", [("usb", slb.MODE_USB), ("lsb", slb.MODE_LSB), ("sat", slb.MODE_USB)])
def test_golden_vectors(name, mode):
    g = np.load(os.path.join(GOLD, "tx_ssb_q15.npz"))
    d = slb.DspIf(1, chain=CH)
    d.DSP_Set_Mode(mode)
    p = d.rx_q15_params()
    assert np.array_equal(np.array(p.taps_i[:], np.int16), g["taps_i"]) and np.array_equal(np.array(p.rel[:], np.int16), g["rel"])
    assert [p.agc_window, p.agc_target, p.agc_floor, p.agc_gmax_q15] == [int(v) for v in g["agc"]]
    if name == "sat":
        hot(d)
    y, iq, gain = run_gpu(d, g["%s_in" % name][None])
    assert np.array_equal(iq[0], g["%s_iq" % name])
    assert np.array_equal(gain[0], g["%s_gain" % name])
    assert np.array_equal(y[0], g["%s_out" % name])


@pytest.mark.parametrize("channels,frames", [(1, 48), (3, 96), (8, 1488), (9, 4800), (33, 9600), (130, 3072)])
def test_vs_oracle_ragged_shapes(port, channels, frames):
    """Mixed modes per channel; an input with L != R gives the same bytes as the same input with R := L (R is ignored)."""
    x = slb.synth_mic(channels, frames)
    rng = np.random.Generator(np.random.PCG64(channels * 7919 + frames))
    x[:, :, 1] = rng.integers(-32768, 32768, (channels, frames))
    d = slb.DspIf(channels, chain=CH); set_modes(d, channels)
    y, iq, gain = run_gpu(d, x)
    check_vs_oracle(port, d, x, y, iq, gain, range(channels))
    x2 = x.copy(); x2[:, :, 1] = x2[:, :, 0]
    e = slb.DspIf(channels, chain=CH); set_modes(e, channels)
    y2, iq2, gain2 = run_gpu(e, x2)
    assert np.array_equal(y, y2) and np.array_equal(iq, iq2) and np.array_equal(gain, gain2)


def test_every_saturation_point(port, rng):
    """Hot taps and a full-scale mic: the FIR's __SSAT and arm_abs_q15 (-32768) fire on many samples; the split-byte tensor-core FIR
    must still equal the 64-bit accumulator. (arm_scale_q15 cannot saturate here: the envelope is never below the block's own peak,
    so no scaled sample exceeds the target — the oracle test holds that bound.) A quiet channel brings the gain limit in."""
    Cn, T = 16, 4800
    d = slb.DspIf(Cn, chain=CH); hot(d); set_modes(d, Cn)
    x = rng.integers(-32768, 32768, (Cn, T, 2)).astype(np.int16)
    x[0, 100:600] = -32768; x[1, 100:600] = 32767; x[2, 100:600, 0] = np.where(np.arange(500) % 24 < 12, 32767, -32768)
    x[3, 1000:2000] = 0; x[4] = (x[4] // 4096).astype(np.int16)
    y, iq, gain = run_gpu(d, x)
    check_vs_oracle(port, d, x, y, iq, gain, range(Cn))
    assert int(np.sum(np.abs(iq.astype(np.int32)) >= 32767)) > 100 and int(np.sum(iq == -32768)) > 0


def test_streaming_two_calls_equal_one(port):
    """The carried raw tail and peak window are the whole state: cuts on and off the 768-frame supertile grid."""
    Cn, T = 6, 48 * 400
    x = slb.synth_mic(Cn, T)
    whole = slb.DspIf(Cn, chain=CH); set_modes(whole, Cn)
    yw, iqw, gw = run_gpu(whole, x)
    for cut in (768 * 3, 48 * 37, 48):
        d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
        parts = [run_gpu(d, np.ascontiguousarray(x[:, a:b])) for a, b in ((0, cut), (cut, T))]
        for j, w in enumerate((yw, iqw, gw)):
            assert np.array_equal(np.concatenate([p_[j] for p_ in parts], 1), w), (cut, j)
    check_vs_oracle(port, whole, x, yw, iqw, gw, (0, 1, 5))


def test_host_path_equals_device_path_when_sliced():
    Cn, T = 13, 1536 * 6 + 48 * 5
    x = slb.synth_mic(Cn, T)
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
    for mode in (slb.MODE_AM, slb.MODE_FM):
        assert lib.SLB_DSP_Set_Mode(h, mode) == ERR_UNSUPPORTED
        assert lib.SLB_DSP_Set_Mode_Channel(h, 1, mode) == ERR_UNSUPPORTED
    before = bytes(d.rx_q15_params())

    def refused(edit):
        p = d.rx_q15_params(); edit(p)
        assert lib.slb_set_rx_q15_params(h, C.byref(p)) == ERR_UNSUPPORTED
        assert bytes(d.rx_q15_params()) == before
    refused(lambda p: setattr(p, "bq_stages", 1))
    refused(lambda p: p.taps_i.__setitem__(7, 32640))                  # (every negative int16 splits: -32768 = 256 (-128) + 0)
    refused(lambda p: p.taps_q.__setitem__(60, 32767))
    refused(lambda p: setattr(p, "agc_window", 18))
    assert lib.slb_set_tune(h, None) == ERR_UNSUPPORTED
    assert lib.slb_set_tune_channel(h, 0, 100.0) == ERR_UNSUPPORTED
    x = torch.zeros((2, 96, 2), dtype=torch.int16, device="cuda"); y = torch.empty_like(x)
    assert lib.slb_rx_process_device(h, x.data_ptr(), y.data_ptr(), 96, None) == ERR_STATE
    xh = np.zeros((2, 96, 2), np.int16); yh = np.empty_like(xh)
    assert lib.slb_rx_process_host(h, xh.ctypes.data, yh.ctypes.data, 96) == ERR_STATE
    assert lib.slb_tx_process_device(h, x.data_ptr(), y.data_ptr(), 40, None) == -1          # frames % 48 != 0
    r = slb.DspIf(2, chain=slb.CHAIN_RX_SSB_Q15)
    assert r.lib.slb_tx_process_device(r.h, x.data_ptr(), y.data_ptr(), 96, None) == ERR_STATE
    with pytest.raises(slb.SeleniteError):
        slb.DspIf(2, fs=96000, chain=CH)


def test_1ms_api_equals_bulk(port):
    """Behind the firmware's 1 ms cadence: each 48-frame mic block is modulated in the call that delivers it (no added latency), then
    rides the ring — the same ring fed with the bulk output."""
    Cn, nblk = 5, 40
    x = slb.synth_mic(Cn, 48 * nblk)
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
    """Same layout and size as RX-SSB-q15 (64 raw frames, the peak window, sidebands); a restored context continues bit for bit."""
    Cn, T = 7, 48 * 60
    x = slb.synth_mic(Cn, T)
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    assert d.state_save().size == slb.DspIf(Cn, chain=slb.CHAIN_RX_SSB_Q15).state_save().size
    y1, _, _ = run_gpu(d, np.ascontiguousarray(x[:, :48 * 23]), want_dbg=False)
    snap = d.state_save()
    y2, iq2, g2 = run_gpu(d, np.ascontiguousarray(x[:, 48 * 23:]))
    e = slb.DspIf(Cn, chain=CH)                                               # modes come back with the checkpoint
    e.state_load(snap)
    z2, zq2, zg2 = run_gpu(e, np.ascontiguousarray(x[:, 48 * 23:]))
    assert np.array_equal(z2, y2) and np.array_equal(zq2, iq2) and np.array_equal(zg2, g2)
    whole = slb.DspIf(Cn, chain=CH); set_modes(whole, Cn)
    yw, _, _ = run_gpu(whole, x, want_dbg=False)
    assert np.array_equal(np.concatenate([y1, y2], 1), yw)


_DROPIN = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import oracle_lib, oracle_tx_q15 as otq, selenite_lite_b200 as slb
from selenite_lite_b200 import _lib
lib = _lib.load()
lib.DSP_Init(); lib.DSP_Set_Mode(slb.MODE_LSB)
x = slb.synth_mic(1, 48 * 30)[0]
prm = slb.dsp_if.q15_params_to_dict(slb.default_rx_q15_params(48000), lsb=1)
exp = otq.tx_ssb_q15(oracle_lib.Oracle("port"), prm, x)[0]
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
    env = dict(os.environ, SELENITE_B200_CHAIN="tx_ssb_q15")
    r = subprocess.run([sys.executable, "-c", _DROPIN, ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "dropin ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_loopback_gpu_equals_oracle(port):
    """TX-SSB-q15 -> RX-SSB-q15 on the GPU (USB and LSB receivers) equals the same loopback through the oracle byte for byte."""
    Cn, T = 4, 48 * 200
    n = np.arange(T)
    m = np.stack([np.rint(0.3 * 32768 * np.cos(2 * np.pi * (800.0 + 400.0 * c) * n / 48000)) for c in range(Cn)]).astype(np.int16)
    x = np.ascontiguousarray(np.stack([m, m], axis=2))
    tx = slb.DspIf(Cn, chain=CH)
    y, _, _ = run_gpu(tx, x, want_dbg=False)
    for rx_mode in (slb.MODE_USB, slb.MODE_LSB):
        rx = slb.DspIf(Cn, chain=slb.CHAIN_RX_SSB_Q15); rx.DSP_Set_Mode(rx_mode)
        audio = torch.zeros((Cn, T), dtype=torch.int16, device="cuda"); rx.set_q15_debug_taps(audio, None)
        z = rx.rx_process(torch.from_numpy(y).cuda()).cpu().numpy(); a = audio.cpu().numpy()
        for c in range(Cn):
            e_y = otq.tx_ssb_q15(port, tx.oracle_params(slb.MODE_USB), x[c])[0]
            e_z, e_a, _, _ = port.rx_ssb_q15(rx.oracle_params(rx_mode), e_y)
            assert np.array_equal(z[c], e_z) and np.array_equal(a[c], e_a), (rx_mode, c)


@pytest.mark.timeout(600, method="thread")
def test_scale_1024_mic_channels_10s(port):
    """1024 mic channels x 10 s (BASELINE config 3's width): whole streams against the oracle on channels spread over the batch."""
    Cn, T = 1024, 480000
    x = slb.synth_mic(8, T)
    x = np.ascontiguousarray(np.tile(x, (Cn // 8, 1, 1)))
    d = slb.DspIf(Cn, chain=CH); set_modes(d, Cn)
    y, _, _ = run_gpu(d, x, want_dbg=False)
    for c in (0, 1, 147, 511, 514, 777, 1022, 1023):
        exp = otq.tx_ssb_q15(port, d.oracle_params(MODES[c % len(MODES)]), x[c])[0]
        assert np.array_equal(y[c], exp), (c, int(np.argmax(np.any(y[c] != exp, axis=1))))


@pytest.mark.timeout(600, method="thread")
def test_scale_8192_channels_2s(port):
    """8192 channels x 2 s: seven channel groups per CTA, the width where the RX kernel once hung. The pre-ALC tap of EVERY channel
    equals slb_st_fir_q15 of L with taps_i / taps_q (an independent kernel) in the rail order of its mode; the output equals the oracle
    on sampled channels."""
    Cn, T = 8192, 96000
    g = torch.Generator(device="cuda"); g.manual_seed(9)
    x = torch.randint(-20000, 20000, (Cn, T, 2), dtype=torch.int16, device="cuda", generator=g)
    d = slb.DspIf(Cn, chain=CH)
    lsb = np.zeros(Cn, bool)
    for c in range(1, Cn, 3):
        d.DSP_Set_Mode(slb.MODE_LSB, channel=c); lsb[c] = True
    iq = torch.zeros((Cn, T, 2), dtype=torch.int16, device="cuda")
    d.set_q15_debug_taps(iq, None)
    y = d.tx_process(x)
    torch.cuda.synchronize()
    d.set_q15_debug_taps(None, None)
    p = d.rx_q15_params()
    st = slb.DspIf(Cn, chain=slb.CHAIN_PASS)
    mic = x[:, :, 0].contiguous()
    rails = []
    for taps in (p.taps_i, p.taps_q):
        c_rev = np.ascontiguousarray(np.array(taps[:64], np.int16)[::-1])
        hist = torch.zeros((Cn, 63), dtype=torch.int16, device="cuda"); out = torch.empty((Cn, T), dtype=torch.int16, device="cuda")
        st.st("fir_q15", c_rev, 64, hist, mic, out, T)
        rails.append(out)
    torch.cuda.synchronize()
    sel = torch.from_numpy(lsb).cuda()[:, None]
    exp_i = torch.where(sel, rails[0], rails[1]); exp_q = torch.where(sel, rails[1], rails[0])
    assert torch.equal(iq[:, :, 0], exp_i) and torch.equal(iq[:, :, 1], exp_q)
    del iq, rails, exp_i, exp_q, mic
    for c in (0, 1, 2, 1023, 4097, 8190, 8191):
        xc = x[c].cpu().numpy()
        exp = otq.tx_ssb_q15(port, d.oracle_params(slb.MODE_LSB if lsb[c] else slb.MODE_USB), xc)[0]
        assert np.array_equal(y[c].cpu().numpy(), exp), c


@pytest.mark.timeout(1500, method="thread")
def test_parity_on_the_stress_build():
    """This file's parity tests on the stress build (random delays at every hand-over), like tests/test_gpu_stress_build.py does for the others."""
    if not os.path.exists(_build.STRESS_LIB_PATH):
        pytest.skip("stress build not present (python __graft_entry__.py builds it)")
    env = dict(os.environ, SELENITE_B200_LIB=_build.STRESS_LIB_PATH)
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "900",
                        os.path.abspath(__file__), "-k", "not stress_build"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1400)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
