"""GPU tests of the all-mode TX chain (SLB_CHAIN_TX_F32, DESIGN.md §3.4): AM and FM channels on the FFT kernel next to SSB-style
channels, against the oracle (oracle/slo_tx_mod.h through tests/oracle_tx_mod.py) and the committed golden vectors.

The FM output cannot be held to the oracle sample by sample: a 1e-7 difference of the baseband is a permanent offset of the integer
phase. It is checked decomposed instead: the increments diff(phi) against the oracle's within the baseband tolerance, the output
bit-identical to the oracle's NCO of the GPU's own phase, and the phase continuing exactly wherever the stream is cut."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_tx_mod as otm
import selenite_lite_b200 as slb
from selenite_lite_b200 import build as _build
from test_golden import GOLD, iq_tolerance
from test_gpu_tx_ssb_f32 import check_int16
from test_tx_am_fm_oracle import LOOPBACK_SNR_DB, loopback_input, worst_case_mics

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIXED = [slb.MODE_AM, slb.MODE_FM, slb.MODE_USB, slb.MODE_LSB, slb.MODE_CW]


def run_gpu(d, x, want_dbg=True):
    """Returns out int16 [C][T][2], pre-ALC baseband f32 [C][T][2], gains [C][T/48], FM phase uint32 [C][T] (0 for other channels)."""
    C, T = x.shape[0], x.shape[1]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    iq = torch.zeros((C, T, 2), dtype=torch.float32, device="cuda") if want_dbg else None
    gain = torch.zeros((C, T // 48), dtype=torch.float32, device="cuda") if want_dbg else None
    ph = torch.zeros((C, T), dtype=torch.int32, device="cuda") if want_dbg else None
    d.set_debug_taps(iq, gain); d.set_phase_tap(ph)
    y = d.tx_process(xd)
    torch.cuda.synchronize()
    d.set_debug_taps(None, None); d.set_phase_tap(None)
    if not want_dbg:
        return y.cpu().numpy(), None, None, None
    return y.cpu().numpy(), iq.cpu().numpy(), gain.cpu().numpy(), ph.cpu().numpy().view(np.uint32)


def make(C, modes, path=slb.RX_PATH_AUTO, chain=slb.CHAIN_TX_F32):
    d = slb.DspIf(C, chain=chain); d.set_rx_path(path)
    for c in range(C):
        d.DSP_Set_Mode(modes[c % len(modes)], channel=c)
    return d


def check_fm(port, prm, x, y, z, gain, phase, phase0=0):
    """(a) increments against the oracle's within 2^31 (2 g tol_a + 2^-22 |u|) + 1 (the baseband difference enters once through
    a and once through the block gain; the product and the division round once each); (b) the output is the NCO of the GPU's phase."""
    _, z_o, g_o, ph_o, _ = otm.tx_mod_f32(port, prm, x)
    tol = iq_tolerance(z_o)[:, 0]
    assert np.all(np.abs(z[:, 0] - z_o[:, 0]) <= tol + 1e-9)
    assert np.allclose(gain, g_o, rtol=2e-5)
    g = np.repeat(g_o.astype(np.float64), 48)
    u = np.abs(z_o[:, 0].astype(np.float64) * g)
    inc = np.diff(np.concatenate([[phase0], phase]).astype(np.uint32)).view(np.int32).astype(np.int64)
    inc_o = np.diff(np.concatenate([[0], ph_o]).astype(np.uint32)).view(np.int32).astype(np.int64)
    bound = 2.0 ** 31 * (2.0 * g * tol + 2.0 ** -22 * u) + 1
    assert np.all(np.abs(inc - inc_o) <= bound), float(np.max(np.abs(inc - inc_o) / bound))
    assert np.array_equal(otm.tx_fm_nco(port, phase, prm["fm_level"]), y)


def check_am(port, prm, x, y, z, gain):
    exp, z_o, g_o, _, _ = otm.tx_mod_f32(port, prm, x)
    tol = iq_tolerance(z_o)
    assert np.all(np.abs(z - z_o) <= tol + 1e-9), float(np.max(np.abs(z - z_o) / (tol + 1e-9)))
    assert np.allclose(gain, g_o, rtol=2e-5)
    assert np.all(y[:, 1] == 0)
    check_int16(y, exp)


def test_golden_vectors(port):
    g = np.load(os.path.join(GOLD, "tx_am_fm_f32.npz"))
    for name, mode in (("am", slb.MODE_AM), ("fm", slb.MODE_FM)):
        d = make(1, [mode])
        assert np.array_equal(d.mask(mode), g["%s_mask" % name])
        y, z, gain, ph = run_gpu(d, g["%s_in" % name][None])
        prm = d.oracle_params(mode)
        err = np.abs(z[0] - g["%s_iq" % name]); tol = iq_tolerance(g["%s_iq" % name])
        assert np.all(err <= tol + 1e-9)
        assert np.allclose(gain[0], g["%s_gain" % name], rtol=2e-5)
        if mode == slb.MODE_AM:
            assert np.all(y[0, :, 1] == 0); check_int16(y[0], g["am_out"])
        else:
            check_fm(port, prm, g["fm_in"], y[0], z[0], gain[0], ph[0])


@pytest.mark.parametrize("channels,frames", [(1, 384), (3, 768), (7, 1920), (33, 4608), (130, 3072)])
def test_vs_oracle_ragged_shapes_mixed_modes(port, best_oracle, channels, frames):
    x = slb.synth_mic(channels, frames)
    d = make(channels, MIXED)
    y, z, gain, ph = run_gpu(d, x)
    ssb = make(channels, [m if m not in (slb.MODE_AM, slb.MODE_FM) else slb.MODE_USB for m in MIXED], chain=slb.CHAIN_TX_SSB_F32)
    y_ssb = run_gpu_ssb(ssb, x)
    for c in range(channels):
        mode = MIXED[c % len(MIXED)]
        prm = d.oracle_params(mode)
        if mode == slb.MODE_AM:
            check_am(port, prm, x[c], y[c], z[c], gain[c])
        elif mode == slb.MODE_FM:
            check_fm(port, prm, x[c], y[c], z[c], gain[c], ph[c])
        else:
            assert np.array_equal(y[c], y_ssb[c]), c                              # SSB-style channels: bit for bit the TX-SSB chain
            exp, z_o, g_o, _ = best_oracle.tx_ssb_f32(prm, x[c])
            assert np.all(np.abs(z[c] - z_o) <= iq_tolerance(z_o) + 1e-9)
            check_int16(y[c], exp)


def run_gpu_ssb(d, x):
    y = d.tx_process(torch.from_numpy(np.ascontiguousarray(x)).cuda()); torch.cuda.synchronize()
    return y.cpu().numpy()


def test_fm_phase_continues_across_cuts_paths_slices_and_checkpoints():
    """One stream of AM / FM / SSB channels: calls cut at hop boundaries, calls served alternately by AUTO and FFT paths, the
    time-sliced host path (channel blocks x time slices) and a mid-stream checkpoint into a fresh context all give the uncut result."""
    C, T = 11, 1536 * 3 + 384
    x = slb.synth_mic(C, T)
    y, _, _, ph = run_gpu(make(C, MIXED), x)
    cuts = [0, 384, 1536, 1536 + 768, 1536 * 3, T]
    d = make(C, MIXED); parts, phs = [], []
    for i in range(len(cuts) - 1):
        d.set_rx_path(slb.RX_PATH_FFT if i % 2 else slb.RX_PATH_AUTO)
        if i == 3:
            snap = d.state_save(); d = make(C, MIXED); d.state_load(snap)
        yy, _, _, pp = run_gpu(d, x[:, cuts[i]:cuts[i + 1]])
        parts.append(yy); phs.append(pp)
    # AM and FM channels are on the FFT kernel on both paths: bit for bit; SSB-style channels change kernel with the path (the
    # tensor-core and FFT kernels agree within 1 LSB, tests/test_gpu_tx_ssb_f32.py)
    ya = np.concatenate(parts, 1)
    for c in range(C):
        if MIXED[c % len(MIXED)] in (slb.MODE_AM, slb.MODE_FM):
            assert np.array_equal(ya[c], y[c]), c
        else:
            check_int16(ya[c], y[c])
    fm = [c for c in range(C) if MIXED[c % len(MIXED)] == slb.MODE_FM]
    assert np.array_equal(np.concatenate(phs, 1)[fm], ph[fm])
    for env in ({"SELENITE_B200_SLICE_BYTES": str(C * 4 * 1536)}, {"SELENITE_B200_SLICE_BYTES": str(4 * 4 * 1536), "SELENITE_B200_SLICE_CHANNELS": "4"}):
        os.environ.update(env)
        try:
            y_host = make(C, MIXED).tx_process(x)
        finally:
            for k in env:
                del os.environ[k]
        assert np.array_equal(y_host, y)


def test_1ms_api_feeder_live_feeder_and_per_channel_cadence():
    """Behind the firmware ring, AM and FM channels go through the same paths as SSB: slb_feeder_run and the live feeder equal the
    per-tick calls, and under per-channel cadence every channel equals a one-channel context that sees only its own events."""
    C, B, ticks = 5, 48, 32
    x = slb.synth_mic(C, 2 * ticks * B + 8 * B)
    a = make(C, MIXED); b = make(C, MIXED); e = make(C, MIXED)
    exp = []
    for t in range(2 * ticks):
        a.DSP_In_Buff_Write(x[:, t * B:(t + 1) * B].reshape(C, -1)); exp.append(a.DSP_In_Buff_Read(4 * B))
    exp = np.stack(exp, 1).reshape(C, -1, 2)
    assert np.any(exp[0] != 0) and np.any(exp[1] != 0)                         # the AM and FM channels did transmit
    n = ticks * B
    got = np.concatenate([b.feeder_run(x[:, :n])[0], b.feeder_run(x[:, n:2 * n])[0]], 1)
    assert np.array_equal(got, exp)
    lv = e.live_open(8, 3, rx=True, tx=False); out = []
    for k in range(2 * ticks // 8):
        if lv.in_flight() == 3:
            out.append(lv.pop()[0])
        lv.push(x[:, k * 8 * B:(k + 1) * 8 * B])
    while lv.in_flight():
        out.append(lv.pop()[0])
    lv.close()
    assert np.array_equal(np.concatenate(out, 1), exp)
    # per-channel cadence against one-channel contexts
    d = make(C, MIXED); single = [make(1, [MIXED[c]]) for c in range(C)]
    pos = [0] * C
    for t in range(60):
        w = np.array([not (c == 1 and t % 7 == 6) and not (c == 3 and t % 5 == 4) for c in range(C)])
        r = np.array([not (c == 0 and t % 11 == 10) and not (c == 4 and t % 3 == 2) for c in range(C)])
        blk = np.zeros((C, 2 * B), np.int16)
        for c in range(C):
            if w[c]:
                blk[c] = x[c, pos[c]:pos[c] + B].reshape(-1); pos[c] += B
        d.DSP_In_Buff_Write_Ch(blk, w.astype(np.uint8)); got = d.DSP_In_Buff_Read_Ch(4 * B, r.astype(np.uint8))
        for c in range(C):
            if w[c]:
                single[c].DSP_In_Buff_Write(blk[c:c + 1])
            ex = single[c].DSP_In_Buff_Read(4 * B)[0] if r[c] else np.zeros(2 * B, np.int16)
            assert np.array_equal(got[c], ex), (t, c)


def test_direction_switch_and_mode_refusals():
    C, B = 3, 48
    x = slb.synth_mic(C, 40 * B)
    a = make(C, [slb.MODE_FM, slb.MODE_AM, slb.MODE_USB]); fresh = make(C, [slb.MODE_FM, slb.MODE_AM, slb.MODE_USB])
    a.DSP_Set_TX()
    for t in range(12):
        a.DSP_In_Buff_Write(x[:, t * B:(t + 1) * B].reshape(C, -1)); a.DSP_In_Buff_Read(4 * B)
    a.DSP_Set_RX(); a.DSP_Set_TX(); fresh.DSP_Set_TX()
    snap_a, snap_f = a.state_save(), fresh.state_save()
    hdr = 4 * 20                                                                  # the header carries the ring pointers, which keep their cadence
    assert np.array_equal(snap_a[hdr:], snap_f[hdr:])
    for t in range(12, 40):
        for d in (a, fresh):
            d.DSP_In_Buff_Write(x[:, t * B:(t + 1) * B].reshape(C, -1))
    y_a = run_gpu(a, x[:, :768], want_dbg=False)[0]; y_f = run_gpu(fresh, x[:, :768], want_dbg=False)[0]
    assert np.array_equal(y_a, y_f)
    ssb = slb.DspIf(1, chain=slb.CHAIN_TX_SSB_F32)
    for mode in (slb.MODE_AM, slb.MODE_FM):
        with pytest.raises(slb.SeleniteError):
            ssb.DSP_Set_Mode(mode)
    with pytest.raises(slb.SeleniteError):
        slb.DspIf(1, chain=slb.CHAIN_TX_F32).DSP_Set_Mode(0x07)
    with pytest.raises(slb.SeleniteError):
        ssb.set_tx_mod_params(slb.default_tx_mod_params())
    p = a.tx_mod_params(); p.am_depth = 1.5
    with pytest.raises(slb.SeleniteError):
        a.set_tx_mod_params(p)


def test_worst_case_mic_inputs(port):
    """Rails, full-scale tone, square wave: no wrap-around anywhere — AM stays inside its envelope bounds, FM increments stay bounded
    (and both follow the oracle as everywhere else), on both paths."""
    x = worst_case_mics(768 * 4)
    for mode in (slb.MODE_AM, slb.MODE_FM):
        for path in (slb.RX_PATH_AUTO, slb.RX_PATH_FFT):
            d = make(x.shape[0], [mode], path)
            y, z, gain, ph = run_gpu(d, x)
            prm = d.oracle_params(mode)
            for c in range(x.shape[0]):
                if mode == slb.MODE_AM:
                    cc, dd = prm["am_carrier"], prm["am_depth"]
                    assert y[c, :, 0].min() >= int(np.floor(cc * (1 - dd) * 32768)) - 1 and y[c, :, 0].max() <= int(np.ceil(cc * (1 + dd) * 32768)) + 1
                    exp = otm.tx_mod_f32(port, prm, x[c])[0]
                    dl = np.abs(y[c].astype(np.int32) - exp.astype(np.int32))
                    assert dl.max() <= 1 and np.all(y[c, :, 1] == 0)
                else:
                    inc = np.diff(np.concatenate([[0], ph[c]]).astype(np.uint32)).view(np.int32).astype(np.int64)
                    assert np.max(np.abs(inc)) <= float(otm.fm_target(prm)) * 2 ** 31 * (1 + 2 ** -22) + 1
                    assert np.array_equal(otm.tx_fm_nco(port, ph[c], prm["fm_level"]), y[c])


@pytest.mark.parametrize("mode", [slb.MODE_AM, slb.MODE_FM])
def test_loopback_tx_into_rx(mode):
    """TX-AM into an RX-SSB-f32 context in AM, TX-FM into one in FM, all on the GPU: the recovered 1 kHz tone's SNR is within 0.1 dB
    of the same loop through the oracle (port TX -> port RX, recorded in test_tx_am_fm_oracle.py)."""
    x = loopback_input()[None]
    y = run_gpu(make(1, [mode]), x, want_dbg=False)[0]
    rx = slb.DspIf(1, chain=slb.CHAIN_RX_SSB_F32); rx.DSP_Set_Mode(mode)
    a = rx.rx_process(torch.from_numpy(y).cuda()).cpu().numpy()
    snr = otm.tone_snr_db(a[0, 384 * 8:, 0], 48000, 1000.0)
    assert abs(snr - LOOPBACK_SNR_DB[mode]) <= 0.1, (snr, LOOPBACK_SNR_DB[mode])


@pytest.mark.timeout(600, method="thread")
def test_scale_1024_channels_2_seconds(port, best_oracle):
    """1024 mic channels x 2 s, AM / FM / USB interleaved, against the oracle on sampled channels."""
    C, T = 1024, 96000
    base = slb.synth_mic(16, T)
    rng = np.random.Generator(np.random.PCG64(9))
    x = np.ascontiguousarray(base[rng.integers(0, 16, C)])
    modes = [slb.MODE_AM, slb.MODE_FM, slb.MODE_USB]
    d = make(C, modes)
    xd = torch.from_numpy(x).cuda(); ph = torch.zeros((C, T), dtype=torch.int32, device="cuda")
    d.set_phase_tap(ph); y = d.tx_process(xd).cpu().numpy(); ph = ph.cpu().numpy().view(np.uint32); d.set_phase_tap(None)
    for c in sorted(set(rng.integers(0, C, 6).tolist()) | {0, 1, C - 1}):
        mode = modes[c % 3]; prm = d.oracle_params(mode)
        if mode == slb.MODE_AM:
            check_int16(y[c], otm.tx_mod_f32(port, prm, x[c])[0])
        elif mode == slb.MODE_USB:
            check_int16(y[c], best_oracle.tx_ssb_f32(prm, x[c])[0])
        elif mode == slb.MODE_FM:
            assert np.array_equal(otm.tx_fm_nco(port, ph[c], prm["fm_level"]), y[c])
            ph_o = otm.tx_mod_f32(port, prm, x[c])[3]
            # the phase follows the oracle's up to the accumulated rounding of the increments
            dphi = (ph[c] - ph_o).view(np.int32).astype(np.float64) / 2.0 ** 32
            assert np.max(np.abs(dphi)) < 1e-2, float(np.max(np.abs(dphi)))


@pytest.mark.timeout(900, method="thread")
def test_parity_on_the_stress_build():
    """This file's parity tests on the stress build (random delays at every hand-over), like tests/test_gpu_stress_build.py does for the others."""
    if not os.path.exists(_build.STRESS_LIB_PATH):
        pytest.skip("stress build not present (python __graft_entry__.py builds it)")
    env = dict(os.environ, SELENITE_B200_LIB=_build.STRESS_LIB_PATH)
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "600",
                        os.path.abspath(__file__), "-k", "not stress_build"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=850)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
