"""GPU parity of the five integer chains away from their default parameters: every AGC window on every kernel path, release tables,
target / floor / gain-limit corners, the TX-Q15 and RX-Q15 mode constants, parameter changes between calls that hand the carried state
from one kernel to another, and CHAN-64-q15 with caller prototypes whose branch FIRs saturate. The gain law is implemented four times
(sl_rx_q15_tc.cu, the mma.sync kernel and q15_agc_kernel of sl_rx_ssb_q15.cu, sl_chan64_q15.cu); each is held BIT-EXACT to the port
with its state carried: output, pre-AGC tap, gain words and the carried peak window (tests/test_q15_agc_law.py pins the port's law to a
NumPy restatement)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_chan_q15 as ocq
import oracle_rx_q15 as orq
import oracle_tx_q15 as otx
import oracle_tx_q15_mod as otq
import selenite_lite_b200 as slb
from oracle_lib import RxQ15State
from selenite_lite_b200 import build as _build
from test_chan64_q15_oracle import np_branches
from test_gpu_chan64_q15 import rails
from test_gpu_rx_ssb_q15 import _q15_audio_biquad
from test_q15_agc_law import block_peaks, gain_law, rel_tables

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_ARG = -1
SSB_MODES = [slb.MODE_USB, slb.MODE_LSB, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG]
ALL_MODES = [slb.MODE_USB, slb.MODE_AM, slb.MODE_LSB, slb.MODE_FM, slb.MODE_CW, slb.MODE_CWR, slb.MODE_DIG, slb.MODE_PKT]
MID = 48 * 9                                                                 # a first call that ends in the middle of a supertile


# ---------------------------------------------------------------------------------------------------------------- the four q15 chains
class Chain:
    """One of the q15 chains of the C ABI with its oracle: run (port, prm, x, state) -> (out, pre-AGC tap, gain words)"""

    def __init__(self, chain, modes, run, state, tx, phase):
        self.chain, self.modes, self.run, self.state, self.tx, self.phase = chain, modes, run, state, tx, phase


CHAINS = {
    "rx_ssb": Chain(slb.CHAIN_RX_SSB_Q15, SSB_MODES, lambda o, p, x, s: o.rx_ssb_q15(p, x, s)[:3], RxQ15State, False, False),
    "tx_ssb": Chain(slb.CHAIN_TX_SSB_Q15, SSB_MODES, lambda o, p, x, s: otx.tx_ssb_q15(o, p, x, s)[:3], RxQ15State, True, False),
    "rx_q15": Chain(slb.CHAIN_RX_Q15, ALL_MODES, lambda o, p, x, s: orq.rx_q15(o, p, x, s)[:3], orq.RxQ15mState, False, False),
    "tx_q15": Chain(slb.CHAIN_TX_Q15, ALL_MODES, lambda o, p, x, s: otq.tx_q15(o, p, x, s)[:3], otq.TxQ15mState, True, True),
}


def make(kind, C):
    ch = CHAINS[kind]
    d = slb.DspIf(C, chain=ch.chain)
    for c in range(C):
        d.DSP_Set_Mode(ch.modes[c % len(ch.modes)], channel=c)
    return d


def set_law(d, rel=None, **kw):
    p = d.rx_q15_params()
    for k, v in kw.items():
        setattr(p, k, v)
    if rel is not None:
        for j in range(32):
            p.rel[j] = int(rel[j])
    d.set_rx_q15_params(p)
    return p


def run_gpu(d, x, tx):
    """one call on the device path: out, the pre-AGC tap (RX [C][T], TX [C][T][2]) and the gain words"""
    C, T = x.shape[0], x.shape[1]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    tap = torch.zeros((C, T, 2) if tx else (C, T), dtype=torch.int16, device="cuda")
    gain = torch.zeros((C, T // 48), dtype=torch.int32, device="cuda")
    d.set_q15_debug_taps(tap, gain)
    y = d.tx_process(xd) if tx else d.rx_process(xd)
    torch.cuda.synchronize()
    d.set_q15_debug_taps(None, None)
    return y.cpu().numpy(), tap.cpu().numpy(), gain.cpu().numpy().view(np.uint32)


def run_cuts(d, x, cuts, tx):
    parts = [run_gpu(d, x[:, a:b], tx) for a, b in zip(cuts[:-1], cuts[1:])]
    return tuple(np.concatenate([p[k] for p in parts], 1) for k in range(3))


def q15_peaks(d, phase=False):
    """the carried peak window of a q15 checkpoint, int16 [C][32] (age a at a - 1): the chain section sits before the 2 x 4 words of ring
    pointers per channel and holds the raw tail [C][64] u32, the peaks, the sidebands [C], the biquad state [C][16] int16 (and TX-Q15's
    phase words [C] u32)"""
    blob = np.frombuffer(bytes(d.state_save()), np.uint8); C = d.channels
    start = blob.size - 2 * C * 16 - C * (64 * 4 + 32 * 2 + 1 + 16 * 2 + (4 if phase else 0))
    return blob[start + 256 * C:start + 320 * C].copy().view(np.int16).reshape(C, 32)


def check(port, kind, d, x, got, cuts, states=None):
    """got = (out, tap, gain) of the GPU over x cut at `cuts`; the oracle runs the same cuts on one carried state per channel (states: a
    list to carry on with). Output, tap, gain words and the carried peak window (ages 1..31) must be equal."""
    ch = CHAINS[kind]
    C = x.shape[0]
    states = [ch.state() for _ in range(C)] if states is None else states
    for c in range(C):
        prm = d.oracle_params(ch.modes[c % len(ch.modes)])
        res = [ch.run(port, prm, x[c, a:b], states[c]) for a, b in zip(cuts[:-1], cuts[1:])]
        exp = [np.concatenate([r[k] for r in res]) for k in range(3)]
        assert np.array_equal(got[1][c], exp[1]), (kind, c, "tap")
        assert np.array_equal(got[2][c], exp[2]), (kind, c, "gain", int(np.argmax(got[2][c] != exp[2])))
        assert np.array_equal(got[0][c], exp[0]), (kind, c, "out")
    pk = q15_peaks(d, ch.phase)
    for c in range(C):
        assert np.array_equal(pk[c, :31], np.ctypeslib.as_array(states[c].peaks)[:31]), (kind, c, "peaks")
    return states


def bursts(C, T, seed, tx=False):
    """Quiet noise (+-300) with a loud burst (one block of full-scale noise) every 17 + c blocks in channel c, so that an aged peak, up to
    the window's oldest, sets the envelope of the blocks after each burst; rail samples in a few channels. TX: the mic, L = R."""
    rng = np.random.Generator(np.random.PCG64(seed))
    x = rng.integers(-300, 301, (C, T, 2))
    for c in range(C):
        gap = 48 * (17 + c % 16)
        for b0 in range(48 * (c % 5), T - 48, gap):
            x[c, b0:b0 + 48] = rng.integers(-32768, 32768, (48, 2))
    x[1::4, ::97] = -32768
    x[2::4, ::89] = 32767
    if tx:
        x[..., 1] = x[..., 0]
    return x.astype(np.int16)


def window_rel(window):
    """a release table that lets every age of the window act: high, falling slowly, different per window"""
    rng = np.random.Generator(np.random.PCG64(100 + window))
    return np.concatenate([[32767], np.sort(rng.integers(20000, 32768, 31))[::-1]])


# ---------------------------------------------------------------------------------------------------------------- 1. RX-SSB-q15, every window
@pytest.mark.parametrize("window", range(1, 18))
def test_rx_ssb_windows_1_to_17_on_both_kernels(port, window, monkeypatch):
    """The tcgen05 kernel (the default) and the mma.sync kernel: each equals the oracle and the two equal each other, checkpoint included.
    200 blocks cut mid-supertile: the second call starts from carried peaks; the mma.sync kernel cuts the launch into segments."""
    C, T = 16, 48 * 200
    x = bursts(C, T, window)
    cuts = [0, MID, T]
    blobs = []
    for legacy in (False, True):
        if legacy:
            monkeypatch.setenv("SELENITE_B200_Q15_PATH", "legacy")
        d = make("rx_ssb", C)
        set_law(d, agc_window=window, rel=window_rel(window))
        check(port, "rx_ssb", d, x, run_cuts(d, x, cuts, False), cuts)
        blobs.append(bytes(d.state_save()))
        monkeypatch.delenv("SELENITE_B200_Q15_PATH", raising=False)
    assert blobs[0] == blobs[1]


@pytest.mark.timeout(300, method="thread")
@pytest.mark.parametrize("window", range(18, 33))
def test_rx_ssb_windows_18_to_32_over_many_segments(port, window):
    """Windows past the tcgen05 kernel's reach run on the mma.sync kernel: 8 channels x 2000 blocks make several time segments, each
    re-deriving the window's peaks before it; the same stream in three ragged calls equals one call, checkpoint included."""
    C, T = 8, 96000
    x = bursts(C, T, window)
    d = make("rx_ssb", C)
    set_law(d, agc_window=window, rel=window_rel(window))
    whole = run_gpu(d, x, False)
    check(port, "rx_ssb", d, x, whole, [0, T])
    e = make("rx_ssb", C)
    set_law(e, agc_window=window, rel=window_rel(window))
    cut = run_cuts(e, x, [0, 48 * 701, 48 * 1403, T], False)
    for k in range(3):
        assert np.array_equal(cut[k], whole[k]), k
    assert bytes(e.state_save()) == bytes(d.state_save())


@pytest.mark.parametrize("legacy", [False, True])
@pytest.mark.parametrize("window", [1, 9, 17, 18, 32])
def test_biquad_path_at_every_window(port, window, legacy, monkeypatch):
    """The optional biquad makes the chain three launches per call (FIR kernel, biquad, q15_agc_kernel), behind either FIR kernel."""
    if legacy:
        monkeypatch.setenv("SELENITE_B200_Q15_PATH", "legacy")
    C, T = 11, 48 * 90
    x = bursts(C, T, 50 + window)
    coeffs, ps = _q15_audio_biquad()
    d = make("rx_ssb", C)
    p = d.rx_q15_params()
    for k in range(12):
        p.bq_coeffs[k] = int(coeffs[k])
    p.bq_stages, p.bq_postshift = 2, ps
    d.set_rx_q15_params(p)
    set_law(d, agc_window=window, rel=window_rel(window))
    cuts = [0, MID, 48 * 40, T]
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        n0 = d.kernel_launches()
        parts.append(run_gpu(d, x[:, a:b], False))
        assert d.kernel_launches() - n0 == 3
    got = tuple(np.concatenate([q[k] for q in parts], 1) for k in range(3))
    check(port, "rx_ssb", d, x, got, cuts)


# ---------------------------------------------------------------------------------------------------------------- 2. the tcgen05-only chains
@pytest.mark.parametrize("window", range(1, 18))
@pytest.mark.parametrize("kind", ["tx_ssb", "rx_q15", "tx_q15"])
def test_tcgen05_only_chains_every_window(port, kind, window):
    C, T = 16, 48 * 100
    x = bursts(C, T, window, tx=CHAINS[kind].tx)
    d = make(kind, C)
    set_law(d, agc_window=window, rel=window_rel(window))
    cuts = [0, MID, T]
    states = check(port, kind, d, x, run_cuts(d, x, cuts, CHAINS[kind].tx), cuts)
    if kind == "tx_q15":
        assert np.array_equal(phases(d), [s.phase for s in states])


def phases(d):
    blob = np.frombuffer(bytes(d.state_save()), np.uint8); C = d.channels
    end = blob.size - 2 * C * 16
    return blob[end - 4 * C:end].copy().view(np.uint32)


@pytest.mark.parametrize("kind", ["rx_ssb", "tx_ssb", "rx_q15", "tx_q15", "chan"])
def test_refusals_leave_the_parameters_unchanged(kind):
    """Window 0 on every chain (and 33 on RX-SSB-q15), a gain limit past 255 << 15, a floor or target of 0 or below: SLB_ERR_ARG, and the
    parameters read back unchanged. 255 << 15 itself is accepted."""
    chan = kind == "chan"
    d = slb.DspIf(1, fs=192000, chain=slb.CHAIN_CHAN64_Q15) if chan else make(kind, 1)
    get, put = (d.chan_q15_params, d.set_chan_q15_params) if chan else (d.rx_q15_params, d.set_rx_q15_params)
    bad = [("agc_window", 0), ("agc_gmax_q15", (255 << 15) + 1), ("agc_floor", 0), ("agc_floor", -1), ("agc_target", 0), ("agc_target", -5)]
    if kind == "rx_ssb":
        bad.append(("agc_window", 33))
    for field, value in bad:
        before = bytes(memoryview(get()))
        p = get(); setattr(p, field, value)
        with pytest.raises(slb.SeleniteError, match="-> %d" % ERR_ARG):
            put(p)
        assert bytes(memoryview(get())) == before, (field, value)
    p = get(); p.agc_gmax_q15 = 255 << 15
    put(p)
    assert get().agc_gmax_q15 == 255 << 15


# ---------------------------------------------------------------------------------------------------------------- 3. AGC constants on every chain
CORNERS = [dict(rel="flat", agc_window=17, agc_target=8192, agc_floor=1, agc_gmax_q15=255 << 15),
           dict(rel="zero", agc_window=9, agc_target=32767, agc_floor=32767, agc_gmax_q15=64 << 15),
           dict(rel="random", agc_window=17, agc_target=16, agc_floor=16, agc_gmax_q15=32768),
           dict(rel="zigzag", agc_window=13, agc_target=32767, agc_floor=8192, agc_gmax_q15=1),
           dict(rel="flat", agc_window=5, agc_target=1, agc_floor=1, agc_gmax_q15=255 << 15),
           dict(rel="random", agc_window=16, agc_target=32767, agc_floor=16, agc_gmax_q15=64 << 15)]


def corner_inputs(C, T, seed, tx):
    """channel c: silence, +-40, rail to rail, or loud bursts followed by quiet stretches (c % 4)"""
    rng = np.random.Generator(np.random.PCG64(seed))
    x = bursts(C, T, seed, tx=False).astype(np.int64)
    x[0::4] = 0
    x[1::4] = rng.integers(-40, 41, x[1::4].shape)
    x[2::4] = rng.integers(-32768, 32768, x[2::4].shape); x[2::4, ::3] = -32768; x[2::4, 1::3] = 32767
    if tx:
        x[..., 1] = x[..., 0]
    return x.astype(np.int16)


def fired(prm, target, tap, gain, tx):
    """which corners acted in one channel's oracle result: the law restated (test_q15_agc_law) from the tap must give the oracle's words"""
    pk = np.maximum(block_peaks(tap[:, 0], 48), block_peaks(tap[:, 1], 48)) if tx else block_peaks(tap, 48)
    q, env, aged = gain_law(pk, prm, target)
    assert np.array_equal(q, gain)
    out = set()
    if np.any(q == prm["agc_gmax_q15"]):
        out.add("gmax")
    if np.any(env < prm["agc_floor"]):
        out.add("floor")
    if np.any(aged):
        out.add("aged-" + next(k for k, v in rel_tables().items() if np.array_equal(v.astype(np.int16), prm["rel"])))
    return out


@pytest.mark.parametrize("kind", ["rx_ssb", "rx_ssb_legacy", "tx_ssb", "rx_q15", "tx_q15"])
def test_agc_corners_on_every_chain(port, kind, monkeypatch):
    if kind == "rx_ssb_legacy":
        monkeypatch.setenv("SELENITE_B200_Q15_PATH", "legacy"); kind = "rx_ssb"
    ch = CHAINS[kind]
    C, T = 16, 48 * 60
    tabs = rel_tables()
    seen = set()
    for i, corner in enumerate(CORNERS):
        x = corner_inputs(C, T, i, ch.tx)
        d = make(kind, C)
        law = dict(corner); rel = tabs[law.pop("rel")]
        set_law(d, rel=rel, **law)
        got = run_gpu(d, x, ch.tx)
        check(port, kind, d, x, got, [0, T])
        for c in range(C):
            mode = ch.modes[c % len(ch.modes)]
            prm = d.oracle_params(mode)
            target = {slb.MODE_AM: "am_depth", slb.MODE_FM: "fm_target"}.get(mode, "agc_target") if kind == "tx_q15" else "agc_target"
            seen |= fired(prm, prm[target], got[1][c], got[2][c], ch.tx)
    assert seen == {"gmax", "floor", "aged-flat", "aged-random", "aged-zigzag"}, seen


# ---------------------------------------------------------------------------------------------------------------- 4. mode constants
TX_MODE_SETS = [dict(am_carrier=0, fm_inc=-65535, fm_level=1.0), dict(am_carrier=32767, fm_inc=-1, fm_level=0.0),
                dict(am_depth=1, fm_target=1, fm_inc=0), dict(fm_inc=1, fm_level=1.0), dict(am_carrier=32767, am_depth=1, fm_inc=65535)]


@pytest.mark.parametrize("i", range(len(TX_MODE_SETS)))
def test_tx_q15_mode_constants(port, i):
    C, T = 16, 48 * 100
    x = bursts(C, T, 70 + i, tx=True)
    d = make("tx_q15", C)
    mp = d.tx_q15_mode_params()
    for k, v in TX_MODE_SETS[i].items():
        setattr(mp, k, v)
    d.set_tx_q15_mode_params(mp)
    cuts = [0, MID, T]
    states = check(port, "tx_q15", d, x, run_cuts(d, x, cuts, True), cuts)
    assert np.array_equal(phases(d), [s.phase for s in states])


@pytest.mark.parametrize("fm_floor", [1, 1 << 18, (1 << 31) - 1])
def test_rx_q15_fm_floor(port, fm_floor):
    C, T = 16, 48 * 100
    x = slb.synth_fm(C, T)
    x[:, ::61] = -32768
    d = make("rx_q15", C)
    mp = d.rx_q15_mode_params(); mp.fm_floor = fm_floor; d.set_rx_q15_mode_params(mp)
    cuts = [0, MID, T]
    check(port, "rx_q15", d, x, run_cuts(d, x, cuts, False), cuts)


# ---------------------------------------------------------------------------------------------------------------- 5. changes between calls
def test_rx_ssb_parameter_schedule_across_kernels_and_checkpoint(port):
    """window 16 (tcgen05) -> 24 (mma.sync) -> 17 (tcgen05) -> 9 with a biquad -> 32 without -> 1 with a new release table. The library
    zeroes the biquad state when the stages or coefficients change; the oracle does the same. A checkpoint after the fourth call, loaded
    into a fresh context with the same parameters, gives the rest of the stream bit for bit."""
    C, seg = 16, 48 * 60
    x = bursts(C, 6 * seg, 99)
    coeffs, ps = _q15_audio_biquad()
    tabs = rel_tables()
    sched = [dict(agc_window=16), dict(agc_window=24), dict(agc_window=17), dict(agc_window=9, bq_stages=2, bq_postshift=ps),
             dict(agc_window=32, bq_stages=0), dict(agc_window=1, rel=tabs["zigzag"])]

    def apply(d, k):
        law = dict(sched[k]); rel = law.pop("rel", window_rel(7))
        p = d.rx_q15_params()
        if law.get("bq_stages"):
            for j in range(12):
                p.bq_coeffs[j] = int(coeffs[j])
        for f, v in law.items():
            setattr(p, f, v)
        for j in range(32):
            p.rel[j] = int(rel[j])
        d.set_rx_q15_params(p)

    d = make("rx_ssb", C)
    states = [RxQ15State() for _ in range(C)]
    outs = []
    for k in range(6):
        apply(d, k)
        if k in (3, 4):                                                       # the filter changed: both sides start it from rest
            for s in states:
                for j in range(16):
                    s.bq[j] = 0
        xs = np.ascontiguousarray(x[:, k * seg:(k + 1) * seg])
        got = run_gpu(d, xs, False)
        check(port, "rx_ssb", d, xs, got, [0, seg], states)
        outs.append(got)
        if k == 3:
            snap = d.state_save()
    e = make("rx_ssb", C)
    apply(e, 3)
    e.state_load(snap)
    for k in (4, 5):
        apply(e, k)
        again = run_gpu(e, np.ascontiguousarray(x[:, k * seg:(k + 1) * seg]), False)
        for j in range(3):
            assert np.array_equal(again[j], outs[k][j]), (k, j)
    assert np.array_equal(q15_peaks(e), q15_peaks(d))


def test_tx_q15_window_and_release_changes(port):
    C, seg = 16, 48 * 40
    x = bursts(C, 3 * seg, 98, tx=True)
    tabs = rel_tables()
    d = make("tx_q15", C)
    states = [otq.TxQ15mState() for _ in range(C)]
    for k, (window, rel) in enumerate(((16, tabs["flat"]), (5, tabs["random"]), (17, tabs["zigzag"]))):
        set_law(d, agc_window=window, rel=rel)
        xs = np.ascontiguousarray(x[:, k * seg:(k + 1) * seg])
        check(port, "tx_q15", d, xs, run_gpu(d, xs, True), [0, seg], states)
    assert np.array_equal(phases(d), [s.phase for s in states])


# ---------------------------------------------------------------------------------------------------------------- 6. CHAN-64-q15
FS = 192000
T_CHAN = 3072 * 3 + 768                                                       # three tiles and a ragged fourth


def chan_run(d, x):
    S, T = x.shape[0], x.shape[1]
    audio = torch.zeros((S, 64, T // 64), dtype=torch.int16, device="cuda")
    gain = torch.zeros((S, 64, T // 192), dtype=torch.int32, device="cuda")
    d.set_q15_debug_taps(audio, gain)
    y = d.chan_process(torch.from_numpy(np.ascontiguousarray(x)).cuda())
    torch.cuda.synchronize()
    d.set_q15_debug_taps(None, None)
    return y.cpu().numpy(), audio.cpu().numpy(), gain.cpu().numpy().view(np.uint32)


def chan_check(port, d, x, got, states):
    exp = ocq.chan_batch(port, d.oracle_params(), x, states)
    for k in range(3):
        for s in range(x.shape[0]):
            assert np.array_equal(got[k][s], exp[k][s]), (k, s)


def chan_ctx(S, proto=None, rel=None, **kw):
    d = slb.DspIf(S, fs=FS, chain=slb.CHAIN_CHAN64_Q15)
    chan_set(d, proto, rel, **kw)
    return d


def chan_set(d, proto=None, rel=None, **kw):
    p = d.chan_q15_params()
    for k, v in kw.items():
        setattr(p, k, v)
    if proto is not None:
        for j in range(512):
            p.proto[j] = int(proto[j])
    if rel is not None:
        for j in range(32):
            p.rel[j] = int(rel[j])
    d.set_chan_q15_params(p)


def chan_inputs():
    x = np.concatenate([rails(T_CHAN), slb.synth_wideband(2, T_CHAN)])
    x[5] = np.clip(x[5].astype(np.int32) * 300, -32768, 32767)                 # wideband at full scale
    return x.astype(np.int16)


def prototypes():
    default = np.array(slb.default_chan_q15_params().proto[:], np.int64)
    e = np.arange(512)
    signs = np.where(((e * 7) // 5) % 3 == 0, -32768, 32767)                    # both signs in every branch
    rng = np.random.Generator(np.random.PCG64(64))
    return {"default_x8": np.clip(8 * default, -32768, 32767), "signs": signs, "random": rng.integers(-32768, 32768, 512)}


@pytest.mark.parametrize("envelope", [0, 1])
@pytest.mark.parametrize("name", ["default_x8", "signs", "random"])
def test_chan_caller_prototypes(port, name, envelope):
    proto = prototypes()[name]
    x = chan_inputs()
    if name != "random":                                                      # the branch FIR's sat16 acts, on both rails' sides
        lo = hi = False
        for s in range(x.shape[0]):
            ai, aq = np_branches(proto, x[s])
            v = np.concatenate([ai.ravel(), aq.ravel()]) >> 15
            lo |= bool(np.any(v < -32768)); hi |= bool(np.any(v > 32767))
        assert lo and hi
    d = chan_ctx(x.shape[0], proto, envelope=envelope)
    chan_check(port, d, x, chan_run(d, x), None)


@pytest.mark.parametrize("window", range(1, 18))
def test_chan_every_window_random_release_and_corners(port, window):
    corner = CORNERS[window % len(CORNERS)]
    rng = np.random.Generator(np.random.PCG64(200 + window))
    rel = rng.integers(-32768, 32768, 32); rel[1:window] = np.abs(rel[1:window]) // 2 + 16384      # random, the window's ages high
    x = chan_inputs()
    x[0] = 0
    x[1] = rng.integers(-40, 41, x[1].shape)
    d = chan_ctx(x.shape[0], prototypes()["random"] if window % 2 else None, rel, envelope=window % 2, agc_window=window,
                 agc_target=corner["agc_target"], agc_floor=corner["agc_floor"], agc_gmax_q15=corner["agc_gmax_q15"])
    chan_check(port, d, x, chan_run(d, x), None)


def test_chan_window_release_and_prototype_changes(port):
    """window 17 -> 4 with a new release table -> 17 with a new prototype; the raw history and the peaks carry across"""
    x = chan_inputs()
    S = x.shape[0]
    tabs = rel_tables(); protos = prototypes()
    d = chan_ctx(S, agc_window=17)
    states = [ocq.ChanQ15State() for _ in range(S)]
    cuts = [0, 3072 + 768, 3072 * 2 + 768, T_CHAN]
    for k, (window, rel, proto) in enumerate(((17, None, None), (4, tabs["random"], None), (17, tabs["flat"], protos["default_x8"]))):
        chan_set(d, proto, rel, agc_window=window)
        xs = np.ascontiguousarray(x[:, cuts[k]:cuts[k + 1]])
        chan_check(port, d, xs, chan_run(d, xs), states)


# ---------------------------------------------------------------------------------------------------------------- 7. the stress build
@pytest.mark.timeout(1500, method="thread")
def test_parity_on_the_stress_build():
    """This file's parity tests on the stress build (random delays at every hand-over of the tensor-core kernels)"""
    if not os.path.exists(_build.STRESS_LIB_PATH):
        pytest.skip("stress build not present (python __graft_entry__.py builds it)")
    env = dict(os.environ, SELENITE_B200_LIB=_build.STRESS_LIB_PATH)
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "900",
                        os.path.abspath(__file__), "-k", "not stress_build"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1400)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
