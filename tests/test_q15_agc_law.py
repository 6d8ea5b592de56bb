"""The gain law shared by the five integer chains (DESIGN.md §3.3 step 5; oracle/slo_api.h), restated in NumPy int64 and held against the
port away from the default constants: every window, release tables that are flat, zero, negative and non-monotone, the target, floor and
gain-limit corners, and inputs that are silent, quiet, noisy and rail to rail. Each chain's pre-AGC tap goes in; the gain words and the
output (the phase steps for FM) must come out bit for bit, over two calls with the peak window carried in the port's state.

  env_b = max (p_b, max_{j=1..W-1} (p_{b-j} rel[j]) >> 15),  q = min ((target << 15) // max (env_b, floor), gmax),
  s = the least shift with q >> s <= 32767,  y = arm_scale_q15 (a, q >> s, s) = sat16 ((a (q >> s)) >> (15 - s))"""
import numpy as np
import pytest

import oracle_chan_q15 as ocq
import oracle_rx_q15 as orq
import oracle_tx_q15 as otx
import oracle_tx_q15_mod as otq
import selenite_lite_b200 as slb
from oracle_lib import RxQ15State
from selenite_lite_b200.dsp_if import chan_q15_params_to_dict, q15_mode_params_to_dict, q15_params_to_dict, tx_q15_mode_params_to_dict

WIN, BLK, CHAN_BLK = 32, 48, 3
TARGETS = FLOORS = (1, 16, 8192, 32767)
GMAXES = (1, 32768, 64 << 15, 255 << 15)


# ------------------------------------------------------------------------------------------------------------------ the law in NumPy
def block_peaks(a, blk):
    """arm_abs_q15 (saturating: |-32768| = 32767), then arm_max_q15 over each block of blk samples along the last axis"""
    a = np.abs(np.asarray(a, np.int64)).clip(max=32767)
    return a.reshape(a.shape[:-1] + (-1, blk)).max(-1)


def gain_law(peaks, prm, target, carried=None):
    """peaks int64 [..., blocks]; carried int16 [..., 32]: the peak window by age before the first block (the port's state: age j + 1 at
    index j). Returns the gain words q, the envelope, and where the envelope came from an aged peak rather than the block's own."""
    peaks = np.asarray(peaks, np.int64)
    nb = peaks.shape[-1]
    old = np.zeros(peaks.shape[:-1] + (WIN,), np.int64) if carried is None else np.asarray(carried, np.int64)[..., ::-1]
    hist = np.concatenate([old, peaks], -1)                                   # hist[..., WIN + b - j] = the peak j blocks before b
    rel = np.asarray(prm["rel"], np.int64)
    aged = np.full(peaks.shape, np.iinfo(np.int64).min)
    for j in range(1, int(prm["agc_window"])):
        aged = np.maximum(aged, (hist[..., WIN - j:WIN - j + nb] * rel[j]) >> 15)
    env = np.maximum(peaks, aged)
    q = np.minimum((int(target) << 15) // np.maximum(env, int(prm["agc_floor"])), int(prm["agc_gmax_q15"]))
    return q, env, aged > peaks


def scale(a, q, blk, saturate=True):
    """arm_scale_q15 (a, q >> s, s) per block of blk samples along the last axis; q int64 [..., blocks] (saturate=False: before the __SSAT)"""
    s = np.zeros_like(q)
    while np.any((q >> s) > 32767):
        s += (q >> s) > 32767
    frac, sh = np.repeat(q >> s, blk, -1), np.repeat(s, blk, -1)
    y = (np.asarray(a, np.int64) * frac) >> (15 - sh)
    return np.clip(y, -32768, 32767).astype(np.int16) if saturate else y


def sat16(v):
    return np.clip(v, -32768, 32767)


# ------------------------------------------------------------------------------------------------------------------ draws and inputs
def rel_tables(seed=7):
    rng = np.random.Generator(np.random.PCG64(seed))
    rnd = rng.integers(-32768, 32768, WIN); rnd[2] = -32768; rnd[5] = -1                 # negatives and the most negative entry
    zig = np.array([32767 if j % 3 == 0 else 4000 * (j % 5) for j in range(WIN)])        # non-monotone: rises again after it falls
    return {"flat": np.full(WIN, 32767), "zero": np.zeros(WIN), "random": rnd, "zigzag": zig}


def draws(max_window):
    """Every window 1..max_window with each release table; the target, floor and gmax corners spread over them so that each value of
    each corner meets every table."""
    out = []
    for t, (name, rel) in enumerate(rel_tables().items()):
        for w in range(1, max_window + 1):
            k = w + 5 * t
            out.append(dict(agc_window=w, rel=rel.astype(np.int16), agc_target=TARGETS[k % 4], agc_floor=FLOORS[(k // 4) % 4],
                            agc_gmax_q15=GMAXES[(k // 2 + t) % 4]))
    return out


def inputs(frames, seed=3):
    """silent, quiet (+-40), noisy (a loud tone, then quiet noise with a burst: the release table decides the gains after it), rail to rail"""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = np.arange(frames)
    w = 2 * np.pi * 700 * n / 48000
    loud = np.stack([np.rint(20000 * np.sin(w)), np.rint(20000 * np.cos(w))], 1)
    noisy = np.where((n < frames // 3)[:, None], loud, rng.integers(-300, 300, (frames, 2)))
    noisy[frames // 2:frames // 2 + 40] = 12000
    rails = rng.integers(-32768, 32768, (frames, 2)); rails[::7] = -32768; rails[3::7] = 32767
    xs = {"silent": np.zeros((frames, 2)), "quiet": rng.integers(-40, 41, (frames, 2)), "noisy": noisy, "rails": rails}
    return {k: v.astype(np.int16) for k, v in xs.items()}


def law(base, d, **extra):
    prm = dict(base); prm.update(d); prm.update(extra)
    return prm


FRAMES, CUT = 48 * 40, 48 * 17                                                 # two calls: 17 blocks, then 23


def over_two_calls(run, prm, x, state):
    """run (prm, x, state) -> (pre-AGC tap, gain words, rest...) over x in two calls on one state; yields each call's results with the
    peak window it started from (None = a fresh state)"""
    first = run(prm, x[:CUT], state)
    carried = np.ctypeslib.as_array(state.peaks).copy()
    second = run(prm, x[CUT:], state)
    yield first, None
    yield second, carried


# ------------------------------------------------------------------------------------------------------------------ the chains
def test_rx_ssb_q15(port):
    base = q15_params_to_dict(slb.default_rx_q15_params())
    for d in draws(32):
        for lsb in (0, 1):
            prm = law(base, d, lsb=lsb)
            for name, x in inputs(FRAMES, seed=d["agc_window"]).items():
                for (y, a, g, _), carried in over_two_calls(port.rx_ssb_q15, prm, x, RxQ15State()):
                    q, _, _ = gain_law(block_peaks(a, BLK), prm, prm["agc_target"], carried)
                    assert np.array_equal(g, q), (d, name)
                    out = scale(a, q, BLK)
                    assert np.array_equal(y[:, 0], out) and np.array_equal(y[:, 1], out), (d, name)


def test_tx_ssb_q15(port):
    base = q15_params_to_dict(slb.default_rx_q15_params())
    run = lambda prm, x, st: otx.tx_ssb_q15(port, prm, x, st)  # noqa: E731
    for d in draws(17):
        prm = law(base, d, lsb=d["agc_window"] % 2)
        for name, x in inputs(FRAMES, seed=d["agc_window"]).items():
            for (y, iq, g, _), carried in over_two_calls(run, prm, x, RxQ15State()):
                q, _, _ = gain_law(np.maximum(block_peaks(iq[:, 0], BLK), block_peaks(iq[:, 1], BLK)), prm, prm["agc_target"], carried)
                assert np.array_equal(g, q), (d, name)
                assert np.array_equal(y[:, 0], scale(iq[:, 0], q, BLK)) and np.array_equal(y[:, 1], scale(iq[:, 1], q, BLK)), (d, name)


@pytest.mark.parametrize("mode", [slb.MODE_USB, slb.MODE_AM, slb.MODE_FM])
def test_rx_q15(port, mode):
    base = q15_mode_params_to_dict(slb.default_rx_q15_params(), slb.default_rx_q15_mode_params(), mode)
    run = lambda prm, x, st: orq.rx_q15(port, prm, x, st)  # noqa: E731
    for d in draws(17):
        prm = law(base, d)
        for name, x in inputs(FRAMES, seed=d["agc_window"]).items():
            for (y, v, g, _), carried in over_two_calls(run, prm, x, orq.RxQ15mState()):
                q, _, _ = gain_law(block_peaks(v, BLK), prm, prm["agc_target"], carried)
                assert np.array_equal(g, q), (d, name)
                out = scale(v, q, BLK)
                assert np.array_equal(y[:, 0], out) and np.array_equal(y[:, 1], out), (d, name)


@pytest.mark.parametrize("mode", [slb.MODE_USB, slb.MODE_AM, slb.MODE_FM])
def test_tx_q15(port, mode):
    """The modulator's target: agc_target (SSB), am_depth (AM), fm_target (FM). AM: I = arm_add_q15 (arm_scale_q15 (y, am_carrier, 0),
    am_carrier), Q = 0; FM: the phase advances by y fm_inc (mod 2^32) per sample."""
    base = tx_q15_mode_params_to_dict(slb.default_rx_q15_params(), slb.default_tx_q15_mode_params(), mode)
    key = {slb.MODE_AM: "am_depth", slb.MODE_FM: "fm_target"}.get(mode, "agc_target")
    for d in draws(17):
        prm = law(base, d)
        prm[key] = d["agc_target"]                                              # the corner drives the modulator's own target
        for name, x in inputs(FRAMES, seed=d["agc_window"]).items():
            st = otq.TxQ15mState()
            phase0 = 0
            for k, (a, b) in enumerate(((0, CUT), (CUT, FRAMES))):
                carried = None if k == 0 else np.ctypeslib.as_array(st.peaks).copy()
                y, iq, g, ph, _ = otq.tx_q15(port, prm, x[a:b], st)
                q, _, _ = gain_law(np.maximum(block_peaks(iq[:, 0], BLK), block_peaks(iq[:, 1], BLK)), prm, prm[key], carried)
                assert np.array_equal(g, q), (d, name)
                yi = scale(iq[:, 0], q, BLK)
                if mode == slb.MODE_AM:
                    car = int(prm["am_carrier"])
                    assert np.array_equal(y[:, 0], sat16(sat16((yi.astype(np.int64) * car) >> 15) + car)) and not y[:, 1].any(), (d, name)
                elif mode == slb.MODE_FM:
                    steps = np.diff(np.concatenate([[phase0], ph.astype(np.int64)])) % (1 << 32)
                    assert np.array_equal(steps, (yi.astype(np.int64) * int(prm["fm_inc"])) % (1 << 32)), (d, name)
                    phase0 = int(ph[-1])
                else:
                    assert np.array_equal(y[:, 0], yi) and np.array_equal(y[:, 1], scale(iq[:, 1], q, BLK)), (d, name)


def test_chan_q15(port):
    """Per bin over 64 bins, AGC blocks of 3 hops; both detectors"""
    base = chan_q15_params_to_dict(slb.default_chan_q15_params())
    for d in draws(17):
        for envelope in (0, 1):
            prm = law(base, d, envelope=envelope)
            for name, x in inputs(768 * 3, seed=d["agc_window"]).items():
                st = ocq.ChanQ15State()
                for k, (a, b) in enumerate(((0, 768), (768, 768 * 3))):
                    carried = None if k == 0 else np.ctypeslib.as_array(st.peaks).reshape(64, WIN).copy()
                    y, aud, g, _ = ocq.chan_q15(port, prm, x[a:b], st)
                    q, _, _ = gain_law(block_peaks(aud, CHAN_BLK), prm, prm["agc_target"], carried)
                    assert np.array_equal(g, q), (d, name, envelope)
                    out = scale(aud, q, CHAN_BLK)
                    assert np.array_equal(y[..., 0], out) and np.array_equal(y[..., 1], out), (d, name, envelope)


def test_the_corners_fire_and_the_scale_never_saturates():
    """The draws above reach what they are for: a gain word at gmax, one set by the floor, one set by an aged peak through each kind of
    table (a zero table never sets it), and the -32768 edge of the output. And the law keeps arm_scale_q15's __SSAT from ever acting:
    |a| <= env gives |a q| >> 15 <= target, so before the saturation every output already lies in int16."""
    xs = inputs(FRAMES)
    seen = set()
    for d in draws(32):
        prm = law({}, d)
        for name, x in xs.items():
            a = x[:, 0]
            q, env, aged = gain_law(block_peaks(a, BLK), prm, prm["agc_target"])
            if np.any(q == prm["agc_gmax_q15"]):
                seen.add("gmax")
            if np.any((env < prm["agc_floor"]) & (q == min((prm["agc_target"] << 15) // prm["agc_floor"], prm["agc_gmax_q15"]))):
                seen.add("floor")
            if np.any(aged):
                seen.add("aged-" + next(k for k, v in rel_tables().items() if np.array_equal(v.astype(np.int16), prm["rel"])))
            y = scale(a, q, BLK, saturate=False)
            assert y.min() >= -32768 and y.max() <= 32767, (d, name)
            if y.min() == -32768:
                seen.add("edge")
    assert seen == {"gmax", "floor", "aged-flat", "aged-random", "aged-zigzag", "edge"}, seen
