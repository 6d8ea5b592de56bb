#!/usr/bin/env python
"""Device-resident throughput of the chains that are not the headline bench line (TX-SSB-f32 = config 3,
CHAN-64-f32 = config 4, RX at other widths, TX AM / FM). Prints one JSON line per chain after a line naming the card, its power
limit and the HBM copy rate measured in the same run (hbm_frac_measured divides by that). Profiling aid, not the bench contract."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import selenite_lite_b200 as slb  # noqa: E402


def timeit(fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn(); ev[i + 1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[-1]) / steps


def measured_copy_gbps(dev, steps=20):
    """HBM roof of this card measured now: a 2 GiB device-to-device copy (bytes read + bytes written per second)."""
    a = torch.empty(1 << 31, dtype=torch.uint8, device=dev); b = torch.empty_like(a)
    ms = timeit(lambda: b.copy_(a), steps)
    del a, b
    return 2 * (1 << 31) / (ms * 1e-3) / 1e9


def card(dev):
    try:
        pl = subprocess.run(["nvidia-smi", "-i", str(dev.index), "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except Exception as exc:  # the number stays unlabelled rather than wrong
        pl = "unknown (%s)" % exc
    return torch.cuda.get_device_name(dev), pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--which", default="tx,chan,rx,q15")
    ap.add_argument("--seconds", type=int, default=10)
    ap.add_argument("--rx-channels", type=int, default=1024)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    peak = 6650.0
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    g = torch.Generator(device=dev); g.manual_seed(1)
    name_, power = card(dev); roof = measured_copy_gbps(dev)
    print(json.dumps({"device": name_, "power_limit": power, "measured_copy_GBps": roof}))
    for which in args.which.split(","):
        if which == "tx":
            C, T = args.rx_channels, 48000 * args.seconds
            m = torch.randint(-8000, 8000, (C, T, 1), dtype=torch.int16, device=dev, generator=g).expand(C, T, 2).contiguous()
            d = slb.DspIf(C, chain=slb.CHAIN_TX_SSB_F32); y = torch.empty_like(m)
            ms = timeit(lambda: d.tx_process(m, y), args.steps); n = C * T; name = "tx_ssb_f32 (config 3: %d mic channels x %d s)" % (C, args.seconds)
        elif which in ("tx_fft", "tx_am", "tx_fm"):
            # TX on the FFT kernel: SSB forced there (the rate AM / FM are measured against), AM and FM (the only kernel that serves them)
            C, T = args.rx_channels, 48000 * args.seconds
            m = torch.randint(-8000, 8000, (C, T, 1), dtype=torch.int16, device=dev, generator=g).expand(C, T, 2).contiguous()
            d = slb.DspIf(C, chain=slb.CHAIN_TX_F32); y = torch.empty_like(m)
            if which == "tx_fft":
                d.set_rx_path(slb.RX_PATH_FFT)
            else:
                d.DSP_Set_Mode(slb.MODE_AM if which == "tx_am" else slb.MODE_FM)
            ms = timeit(lambda: d.tx_process(m, y), args.steps); n = C * T
            name = "%s (tx_f32, FFT kernel: %d mic channels x %d s)" % ({"tx_fft": "ssb", "tx_am": "am", "tx_fm": "fm"}[which], C, args.seconds)
        elif which == "chan":
            S, T = 64, 192000 * args.seconds // 768 * 768
            x = torch.randint(-3000, 3000, (S, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(S, fs=192000, chain=slb.CHAIN_CHAN64_F32); y = torch.empty((S, 64, T // 64, 2), dtype=torch.int16, device=dev)
            ms = timeit(lambda: d.chan_process(x, y), args.steps); n = S * T; name = "chan64_f32 (config 4: 64 x 192 kHz streams -> 4096 channels, %d s)" % args.seconds
        elif which == "q15":
            C, T = args.rx_channels, 48000 * args.seconds
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_RX_SSB_Q15); y = torch.empty_like(x)
            ms = timeit(lambda: d.rx_process(x, y), args.steps); n = C * T; name = "rx_ssb_q15 (%d channels x %d s)" % (C, args.seconds)
        elif which == "pass":
            C, T = args.rx_channels, 48000 * args.seconds // 384 * 384
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_PASS); y = torch.empty_like(x)
            ms = timeit(lambda: d.rx_process(x, y), args.steps); n = C * T; name = "pass (the firmware as shipped: bit-exact copy, %d channels x %d s)" % (C, args.seconds)
        elif which == "am":
            C, T = args.rx_channels, 48000 * args.seconds // 384 * 384
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_RX_SSB_F32); d.DSP_Set_Mode(slb.MODE_AM); y = torch.empty_like(x)
            ms = timeit(lambda: d.rx_process(x, y), args.steps); n = C * T
            name = "rx am (%s, %d channels x %d s)" % ("complex-detector tensor-core kernel" if os.environ.get("SELENITE_B200_AM_PATH") == "tc" else "FFT kernel", C, args.seconds)
        elif which == "fm":
            C, T = args.rx_channels, 48000 * args.seconds // 384 * 384
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_RX_SSB_F32); d.DSP_Set_Mode(slb.MODE_FM); y = torch.empty_like(x)
            ms = timeit(lambda: d.rx_process(x, y), args.steps); n = C * T; name = "rx fm (complex-detector tensor-core kernel, %d channels x %d s)" % (C, args.seconds)
        else:
            C, T = args.rx_channels, 48000 * args.seconds // 384 * 384
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_RX_SSB_F32); y = torch.empty_like(x)
            ms = timeit(lambda: d.rx_process(x, y), args.steps); n = C * T; name = "rx_ssb_f32 (%d channels x %d s)" % (C, args.seconds)
        gs = n / (ms * 1e-3) / 1e9
        print(json.dumps({"chain": name, "ms_per_step": ms, "Gsamples_per_s": gs, "algorithmic_GBps": gs * 8, "hbm_frac": gs * 8 / peak,
                          "hbm_frac_measured": gs * 8 / roof}))
        del d


if __name__ == "__main__":
    main()
