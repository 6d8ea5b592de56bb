#!/usr/bin/env python
"""Device-resident throughput of the chains that are not the headline bench line (TX-SSB-f32 = config 3,
CHAN-64-f32 = config 4, RX at other widths, TX AM / FM, TX-SSB-q15, RX-Q15 AM / FM, TX-Q15 AM / FM, tuned channels, CHAN-64-q15).
Prints one JSON line per chain after a line naming the card, its power limit and the HBM copy rate measured in the same run
(hbm_frac_measured divides by that). Profiling aid, not the bench contract."""
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
        elif which in ("chan64_q15", "chan64_q15_1024", "chan_1024"):
            # CHAN-64-q15 (DESIGN.md §3.10) at config 4's width and at 1024 streams; chan_1024 = CHAN-64-f32 at 1024 streams beside it
            S, T = (1024 if which.endswith("1024") else 64), 192000 * args.seconds // 768 * 768
            x = torch.randint(-3000, 3000, (S, T, 2), dtype=torch.int16, device=dev, generator=g)
            q15 = which.startswith("chan64_q15")
            d = slb.DspIf(S, fs=192000, chain=slb.CHAIN_CHAN64_Q15 if q15 else slb.CHAIN_CHAN64_F32)
            y = torch.empty((S, 64, T // 64, 2), dtype=torch.int16, device=dev)
            ms = timeit(lambda: d.chan_process(x, y), args.steps); n = S * T
            name = "%s (%d x 192 kHz streams -> %d channels, %d s)" % ("chan64_q15" if q15 else "chan64_f32", S, 64 * S, args.seconds)
            del x, y
        elif which == "q15":
            C, T = args.rx_channels, 48000 * args.seconds
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_RX_SSB_Q15); y = torch.empty_like(x)
            ms = timeit(lambda: d.rx_process(x, y), args.steps); n = C * T; name = "rx_ssb_q15 (%d channels x %d s)" % (C, args.seconds)
        elif which == "txq15":
            C, T = args.rx_channels, 48000 * args.seconds
            m = torch.randint(-8000, 8000, (C, T, 1), dtype=torch.int16, device=dev, generator=g).expand(C, T, 2).contiguous()
            d = slb.DspIf(C, chain=slb.CHAIN_TX_SSB_Q15); y = torch.empty_like(m)
            ms = timeit(lambda: d.tx_process(m, y), args.steps); n = C * T; name = "tx_ssb_q15 (%d mic channels x %d s)" % (C, args.seconds)
        elif which in ("tx_q15_am", "tx_q15_fm", "tx_q15_ssb"):
            # TX-Q15 (DESIGN.md §3.9) with every mic channel in AM, FM or USB (the USB form is the TX-SSB-q15 kernel on the same context)
            C, T = args.rx_channels, 48000 * args.seconds
            m = torch.randint(-8000, 8000, (C, T, 1), dtype=torch.int16, device=dev, generator=g).expand(C, T, 2).contiguous()
            d = slb.DspIf(C, chain=slb.CHAIN_TX_Q15); y = torch.empty_like(m)
            d.DSP_Set_Mode({"tx_q15_am": slb.MODE_AM, "tx_q15_fm": slb.MODE_FM, "tx_q15_ssb": slb.MODE_USB}[which])
            ms = timeit(lambda: d.tx_process(m, y), args.steps); n = C * T; name = "%s (%d mic channels x %d s)" % (which, C, args.seconds)
        elif which in ("rx_q15_am", "rx_q15_fm", "rx_q15_ssb"):
            # RX-Q15 (DESIGN.md §3.8) with every channel in AM, FM or USB (the USB form is the RX-SSB-q15 kernel on the same context)
            C, T = args.rx_channels, 48000 * args.seconds
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_RX_Q15); y = torch.empty_like(x)
            d.DSP_Set_Mode({"rx_q15_am": slb.MODE_AM, "rx_q15_fm": slb.MODE_FM, "rx_q15_ssb": slb.MODE_USB}[which])
            ms = timeit(lambda: d.rx_process(x, y), args.steps); n = C * T; name = "%s (%d channels x %d s)" % (which, C, args.seconds)
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
        elif which in ("rx_tuned", "rx_half_tuned", "tx_usb", "tx_usb_tuned"):
            # per-channel tuning (DESIGN.md §3.5): every / every other channel offset by 7.3 kHz; TX-F32 in USB untuned and tuned
            C, T = args.rx_channels, 48000 * args.seconds // 384 * 384
            tx = which.startswith("tx")
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_TX_F32 if tx else slb.CHAIN_RX_SSB_F32); y = torch.empty_like(x)
            if which != "tx_usb":
                hz = torch.full((C,), 7300.0, dtype=torch.float64)
                if which == "rx_half_tuned":
                    hz[1::2] = 0.0
                d.set_tune(hz.numpy())
            ms = timeit(lambda: (d.tx_process if tx else d.rx_process)(x, y), args.steps); n = C * T
            name = "%s (%d channels x %d s)" % ({"rx_tuned": "rx_ssb_f32 USB, all channels tuned", "rx_half_tuned": "rx_ssb_f32 USB, half the channels tuned",
                                                 "tx_usb": "tx_f32 USB untuned", "tx_usb_tuned": "tx_f32 USB, all channels tuned"}[which], C, args.seconds)
        elif which == "tune_kernel":
            # the mixer's own time, from a torch.profiler run of its own: an RX call with every channel tuned (8 B per tuned sample)
            C, T = args.rx_channels, 48000 * args.seconds // 384 * 384
            x = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g)
            d = slb.DspIf(C, chain=slb.CHAIN_RX_SSB_F32); y = torch.empty_like(x); d.set_tune([7300.0] * C)
            d.rx_process(x, y); torch.cuda.synchronize()
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    d.rx_process(x, y)
                torch.cuda.synchronize()
            us = [e.device_time_total for e in prof.key_averages() if "tune_mix_kernel" in e.key]
            us_adv = [e.device_time_total for e in prof.key_averages() if "tune_advance_kernel" in e.key]
            ms = sum(us) / 1e3 / args.steps; n = C * T
            gbps = n * 8 / (ms * 1e-3) / 1e9
            print(json.dumps({"kernel": "tune_mix_kernel (RX, %d channels x %d s, all tuned)" % (C, args.seconds), "ms_per_call": ms,
                              "advance_ms_per_call": sum(us_adv) / 1e3 / args.steps, "GBps_at_8B_per_sample": gbps, "frac_of_measured_copy": gbps / roof}))
            del d
            continue
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
