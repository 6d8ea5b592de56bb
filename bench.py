#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: complex Msamples/s of the fused RX chain, whole box, + HBM roofline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the hot path (slb_rx_process_device, RX-SSB-f32 chain) over one batch of synthetic I/Q.
  N = 1: BASELINE configs[1], 1024 independent 48 kHz channels x 10 s (480 000 frames) = 1.97 GB in + 1.97 GB out per step.
  N > 1 (torchrun, one rank per GPU): BASELINE configs[4], 65 536 channels x 1 s sharded as contiguous ranges of 65 536 / N
         channels per GPU with NO data-path collective ("scaling": "strong"); after the timed compute the optional NCCL
         all-gather of the decoded audio (shard.gather_audio) is timed on its own and reported under "gather".
Both are far larger than the 126 MB L2. `value` has inputs resident in HBM; `e2e` is the same batch through the host-buffer
C-ABI call (slb_rx_process_host: pinned host memory -> H2D -> kernel -> D2H, sliced and overlapped) with the plain pinned
cudaMemcpyAsync duplex ceiling of the same bytes measured beside it on every rank at once (`e2e.pcie_ceiling_gbs`).
--dump-outputs DIR writes, after the timed steps, what the last of them returned (see dump_outputs), so that two builds can be
compared output for output: the inputs and the number of calls are fixed by the arguments.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "complex Msamples/s (whole box) RX chain"
UNIT = "Msamples/s"
CHANNELS_PER_GPU = 1024
FS = 48000
SECONDS = 10
FRAMES = FS * SECONDS          # 480 000 = 1250 hops of 384
BYTES_PER_SAMPLE = 8           # 4 B int16 I/Q in + 4 B int16 L/R out (SURVEY.md §8d)
CHAIN_NOTE = "RX-SSB-f32 chain (overlap-save SSB demod + 2-stage biquad + AGC; filter and biquad block response evaluated as one exact integer contraction on tcgen05: int8 digit planes x int8 digit planes -> int32, then float32)"
WORKLOAD = "configs[1]: 1024 independent 48 kHz I/Q channels x 10 s on one GPU, " + CHAIN_NOTE
CONFIG5_CHANNELS = 65536       # BASELINE configs[4]: "65536-channel RX chain sharded across 2/4/8 B200, optional NCCL gather of decoded audio"
CONFIG5_SECONDS = 1
WORKLOAD5 = "configs[4]: 65536 independent 48 kHz I/Q channels x 1 s sharded over %d GPUs (%d channels per GPU, contiguous ranges, no data-path collective), " + CHAIN_NOTE


def workload_for(world, seconds):
    """(channels per GPU, frames per step, workload string, scaling)."""
    if world == 1:
        return CHANNELS_PER_GPU, FS * seconds, WORKLOAD, "weak"
    c = CONFIG5_CHANNELS // world
    return c, FS * CONFIG5_SECONDS, WORKLOAD5 % (world, c), "strong"


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True); self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for k, n in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def synth_on_gpu(torch, channels, frames, device, first_channel):
    """Tone + complex Gaussian noise per channel (SURVEY.md §8d amplitudes and tone placement), generated on the device."""
    import selenite_lite_b200 as slb
    g = torch.Generator(device=device); g.manual_seed(slb.signals.SEED + first_channel)
    f0 = torch.tensor([slb.channel_tone_hz(first_channel + c) for c in range(channels)], device=device, dtype=torch.float64)
    out = torch.empty((channels, frames, 2), dtype=torch.int16, device=device)
    step = 64
    n = torch.arange(frames, device=device, dtype=torch.float64)
    for c0 in range(0, channels, step):
        c1 = min(channels, c0 + step)
        ph = (2.0 * torch.pi / FS) * f0[c0:c1, None] * n[None, :]
        iq = torch.stack([torch.cos(ph), torch.sin(ph)], -1).float() * 0.25
        iq += 0.01 * torch.randn(iq.shape, device=device, generator=g)
        out[c0:c1] = torch.clamp(torch.round(iq * 32768.0), -32768, 32767).to(torch.int16)
    return out


DUMP_BYTES = 60 * 10**6        # .npy payload of one --dump-outputs run, all ranks together (under 64 MB with the headers)


def dump_outputs(out_dir, y, rank, world):
    """Writes a fixed sample of y (int16 [channels][frames][2], this rank's output of the last timed step) as float32
    [n][frames][2] to out_dir/rx_out.npy (rx_out_rank<r>.npy when several ranks run): the n channels are drawn without
    replacement by numpy's default_rng(0) from this rank's channel range and kept in ascending order, so row i is global
    channel rank * channels_per_gpu + ch[i]; n is the most whole channels that fit this rank's share of DUMP_BYTES (at least
    one, cut to the frames that fit)."""
    import numpy as np
    import torch
    C, T, _ = y.shape
    budget = DUMP_BYTES // world
    n = max(1, min(C, budget // (T * 2 * 4)))
    frames = min(T, budget // (n * 2 * 4))
    ch = np.sort(np.random.default_rng(0).choice(C, n, replace=False))
    sample = y[torch.from_numpy(ch).to(y.device), :frames].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rx_out.npy" if world == 1 else "rx_out_rank%d.npy" % rank), sample)


def cpu_reference_run(threads, budget_s):
    """The reference's own CPU implementation of the path (oracle/_ref: CMSIS-DSP V1.5.3 compiled for this host; the
    port when that library is absent), channels split statically over `threads` pthreads, on a bounded sample."""
    import numpy as np
    import oracle_lib
    import selenite_lite_b200 as slb
    oracle_lib.build_oracles(want_ref=False)
    try:
        orc = oracle_lib.Oracle("ref"); kind = "reference"
    except (FileNotFoundError, OSError):
        orc = oracle_lib.Oracle("port"); kind = "port"
    p = slb.default_rx_f32_params(FS)
    prm = slb.dsp_if.params_to_dict(p, slb.default_mask(FS, p.fft_len, slb.MODE_USB))
    frames = 384 * 125                                       # 1 s per channel
    channels = threads * 8
    x = slb.synth_iq(min(channels, 8), frames)
    x = np.ascontiguousarray(np.tile(x, ((channels + x.shape[0] - 1) // x.shape[0], 1, 1))[:channels])
    orc.rx_ssb_f32_batch(prm, x[:threads], nthreads=threads)            # warm the caches / page in the library
    states, n_calls = None, 0
    t0 = time.perf_counter()
    while True:                                              # a continuing stream: state carries from call to call
        _, states = orc.rx_ssb_f32_batch(prm, x, states, nthreads=threads)
        n_calls += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s:
            break
    return {"value": n_calls * channels * frames / dt / 1e6, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": "%d calls x %d channels x %d frames (1 s each) of the same chain and signal model, gcc -O2 -ffp-contract=off, %d pthreads, %.1f s"
                      % (n_calls, channels, frames, threads, dt)}, n_calls * channels * frames, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    times = []
    base = None
    budget = max(1.0, min(10.0, 60.0 / (args.warmup + args.steps)))     # whole run ends within about a minute
    for i in range(args.warmup + args.steps):
        base, n, dt = cpu_reference_run(threads, budget_s=budget)
        if i >= args.warmup:
            times.append((n, dt))
    tot_s = sum(t for _, t in times); tot_n = sum(n for n, _ in times)
    v = tot_n / tot_s / 1e6
    base["value"] = v
    world = max(1, int(os.environ.get("WORLD_SIZE", args.gpus)))
    _, _, workload, scaling = workload_for(world, SECONDS)
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / len(times), "higher_is_better": True, "scaling": scaling,
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": workload, "note": "CPU arm: each step is a bounded sample (%s)" % base["sample"]},
                      "cpu_baseline": base, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}))


def measure_traffic(args):
    """DRAM bytes of ONE launch of the dominant kernel at the bench configuration, measured now, on this box: a short ncu pass
    over this very script (--traffic-probe: build the same batch, launch the kernel a few times) that collects only
    dram__bytes_read.sum and dram__bytes_write.sum. Returns (bytes, note)."""
    import csv
    import io
    import shutil
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found on this box"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k", "regex:rx_ssb_tc", "-s", "2", "-c", "1",
           "--csv", sys.executable, os.path.abspath(__file__), "--traffic-probe", "--seconds", str(args.seconds)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, BENCH_NO_SAMPLER="1")).stdout
        tot, seen = 0.0, 0
        rows = [r for r in csv.reader(io.StringIO(out[out.index('"ID"'):]))]
        hdr = rows[0]
        for r in rows[1:]:
            d = dict(zip(hdr, r))
            if d.get("Metric Name") in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[d["Metric Unit"]]
                tot += float(d["Metric Value"].replace(",", "")) * mult; seen += 1
        if seen != 2:
            return None, "ncu pass returned %d of 2 counters" % seen
        return tot, "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu pass inside this bench run"
    except Exception as exc:  # noqa: BLE001  (a profiler failure must not take the bench line down)
        return None, "ncu pass failed: %s" % (str(exc)[:120])


def traffic_probe(args):
    """Child of measure_traffic(): the bench batch, a few launches, nothing else."""
    import torch
    import selenite_lite_b200 as slb
    dev = torch.device("cuda", 0)
    C, T, _, _ = workload_for(1, args.seconds)
    d = slb.DspIf(C, fs=FS, chain=slb.CHAIN_RX_SSB_F32, device=0)
    x = synth_on_gpu(torch, C, T, dev, first_channel=0)
    y = torch.empty_like(x)
    for _ in range(4):
        d.rx_process(x, y)
    torch.cuda.synchronize()


def pin_rank_to_cores(local, world):
    """Every rank gets its own slice of the host cores (the staging threads of 8 ranks otherwise migrate over one NUMA node)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // max(1, world))
        mine = cores[local * per:(local + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return len(mine)
    except Exception:
        return None


def run_ours(args):
    import torch
    import selenite_lite_b200 as slb
    rank, world, local = slb.shard.env_rank_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    cores_per_rank = pin_rank_to_cores(local, world) if world > 1 else None

    C, T, workload, scaling = workload_for(world, args.seconds)
    lo = rank * C                                             # this rank's contiguous channel range [lo, lo + C)
    d = slb.DspIf(C, fs=FS, chain=slb.CHAIN_RX_SSB_F32, device=local)
    x = synth_on_gpu(torch, C, T, dev, first_channel=lo)
    y = torch.empty_like(x)
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        d.rx_process(x, y)
    barrier()
    sampler = ClockSampler(local)
    if not os.environ.get("BENCH_NO_SAMPLER"):
        sampler.start()
    time.sleep(0.3)
    launches0 = d.kernel_launches()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    torch.cuda.profiler.start()                              # ncu --profile-from-start off sees exactly the timed region
    evs[0].record()
    for i in range(args.steps):
        d.rx_process(x, y)
        evs[i + 1].record()
    barrier()
    torch.cuda.profiler.stop()
    clocks = sampler.stop()
    launches = d.kernel_launches() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y, rank, world)
    step_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    if os.environ.get("BENCH_DEBUG"):
        print("step_ms", [round(v, 3) for v in step_ms], file=sys.stderr)
    total_ms = max_over_ranks(evs[0].elapsed_time(evs[-1]))
    if dist is not None:
        ln = torch.tensor([launches], device=dev, dtype=torch.int64); dist.all_reduce(ln); launches = int(ln.item())
    samples_per_step = C * T * world
    value = samples_per_step * args.steps / (total_ms * 1e-3) / 1e6

    # roofline of the dominant (only) kernel: algorithmic bytes per launch / mean launch duration on this rank
    peak, peak_src = load_peaks()
    kern_ms = sum(step_ms) / len(step_ms)
    achieved = C * T * BYTES_PER_SAMPLE / (kern_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "peak_source": peak_src, "kernel": "rx_ssb_tc_kernel (sl_rx_ssb_tc.cu: tcgen05.mma kind::i8 FIR + biquad/AGC epilogue)", "algorithmic_bytes_per_launch": C * T * BYTES_PER_SAMPLE,
                "note": "1 launch per step; frac vs the nominal 8 TB/s = %.3f; the kernel is bound by the SM's L1 / shared-memory data pipe (tensor-core operand reads ~50 %% of its cycles + LSU wavefronts of converters, epilogue and output stores ~40 %%: profiles/r02_summary.md), not by HBM (DESIGN.md §4A)" % (achieved / 8000.0)}

    # optional gather of the decoded audio over NCCL / NVLink (configs[4]), timed on its own AFTER the timed compute
    gather = None
    if dist is not None:
        full = torch.empty((C * world, T, 2), dtype=torch.int16, device=dev)
        for _ in range(2):
            slb.shard.gather_audio(y, C * world, out=full)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_g = 3
        g0.record()
        for _ in range(n_g):
            slb.shard.gather_audio(y, C * world, out=full)
        g1.record()
        barrier()
        g_ms = max_over_ranks(g0.elapsed_time(g1) / n_g)
        ok = bool(torch.equal(full[lo:lo + C], y))           # this rank's own shard sits where it belongs
        recv = (world - 1) * C * T * 4                       # bytes every GPU receives over NVLink per gather
        gather = {"op": "ncclAllGather of int16 audio [channels][frames][2] (one frame = one int32 word), every rank ends with all %d channels" % (C * world),
                  "bytes_per_rank_in": C * T * 4, "bytes_per_rank_received": recv, "ms": g_ms, "recv_GBps_per_gpu": recv / (g_ms * 1e-3) / 1e9,
                  "algbw_GBps": C * world * T * 4 / (g_ms * 1e-3) / 1e9, "own_shard_in_place": ok,
                  "note": "after the timed compute, not part of `value`; NVLink peer-copy reference on this pool 770 GB/s per direction per GPU"}
        del full

    # end to end through the host-buffer C-ABI call, and the plain-copy ceiling of the same bytes beside it
    e2e = None
    if not args.no_e2e:
        xh = torch.empty((C, T, 2), dtype=torch.int16).pin_memory(); yh = torch.empty((C, T, 2), dtype=torch.int16).pin_memory()
        xh.copy_(x); torch.cuda.synchronize()
        d2 = slb.DspIf(C, fs=FS, chain=slb.CHAIN_RX_SSB_F32, device=local)
        for _ in range(2):
            d2.rx_process_pinned(xh, yh)
        barrier()
        t0 = time.perf_counter()
        n_e2e = max(3, min(args.steps, 5))
        e2e_steps = []
        for _ in range(n_e2e):
            t1 = time.perf_counter()
            d2.rx_process_pinned(xh, yh)                     # returns after the D2H copy of the result has landed
            e2e_steps.append(time.perf_counter() - t1)
        barrier()
        # per-step wall times of this rank; the reported figure uses the MEDIAN step (max over ranks), so that one step hit by another
        # tenant of the host (seen once: 62 ms instead of 42) does not decide the number; the mean is kept beside it
        dt_mean = max_over_ranks(time.perf_counter() - t0)
        dt = max_over_ranks(sorted(e2e_steps)[len(e2e_steps) // 2]) * n_e2e
        if os.environ.get("BENCH_DEBUG"):
            print("e2e step ms", [round(v * 1e3, 2) for v in e2e_steps], file=sys.stderr)
        # ceiling: the same bytes as ONE contiguous pinned cudaMemcpyAsync each way, both directions at once, all ranks at once
        s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

        def duplex():
            with torch.cuda.stream(s_in):
                x.copy_(xh, non_blocking=True)
            with torch.cuda.stream(s_out):
                yh.copy_(y, non_blocking=True)
        duplex(); barrier()
        dt_c = None
        for _ in range(3):                                   # a ceiling is the best the link does: best of three rounds (a round disturbed by
            t0 = time.perf_counter()                         # another process's driver call once read 33 GB/s next to an e2e of 44)
            for _ in range(n_e2e):
                duplex()
            barrier()
            r = max_over_ranks(time.perf_counter() - t0)
            dt_c = r if dt_c is None else min(dt_c, r)
        ceil_gbs = C * T * 4 * n_e2e / dt_c / 1e9            # per GPU, each way
        e2e_val = samples_per_step * n_e2e / dt / 1e6
        ceil_val = samples_per_step * n_e2e / dt_c / 1e6
        e2e = {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": C * T * 4 * world, "d2h_bytes_per_step": C * T * 4 * world,
               "steps": n_e2e, "statistic": "median step (max over ranks); mean-based value in value_mean", "value_mean": samples_per_step * n_e2e / dt_mean / 1e6,
               "pcie_ceiling_gbs": ceil_gbs, "pcie_ceiling_msamples": ceil_val, "frac_of_ceiling": e2e_val / ceil_val,
               "ceiling_how": "same bytes as one contiguous pinned cudaMemcpyAsync H2D + one D2H per step on two streams, every rank at once, GB/s per GPU each way, best of three rounds",
               "host_cores_per_rank": cores_per_rank,
               "path": "slb_rx_process_host: pinned host -> strided H2D -> rx_ssb_tc_kernel -> strided D2H, time slices of all channels, copies and kernels on 3 streams"}
        del xh, yh, d2

    # the other chains of the library at the same width, device-resident, for context (not the headline metric)
    other = None
    if rank == 0 and world == 1 and not args.no_other:
        other = {}
        del x, y
        torch.cuda.empty_cache()
        g = torch.Generator(device=dev); g.manual_seed(1)

        def timed(fn, n=5):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record(); torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n
        xi = torch.randint(-8000, 8000, (C, T, 2), dtype=torch.int16, device=dev, generator=g); yo = torch.empty_like(xi)
        for name, chain, call in (("rx_ssb_q15", slb.CHAIN_RX_SSB_Q15, "rx_process"), ("tx_ssb_f32", slb.CHAIN_TX_SSB_F32, "tx_process")):
            dd = slb.DspIf(C, fs=FS, chain=chain, device=local)
            ms = timed(lambda: getattr(dd, call)(xi, yo))
            other[name] = {"Msamples_per_s": C * T / (ms * 1e-3) / 1e6, "hbm_frac": C * T * BYTES_PER_SAMPLE / (ms * 1e-3) / 1e9 / peak,
                           "note": "bit-exact integer chain: rx_q15_tc_kernel (tcgen05 kind::i8 FIRs, integer epilogue)" if name == "rx_ssb_q15" else "config 3: tx_ssb_tc_kernel (tcgen05 FIR, two rails)"}
            del dd
        del xi, yo
        S, Tw = 64, 192000 * args.seconds // 768 * 768
        xw = torch.randint(-3000, 3000, (S, Tw, 2), dtype=torch.int16, device=dev, generator=g)
        yw = torch.empty((S, 64, Tw // 64, 2), dtype=torch.int16, device=dev)
        dd = slb.DspIf(S, fs=192000, chain=slb.CHAIN_CHAN64_F32, device=local)
        ms = timed(lambda: dd.chan_process(xw, yw))
        other["chan64_f32"] = {"Msamples_per_s": S * Tw / (ms * 1e-3) / 1e6, "hbm_frac": S * Tw * BYTES_PER_SAMPLE / (ms * 1e-3) / 1e9 / peak,
                               "note": "config 4: 64 x 192 kHz wideband streams -> 4096 narrowband channels"}
        del dd, xw, yw
        torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu_baseline = cpu_reference_run(os.cpu_count() or 1, budget_s=12.0)[0]
    if rank == 0 and world == 1 and not args.no_traffic:
        roofline["traffic"], roofline["traffic_how"] = measure_traffic(args)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()
    if rank != 0:
        return
    print(json.dumps({
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload, "channels_per_gpu": C, "channels_total": C * world, "frames_per_step": T, "fs": FS, "chain": "rx_ssb_f32",
                   "arithmetic": "filter + biquad block response: int8 x int8 -> int32 digit products of int16 samples and a 32-bit-quantised map (exact for that map; the high data byte meets all four map digits); state chain, AGC, pack: float32",
                   "l2_policy": "inputs larger than L2 (%.1f GB touched per step per GPU vs 126 MB L2)" % (C * T * 8 / 1e9), "parallelism": "channels sharded, no collective"},
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gather": gather, "gpu_launches": launches, "clocks": clocks, "other_chains": other}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-other", action="store_true", help="skip the context measurements of the other chains")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu pass that measures the kernel's DRAM traffic")
    ap.add_argument("--traffic-probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--seconds", type=int, default=SECONDS, help="signal seconds per channel per step (profiling runs only; the headline uses the default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's output to DIR/rx_out.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's output (--impl ours)")
    if args.traffic_probe:
        traffic_probe(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
