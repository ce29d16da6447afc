#!/usr/bin/env python
"""bench.py — Msamples/s of the resample -> effects -> mix pipeline (BASELINE.json metric).

Workload (config.workload = "cfg3_pipeline"): per GPU 4096 mono 44.1 kHz f32 streams of `--seconds`
seconds, each `UniformSourceIterator(1 ch, 48 kHz) -> low_pass(200) -> amplify(1.2)`, summed by
`mixer(1, 48000)` — the benches/pipeline.rs shape of BASELINE.json configs[2], which is the
configuration the metric is quoted on and fits one GPU.  A step = one drain of the MixerSource over the
whole batch.  "samples" = sum over streams of post-resample, pre-mix samples (SURVEY.md §8d).

  python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
  python bench.py ... --dump-outputs DIR                        # also writes the last timed step's mix to DIR/mix.npy
  python bench.py --impl reference ...                          # the reference's CPU algorithm (oracle port,
                                                                # all host threads; rodio is Rust and cannot be built here)
Under torchrun (N>1) every rank renders its own 4096 streams (weak scaling), the partial mixes are
all-reduced (NCCL) inside the timed region, time = max over ranks of the CUDA-event time.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MIX_CH, MIX_RATE, IN_RATE = 1, 48000, 44100
LOW_PASS_HZ, AMPLIFY = 200, 1.2
DUMP_MAX_SAMPLES = 1 << 23      # 32 MB of float32: a longer mix is dumped as a fixed, seeded sample of its samples


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="streams per GPU")
    ap.add_argument("--seconds", type=float, default=2.0, help="audio seconds per stream")
    ap.add_argument("--flags", type=int, default=0, help="rb_batch_create flags (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the mix of the last timed step to DIR/mix.npy (float32), for comparing two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def measured_traffic(workload: str, streams: int, seconds: float):
    """dram bytes per launch of the dominant kernel from the committed ncu capture of this exact config."""
    try:
        with open(os.path.join(ROOT, "profiles", "r1_traffic.json")) as f:
            t = json.load(f)[workload]
        if t["streams_per_gpu"] == streams and abs(t["seconds"] - seconds) < 1e-9:
            return t["traffic"], t["source"]
    except Exception:
        pass
    return None, None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# clocks sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def make_sources(rb, n_streams: int, frames: int, pcm=None):
    """cfg3 sources.  `pcm` (n_streams x frames float32) may be None: the bench fills HBM directly."""
    srcs = []
    dummy = np.zeros(frames, dtype=np.float32)
    for s in range(n_streams):
        x = dummy if pcm is None else pcm[s]
        srcs.append(rb.UniformSourceIterator(rb.TestSource(x, 1, IN_RATE), MIX_CH, MIX_RATE)
                    .low_pass(LOW_PASS_HZ).amplify(AMPLIFY))
    return srcs


def resampled_frames(L: int, from_rate: int, to_rate: int) -> int:
    """Closed form of SampleRateConverter's output length on L frames (DESIGN.md section 3; src/conversions/sample_rate.rs:157-199)."""
    import math
    g = math.gcd(from_rate, to_rate)
    fr, to = from_rate // g, to_rate // g
    if L <= 1 or fr == to:
        return L
    n = -((-(L - 1) * to) // fr)
    return n + (1 if n * fr < L * to else 0)


def cpu_streams(n_streams: int, frames: int, seed: int = 1234):
    """cfg3 streams in the oracle's own terms -- nothing of the product package is imported on this path."""
    import oracle
    rng = np.random.default_rng(seed)
    chain = [oracle.fx(oracle.FX_UNIFORM, u32=[MIX_CH, MIX_RATE]), oracle.fx(oracle.FX_LOW_PASS, u32=[LOW_PASS_HZ], f32=[0.5]),
             oracle.fx(oracle.FX_AMPLIFY, f32=[AMPLIFY])]
    out = []
    for _ in range(n_streams):
        out.append(oracle.Stream(rng.uniform(-1, 1, frames).astype(np.float32), 1, IN_RATE, chain, 0))
    return out


def cpu_reference(streams, frames: int, threads: int):
    """The reference's CPU algorithm (oracle port, pull iterators, monomorphised chain like rustc's), streams sharded
    over `threads` host threads.  Returns (Msamples/s, seconds, samples)."""
    import oracle
    out_frames = resampled_frames(frames, IN_RATE, MIX_RATE)
    _, secs = oracle.mixer_mt(streams, MIX_CH, MIX_RATE, threads, out_frames + 16, static_dispatch=True)
    samples = len(streams) * out_frames
    return samples / secs / 1e6, secs, samples


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def run_reference(args):
    """bench.py --impl reference: rodio's CPU path (C++ restatement: the Rust toolchain is not in the image) on the SAME
    configuration -- args.streams streams of args.seconds seconds -- with all host threads.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import oracle
    oracle.build()
    threads = host_threads()
    frames = int(round(args.seconds * IN_RATE))
    n_streams = args.streams
    streams = cpu_streams(n_streams, frames)
    cpu_reference(streams[:max(1, min(n_streams, threads))], frames, threads)          # warm-up (page in, spawn)
    steps = args.steps
    runs = [cpu_reference(streams, frames, threads) for _ in range(steps)]
    vals = sorted(r[0] for r in runs)
    value = statistics.median(vals)
    secs_all = sum(r[1] for r in runs)
    sample = (f"the full configuration: {n_streams} streams x {args.seconds} s, {steps} timed drains, {threads} host threads; "
              f"Msamples/s min/median/max {vals[0]:.1f}/{value:.1f}/{vals[-1]:.1f}")
    line = {
        "impl": "reference", "metric": "Msamples/s resample->low_pass->amplify->mix", "value": value,
        "unit": "Msamples/s", "n_gpus": args.gpus, "steps": steps, "warmup": 1,
        "ms_per_step": 1e3 * secs_all / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg3_pipeline", "streams_per_gpu": args.streams, "seconds": args.seconds,
                   "in_rate": IN_RATE, "mixer": [MIX_CH, MIX_RATE], "low_pass_hz": LOW_PASS_HZ, "amplify": AMPLIFY,
                   "note": "C++ restatement of rodio's CPU pull-iterator path (Rust toolchain unavailable)"},
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": threads, "kind": "port", "sample": sample,
                         "runs_msamples_per_s": [round(r[0], 1) for r in runs]},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist

    import rodio_b200 as rb
    from rodio_b200 import build as rb_build
    from rodio_b200 import dist as rbd

    rank, local_rank, world = rbd.env_rank()
    if not os.path.exists(rb.capi.LIB_PATH):
        rb_build.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: rodio_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctx = rb.Context(local_rank)
    ext = torch.cuda.ExternalStream(ctx.cuda_stream, device=dev)
    comm = None
    if world > 1:
        # torch.distributed is the plumbing (barrier, max over ranks, handing out the communicator id); the data-path
        # collective is the library's own: rb_batch_render_mix_allreduce = render + k_mix_exchange over NVLink peer memory (NCCL's
        # all-reduce where the ranks cannot map each other's memory; RB_COMM_NCCL_ONLY=1 forces it for A/B runs)
        rbd.init_process_group("nccl")
        ids = [rb.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = rb.Comm(ctx, world, rank, ids[0])

    S = args.streams
    frames = int(round(args.seconds * IN_RATE))
    srcs = make_sources(rb, S, frames)
    batch = rb.Batch(srcs, MIX_CH, MIX_RATE, flags=args.flags, ctx=ctx)
    out_frames = batch.stream_out_len(0)
    mix_len = batch.mix_len
    samples_per_step = S * out_frames * world
    algo_bytes = batch.algorithmic_bytes
    launches = batch.launches_per_render
    try:
        family = batch.kernel_family
    except Exception:   # an older library without the query: the default plan is the HOT kernel
        family = 1
    kernel_label = {2: "k_fused_lanes + k_sum_groups (2 launches per step)", 3: "k_fused_duo + k_sum_groups (2 launches per step)",
                    4: "k_fused_duo over timeline segments + k_sum_groups (2 launches per step)",
                    1: "k_fused_hot + k_sum_partials (2 launches per step)"}.get(family, "kernel family %d" % family)

    # ---- inputs resident in HBM before the timed region (seeded, distinct per rank) ----
    p0, _ = batch.input_device_ptr(0)
    pitch = (batch.input_device_ptr(1)[0] - p0) // 4 if S > 1 else frames
    for i in range(S):
        batch.input_device_ptr(i)          # marks every stream as provided
    arena = torch.as_tensor(rbd.DeviceArray(p0, pitch * (S - 1) + frames), device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x5EED + rank)
    with torch.cuda.stream(ext):
        # drawn as a packed (streams, frames) block and copied into the batch's pitched rows: the same seed gives every stream
        # the same samples whatever padding the library puts between streams
        arena.as_strided((S, frames), (pitch, 1)).copy_(torch.empty(S, frames, device=dev).uniform_(-1.0, 1.0, generator=gen))
    mix = torch.as_tensor(rbd.DeviceArray(batch.mix_device_ptr, max(1, mix_len)), device=dev)

    def step():
        if comm is not None:
            comm.render_mix_allreduce(batch)
        else:
            batch.render_mix_device()

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(3, args.warmup)):
        step()
    fence()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    e0.record(ext)
    for _ in range(args.steps):
        step()
    e1.record(ext)
    fence()
    # what the last timed step handed its caller, copied before the loops below render into the same buffer
    last_mix = mix[:mix_len].cpu().numpy() if args.dump_outputs else None
    ms_total = e0.elapsed_time(e1)
    ms_total = rbd.max_over_ranks(ms_total, dev)
    ms_step = ms_total / args.steps
    value = samples_per_step / (ms_step * 1e-3) / 1e6

    # ---- roofline of the dominant kernel: timed alone (no collective), CUDA events on its stream ----
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    k0.record(ext)
    for _ in range(args.steps):
        batch.render_mix_device()
    k1.record(ext)
    torch.cuda.synchronize(dev)
    ms_kernel = k0.elapsed_time(k1) / args.steps
    peak, peak_src = peaks()
    achieved = algo_bytes / (ms_kernel * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic("cfg3_pipeline", S, args.seconds)

    # ---- end to end through the public API with HOST buffers (H2D + render + D2H every step) ----
    e2e = None
    if not args.no_e2e:
        host_in = torch.empty(S * frames, dtype=torch.float32, pin_memory=True)
        with torch.cuda.stream(ext):
            tmp = torch.empty(S * frames, dtype=torch.float32, device=dev)
            tmp.uniform_(-1.0, 1.0, generator=gen)
            host_in.copy_(tmp, non_blocking=False)
        del tmp
        host_out = torch.empty(max(1, mix_len), dtype=torch.float32, pin_memory=True)

        def e2e_step():
            batch.upload_packed(host_in.data_ptr(), S * frames)
            if world > 1:
                comm.render_mix_allreduce(batch)
                with torch.cuda.stream(ext):
                    host_out.copy_(mix, non_blocking=True)
                ctx.sync()
            else:
                batch.render_mix_into(host_out.data_ptr(), mix_len)

        e2e_steps = max(3, min(args.steps, 10))
        for _ in range(2):
            e2e_step()
        fence()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(ext)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        f1.record(ext)
        fence()
        wall_ms = (time.perf_counter() - t0) * 1e3
        e2e_ms = rbd.max_over_ranks(max(f0.elapsed_time(f1), wall_ms) / e2e_steps, dev)
        e2e = {"value": samples_per_step / (e2e_ms * 1e-3) / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": S * frames * 4, "d2h_bytes_per_step": mix_len * 4, "ms_per_step": e2e_ms,
               "steps": e2e_steps, "note": "pinned host PCM -> rb_batch_upload_packed -> render -> host mix, per step"}
        # the same through s16 host PCM (what rodio's decoders yield: src/decoder/wav.rs:119-151, converted by
        # SampleTypeConverter, src/conversions/sample.rs:42-44): half the bytes over PCIe, converted on the device at upload
        try:
            srcs16 = [rb.UniformSourceIterator(rb.TestSource(np.zeros(frames, np.int16), 1, IN_RATE), MIX_CH, MIX_RATE)
                      .low_pass(LOW_PASS_HZ).amplify(AMPLIFY) for _ in range(S)]
            batch16 = rb.Batch(srcs16, MIX_CH, MIX_RATE, flags=args.flags, ctx=ctx)
            host16 = torch.empty(S * frames, dtype=torch.int16, pin_memory=True)
            with torch.cuda.stream(ext):
                tmp = torch.empty(S * frames, dtype=torch.float32, device=dev)
                tmp.uniform_(-30000.0, 30000.0, generator=gen)
                host16.copy_(tmp.to(torch.int16), non_blocking=False)
            del tmp
            mix16 = torch.as_tensor(rbd.DeviceArray(batch16.mix_device_ptr, max(1, mix_len)), device=dev)

            def e2e16_step():
                batch16.upload_packed(host16.data_ptr(), S * frames)
                if world > 1:
                    comm.render_mix_allreduce(batch16)
                    with torch.cuda.stream(ext):
                        host_out.copy_(mix16, non_blocking=True)
                    ctx.sync()
                else:
                    batch16.render_mix_into(host_out.data_ptr(), mix_len)
            for _ in range(2):
                e2e16_step()
            fence()
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record(ext)
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e16_step()
            h1.record(ext)
            fence()
            wall16 = (time.perf_counter() - t0) * 1e3
            ms16 = rbd.max_over_ranks(max(h0.elapsed_time(h1), wall16) / e2e_steps, dev)
            e2e["s16_input"] = {"value": samples_per_step / (ms16 * 1e-3) / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": S * frames * 2,
                                "d2h_bytes_per_step": mix_len * 4, "ms_per_step": ms16, "kernel_family": batch16.kernel_family,
                                "note": "pinned host s16 PCM -> rb_batch_upload_packed -> k_convert (device) -> render -> host mix, per step"}
            batch16.close()
            del host16
        except Exception as exc:   # noqa: BLE001
            e2e["s16_input"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- the other BASELINE configurations beside it (N=1 only): every entry is one render of resident inputs, CUDA events on
    # the render stream, its own algorithmic bytes and roofline fraction; a failure is reported in place, never fatal ----
    also = None
    if world == 1 and not args.no_e2e:
        also = {}

        def timed(name, workload, srcs, mixer_ch, flags, steps, kernel_names, fill=True):
            try:
                b2 = rb.Batch(srcs, mixer_ch, MIX_RATE, flags=flags, ctx=ctx)
                n2 = len(srcs)
                if fill:
                    q0, cap0 = b2.input_device_ptr(0)
                    pitch2 = (b2.input_device_ptr(1)[0] - q0) // 4 if n2 > 1 else cap0
                    for i in range(n2):
                        b2.input_device_ptr(i)
                    with torch.cuda.stream(ext):
                        torch.as_tensor(rbd.DeviceArray(q0, pitch2 * (n2 - 1) + cap0), device=dev).uniform_(-0.5, 0.5, generator=gen)
                for _ in range(3):
                    b2.render_mix_device()
                torch.cuda.synchronize(dev)
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record(ext)
                for _ in range(steps):
                    b2.render_mix_device()
                g1.record(ext)
                torch.cuda.synchronize(dev)
                ms2 = g0.elapsed_time(g1) / steps
                fam = b2.kernel_family
                samples2 = n2 * b2.stream_out_len(0)      # every stream of these configurations has the same shape
                gbs = b2.algorithmic_bytes / (ms2 * 1e-3) / 1e9
                also[name] = {"workload": workload, "value": samples2 / (ms2 * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms2,
                              "steps": steps, "launches": b2.launches_per_render,
                              "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                                           "kernel": kernel_names.get(fam, "kernel family %d" % fam)}}
                b2.close()
            except Exception as exc:   # noqa: BLE001 -- the headline line must survive whatever happens here
                also[name] = {"workload": workload, "error": f"{type(exc).__name__}: {exc}"[:300]}

        FAM = {-1: "general path (one kernel per adapter)", 0: "k_fused_biquad", 1: "k_fused_hot + k_sum_partials", 2: "k_fused_lanes + k_sum_groups",
               3: "k_fused_duo + k_sum_groups", 4: "k_fused_duo over timeline segments + k_sum_groups", 5: "k_fused_fx + k_fx_sum_partials",
               6: "k_lerp_mix + k_sum_groups"}
        z = lambda n: np.zeros(n, np.float32)
        steps2 = max(3, min(args.steps, 10))
        timed("cfg2_dynamic_mixer", "mixer(1, 48000) of 1024 mono 48 kHz f32 sources x 10 s, summed in insertion order (bit-exact)",
              [rb.TestSource(z(48000 * 10), 1, MIX_RATE) for _ in range(1024)], 1, args.flags, args.steps, {-1: "k_mix_ordered"})
        timed("cfg2_from_generators", "BASELINE configs[1] as the reference states it: 1024 SineWave sources (110 Hz * 2^(s/128)) x 10 s handed to "
              "mixer(1, 48000) -- generated on the device (k_siggen: f32 phase recurrence per source, glibc's sinf in FP64) AND summed in "
              "insertion order, nothing uploaded; latency-bound by the 480 000 serial phase steps per source",
              [rb.SineWave(min(110.0 * 2.0 ** (s / 128.0), 19999.0)).take(48000 * 10) for s in range(1024)], 1, args.flags, 3,
              {-1: "k_siggen + k_mix_ordered"}, fill=False)
        one2 = z(2 * IN_RATE)
        timed("cfg3_low_pass_1000_time_parallel",
              "cfg3 shape at low_pass(1000) with RB_BIQUAD_TIME_PARALLEL (SURVEY 8d cfg3: the scan variant beside the exact one): 4096 mono "
              "streams x 2 s, timeline segments with a warm-up; <= 1e-5 * peak of the reference (tests), most segments bit-identical",
              [rb.UniformSourceIterator(rb.TestSource(one2, 1, IN_RATE), 1, MIX_RATE).low_pass(1000).amplify(AMPLIFY) for _ in range(4096)],
              1, rb.capi.RB_BIQUAD_TIME_PARALLEL, steps2, FAM)
        timed("cfg3_exact_order", "the headline batch (4096 mono x 2 s, 44.1 -> 48 kHz -> low_pass(200) -> amplify -> mix) with RB_MIX_EXACT_ORDER: "
              "k_fused_hot hands the running sum of every tile from CTA to CTA, so the WHOLE mix is the reference's sequential sum over "
              "all 4096 sources bit for bit (tests/test_bench_geometries_gpu.py::test_exact_order_*); the default grouping above is <= 1e-5 * peak",
              [rb.UniformSourceIterator(rb.TestSource(one2, 1, IN_RATE), 1, MIX_RATE).low_pass(LOW_PASS_HZ).amplify(AMPLIFY) for _ in range(4096)],
              1, rb.capi.RB_MIX_EXACT_ORDER, steps2, {1: "k_fused_hot<1, true, CHAIN> (one launch)"})
        timed("cfg3_no_filter", "4096 mono streams x 2 s, 44.1 -> 48 kHz -> amplify(1.2) -> mix (bit-exact per stream)",
              [rb.UniformSourceIterator(rb.TestSource(one2, 1, IN_RATE), 1, MIX_RATE).amplify(AMPLIFY) for _ in range(4096)], 1, 0, steps2, FAM)
        timed("cfg4_effect_chain", "512 stereo 48 kHz sources x 1 s: Spatial -> reverb(50 ms, 0.3) -> automatic_gain_control -> mix(2 ch); "
              "latency-bound: three serial recurrences per stream, 100 800 steps of >= 22 cycles",
              [rb.Spatial(rb.TestSource(z(2 * 48000), 2, MIX_RATE), [float(s % 7 - 3), 1.0, 0.0], [-1, 0, 0], [1, 0, 0])
               .reverb(rb.Duration.from_millis(50), 0.3).automatic_gain_control() for s in range(512)], 2, 0, 3, FAM)
        timed("cfg4_exact_order", "cfg4 with RB_MIX_EXACT_ORDER: k_fused_fx hands the running sum from CTA to CTA -- the whole stereo mix is the "
              "reference's sequential sum bit for bit (tests/test_bench_geometries_gpu.py::test_exact_order_effect_chain_cfg4)",
              [rb.Spatial(rb.TestSource(z(2 * 48000), 2, MIX_RATE), [float(s % 7 - 3), 1.0, 0.0], [-1, 0, 0], [1, 0, 0])
               .reverb(rb.Duration.from_millis(50), 0.3).automatic_gain_control() for s in range(512)], 2, rb.capi.RB_MIX_EXACT_ORDER, 3,
              {5: "k_fused_fx<2, CHAIN> (one launch)"})
        one1 = z(IN_RATE)
        sweep = {}
        for n3 in (1, 16, 256, 1024, 4096, 16384, 65536):
            timed("_sweep", f"{n3} mono streams x 1 s, 44.1 -> 48 kHz -> low_pass(200) -> amplify(1.2) -> mix",
                  [rb.UniformSourceIterator(rb.TestSource(one1, 1, IN_RATE), 1, MIX_RATE).low_pass(LOW_PASS_HZ).amplify(AMPLIFY) for _ in range(n3)],
                  1, args.flags, 5 if n3 >= 16384 else steps2, FAM)
            r = also.pop("_sweep")
            sweep[str(n3)] = {"ms": r.get("ms_per_step"), "Msamples_s": r.get("value"), "frac": (r.get("roofline") or {}).get("frac"),
                              "kernel": (r.get("roofline") or {}).get("kernel"), **({"error": r["error"]} if "error" in r else {})}
        also["cfg5_sweep"] = {"workload": "BASELINE configs[4]: batch 1 -> 65536 x 1 s@44.1 kHz f32 through the fused pipeline (exact biquad), default planner",
                              "streams": sweep}
        if "65536" in sweep and sweep["65536"].get("frac") is not None:
            also["cfg5_65536_streams"] = {"workload": "65536 mono streams x 1 s, 44.1 -> 48 kHz -> low_pass(200) -> amplify(1.2) -> mix, inputs 11.6 GB resident",
                                          "value": sweep["65536"]["Msamples_s"], "unit": "Msamples/s", "ms_per_step": sweep["65536"]["ms"],
                                          "roofline": {"bound": "hbm", "achieved": sweep["65536"]["frac"] * peak, "peak": peak, "unit": "GB/s",
                                                       "frac": sweep["65536"]["frac"], "kernel": sweep["65536"]["kernel"]}}

    # ---- strong scaling beside the weak-scaling headline: a FIXED total batch sharded over the ranks (SURVEY 8d cfg3 is 4096
    # streams in total on 8 GPUs; cfg5's large end 65 536).  Exact biquad, all-reduce inside the timed region, max over ranks. ----
    strong = None
    if not args.no_e2e:
        strong = {}
        for total, secs in ((4096, args.seconds), (65536, 1.0)):
            try:
                lo, hi = rbd.shard_range(total, rank, world)
                fr = int(round(secs * IN_RATE))
                bs = rb.Batch(make_sources(rb, hi - lo, fr), MIX_CH, MIX_RATE, flags=args.flags, ctx=ctx)
                s0, cap0 = bs.input_device_ptr(0)
                pitch_s = (bs.input_device_ptr(1)[0] - s0) // 4 if hi - lo > 1 else cap0
                for i in range(hi - lo):
                    bs.input_device_ptr(i)
                with torch.cuda.stream(ext):
                    torch.as_tensor(rbd.DeviceArray(s0, pitch_s * (hi - lo - 1) + cap0), device=dev).uniform_(-1.0, 1.0, generator=gen)
                run = (lambda: comm.render_mix_allreduce(bs)) if comm is not None else bs.render_mix_device
                for _ in range(3):
                    run()
                fence()
                st = max(3, min(args.steps, 10))
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record(ext)
                for _ in range(st):
                    run()
                t1.record(ext)
                fence()
                ms_s = rbd.max_over_ranks(t0.elapsed_time(t1) / st, dev)
                r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                r0.record(ext)
                for _ in range(st):
                    bs.render_mix_device()
                r1.record(ext)
                fence()
                ms_r = rbd.max_over_ranks(r0.elapsed_time(r1) / st, dev)
                strong[f"{total}_streams_total"] = {
                    "streams_per_gpu": hi - lo, "seconds": secs, "ms_per_step": ms_s, "render_only_ms": ms_r, "allreduce_ms": max(0.0, ms_s - ms_r),
                    "value": total * bs.stream_out_len(0) / (ms_s * 1e-3) / 1e6, "unit": "Msamples/s", "kernel_family": bs.kernel_family,
                    "limiter": ("recurrence latency: a stream of %d samples is a serial chain of >= 13 cycles per sample whatever the shard size" % bs.stream_out_len(0))
                               if bs.kernel_family == 1 and hi - lo <= 4096 else "see roofline of the shard size"}
                bs.close()
            except Exception as exc:   # noqa: BLE001
                strong[f"{total}_streams_total"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    clocks = sampler.stop()   # sampled over the timed region, the kernel-only loop and the end-to-end loop

    # ---- CPU baseline beside it (rank 0, N=1): bounded sample of the same workload ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle
        oracle.build()
        threads = host_threads()
        n_cpu = max(threads, min(S, 64 * threads))
        cs = cpu_streams(n_cpu, IN_RATE)
        cpu_reference(cs[:threads], IN_RATE, threads)
        v, secs, smp = max(cpu_reference(cs, IN_RATE, threads) for _ in range(3))
        cpu = {"value": v, "unit": "Msamples/s", "cores": threads, "kind": "port",
               "sample": f"{n_cpu} streams x 1 s of the same chain, best of 3 drains ({secs:.2f} s wall), oracle port "
                         f"(pull iterators) sharded over {threads} host threads"}

    if rank == 0:
        line = {
            "metric": "Msamples/s resample->low_pass->amplify->mix", "value": value, "unit": "Msamples/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg3_pipeline", "streams_per_gpu": S, "seconds": args.seconds, "in_rate": IN_RATE,
                       "mixer": [MIX_CH, MIX_RATE], "low_pass_hz": LOW_PASS_HZ, "amplify": AMPLIFY,
                       "biquad": "exact sequential f32 order (bit-exact with the reference)",
                       "l2": f"inputs {S * frames * 4 / 1e9:.2f} GB per GPU, larger than the 126 MB L2 (no flush needed)",
                       "flags": args.flags},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel_ms": ms_kernel, "kernel": kernel_label,
                         "algorithmic_bytes_per_step": algo_bytes,
                         "note": "whole render (all launches of one step) timed with CUDA events on the launch stream"},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "also": also,
            "strong_scaling": strong,
            "allreduce": None if world == 1 else {"impl": "rb_batch_render_mix_allreduce: " + comm.transport, "floats": mix_len,
                                                  "ms": max(0.0, ms_step - ms_kernel)},
            "gpu_launches": launches * args.steps,
            "clocks": clocks,
        }
        if args.dump_outputs:
            if last_mix.size > DUMP_MAX_SAMPLES:
                last_mix = last_mix[np.sort(np.random.default_rng(0).choice(last_mix.size, DUMP_MAX_SAMPLES, replace=False))]
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "mix.npy"), last_mix)
        print(json.dumps(line), flush=True)
    batch.close()
    if world > 1:
        dist.barrier()
        comm.close()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
