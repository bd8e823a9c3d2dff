#!/usr/bin/env python
"""bench.py — 44.1 kHz output samples/s of the so-vits-svc waveform-generation hot path on B200.

A step = one ``SynthesizerTrn.infer`` over a batch of synthetic utterances (BASELINE config 2 by default:
8 x 862 frames = 8 x 10 s; ContentVec-768 features, f0, uv, speaker id; seeded random-init weights).
  value : whole-job samples/s with inputs resident in HBM when the timed region starts
  e2e   : same through the public API with pinned HOST inputs (H2D inside the timed region) and the
          waveform read back to the host every step
  roofline     : dominant kernel (tcgen05 ResBlock pair), CUDA-event device time inside this script
  cpu_baseline : the oracle port of the reference path on the host cores (bounded sample)
``--impl reference`` times that CPU port as the reference arm (the reference is pure Python/PyTorch; there is
no compiled reference to build).
``--impl reference-cuda`` times the same reference ops as plain PyTorch on the B200 (cuDNN/ATen, TF32 default) - the
denominator of BASELINE.json's ">= 5x the reference's PyTorch-CUDA infer" target.
Other BASELINE configs: ``--vocoder nsf-snake-hifigan`` (config 4) and ``--workload flow5`` (config 5: flow-only
microbench, z_p[1,192,100000]; reported in frames/s with the roofline in both FLOP and HBM units).
``--dump-outputs DIR`` writes what the last timed step returned as ``DIR/<name>.npy`` (float32): ``audio`` and ``f0`` of
``infer`` for config 2 / 4, ``z`` of the flow for config 5.  Weights, inputs and noise are seeded, so two builds run with
the same arguments can be compared output for output.
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

METRIC = "44.1 kHz audio samples/sec"
UNIT = "samples/s"
FLOP_PER_SAMPLE_DEC = 1269530.0      # SURVEY §8d: generator FLOPs per output sample
WORKLOAD = "config2: configs/config.json NSF-HiFiGAN 44.1 kHz, ContentVec768 synthetic feats, batch 8 x 10 s (862 frames)"
WORKLOAD_SNAKE = "config4: vdecoder/hifiganwithsnake Generator variant (nsf-snake-hifigan), batch 8 x 10 s (862 frames)"
WORKLOAD_FLOW5 = "config5: flow-only microbench, ResidualCouplingBlock WN stack 192ch x 4 flows, z_p[1,192,100000], g[1,768,1]"
FLOW_FLOP_PER_FRAME = 14.156e6       # SURVEY §8d: 1 415.6 GFLOP at T = 100 000
FLOW_BYTES_PER_FRAME_LAYER = 1152.0  # SURVEY §8d: per coupling layer, read 192 ch + write 96 ch fp32
DUMP_BYTES = 60 << 20                # --dump-outputs: array data in all (< 64 MB with the .npy headers)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cuda"])
    ap.add_argument("--vocoder", default="nsf-hifigan", choices=["nsf-hifigan", "nsf-snake-hifigan"])
    ap.add_argument("--workload", default="config2", choices=["config2", "flow5"])
    ap.add_argument("--precision", default=os.environ.get("SVB_BENCH_PRECISION", "tc"), choices=["tc", "fp32"])
    ap.add_argument("--batch", type=int, default=8, help="utterances per GPU")
    ap.add_argument("--frames", type=int, default=862)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of this project's path (--impl b200)")
    return args


def dump_outputs(out_dir, arrays, seed=0):
    """Write each array as <out_dir>/<name>.npy in float32.  One larger than its share of DUMP_BYTES keeps a fixed, seeded
    subset of its last (time) axis, in order, so that the dumps of two builds still compare element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[-1])
            a = a[..., np.sort(np.random.default_rng(seed).choice(a.shape[-1], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def pick_threads(cfg, sd):
    """MKL-DNN on a 128-core host is slowest with all threads at this problem size; probe a short clip with a few
    thread counts and keep the fastest ("all the host threads it can use")."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import svc_oracle as O
    from sovits_b200 import synth
    ncpu = os.cpu_count() or 1
    cands = sorted({t for t in (8, 16, 32, 64, ncpu) if t <= ncpu})
    c, f0, uv, sid = synth.synth_inputs(cfg, 1, 64)
    noise = synth.draw_noise(1, 64, cfg)
    best, best_t = cands[0], float("inf")
    for t in cands:
        torch.set_num_threads(t)
        O.infer(sd, cfg, c, f0, uv, sid, noise, noice_scale=0.4)
        t0 = time.perf_counter()
        O.infer(sd, cfg, c, f0, uv, sid, noise, noice_scale=0.4)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = t, dt
    return best


def cpu_oracle_rate(cfg, sd, T, runs, warmup, threads, B=1):
    """Oracle port of the reference infer on the host cores, B utterances of T frames per step."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import svc_oracle as O
    from sovits_b200 import synth
    torch.set_num_threads(threads)
    c, f0, uv, sid = synth.synth_inputs(cfg, B, T)
    noise = synth.draw_noise(B, T, cfg)
    times = []
    for i in range(warmup + runs):
        t0 = time.perf_counter()
        O.infer(sd, cfg, c, f0, uv, sid, noise, noice_scale=0.4)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    N = B * T * cfg.hop
    return N / (sum(times) / len(times)), times


def load_cfg(args):
    from sovits_b200.config import load_config
    cfg = load_config()
    if args.vocoder != "nsf-hifigan":
        cfg.vocoder_name = args.vocoder
    return cfg


def run_reference_cuda(args):
    """The reference's own ops (oracle port = F.conv1d / conv_transpose1d / cumsum / sin through cuDNN + ATen, weight norm
    recomputed every forward like the reference) on cuda:0 with torch defaults (TF32 convolutions)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    import sovits_b200  # noqa: F401
    from sovits_b200 import synth
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import svc_oracle as O
    cfg = load_cfg(args)
    dev = torch.device("cuda:0")
    sd = {k: v.to(dev) for k, v in synth.synth_state_dict(cfg).items()}
    B, T = args.batch, args.frames
    c, f0, uv, sid = [t.to(dev) for t in synth.synth_inputs(cfg, B, T)]
    N = T * cfg.hop
    torch.manual_seed(52468)
    noise = {"z_noise": torch.randn(B, cfg.inter_channels, T, device=dev), "rand_ini": torch.rand(B, cfg.n_harmonics, device=dev),
             "har_noise": torch.randn(B, N, cfg.n_harmonics, device=dev)}
    torch.backends.cudnn.benchmark = True
    for _ in range(max(2, args.warmup)):
        O.infer(sd, cfg, c, f0, uv, sid, noise, noice_scale=0.4)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        O.infer(sd, cfg, c, f0, uv, sid, noise, noice_scale=0.4)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    rate = B * N / (ms * 1e-3)
    line = {"impl": "reference-cuda", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(2, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "tf32 convolutions (cuDNN default) / f32", "data": "synthetic",
            "config": {"workload": WORKLOAD if args.vocoder == "nsf-hifigan" else WORKLOAD_SNAKE, "global_batch": B, "frames": T,
                       "samples_per_item": N, "what": "oracle port of the reference ops on cuda:0 (cuDNN + ATen), cudnn.benchmark on"},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_flow5(args):
    """BASELINE config 5: the flow alone (4 coupling layers, reverse) on z_p[1,192,100000], g[1,768,1], mask = ones."""
    import torch
    import sovits_b200  # noqa: F401
    from sovits_b200 import synth
    from sovits_b200.engine import TailEngine
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    cfg = load_cfg(args)
    sd = synth.synth_state_dict(cfg)
    eng = TailEngine(cfg, dev, args.precision)
    eng.load_state_dict(sd)
    T = 100_000
    gen = torch.Generator().manual_seed(1234)
    z_host = torch.randn((1, cfg.inter_channels, T), generator=gen).pin_memory()
    g_host = torch.randn((1, cfg.gin_channels, 1), generator=gen).pin_memory()
    z_p, g = z_host.to(dev), g_host.to(dev)
    out_host = torch.empty((1, cfg.inter_channels, T)).pin_memory()
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def step_dev():
        flush.zero_()
        return eng.flow_reverse(z_p, g)

    def step_e2e():
        flush.zero_()
        o = eng.flow_reverse(z_host.to(dev, non_blocking=True), g_host.to(dev, non_blocking=True))
        out_host.copy_(o, non_blocking=True)

    def timed(fn, steps):
        # the L2 flush is part of the loop but not of the metric: time it alone and subtract
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        for _ in range(steps):
            flush.zero_()
        e[1].record()
        for _ in range(steps):
            last = fn()
        e[2].record()
        torch.cuda.synchronize()
        return (e[1].elapsed_time(e[2]) - e[0].elapsed_time(e[1])) / steps, last

    for _ in range(max(args.warmup, 3)):
        step_dev()
    step_e2e()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = eng.launch_count
    ms, z_last = timed(step_dev, args.steps)
    launches = eng.launch_count - l0
    ms_e2e, _ = timed(step_e2e, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"z": z_last})
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        with open(pk_path) as f:
            peaks = json.load(f)
    tf_peak, hbm_peak = peaks.get("bf16_tflops", 1590.0), peaks.get("hbm_gbs", 6650.0)
    flops = FLOW_FLOP_PER_FRAME * T
    byts = FLOW_BYTES_PER_FRAME_LAYER * 4 * T
    ach_tf = flops / (ms * 1e-3) / 1e12
    ach_gb = byts / (ms * 1e-3) / 1e9
    line = {"metric": "flow frames/sec (config 5 microbench)", "value": T / (ms * 1e-3), "unit": "frames/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands / f32 accumulate (tcgen05)" if args.precision == "tc" else "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_FLOW5, "frames": T, "precision": args.precision,
                       "l2": "160 MB flush buffer written before every step (its time is measured and subtracted)"},
            "e2e": {"value": T / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": z_host.numel() * 4 + g_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4},
            "gpu_launches": int(launches), "ffma_fallbacks_in_tc": eng.fallback_count, "clocks": clocks,
            "roofline": {"kernel": "flow (whole coupling block)", "bound": "tensor", "achieved": ach_tf, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": ach_tf / tf_peak, "traffic": None,
                         "peak_source": "measured burst bf16==fp16 (kernel timed alone)" if peaks else "fallback"},
            "roofline_hbm": {"bound": "hbm", "achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gb / hbm_peak,
                             "algorithmic_bytes": byts, "note": "SURVEY 8d per-layer figure: 1152 B/frame/layer x 4 layers"}}
    print(json.dumps(line), flush=True)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    import sovits_b200  # noqa: F401
    from sovits_b200 import synth
    cfg = load_cfg(args)
    sd = synth.synth_state_dict(cfg)
    cores = pick_threads(cfg, sd)
    # BASELINE.md §3: the CPU arm runs the whole config-2 batch (B utterances x T frames) per step; 1 warm-up
    rate, times = cpu_oracle_rate(cfg, sd, args.frames, args.steps, 1, cores, B=args.batch)
    ms = 1000.0 * sum(times) / len(times)
    sample = (f"each step = the full batch, {args.batch} utterances x {args.frames} frames, on {cores} host threads "
              f"(fastest of 8/16/32/64/{os.cpu_count()} on a short probe); 1 warm-up step")
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD if args.vocoder == "nsf-hifigan" else WORKLOAD_SNAKE, "global_batch": args.batch,
                       "frames": args.frames, "samples_per_item": args.frames * cfg.hop, "parallelism": "host cpu",
                       "note": "rank 0 only; the CPU arm does not scale with --gpus"},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- GPU arm
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.impl == "reference-cuda":
        run_reference_cuda(args)
        return
    if args.workload == "flow5":
        run_flow5(args)
        return
    import torch
    import torch.distributed as dist
    import sovits_b200
    from sovits_b200 import models, synth
    from sovits_b200 import dist as sdist
    from sovits_b200.config import load_config

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    cfg = load_cfg(args)
    snake = args.vocoder != "nsf-hifigan"
    B, T = args.batch, args.frames
    N = T * cfg.hop
    # ---- weights: rank 0 makes them, one NCCL broadcast (the path's only collective, SURVEY §8e)
    if world > 1:
        shapes = synth.param_shapes(cfg)
        sd = synth.synth_state_dict(cfg) if rank == 0 else None
        sd = sdist.broadcast_state_dict(sd, shapes, src=0, device=dev)
    else:
        sd = synth.synth_state_dict(cfg)
    with open(sovits_b200.DEFAULT_CONFIG) as f:
        kw = json.load(f)["model"]
    kw["vocoder_name"] = args.vocoder
    net = models.SynthesizerTrn(1025, 20, **kw).eval()
    net.load_state_dict(sd)
    net = net.to(dev)
    net.set_precision(args.precision)

    # ---- inputs: the global batch, sharded by contiguous blocks
    c, f0, uv, sid = synth.synth_inputs(cfg, B * world, T)
    lo, hi = sdist.shard_range(B * world, rank, world)
    host = [t[lo:hi].contiguous().pin_memory() for t in (c, f0, uv, sid)]
    devin = [t.to(dev) for t in host]
    out_host = torch.empty((B, 1, N), dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in host)
    d2h = out_host.numel() * out_host.element_size()

    def step_dev():
        return net.infer(devin[0], devin[1], devin[2], g=devin[3], noice_scale=0.4)

    from sovits_b200.pipeline import HostPipeline
    pipe = HostPipeline(net, dev, depth=2)

    def step_e2e():
        # the repo's public host-buffer entry point: pinned HOST features in, pinned HOST waveform out; the upload of step
        # i+1 and the read-back of step i-1 overlap the kernels of step i (two copy streams ordered by events)
        return pipe.submit(host[0], host[1], host[2], host[3], noice_scale=0.4)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for _ in range(steps):
            last = fn()
        if isinstance(last, tuple) and isinstance(last[1], torch.cuda.Event):
            torch.cuda.current_stream().wait_event(last[1])      # e2e: the timed region ends when the LAST waveform is on the host
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item()), last

    # clocks are sampled from before the warm-up until after both timed regions (nvidia-smi needs ~0.2 s to produce its first
    # row; the timed regions are only ~0.1 s each), every 100 ms
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_dev()
    for _ in range(max(args.warmup, 3)):     # every pipeline slot allocates its pinned / device buffers on first use
        step_e2e()
    eng = net._b200_engine
    if sampler:
        t_wait = time.time()
        while not sampler.rows and time.time() - t_wait < 3.0:       # make sure the sampler is running before timing starts
            step_dev()
    l0 = eng.launch_count
    ms_dev, (audio_last, f0_last) = timed(step_dev, args.steps)
    launches = (eng.launch_count - l0)
    ms_e2e, _ = timed(step_e2e, args.steps)
    clocks = sampler.stop() if sampler else None

    # ---- roofline: CUDA events around every launch of each kernel family, on the launching stream (svb_profile_enable)
    roof, secondary = None, []
    fb0 = eng.fallback_count
    eng.profile_enable(True)
    nprof = min(args.steps, 3)
    for _ in range(nprof):
        step_dev()
    torch.cuda.synchronize()
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        with open(pk_path) as f:
            peaks = json.load(f)
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "measured (MEASURED_PEAKS.json, sustained bf16==fp16 rate)" if peaks else "fallback"
    traffic_db = {}
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic_db = json.load(open(tpath))
        except Exception:
            traffic_db = {}

    def tensor_entry(name):
        pr = eng.profile_read(name)
        if not pr or pr["ms"] <= 0 or pr["flops"] <= 0:
            return None
        ach = pr["flops"] / (pr["ms"] * 1e-3) / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak,
                "traffic": traffic_db.get(name), "launches_per_step": pr["count"] / nprof, "avg_launch_ms": pr["ms"] / pr["count"],
                "ms_per_step": pr["ms"] / nprof, "peak_source": peak_src,
                "hbm_gbs_algorithmic": pr["bytes"] / (pr["ms"] * 1e-3) / 1e9}

    def hbm_entry(name):
        pr = eng.profile_read(name)
        if not pr or pr["ms"] <= 0 or pr["bytes"] <= 0:
            return None
        a = pr["bytes"] / (pr["ms"] * 1e-3) / 1e9
        return {"kernel": name, "bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s", "frac": a / hbm_peak,
                "traffic": traffic_db.get(name), "launches_per_step": pr["count"] / nprof, "ms_per_step": pr["ms"] / nprof}

    if args.precision == "tc":
        tensor_names = ["pair_tc", "resblock_tc", "ups_tc", "flow_tc", "enc_gemm", "enc_attn"]
        if snake:
            tensor_names.insert(0, "snake_conv")
    else:
        tensor_names = ["pair_f32"]
    entries = [e for e in (tensor_entry(n) for n in tensor_names) if e]
    if entries:
        entries.sort(key=lambda e: -e["ms_per_step"])
        roof = entries[0]                      # the dominant kernel family of this step
        secondary.extend(entries[1:])
    for n in ("nsf_source", "conv_post"):
        e = hbm_entry(n)
        if e:
            secondary.append(e)
    for nm in ("enc_p", "flow", "generator"):
        pp = eng.profile_read(nm)
        if pp:
            secondary.append({"kernel": nm, "ms_per_step": pp["ms"] / max(1, pp["count"])})
    eng.profile_enable(False)
    fallbacks = eng.fallback_count - fb0

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sd_cpu = {k: v.cpu() for k, v in sd.items()}
        cores = pick_threads(cfg, sd_cpu)
        cpu_oracle_rate(cfg, sd_cpu, 64, runs=1, warmup=0, threads=cores, B=1)      # short warm-up
        rate, times = cpu_oracle_rate(cfg, sd_cpu, T, runs=1, warmup=0, threads=cores, B=B)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"oracle port of SynthesizerTrn.infer, the full batch ({B} utterances x {T} frames) once after a short "
                         f"warm-up ({sum(times):.1f} s of CPU work)"}

    if args.dump_outputs:
        outs = {"audio": audio_last, "f0": f0_last}
        if world > 1:                          # every rank holds its block of the global batch
            for k, t in outs.items():
                parts = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(parts, t.contiguous())
                outs[k] = torch.cat(parts)
        if rank == 0:
            dump_outputs(args.dump_outputs, outs)

    if rank == 0:
        total_samples = float(B * world * N)
        value = total_samples * args.steps / (ms_dev * 1e-3)
        e2e_v = total_samples * args.steps / (ms_e2e * 1e-3)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16 operands / f32 accumulate (tcgen05)" if args.precision == "tc" else "f32",
                "data": "synthetic",
                "config": {"workload": WORKLOAD_SNAKE if snake else WORKLOAD, "global_batch": B * world, "frames": T, "samples_per_item": N,
                           "parallelism": f"dp{world}", "precision": args.precision,
                           "l2": "per-step working set (>1 GB of activations) exceeds the 126 MB L2; no explicit flush",
                           "rtf": value / 44100.0},
                "e2e": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "ffma_fallbacks_in_tc": int(fallbacks), "clocks": clocks, "roofline": roof,
                "roofline_secondary": secondary, "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
