#!/usr/bin/env python
"""bench.py -- throughput of the B200-native FastSpeech2 + HiFi-GAN inference path (driver contract in the task brief).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference [...]                          CPU reference arm (oracle port of the reference, host cores)

A "step" is one pass of the hot path over one synthetic batch per GPU: FastSpeech2.forward (phonemes -> mel, including the
single host sync on max(mel_len)) followed by hifigan Generator.forward (mel -> 22.05 kHz fp32 waveform), i.e.
BASELINE.json configs[2]; the mel-only configs[1] number is reported in `extra`.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HOP = 256
FS2_FLOPS = lambda L, T: 4 * L * (5767168 + 1024 * L) + 2360832 * L + 6 * T * (5767168 + 1024 * T) + 8724480 * T  # BASELINE.md section 3
HIFIGAN_FLOPS_PER_FRAME = 614105088


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sampler-period-ms", type=float, default=100.0, help="clock / power sampling period during the timed region (0 = no sampler; diagnosis only)")
    ap.add_argument("--sampler-queries", choices=["all", "clocks"], default="all", help="'clocks': SM clock every sample, power and event reasons every 5th")
    ap.add_argument("--prime", type=int, default=2, help="untimed calls of the timed function right before each timed region (counted in `warmup`)")
    ap.add_argument("--warm-seconds", type=float, default=1.0, help="minimum wall time of the untimed warm-up (steps are added to --warmup until it is reached)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="utterances per GPU per step")
    ap.add_argument("--phonemes", type=int, default=128)
    ap.add_argument("--cpu-sample", type=int, default=2, help="utterances in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cpu-full-batch", action="store_true", help="skip the one cold CPU pass over the whole batch (~45 s)")
    ap.add_argument("--headline-only", action="store_true", help="skip the extra BASELINE.json configs (0, 1, 3, 4-shard)")
    ap.add_argument("--voc-f8-mask", type=int, default=None, help="override hifigan.Generator.f8_mask (A/B of the operand split)")
    ap.add_argument("--voc-fused-mask", type=int, default=None, help="override hifigan.Generator.fused_mask (A/B of the fused ResBlock-group kernel)")
    ap.add_argument("--voc-pair-kmax", type=int, default=None, help="override hifigan.Generator.pair_kmax (largest kernel size run as fused pairs)")
    ap.add_argument("--voc-pair-mask", type=int, default=None, help="override hifigan.Generator.pair_mask (A/B of the per-pair fused launches)")
    ap.add_argument("--fs2-f8", type=int, default=None, choices=[0, 1], help="override the decoder / PostNet operand split (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (rank 0) as DIR/<name>.npy, to compare two builds output for output")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


_NVML_LOOP = r"""
import sys, time
import pynvml as N
N.nvmlInit()
h = N.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
period, light = float(sys.argv[3]) / 1e3, sys.argv[4] == "clocks"
mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
out = open(sys.argv[2], "w")
k = 0
while True:
    t0 = time.perf_counter()
    full = not light or k % 5 == 0          # "clocks": power and event reasons on every 5th sample only
    r = get_reasons(h) if full else -1
    pw = N.nvmlDeviceGetPowerUsage(h) / 1000.0 if full else -1.0
    c = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
    out.write("%d,%d,%d,%.1f,%d,%.2f\n" % (int(sys.argv[1]), c, mx, pw, r, (time.perf_counter() - t0) * 1e3))
    out.flush()
    k += 1
    time.sleep(period)
"""


class ClockSampler:
    """SM clock, power and clock-event reasons every 100 ms while the bench runs.  NVML in a helper process (a handful of light driver
    queries per sample); `nvidia-smi -lms` is the fallback -- its full query every 100 ms was observed to perturb the very region it
    samples (device-timed step up to 1.5x the undisturbed one on some hosts), hence 500 ms there."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index: int, period_ms: float = 100.0, queries: str = "all"):
        self.path = os.path.join(tempfile.mkdtemp(), "clocks.csv")
        self.proc, self.mode = None, None
        phys = gpu_index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                phys = int(vis.split(",")[gpu_index])
            except Exception:
                phys = gpu_index
        try:
            import pynvml  # noqa: F401
            self.proc = subprocess.Popen([sys.executable, "-c", _NVML_LOOP, str(phys), self.path, str(period_ms), queries], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            self.mode = "nvml"
        except Exception:
            try:
                self.f = open(self.path, "w")
                self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "500",
                                              "-i", str(phys)], stdout=self.f, stderr=subprocess.DEVNULL)
                self.mode = "nvidia-smi"
            except Exception:
                self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no sampler available"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons, qms = [], [], [], set(), []
        try:
            lines = open(self.path).read().splitlines()
        except Exception:
            lines = []
        for line in lines:
            parts = [x.strip() for x in line.split(",")]
            try:
                if self.mode == "nvml":
                    if len(parts) < 5:
                        continue
                    sm.append(float(parts[1])); mx.append(float(parts[2]))
                    pw.append(float(parts[3]) if float(parts[3]) >= 0 else (pw[-1] if pw else 0.0))
                    bits = max(int(parts[4]), 0)
                    for b, n in self.BITS.items():
                        if bits & b:
                            reasons.add(n)
                    if len(parts) > 5:
                        qms.append(float(parts[5]))
                else:
                    if len(parts) < 8:
                        continue
                    sm.append(float(parts[1])); mx.append(float(parts[2])); pw.append(float(parts[3]))
                    for n, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], parts[4:8]):
                        if v.lower().startswith("active"):
                            reasons.add(n)
            except ValueError:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "sampler": self.mode}
        busy = [c for c, w in zip(sm, pw) if w > 250.0] or sm          # samples taken under load (idle draw is ~150 W)
        return {"sm_mhz": statistics.median(busy), "sm_mhz_min": min(busy), "sm_mhz_last_samples": busy[-4:], "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "samples_under_load": len(busy),
                "reasons": sorted(reasons), "sampler": self.mode, "query_ms_max": max(qms) if qms else None}


OUTPUT_NAMES = ("mel", "postnet_mel", "p_pred", "e_pred", "log_d_pred", "d_rounded", "src_masks", "mel_masks", "src_lens", "mel_lens")
DUMP_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """Write each array as `directory/<name>.npy`: floating point as float32, integers and masks as float64 (exact).  If they come to
    more than 64 MB in all, every array above 1 MB is cut to the same fraction of its elements, taken evenly spaced over the flattened
    array, so that runs with the same arguments sample the same positions."""
    import numpy as np
    arrays = {k: v.astype(np.float32 if np.issubdtype(v.dtype, np.floating) else np.float64) for k, v in arrays.items()}
    big = {k for k, a in arrays.items() if a.nbytes > 1 << 20}
    room = DUMP_BYTES - 4096 * len(arrays) - sum(a.nbytes for k, a in arrays.items() if k not in big)     # (4 KB per .npy header)
    keep = min(1.0, room / max(1, sum(arrays[k].nbytes for k in big)))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        if name in big and keep < 1.0:
            a = a.reshape(-1)[np.linspace(0, a.size - 1, int(a.size * keep)).astype(np.int64)]
        np.save(os.path.join(directory, name + ".npy"), a)


def workload_config(args, world, frames_per_utt):
    return {"workload": f"configs[2]: LJSpeech config, batch={args.batch}/GPU x {args.phonemes} phonemes -> ~{frames_per_utt:.0f} mel frames "
                        "each (free-running, duration-steered random-init weights), FastSpeech2 + HiFi-GAN end to end, fp32 22.05 kHz waveform",
            "batch_per_gpu": args.batch, "global_batch": args.batch * world, "phonemes": args.phonemes,
            "mel_frames_per_utt": round(frames_per_utt, 1),
            "parallelism": f"dp{world}: utterance shards, weights replicated, no data-path collective; asynchronous NCCL gather of the waveforms to rank 0 only",
            "l2": "per-step activation working set (>2 GB) and weights (196 MB) exceed the 126 MB L2; no explicit flush"}


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_run(args, n_utt, steps, warmup):
    """The reference's CPU implementation of the path (oracle port: the same ATen CPU kernels the reference calls),
    all host threads, on a bounded sample of the workload.  Returns (samples/s, frames/s, seconds/step, cores, frames)."""
    import torch
    from fastspeech2_b200 import configs, synth
    from oracle import fs2_oracle as O
    ncpu = os.cpu_count() or 1
    pc, mc = configs.make_configs("LJSpeech", tempfile.mkdtemp())
    sd = synth.fastspeech2_state_dict(pc, mc, seed=0)
    hsd = O.fold_weight_norm(synth.hifigan_state_dict(configs.HIFIGAN_CONFIG, seed=0))
    spk, texts, lens, L = synth.make_batch(args.batch, args.phonemes, seed=0)
    spk, texts, lens = spk[:n_utt], texts[:n_utt], lens[:n_utt]
    # "all the host threads it can use": more threads than the problem can feed SLOW ATen down on many-core hosts, so the
    # thread count is the best of {all, half, 32, 16} logical CPUs, picked on one short vocoder call (the dominant part).
    cands = sorted({c for c in (ncpu, max(1, ncpu // 2), 32, 16) if c <= ncpu}, reverse=True)
    probe = synth.make_mel(1, 64, seed=0)
    best, cores = None, ncpu
    for c in cands:
        torch.set_num_threads(c)
        O.hifigan_forward(hsd, probe)
        t0 = time.perf_counter()
        O.hifigan_forward(hsd, probe)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, c
    torch.set_num_threads(cores)

    def step():
        out = O.fastspeech2_forward(sd, spk, texts, lens, L)
        t1 = time.perf_counter()
        wav = O.hifigan_forward(hsd, out[1].transpose(1, 2))
        return int(out[9].sum()), t1, wav

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    frames = 0
    fs2_s = 0.0
    for _ in range(steps):
        ts = time.perf_counter()
        f, t1, _ = step()
        fs2_s += t1 - ts
        frames += f
    dt = time.perf_counter() - t0
    return frames * HOP / dt, frames / max(fs2_s, 1e-9), dt / steps, cores, frames // steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = max(1, min(args.cpu_sample, args.batch))
    sps, fps, sec, cores, frames = cpu_reference_run(args, n, args.steps, min(args.warmup, 1))
    line = {"impl": "reference", "metric": "audio_samples_per_s", "value": sps, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, 1, frames / n),
            "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port",
                             "sample": f"{n} of the {args.batch} utterances per step ({frames} mel frames), oracle port of the reference "
                                       "(same ATen CPU kernels), fp32, best of {all, half, 32, 16} host threads"},
            "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mel_frames_per_s": sps / HOP,
            "extra": {"mel_frames_per_s_fastspeech2_only": fps}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- GPU arm
def fs2_flops_batch(src_lens, mel_lens):
    """Algorithmic FastSpeech2 FLOPs of a batch with valid lengths (BASELINE.md section 3, per utterance)."""
    return float(sum(FS2_FLOPS(int(l), int(t)) for l, t in zip(src_lens, mel_lens)))


def run_ours(args):
    import contextlib
    import ctypes as C
    import io

    import torch
    import torch.distributed as dist

    from fastspeech2_b200 import _lib, configs, synth
    from fastspeech2_b200.hifigan import AttrDict, Generator
    from fastspeech2_b200.model import FastSpeech2
    from fastspeech2_b200.parallel import Rank0Gather

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=datetime.timedelta(seconds=180))
    lib = _lib.lib()
    pk = peaks()
    scratch = tempfile.mkdtemp()

    def acoustic(dataset):
        pc, mc = configs.make_configs(dataset, scratch)
        model = FastSpeech2(pc, mc)
        model.load_state_dict(synth.fastspeech2_state_dict(pc, mc, seed=0))
        if args.fs2_f8 is not None:
            f8_bits = _lib.TC_DECODER_F8 | _lib.TC_POSTNET_F8
            model.tc_mask = (model.tc_mask & ~f8_bits) | (f8_bits if args.fs2_f8 else 0)
        return model.to(dev).eval()

    model = acoustic("LJSpeech")
    voc = Generator(AttrDict(configs.HIFIGAN_CONFIG))
    voc.load_state_dict(synth.hifigan_state_dict(configs.HIFIGAN_CONFIG, seed=0))
    if args.voc_f8_mask is not None:
        voc.f8_mask = args.voc_f8_mask
    if args.voc_fused_mask is not None:
        voc.fused_mask = args.voc_fused_mask
    if args.voc_pair_mask is not None:
        voc.pair_mask = args.voc_pair_mask
    if args.voc_pair_kmax is not None:
        voc.pair_kmax = args.voc_pair_kmax
    voc.eval()
    with contextlib.redirect_stdout(io.StringIO()):
        voc.remove_weight_norm()
    voc.to(dev)

    def inputs(batch, phonemes, seed, n_speakers=1, min_len=None):
        spk, texts, lens, L = synth.make_batch(batch, phonemes, seed=seed, n_speakers=n_speakers, min_len=min_len)
        host = tuple(t.pin_memory() for t in (spk, texts, lens))
        return host, tuple(t.to(dev) for t in host), L

    def timed(fn, steps, collective=True, prime=None):
        """`steps` calls of fn bracketed by barrier + synchronize, CUDA events on the launch stream, max over ranks.  `prime` untimed
        calls of the same fn run right before the opening barrier (they are warm-up steps: the caller adds them to `warmup`), so that
        the timed region starts from the loop's own steady state and not after a pause of host-side bookkeeping."""
        prime = args.prime if prime is None else prime
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]      # one event record per step: the per-step spread, for diagnosis
        gc_was = gc.isenabled()
        gc.collect()
        gc.disable()                             # (as timeit does) no cyclic-GC pause on the launching thread inside the timed region
        last = None
        for _ in range(prime):
            last = None
            last = fn()
        if world > 1 and collective:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.fs2_kernel_launch_count()
        mallocs0 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0)
        host = [time.perf_counter()]
        e0.record()
        for i in range(steps):
            last = None                          # at most one previous result set alive, as in the warm-up
            last = fn()
            marks[i].record()
            host.append(time.perf_counter())
        e1.record()
        torch.cuda.synchronize()
        if gc_was:
            gc.enable()
        if world > 1 and collective:
            dist.barrier()
        each = [a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks)]
        per = sorted(each)
        slow = each.index(per[-1])
        timed.spread = {"min": round(per[0], 3), "median": round(per[len(per) // 2], 3), "max": round(per[-1], 3), "slowest_step_index": slow,
                        "slowest_step_host_ms": round((host[slow + 1] - host[slow]) * 1e3, 3),
                        "cudaMallocs_in_region": int(torch.cuda.memory_stats(dev).get("num_device_alloc", 0) - mallocs0)}
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        launches = torch.tensor([lib.fs2_kernel_launch_count() - n0], device=dev, dtype=torch.int64)
        if world > 1 and collective:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(launches, op=dist.ReduceOp.SUM)
        return ms.item(), int(launches.item()), last

    def all_sum(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ------------------------------------------------------------------ headline: configs[2], one micro-batch of `--batch` utterances per GPU per step
    (spk_h, texts_h, lens_h), (spk, texts, lens), L = inputs(args.batch, args.phonemes, seed=rank)
    gather = Rank0Gather() if world > 1 else None

    def step_local():                               # no collectives: safe to run on a single rank
        out = model(spk, texts, lens, L)
        wav = voc(out[1].transpose(1, 2))
        return out, wav

    def step_device():
        out, wav = step_local()
        if gather is not None:
            gather.submit(wav[:, 0], out[9])         # async, rank 0 receives; overlaps the next step
        return out, wav

    wav_host = {}

    def step_e2e():
        s_d, t_d, l_d = spk_h.to(dev, non_blocking=True), texts_h.to(dev, non_blocking=True), lens_h.to(dev, non_blocking=True)
        out = model(s_d, t_d, l_d, L)
        wav = voc(out[1].transpose(1, 2))
        if gather is not None:
            gather.submit(wav[:, 0], out[9])
        key = tuple(wav.shape)
        if key not in wav_host:
            wav_host[key] = torch.empty(wav.shape, dtype=wav.dtype).pin_memory()
        wav_host[key].copy_(wav, non_blocking=True)
        mel_lens_host = out[9].cpu()          # the step's result lengths (also the stream sync for the waveform copy)
        return out, wav, mel_lens_host

    # Warm-up: at least `--warmup` (>= 3) steps AND at least ~1 s of work, so that the first timed region does not sit on the clock /
    # power ramp of a cold GPU (observed: a region timed right after 3 steps of a fresh process can read 20 % slow).  The clock
    # sampler starts before the warm-up so that its own start-up is not inside the timed region either.
    sampler = ClockSampler(local, args.sampler_period_ms, args.sampler_queries) if rank == 0 and args.sampler_period_ms > 0 else None
    warm_steps = max(args.warmup, 3)
    out, wav = step_device()                          # first call: one-time weight packing / workspace allocation
    torch.cuda.synchronize()
    t_w0 = time.perf_counter()
    for _ in range(warm_steps - 1):
        out, wav = step_device()
        torch.cuda.synchronize()
    dt = time.perf_counter() - t_w0
    extra = torch.tensor([min(200, max(0, int((args.warm_seconds - dt) / max(dt / (warm_steps - 1), 1e-4)) + 1)) if dt < args.warm_seconds else 0], device=dev)
    if world > 1:                                     # every rank runs the same number of (collective-carrying) steps
        dist.all_reduce(extra, op=dist.ReduceOp.MAX)
    for _ in range(int(extra.item())):
        out, wav = step_device()
    warm_steps += int(extra.item())
    if gather is not None:
        gather.flush()
    torch.cuda.synchronize()
    frames_step = int(all_sum(float(out[9].sum().item())))          # all ranks, one step
    samples_step = frames_step * HOP
    fs2_flop_step = all_sum(fs2_flops_batch(lens_h.tolist(), out[9].tolist()))
    d2h = int(wav.numel() * 4 + out[9].numel() * 8)
    del out, wav                                      # (timed() keeps at most one previous result set alive, like the warm-up loop)

    # N > 1: the asynchronous gather of the last step completes inside the timed region (flush before the closing event)
    ms_total, launches, last = timed(step_device, args.steps) if gather is None else _timed_with_flush(timed, step_device, gather, args.steps, args.prime)
    clocks = sampler.stop() if sampler else None
    spread_device = dict(timed.spread)
    if args.dump_outputs and rank == 0:
        out, wav = last
        dump_outputs(args.dump_outputs, {**{n: t.cpu().numpy() for n, t in zip(OUTPUT_NAMES, out)}, "wav": wav.cpu().numpy()})
        del out, wav
    del last
    value = samples_step * args.steps / (ms_total * 1e-3)

    ms_mel, _, _ = timed(lambda: model(spk, texts, lens, L), args.steps)
    mel_fps = frames_step * args.steps / (ms_mel * 1e-3)

    ms_e2e, _, _ = timed(step_e2e, args.steps) if gather is None else _timed_with_flush(timed, step_e2e, gather, args.steps, args.prime)
    e2e_value = samples_step * args.steps / (ms_e2e * 1e-3)
    spread_e2e = dict(timed.spread)
    h2d = spk_h.numel() * 8 + texts_h.numel() * 8 + lens_h.numel() * 8

    def class_profile(fn):
        """One extra, untimed pass with CUDA events around every launch: per-class ms / flops / launches (fs2_profile_begin/end)."""
        lib.fs2_profile_begin()
        fn()
        torch.cuda.synchronize()
        n = _lib.PROF_CLASSES
        ms = (C.c_double * n)(); fl = (C.c_double * n)(); cnt = (C.c_int64 * n)()
        lib.fs2_profile_end(ms, fl, cnt)
        return list(ms), list(fl), list(cnt)

    def tensor_roofline(fn, ms_step):
        """Roofline of the dominant kernel class = the tcgen05 kernels (implicit-GEMM conv1d + fused ResBlock group).  Bracketing every
        launch with two events costs a bubble per launch, so the class's duration inside the TIMED region is its share of the
        bracketed pass times the event-timed step; the raw bracketed figure is reported next to it."""
        ms, fl, cnt = class_profile(fn)
        share = ms[0] / max(sum(ms), 1e-9)
        cls_ms = share * ms_step
        achieved = fl[0] / (cls_ms * 1e-3) / 1e12 if cls_ms > 0 else 0.0
        return {"achieved": achieved, "frac": achieved / pk["tflops_sustained"], "share_of_step": share, "launches_per_step": int(cnt[0]),
                "avg_launch_ms": cls_ms / max(int(cnt[0]), 1), "algorithmic_tflop_per_step": fl[0] / 1e12,
                "achieved_event_bracketed": fl[0] / (ms[0] * 1e-3) / 1e12 if ms[0] > 0 else 0.0,
                "other_classes_ms": {"attention": ms[1], "layernorm": ms[2], "other": ms[3], "conv1d_fp32_cuda_cores": ms[4]},
                "other_classes_launches": {"attention": int(cnt[1]), "layernorm": int(cnt[2]), "other": int(cnt[3]), "conv1d_fp32_cuda_cores": int(cnt[4])}}

    roof = None
    if rank == 0:
        r = tensor_roofline(step_local, ms_total / args.steps)
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02", "step_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("tcgen05_class_dram_bytes_per_launch"), tj.get("source")
        roof = {"kernel": "tcgen05 kernel class: conv_tc_kernel (implicit-GEMM conv1d: FFT-block projections / conv-FFN of encoder and decoder, "
                          "variance predictors, PostNet, HiFi-GAN convs) + resstack_kernel (fused ResBlock group / pairs); attention, layer norm "
                          "and the few fp32 CUDA-core launches are separate classes (other_classes_ms) and NOT counted",
                "bound": "tensor", "achieved": r["achieved"], "peak": pk["tflops_sustained"], "unit": "TFLOP/s", "frac": r["frac"],
                "peak_source": pk["source"] + ", bf16 sustained (kernels timed inside a long step); two MMAs per useful MMA-equivalent in the "
                                              "f16+f8 operand split, three in the split-fp16 one: 0.50 / 0.33 of the peak is the ceiling",
                "traffic": traffic, "traffic_source": traffic_src,
                "timing": "class share from one untimed step with CUDA events around every launch x the event-timed step", **{k: v for k, v in r.items() if k not in ("achieved", "frac")}}

    # ------------------------------------------------------------------ the other BASELINE.json configs (N = 1: all of them; N > 1: the configs[4] shard)
    extra_cfg = {}

    def measure(name, workload, fn, flops_fn, steps, frames_fn, with_voc):
        for _ in range(3):
            o = fn()
        torch.cuda.synchronize()
        ms, _, o = timed(fn, steps)
        frames = all_sum(frames_fn(o))
        ms_step = ms / steps
        flop = all_sum(flops_fn(o))
        d = {"workload": workload, "ms_per_step": ms_step, "steps": steps, "mel_frames_per_s": frames / (ms_step * 1e-3),
             "useful_tflops": flop / (ms_step * 1e-3) / 1e12, "frac_of_bf16_sustained_peak": flop / (ms_step * 1e-3) / 1e12 / pk["tflops_sustained"] / world}
        if with_voc:
            d["audio_samples_per_s"] = frames * HOP / (ms_step * 1e-3)
        extra_cfg[name] = d

    if not args.headline_only:
        B4 = 64
        (_, _, lens4_h), (spk4, texts4, lens4), L4 = inputs(B4, args.phonemes, seed=100 + rank)

        def step_c4():
            o = model(spk4, texts4, lens4, L4)
            w = voc(o[1].transpose(1, 2))
            return o

        measure("configs[4]_shard", f"LJSpeech, {B4} utterances per GPU x {args.phonemes} phonemes (one GPU's shard of the batch-512 job; x{world} GPUs here), "
                                    "FastSpeech2 + HiFi-GAN", step_c4,
                lambda o: fs2_flops_batch(lens4_h.tolist(), o[9].tolist()) + HIFIGAN_FLOPS_PER_FRAME * float(o[9].sum().item()),
                max(2, args.steps // 2), lambda o: float(o[9].sum().item()), True)
        del spk4, texts4, lens4
    if not args.headline_only and world == 1:
        (_, _, lens1_h), (spk1, texts1, lens1), L1 = inputs(1, args.phonemes, seed=7)

        def step_c0():
            o = model(spk1, texts1, lens1, L1)
            voc(o[1].transpose(1, 2))
            return o

        measure("configs[0]", f"LJSpeech, batch=1 x {args.phonemes} phonemes, FastSpeech2 + HiFi-GAN (latency case; the reference's CPU-runnable config)", step_c0,
                lambda o: fs2_flops_batch(lens1_h.tolist(), o[9].tolist()) + HIFIGAN_FLOPS_PER_FRAME * float(o[9].sum().item()),
                args.steps * 2, lambda o: float(o[9].sum().item()), True)
        extra_cfg["configs[1]"] = {"workload": f"LJSpeech, batch={args.batch} x {args.phonemes} phonemes, FastSpeech2 only (mel, no vocoder)",
                                   "ms_per_step": ms_mel / args.steps, "steps": args.steps, "mel_frames_per_s": mel_fps,
                                   "useful_tflops": fs2_flop_step / (ms_mel / args.steps * 1e-3) / 1e12,
                                   "frac_of_bf16_sustained_peak": fs2_flop_step / (ms_mel / args.steps * 1e-3) / 1e12 / pk["tflops_sustained"]}
        libri = acoustic("LibriTTS")
        (_, _, lens3_h), (spk3, texts3, lens3), L3 = inputs(64, 256, seed=11, n_speakers=904, min_len=64)

        def step_c3():
            return libri(spk3, texts3, lens3, L3)

        measure("configs[3]", "LibriTTS multi-speaker (904-speaker embedding), batch=64, mixed 64-256 phonemes with padding masks, FastSpeech2 only; "
                              "frames = VALID mel frames", step_c3,
                lambda o: fs2_flops_batch(lens3_h.tolist(), o[9].tolist()), max(2, args.steps // 2), lambda o: float(o[9].sum().item()), False)
        extra_cfg["configs[3]"]["padded_frames_per_step"] = int(step_c3()[0].shape[0] * step_c3()[0].shape[1])
        del libri

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            n = max(1, min(args.cpu_sample, args.batch))
            sps, fps, sec, cores, frames = cpu_reference_run(args, n, 1, 1)
            cpu = {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port",
                   "sample": f"{n} of the {args.batch} utterances ({frames} mel frames), 1 warm-up + 1 timed pass ({sec:.1f} s), oracle port of "
                             "the reference (same ATen CPU kernels), fp32, best of {all, half, 32, 16} host threads",
                   "mel_frames_per_s_fastspeech2_only": fps}
            if not args.no_cpu_full_batch:
                sps_f, fps_f, sec_f, cores_f, frames_f = cpu_reference_run(args, args.batch, 1, 0)
                cpu["full_batch_once"] = {"value": sps_f, "unit": "samples/s", "utterances": args.batch, "mel_frames": frames_f, "seconds": sec_f,
                                          "cores": cores_f, "note": "the WHOLE configs[2] batch, one cold pass (no warm-up), same port"}
        line = {"metric": "audio_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": warm_steps + args.prime, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(args, world, frames_step / (args.batch * world)),
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": launches,
                "mel_frames_per_s": frames_step * args.steps / (ms_total * 1e-3),          # the other half of BASELINE.json's metric, same timed region
                "roofline": roof, "cpu_baseline": cpu,
                "extra": {"step_ms_spread": {"device_timed": spread_device, "e2e": spread_e2e, "note": "this rank's per-step CUDA-event durations"},
                          "mel_frames_per_s": frames_step * args.steps / (ms_total * 1e-3),
                          "fastspeech2_only_mel_frames_per_s": mel_fps, "fastspeech2_only_ms_per_step": ms_mel / args.steps,
                          "algorithmic_tflop_per_step": (fs2_flop_step + HIFIGAN_FLOPS_PER_FRAME * frames_step) / 1e12,
                          "useful_tflops_whole_step": (fs2_flop_step + HIFIGAN_FLOPS_PER_FRAME * frames_step) / (ms_total / args.steps * 1e-3) / 1e12,
                          "configs": extra_cfg,
                          "operand_split": {"vocoder_f8_mask": int(voc.f8_mask), "vocoder_fused_stage_mask": int(voc.fused_mask), "vocoder_pair_stage_mask": int(voc.pair_mask),
                                            "fs2_tc_mask": int(model.tc_mask)},
                          "build": lib.fs2_build_info().decode()}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _timed_with_flush(timed, step, gather, steps, prime):
    """Timed region for N > 1: the asynchronous rank-0 gather of the LAST step must complete inside the region."""
    count = {"i": 0}

    def fn():
        r = step()
        count["i"] += 1
        if count["i"] == steps + prime:         # (timed() first makes `prime` untimed calls)
            gather.flush()
        return r
    return timed(fn, steps)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.gpus > 1 and "RANK" not in os.environ:
        port = 29000 + os.getpid() % 1000
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    run_ours(args)


if __name__ == "__main__":
    main()
