#!/usr/bin/env python
"""bench.py -- audio-seconds per second of ToneColorConverter.convert on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 32] [--secs 10] [--impl native|reference]

A "step" is one pass of the hot path over one batch of synthetic utterances.  The default
workload is BASELINE.json configs[1]: batch 32 x 10 s clips at 22.05 kHz on one B200, in the
default arithmetic mode (--precision f16x3: split-precision fp16 tensor-core convolutions, fp32-grade
results -- stricter than the config's "fp16"; fp32 = CUDA cores only, f16 = single pass).  The
other modes are timed briefly in the same run and reported under "modes_audio_s_per_s".  For N > 1 launch under torchrun: one rank per
GPU, every rank converts its own `batch` clips (weak scaling, no data-path collective; NCCL only
broadcasts the checkpoint and, in the end-to-end leg, gathers the output waveforms on rank 0).

One JSON line on stdout (rank 0):
  value      device-resident: waveforms already in HBM -> ovc_convert_waveform (STFT + voice_conversion), CUDA events
  e2e        HOST numpy waveforms in, HOST numpy waveforms out, all inside the timed region, through
             openvoice_b200.distributed.convert_sharded_async at every N (each rank stages, uploads from pinned memory
             and converts its shard; N > 1: results gathered GPU-to-GPU over NCCL; rank 0 downloads; one call in flight
             behind the current one, so a step's download overlaps the next step's kernels).  At N = 1 the synchronous
             ToneColorConverter.convert_batch is timed beside it (`e2e_convert_batch`)
  roofline   generator ResBlock conv family (90 % of the FLOPs), timed live with CUDA events around every launch:
             ALGORITHMIC TFLOP/s (2*MAC of the reference's convs, no credit for the 3 split-precision passes) over
             the measured dense fp16/bf16 tensor peak; pipe occupancy, HBM figures and a per-kernel table beside it
  cudnn_baseline  the reference's own torch graph (oracle port, F.conv1d -> cuDNN) on this GPU, TF32 on and off
  cpu_baseline  the oracle port of the reference's CPU path on this box's host cores (N=1 only)
--impl reference times that CPU path alone (the reference arm).

--dump-outputs DIR writes what the last timed device-resident step returned (rank 0's o_hat and frames) as DIR/<name>.npy,
so that two builds run with the same arguments, hence on the same seeded inputs, can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree as it found it (which may be read-only)

SR = 22050
HOP = 256
GFLOP_PER_FRAME = 0.65766          # SURVEY.md section 8d: 657.66 MFLOP per spectrogram frame
FFMA_PEAK_TFLOPS = 74.4            # nominal 148 SM x 128 lanes x 2 x 1.965 GHz (fallback)
DUMP_BYTES = 60_000_000            # --dump-outputs: o_hat + frames written whole up to this size ...
DUMP_SAMPLE = 4_000_000            # ... else this many seeded samples of o_hat (values + float64 indices: 48 MB)


def ffma_peak():
    """fp32 FMA peak of this pool's B200s as tools/ffma_bench.cu measured it (profiles/r02_ffma_peak.json), else nominal"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_ffma_peak.json")))
        return float(d["ffma_peak_tflops"]), "measured (tools/ffma_bench.cu, profiles/r02_ffma_peak.json)"
    except Exception:
        return FFMA_PEAK_TFLOPS, "nominal 148 SM x 128 lanes x 2 x 1.965 GHz"


def synth_wave(i, secs):
    rng = np.random.default_rng(1000 + i)
    L = int(round(secs * SR))
    return (0.5 * (2.0 * rng.random(L, dtype=np.float32) - 1.0)).astype(np.float32)


def synth_se(i, base):
    import torch
    return 0.1 * torch.randn(1, 256, 1, generator=torch.Generator().manual_seed(base + i))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            self.path = tempfile.mktemp(suffix=".csv")
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, mx = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 7:
                    continue
                sm.append(float(p[0]))
                mx = float(p[1])
                for n, v in zip(names, p[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def host_cores():
    """Usable host cores: scheduler affinity, capped by the cgroup CPU quota (a container on a big
    host reports every core in os.cpu_count(); oversubscribing MKLDNN with them is far slower)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return max(1, min(n, 64))


def pin_to_gpu_numa(local):
    """Multi-rank runs: keep this rank's host threads (staging copies, NCCL proxy) on the NUMA node its GPU hangs off.
    Best effort: returns a short description, or None when sysfs does not say."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return f"numa node {node}, {len(cpus)} cpus"
    except Exception:
        return None


def cpu_reference_throughput(n_clips, secs, threads=None, budget_s=25.0):
    """Time the oracle port of the reference's convert() arithmetic (spectrogram + voice_conversion,
    batch 1 per utterance like openvoice/api.py:141-155) on the host cores."""
    import torch
    from oracle import vc_oracle as O
    threads = threads or host_cores()
    torch.set_num_threads(threads)
    sd = O.synthetic_state_dict(1234)
    waves = [torch.from_numpy(synth_wave(i, secs)) for i in range(n_clips)]
    done = []
    with torch.no_grad():
        O.convert_waveform(sd, waves[0][: SR], synth_se(0, 2000), synth_se(0, 3000), None, 0.3)   # warm-up
        t0 = time.perf_counter()
        for i, w in enumerate(waves):
            T = w.shape[0] // HOP
            noise = torch.randn(1, 192, T)
            O.convert_waveform(sd, w, synth_se(i, 2000), synth_se(i, 3000), noise, 0.3)
            done.append(w)
            if time.perf_counter() - t0 > budget_s:   # bounded sample
                break
        dt = time.perf_counter() - t0
    audio_s = sum((w.shape[0] // HOP) * HOP for w in done) / SR
    return audio_s / dt, dt, torch.get_num_threads(), len(done)


def workload_config(B, secs, world):
    """the `config` object both arms report: BASELINE.json configs[1] unless --batch / --secs say otherwise"""
    T = int(round(secs * SR)) // HOP
    return {"workload": f"ToneColorConverter.convert_batch, batch {B} x {secs:g} s clips @ {SR} Hz per GPU "
                        "(BASELINE configs[1]), seeded synthetic checkpoint, tau 0.3, in-kernel Philox noise",
            "batch_per_gpu": B, "global_batch": B * world, "secs": secs, "frames": T}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_clips = max(1, min(args.batch, args.ref_clips))
    times, vals = [], []
    val = None
    for s in range(args.warmup + args.steps):
        v, dt, threads, done = cpu_reference_throughput(n_clips, args.secs)
        if s >= args.warmup:
            times.append(dt)
            vals.append(v)
            val = float(np.mean(vals))
    sample = f"{n_clips} x {args.secs:g} s clips per step, batch 1 each (convert semantics), fp32, torch CPU ({threads} threads)"
    line = {
        "impl": "reference", "metric": "audio_seconds_per_second", "value": val, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args.batch, args.secs, args.gpus),
                       sample=f"each step converts {n_clips} of the {args.batch} clips (bounded sample; the metric is a rate)",
                       parallelism=f"{threads} host threads", e2e_api="oracle port of ToneColorConverter.convert (torch CPU)"),
        "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_REAL_STDOUT = None


def emit(line):
    """The one JSON line goes to the real stdout; everything else any library prints on fd 1
    (e.g. NCCL's version banner) has been redirected to stderr by quiet_stdout()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def quiet_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def cudnn_reference(B, secs, steps=3):
    """SURVEY section 8d's third column: the reference's own PyTorch graph on THIS GPU (cuDNN convolutions; the oracle
    port issues the same F.conv1d / conv_transpose1d calls as openvoice/models.py), batch B x secs padded batch,
    explicit noise, TF32 on (torch's cudnn default) and off.  Never part of the product path."""
    import torch
    from oracle import vc_oracle as O
    dev = "cuda"
    sd = {k: v.to(dev) for k, v in O.synthetic_state_dict(1234).items()}
    wav = torch.from_numpy(np.stack([synth_wave(i, secs) for i in range(B)])).to(dev)
    T = wav.shape[1] // HOP
    gs = torch.cat([synth_se(i, 2000) for i in range(B)]).to(dev)
    gt = torch.cat([synth_se(i, 3000) for i in range(B)]).to(dev)
    lengths = torch.full((B,), T, dtype=torch.int64, device=dev)
    noise = torch.randn(B, 192, T, device=dev)
    out = {}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        torch.backends.cudnn.benchmark = True
        for tf32 in (True, False):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32

            def step():
                with torch.no_grad():
                    spec = O.spectrogram(wav)
                    return O.voice_conversion(sd, spec, lengths, gs, gt, noise, 0.3)[0]
            step(); step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                o = step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out["tf32_on" if tf32 else "tf32_off"] = {"audio_s_per_s": B * T * HOP / SR / (ms * 1e-3), "ms_per_step": ms}
            del o
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
        torch.cuda.empty_cache()
    out["what"] = (f"oracle port of the reference graph (F.conv1d -> cuDNN, weight-norm folded every call like the reference), "
                   f"padded batch {B} x {secs:g} s, torch {torch.__version__}, cudnn.benchmark on, CUDA events, {steps} steps")
    return out


def dump_outputs(path, o_hat, frames):
    """What the last timed step returned: path/o_hat.npy (float32 [B, hop * T]) and path/frames.npy (float64 [B]).
    An o_hat too large for DUMP_BYTES is written as a fixed, seeded sample of DUMP_SAMPLE of its elements instead:
    o_hat.npy holds the values, o_hat_index.npy their flat indices (float64, exact below 2**53)."""
    os.makedirs(path, exist_ok=True)
    o = o_hat.cpu().numpy()
    out = {"frames": frames.cpu().numpy().astype(np.float64)}
    if o.nbytes + out["frames"].nbytes <= DUMP_BYTES:
        out["o_hat"] = o
    else:
        idx = np.sort(np.random.default_rng(0).choice(o.size, DUMP_SAMPLE, replace=False))
        out["o_hat"] = o.reshape(-1)[idx]
        out["o_hat_index"] = idx.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def latency_config1(conv, secs_list=(3.0, 10.0), iters=20):
    """BASELINE configs[0] on the GPU: ToneColorConverter.convert of ONE clip (batch 1), host array in, host array
    out, median wall time."""
    import torch
    out = {}
    src, tgt = synth_se(0, 2000), synth_se(0, 3000)
    for secs in secs_list:
        w = synth_wave(0, secs)
        for _ in range(3):
            conv.convert(w, src, tgt, tau=0.3)
        ts = []
        for _ in range(iters):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            conv.convert(w, src, tgt, tau=0.3)
            ts.append((time.perf_counter() - t0) * 1e3)
        ms = float(np.median(ts))
        out[f"{secs:g}s"] = {"ms": ms, "audio_s_per_s": (len(w) // HOP * HOP / SR) / (ms * 1e-3),
                             "launches": int(conv.model.native.last_launch_count)}
    out["what"] = "ToneColorConverter.convert, batch 1, host numpy in/out, median of %d wall-clock calls" % iters
    return out


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--secs", type=float, default=10.0)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--ref-clips", type=int, default=4, help="clips per step of the CPU reference arm")
    ap.add_argument("--cpu-clips", type=int, default=8, help="clips in the cpu_baseline sample of the native arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--precision", default=os.environ.get("OVC_PRECISION", "f16x3"), choices=["fp32", "f16x3", "f16"],
                    help="conv arithmetic: f16x3 = split-precision fp16 tensor cores (default, fp32-grade), "
                         "fp32 = CUDA-core FFMA2, f16 = single-pass fp16 (11-bit operands, the reference's own GPU default class)")
    ap.add_argument("--wide-variant", type=int, default=None, help="tiling of the 128-column tensor-core kernel (ovc_set_option)")
    ap.add_argument("--no-config3", action="store_true", help="skip the BASELINE config-3 side measurement (V1 TTS + convert, batch 16)")
    ap.add_argument("--no-modes", action="store_true", help="skip the short side measurements of the other precisions")
    ap.add_argument("--no-cudnn", action="store_true", help="skip the reference-on-this-GPU (PyTorch / cuDNN) column")
    ap.add_argument("--no-sides", action="store_true", help="skip every side measurement (modes, config1/3/4, cudnn, cpu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed device-resident step returned (o_hat, frames) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs: only the native arm has a device-resident timed path")
    if args.impl == "reference":
        return run_reference(args)
    if args.no_sides:
        args.no_config3 = args.no_modes = args.no_cudnn = args.no_cpu_baseline = True

    import torch
    import torch.distributed as dist
    from oracle import vc_oracle as O          # synthetic checkpoint recipe + cpu_baseline / cudnn_baseline only
    from openvoice_b200 import distributed as D
    from openvoice_b200.api import ToneColorConverter

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path)"
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    numa = pin_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun"

    # ---- model: rank 0 owns the checkpoint, NCCL broadcasts it (north_star)
    sd = D.broadcast_state_dict(O.synthetic_state_dict(1234) if rank == 0 else None, device=dev)

    def make_converter(zero_g=False):
        import copy
        hp = copy.deepcopy(O.DEFAULT_HPARAMS)
        hp["model"]["zero_g"] = zero_g
        with tempfile.TemporaryDirectory() as td:
            cfg = os.path.join(td, "config.json")
            json.dump(hp, open(cfg, "w"))
            cv = ToneColorConverter(cfg, device=dev, enable_watermark=False, precision=args.precision)
        cv.model.load_state_dict(sd)
        if args.wide_variant is not None:
            cv.model.native.set_option("wide_variant", args.wide_variant)
        return cv

    conv = make_converter()
    B, secs = args.batch, args.secs
    waves = [synth_wave(rank * B + i, secs) for i in range(B)]
    L = len(waves[0])
    T = L // HOP
    audio_s_step = B * T * HOP / SR
    src = torch.cat([synth_se(rank * B + i, 2000) for i in range(B)]).to(dev)
    tgt = torch.cat([synth_se(rank * B + i, 3000) for i in range(B)]).to(dev)
    wav_dev = torch.from_numpy(np.stack(waves)).to(dev)
    wav_len = torch.full((B,), L, dtype=torch.int64, device=dev)

    out_dev = torch.empty(B, T * HOP, device=dev)
    frames_dev = torch.empty(B, dtype=torch.int64, device=dev)

    def device_step(seed):      # every buffer at a stable address: the library replays the call from a CUDA graph
        return conv.model.native.convert_waveform(wav_dev, wav_len, src, tgt, tau=0.3, seed=seed, out=out_dev, frames_out=frames_dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident leg
    for s in range(args.warmup):
        device_step(s)
    native = conv.model.native
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        last = device_step(1000 + s)
    e1.record()
    barrier()
    ms_dev = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches_per_call = native.last_launch_count
    if args.dump_outputs and rank == 0:     # before the legs below reuse the output buffers
        dump_outputs(args.dump_outputs, *last)

    # ---- per-kernel leg (roofline): the same steps again with CUDA events around every conv launch
    native.profile_enable(True)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for s in range(args.steps):
        device_step(2000 + s)
    p1.record()
    torch.cuda.synchronize()
    ms_prof_step = p0.elapsed_time(p1) / args.steps
    detail = native.profile_detail(1 << 16)
    prof = native.profile_read()
    native.profile_enable(False)

    # ---- the other arithmetic modes, short (2 timed steps), device-resident only
    modes = {}
    if not args.no_modes:
        for mode in ("fp32", "f16x3", "f16"):
            if mode == args.precision:
                continue
            native.set_precision(mode)
            device_step(1)
            barrier()
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            m0.record()
            device_step(2); device_step(3)
            m1.record()
            barrier()
            modes[mode] = world * audio_s_step / (max_over_ranks(m0.elapsed_time(m1)) / 2 * 1e-3)
        native.set_precision(args.precision)

    # ---- end-to-end leg: host numpy in, host numpy out, through the public API.  The same pipelined call at every N:
    # openvoice_b200.distributed.convert_sharded_async -- each rank stages + uploads + converts its shard, the results are
    # gathered GPU-to-GPU (N > 1) and downloaded on rank 0, ONE call in flight behind the current one, so step i's
    # download overlaps step i+1's kernels; every step's inputs cross PCIe from pinned memory and every step's results
    # land in host memory inside the timed region.  (The synchronous ToneColorConverter.convert_batch is timed beside
    # it at N = 1 as `e2e_convert_batch`.)
    all_waves = waves if world == 1 else [synth_wave(i, secs) for i in range(world * B)]
    all_src = [synth_se(i, 2000) for i in range(world * B)]
    all_tgt = [synth_se(i, 3000) for i in range(world * B)]

    def e2e_run(n):
        res, prev = None, None
        for _ in range(n):
            job = D.convert_sharded_async(conv, all_waves, all_src, all_tgt, tau=0.3)
            if prev is not None:
                res = prev.result()      # step i's waveforms are on the host while step i+1 computes
            prev = job
        res = prev.result()
        return res
    h2d, d2h = int(B * L * 4 + B * 8), int(world * B * T * HOP * 4)
    e2e_api = "openvoice_b200.distributed.convert_sharded_async (one call in flight; d2h on rank 0 only)"

    # untimed: W steps, and at least enough for both upload slots of the sharded path to have captured their CUDA graph
    # (a launch signature is captured the second time it is seen; a capture + instantiation costs ~10 ms once)
    e2e_run(max(args.warmup, 6))
    barrier()
    t0 = time.perf_counter()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    res = e2e_run(args.steps)
    g1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms_e2e = max_over_ranks(max(g0.elapsed_time(g1), wall_ms)) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        assert len(res) == world * B and res[0].shape[0] == T * HOP and np.isfinite(res[0]).all() and np.isfinite(res[-1]).all()
    e2e_sync = None
    if world == 1:
        for _ in range(3):
            conv.convert_batch(waves, src, tgt, tau=0.3, max_batch=B)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for _ in range(max(2, args.steps // 2)):
            conv.convert_batch(waves, src, tgt, tau=0.3, max_batch=B)
        ms_sync = (time.perf_counter() - t1) * 1e3 / max(2, args.steps // 2)
        e2e_sync = {"value": audio_s_step / (ms_sync * 1e-3), "unit": "audio-s/s", "ms_per_step": ms_sync,
                    "what": "ToneColorConverter.convert_batch (synchronous: stage, upload, convert, download, unpack per call)"}

    # ---- config 4 (V2 converter: zero_g, 16 clips of 10 s per GPU, sharded): side key
    config4 = None
    if not args.no_sides:
        try:
            conv4 = make_converter(zero_g=True)
            n4 = 16 * world
            w4 = [synth_wave(5000 + i, 10.0) for i in range(n4)]
            s4 = [synth_se(5000 + i, 2000) for i in range(n4)]
            t4 = [synth_se(5000 + i, 3000) for i in range(n4)]

            def run4(n):
                prev, out = None, None
                for _ in range(n):
                    job = D.convert_sharded_async(conv4, w4, s4, t4, tau=0.3)
                    if prev is not None:
                        out = prev.result()
                    prev = job
                return prev.result()
            run4(6)      # both upload slots captured before the timed calls
            barrier()
            c0 = time.perf_counter()
            r4 = run4(3)
            barrier()
            ms4 = max_over_ranks((time.perf_counter() - c0) * 1e3) / 3
            a4 = n4 * (len(w4[0]) // HOP * HOP) / SR
            config4 = {"workload": f"V2 converter (zero_g), global batch {n4} = 16 x 10 s per GPU, convert_sharded_async, host in / host out",
                       "ms_per_step": ms4, "audio_s_per_s": a4 / (ms4 * 1e-3)}
            del conv4
        except Exception as e:      # a side measurement must never cost the headline line
            config4 = {"error": f"{type(e).__name__}: {e}"[:240]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured" if "hbm_gbs" in peaks else "fallback"
    k_ms = prof["ms"] / max(1, prof["launches"])
    ach_gbs = prof["bytes"] / max(1e-9, prof["ms"] * 1e-3) / 1e9
    ach_tf = prof["flops"] / max(1e-9, prof["ms"] * 1e-3) / 1e12

    # per-kernel table of the generator ResBlock family (family flag 1): name -> [launches, ms, flops, bytes]
    fam = {}
    for name, ms, fl, by, f in detail:
        if not f:
            continue
        key = {"T128": "tcconv_wide_kernel<1> / tcconv_kernel<128> (C >= 128)", "T64c": "tcconv_kernel<64> (C = 64)",
               "T32c": "tcconv_kernel<32> (C = 32)", "P32k": "tcpair_kernel<32> (C = 32, fused k = 3 conv pairs; 2 convs per launch)",
               "P64k": "tcpair_kernel<64> (C = 64, fused k = 3 conv pairs; 2 convs per launch)"
               }.get(name[:4], "conv1d_f32 (CUDA cores)")
        a = fam.setdefault(key, [0, 0.0, 0.0, 0.0])
        a[0] += 1; a[1] += ms; a[2] += fl; a[3] += by

    def ncu_traffic(pattern):
        """dram read + write bytes of one launch of the dominant kernel from the committed ncu --set full capture"""
        import glob
        for path in sorted(glob.glob(os.path.join(ROOT, "profiles", pattern))):
            try:
                cap = json.load(open(path))
                cap = cap[0] if isinstance(cap, list) else cap
                rd, wr = cap["dram__bytes_read.sum"].split(), cap["dram__bytes_write.sum"].split()
                unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                return ((float(rd[0]) * unit.get(rd[1], 1.0) + float(wr[0]) * unit.get(wr[1], 1.0)),
                        f"{os.path.basename(path)}: {cap.get('what', 'ncu --set full, one launch')}")
            except Exception:
                continue
        return None, None

    def ncu_dram_pass():
        """average DRAM bytes per ResBlock conv launch from the committed single-pass ncu run of THIS workload (batch 32 x 10 s,
        f16x3: tools/gpu_ncu.sh -> tools/summarize_ncu.py dram); only valid for the default batch / length / precision"""
        import glob
        if (B, secs, args.precision) != (32, 10.0, "f16x3"):
            return None, "no ncu DRAM pass for this batch / length / precision (committed one: batch 32 x 10 s, f16x3)"
        paths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r02*_ncu_dram_b32_f16x3.json")))
        if not paths:
            return None, None
        cap = json.load(open(paths[-1]))
        return cap["dram_bytes_per_launch_avg"], f"{os.path.basename(paths[-1])}: {cap['what']} (average over the 72 launches)"

    if args.precision == "fp32":
        traffic, traffic_note = ncu_traffic("r0*_ncu_full_A_K11D1_ffma2.json")
        roofline = {
            "kernel": "conv1d_f32<EPI_LINEAR> (generator ResBlock1 convs, 72 launches per call)",
            "bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
            "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
            "avg_launch_ms": k_ms, "launches": prof["launches"], "share_of_step": prof["ms"] / args.steps / ms_prof_step,
            "binding": "fp32 FFMA (dense contraction, SURVEY.md section 8d)",
            "ffma": {"achieved": ach_tf, "peak": ffma_peak()[0], "unit": "TFLOP/s", "frac": ach_tf / ffma_peak()[0],
                     "peak_source": ffma_peak()[1]},
        }
    else:
        # tensor-core modes.  achieved = ALGORITHMIC FLOPs (2*MAC of the reference's convs) / CUDA-event time; the split
        # precision spends 3 tensor FLOPs per algorithmic FLOP, which shows up as pipe_occupancy, not as achieved work.
        passes = 3 if args.precision == "f16x3" else 1
        tc_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        traffic, traffic_note = ncu_dram_pass()
        roofline = {
            "kernel": "tcconv_kernel<128|64|32> + tcconv_wide_kernel<1> (C = 256, k >= 7) + tcpair_kernel<64|32> (fused k = 3 conv pairs): "
                      f"the 72 generator ResBlock1 convs on tcgen05, {prof['launches'] // max(1, args.steps)} launches per call",
            "bound": "tensor", "achieved": ach_tf, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach_tf / tc_peak,
            "frac_note": "algorithmic FLOPs / time / measured dense 16-bit tensor peak; the fp32-grade split precision needs "
                         "3 MMA passes, so 1/3 is the ceiling of this mode",
            "mma_passes": passes, "pipe_occupancy": ach_tf * passes / tc_peak,
            "traffic": traffic, "traffic_note": traffic_note, "algorithmic_bytes_per_launch": prof["bytes"] / max(1, prof["launches"]),
            "peak_source": ("measured" if "bf16_tflops_sustained" in peaks else "fallback") + " dense bf16/fp16 sustained (MEASURED_PEAKS.json)",
            "avg_launch_ms": k_ms, "launches": prof["launches"], "share_of_step": prof["ms"] / args.steps / ms_prof_step,
            "hbm": {"achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak, "peak_source": peak_src,
                    "note": "layer-granular algorithmic bytes (SURVEY 8d tier T2: in + out per conv) / time"},
        }
    roofline["kernels"] = {
        k: {"launches_per_step": a[0] // args.steps, "ms_per_step": a[1] / args.steps, "algorithmic_tflops": a[2] / a[1] / 1e9,
            "algorithmic_gbs": a[3] / a[1] / 1e6} for k, a in sorted(fam.items(), key=lambda kv: -kv[1][1])}
    value = world * audio_s_step / (ms_dev * 1e-3)
    e2e_val = world * audio_s_step / (ms_e2e * 1e-3)
    line = {
        "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "f16x3": "f32 (3xFP16 split-precision tensor-core convs with fp32 accumulation, fp32 FFMA2 elsewhere)",
                  "f16": "f16 operands, f32 accumulation (single-pass tensor-core convs, fp32 elsewhere)"}[args.precision],
        "data": "synthetic", "precision": args.precision, "modes_audio_s_per_s": modes,
        "config": dict(workload_config(B, secs, world),
                       l2="activations per step (>3 GB) exceed the 126 MB L2; no explicit flush",
                       parallelism=f"replicas x{world}" + (f", rank 0 pinned to {numa}" if numa else ""), e2e_api=e2e_api),
        "tflops_algorithmic": world * B * T * GFLOP_PER_FRAME / ms_dev,
        "e2e": {"value": e2e_val, "unit": "audio-s/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches_per_call * args.steps * 3),
        "launches_per_call": int(launches_per_call),
        "roofline": roofline, "clocks": clocks,
    }
    if e2e_sync is not None:
        line["e2e_convert_batch"] = e2e_sync
    if config4 is not None:
        line["config4"] = config4
    if world == 1 and not args.no_sides:
        try:
            line["config1"] = latency_config1(conv)
        except Exception as e:
            line["config1"] = {"error": f"{type(e).__name__}: {e}"[:240]}
    if world == 1 and not args.no_cudnn:
        try:
            line["cudnn_baseline"] = cudnn_reference(B, secs)
        except Exception as e:
            line["cudnn_baseline"] = {"error": f"{type(e).__name__}: {e}"[:240]}
    if world == 1 and not args.no_cpu_baseline:
        v, dt, threads, done = cpu_reference_throughput(args.cpu_clips, secs)
        line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": threads, "kind": "port",
                                "sample": f"{done} x {secs:g} s clips, batch 1 each (convert semantics), fp32 torch CPU, {dt:.1f} s"}
    if world == 1 and not args.no_config3:
        # BASELINE.json configs[2] (V1 BaseSpeakerTTS.tts + convert, batch 16): a side measurement, never the headline
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location(
                "tts_pipeline_bench", os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "tts_pipeline_bench.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            r3 = mod.measure(batch=16, tokens=121, iters=3, cpu=False, precision=args.precision)
            line["config3"] = {k: r3[k] for k in ("workload", "audio_s_per_batch", "tts_ms", "convert_ms", "e2e_ms",
                                                  "tts_audio_s_per_s", "pipeline_audio_s_per_s", "text_front_launches")}
        except Exception as e:      # a side measurement must never cost the headline line
            line["config3"] = {"error": f"{type(e).__name__}: {e}"[:240]}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
