#!/usr/bin/env python
"""Benchmark of the stylization hot path (BASELINE.json metric: stylized frames/s @512x512).

    python bench.py --gpus N --steps K --warmup W                 # this repo's B200 engine, BASELINE configs[1]
    python bench.py --config c3|c4|c5 --gpus N ...                # the other BASELINE configs (528^2 / 8 characters / 1024^2 stage 1)
    python bench.py --impl reference --gpus N --steps K ...       # the reference's CPU path (oracle port) on the host cores
    python bench.py --gpus 1 --steps K --dump-outputs DIR         # also save what the timed path returned in its last step

One *step* = one pass of stage 1 -> uint8 -> edge burn-in -> stage 2 -> uint8 RGBA over the rank's synthetic
frame stack.  With N > 1 (torchrun, one rank per GPU) every rank owns its own frame range, weights are broadcast
once over NCCL and there is no per-frame collective.  Prints ONE JSON line on rank 0.

What the line reports (round-2 contract):
* ``value`` / ``e2e`` / ``roofline``: the PARITY-GRADE mode (split-fp16 "fp16x3", <= 1e-3 max-abs against the fp32
  reference forward) - the number and the parity claim refer to the same mode;
* ``config.parity``: the in-process parity gate - one 512x512 frame through both stages, engine vs an fp32 reference
  forward (the oracle port run on cuda with TF32 off), before anything is timed; a failing gate exits non-zero;
* ``config.fast_mode``: the single-pass fp16 mode (same operand class as the reference's own default GPU path,
  which runs its convolutions in TF32 = 10-bit mantissa) with its measured error, fps, e2e and roofline;
* ``config.gpu_baseline``: the reference's forward on the same B200 (torch cuDNN + torchvision deform_conv2d CUDA
  kernels; batch 1 as test_stage1.py:57-63 runs it, and batch 16), fps and its own error against true fp32;
* ``cpu_baseline``: the reference's CPU path on the host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "stylized frames/sec @512x512 (stage1+stage2)"
UNIT = "frames/s"
TOL = 1e-3          # BASELINE.json north_star: max-abs fp32 against the reference's own forward
DUMP_BYTES = 60 * 10**6   # float32 payload of --dump-outputs: with the .npy headers the dump stays under 64 MB

CONFIGS = {
    # name: (workload description, frame size, total frames (None = per-GPU), characters, stage-1 only, scaling)
    "c2": ("stage1+stage2 inference, 64-frame synthetic dab-like sequence, 512x512 (BASELINE configs[1])", 512, None, 1, False, "weak"),
    "c3": ("stage1+stage2, 256-frame synthetic jumping-like sequence at its real size 528x528, batch 16, frame-shard (BASELINE configs[2])",
           528, 256, 1, False, "strong"),
    "c4": ("8 characters (8 distinct checkpoints) x 128 synthetic frames, stage1+stage2, character -> GPU (BASELINE configs[3])",
           512, 8 * 128, 8, False, "strong"),
    "c5": ("1024x1024 synthetic frame stream, 512 frames, stage 1 only, frame-shard HBM stress (BASELINE configs[4])",
           1024, 512, 1, True, "strong"),
}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def usable_cores():
    """Host cores this process may really use: scheduler affinity, cgroup CPU quota and physical cores (one thread per
    core - SMT siblings only add contention to oneDNN / the im2col loop), whichever is smallest."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    try:
        cores = set()
        phys = core = None
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("physical id"):
                    phys = line.split(":")[1].strip()
                elif line.startswith("core id"):
                    core = line.split(":")[1].strip()
                elif not line.strip():
                    if phys is not None and core is not None:
                        cores.add((phys, core))
                    phys = core = None
        if cores:
            n = min(n, len(cores))
    except Exception:
        pass
    return max(1, n)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.tmp = None

    def start(self):
        try:
            self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=self.tmp, stderr=subprocess.DEVNULL)
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
        self.tmp.flush()
        self.tmp.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.tmp.read().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.tmp.name)
        except OSError:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------ reference arms
def _weights(seed):
    from drawingspinup_b200 import synth
    return (synth.to_torch_state_dict(synth.make_state_dict(1, seed=seed, out_gain=0.25)),
            synth.to_torch_state_dict(synth.make_state_dict(2, seed=seed, out_gain=0.25)))


def cpu_reference(size: int, reps: int, warmup: int, threads: int, seed: int = 1234, budget_s: float = 1e9):
    """The reference's CPU path (oracle port: torch fp32 convolutions + torchvision deform_conv2d, models.py:113-129 /
    293-356 and the uint8 steps of test_stage1.py:60-70 / test_stage2.py:67-78): one ``size`` x ``size`` frame through
    stage 1 + stage 2 per repetition.  Returns (seconds per frame [median of the timed reps], list of rep times, threads)."""
    import numpy as np
    import torch
    from drawingspinup_b200 import synth
    from oracle import reference_port as rp
    torch.set_num_threads(threads)
    sd1, sd2 = _weights(seed)
    color, pos, edge = synth.make_frames(1, size, size, seed=seed)

    def one():
        with torch.no_grad():
            x1 = torch.from_numpy(rp.frame_to_tensor(color[0], pos[0])[0])[None]
            y1 = rp.generator_j_ric_forward(sd1, x1, use_torchvision=True)
            r1 = rp.compose_rgba(y1[0].numpy(), rp.frame_to_tensor(color[0], pos[0])[1])
            x2 = torch.from_numpy(rp.frame_to_tensor(r1, pos[0], edge[0])[0])[None]
            y2 = rp.generator_j_forward(sd2, x2)
            return rp.compose_rgba(y2[0].numpy(), rp.frame_to_tensor(color[0], pos[0])[1])

    t_start = time.perf_counter()
    for _ in range(warmup):
        one()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s and len(times) >= 1:
            break
    times_sorted = sorted(times)
    return times_sorted[len(times_sorted) // 2], times, torch.get_num_threads()


def pick_cpu_size(threads: int, n_frames: int, budget_s: float, start: int = 256):
    """Largest sample frame size in {start, start/2, ...} >= 64 for which ``n_frames`` frames fit in ``budget_s`` on this host
    (one probe frame at 64x64 scaled by pixel count; the deformable im2col loop is linear in pixels)."""
    spf64, _, _ = cpu_reference(64, 1, 1, threads)
    size = start
    while size > 64 and spf64 * (size / 64.0) ** 2 * n_frames > budget_s:
        size //= 2
    return size, spf64


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores, same metric /
    unit / config as the engine's arm; every step is one bounded-sample frame (size picked so that the whole run ends
    within a few minutes), frames/s scaled to the 512x512 workload by pixel count."""
    if rank != 0:
        return
    threads = usable_cores()
    size, spf64 = pick_cpu_size(threads, args.steps + args.warmup, budget_s=240.0, start=args.cpu_size)
    spf, times, threads = cpu_reference(size, args.steps, args.warmup, threads)
    S = CONFIGS[args.config][1]
    scale = (size * size) / float(S * S)
    val = scale / spf
    sample = ("%d warm-up + %d timed step(s), each 1 frame %dx%d through stage1+stage2 (oracle port of models.py:113-129/293-356: "
              "torch CPU fp32 + torchvision deform_conv2d), %d threads = usable physical cores; median %.2f s/frame at the sample "
              "size (min %.2f, max %.2f), frames/s scaled by pixel count to %dx%d"
              % (args.warmup, len(times), size, size, threads, spf, min(times), max(times), S, S))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": spf * 1e3, "higher_is_better": True, "scaling": CONFIGS[args.config][5],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": CONFIGS[args.config][0], "frames_per_gpu": args.frames, "height": S, "width": S,
                       "sample_height": size, "sample_width": size},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def gpu_reference(dev, size, sd1, sd2, color, pos, edge, frames=2):
    """The reference's forward on THIS GPU (what test_stage1.py:59-63 / test_stage2.py:66-70 dispatch with device 'cuda:0'):
    torch's cuDNN convolutions + torchvision's CUDA deform_conv2d, fp32, batch 1 and batch 16, with the library default
    (cudnn.allow_tf32 = True: stage-2 convolutions run in TF32) and with TF32 off (true fp32, also the checker of the
    parity gate).  The live reference classes are used when /root/reference is importable, else the oracle port on cuda."""
    import numpy as np
    import torch
    from oracle import reference_port as rp
    out = {"impl": "oracle port on cuda: torch cuDNN conv2d + torchvision.ops.deform_conv2d CUDA kernels, fp32 "
                   "(reference call sites training/models.py:113-129, 293-356)",
           "height": size, "width": size}
    sd1d = {k: v.to(dev) for k, v in sd1.items()}
    sd2d = {k: v.to(dev) for k, v in sd2.items()}
    x1 = torch.from_numpy(np.stack([rp.frame_to_tensor(color[i], pos[i])[0] for i in range(16)])).to(dev)
    x2 = torch.from_numpy(np.stack([rp.frame_to_tensor(color[i], pos[i], edge[i])[0] for i in range(16)])).to(dev)

    def timed(fn, n):
        fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n

    results = {}
    old_c, old_m = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    try:
        with torch.no_grad():
            for tag, tf32 in (("tf32_off", False), ("library_default", None)):
                if tf32 is None:
                    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_c, old_m
                else:
                    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
                ent = {"cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32),
                       "matmul_allow_tf32": bool(torch.backends.cuda.matmul.allow_tf32)}
                for b in (1, 16):
                    try:
                        ms1 = timed(lambda: rp.generator_j_ric_forward(sd1d, x1[:b], use_torchvision=True), frames)
                        ms2 = timed(lambda: rp.generator_j_forward(sd2d, x2[:b]), frames)
                        ent["batch%d" % b] = {"stage1_ms": ms1, "stage2_ms": ms2, "fps": b * 1e3 / (ms1 + ms2)}
                    except RuntimeError as exc:          # e.g. out of memory for the batch-16 columns buffer
                        ent["batch%d" % b] = {"error": str(exc).splitlines()[0][:160]}
                        torch.cuda.empty_cache()
                y1 = rp.generator_j_ric_forward(sd1d, x1[:1], use_torchvision=True)
                y2 = rp.generator_j_forward(sd2d, x2[:1])
                results[tag] = (y1, y2)
                out[tag] = ent
        e1 = (results["library_default"][0] - results["tf32_off"][0]).abs().max().item()
        e2 = (results["library_default"][1] - results["tf32_off"][1]).abs().max().item()
        out["library_default"]["max_abs_err_vs_fp32"] = {"stage1": e1, "stage2": e2}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_c, old_m
    del sd1d, sd2d, x1, x2, results
    torch.cuda.empty_cache()
    return out


def parity_gate(pipes, dev, size, sd1, sd2, seed):
    """One ``size`` x ``size`` frame through both stages, each engine mode against the fp32 reference forward on identical
    inputs (oracle port on cuda, TF32 off = true fp32; tests/test_gpu_parity.py holds the same frame to the CPU oracle).
    Stage 2 is checked on the engine's own stage-1 bytes, as test_stage2.py would read them back from disk."""
    import numpy as np
    import torch
    from drawingspinup_b200 import synth
    from oracle import reference_port as rp
    color, pos, edge = synth.make_frames(1, size, size, seed=seed + 77)
    c_d, p_d, e_d = (torch.from_numpy(a).to(dev) for a in (color, pos, edge))
    sd1d = {k: v.to(dev) for k, v in sd1.items()}
    sd2d = {k: v.to(dev) for k, v in sd2.items()}
    res = {}
    old_c, old_m = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            for mode, pipe in pipes.items():
                r1, y1 = pipe.g1.forward_frames(c_d, p_d, None, return_float=True)
                y2 = None
                if pipe.g2 is not None:
                    _, y2 = pipe.g2.forward_frames(r1, p_d, e_d, return_float=True)
                torch.cuda.synchronize(dev)
                x1 = torch.from_numpy(rp.frame_to_tensor(color[0], pos[0])[0])[None].to(dev)
                ref1 = rp.generator_j_ric_forward(sd1d, x1, use_torchvision=True)
                err = {"stage1": (y1 - ref1).abs().max().item()}
                if y2 is not None:
                    x2 = torch.from_numpy(rp.frame_to_tensor(r1[0].cpu().numpy(), pos[0], edge[0])[0])[None].to(dev)
                    ref2 = rp.generator_j_forward(sd2d, x2)
                    err["stage2"] = (y2 - ref2).abs().max().item()
                res[mode] = err
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_c, old_m
    del sd1d, sd2d
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------ engine arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--frames", type=int, default=64, help="frames per GPU per step (config c2; the others fix the total)")
    ap.add_argument("--batch", type=int, default=16, help="frames per kernel launch")
    ap.add_argument("--precision", default="fp16x3", choices=["fp16", "fp16x3"],
                    help="mode reported as `value` (default: the parity-grade split-fp16 mode)")
    ap.add_argument("--cpu-size", type=int, default=256, help="largest frame size of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-fast", action="store_true", help="skip the secondary single-pass fp16 measurement")
    ap.add_argument("--no-parity-gate", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the uint8 RGBA frames the timed path returned in its last step as "
                         "DIR/rgba_char<c>.npy (float32 [k,H,W,4]; rank 0; k frames per character chosen by a fixed seed "
                         "so that the dump stays under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return 0
    args.warmup = max(args.warmup, 3)
    workload, S, total_frames, n_chars, stage1_only, scaling = CONFIGS[args.config]

    # stdout must carry exactly ONE JSON line: everything printed before it (e.g. banners written from C) goes to
    # stderr, the real stdout is restored just for the result line.  NCCL_DEBUG is left to the caller / driver.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist
    from drawingspinup_b200 import synth
    from drawingspinup_b200.pipeline import StylizationPipeline, assign_work, broadcast_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 engine has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    # ---- work assignment: characters (weight sets) and frames of this rank
    if total_frames is None:
        F = args.frames                                   # weak scaling: every rank owns its own F-frame stack
        my_chars = [0]
        frames_of = {0: F}
        seeds = {0: 1234 + rank}
    else:
        frames_of = assign_work(total_frames, n_chars, rank, world)   # character -> GPU, or a frame shard of the one clip
        my_chars = sorted(frames_of)
        seeds = {c: 1234 + 17 * c + rank for c in my_chars}
    my_frames = sum(frames_of.values())
    all_frames = my_frames
    if world > 1:
        t = torch.tensor([my_frames], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        all_frames = int(t.item())

    # ---- weights: one character's checkpoint is broadcast once from rank 0 (single-character configs); with several
    # characters every rank builds (= "loads") the checkpoints of its own characters and nothing is broadcast
    weights = {}
    if n_chars == 1:
        sd1, sd2 = _weights(1234) if rank == 0 else (None, None)
        weights[0] = (broadcast_state_dict(sd1, 0, dev), broadcast_state_dict(sd2, 0, dev))
    else:
        for c in my_chars:
            weights[c] = _weights(1234 + c)

    stacks = {}
    for c in my_chars:
        color, pos, edge = synth.make_frames(frames_of[c], S, S, seed=seeds[c])
        h = tuple(torch.from_numpy(a).pin_memory() for a in (color, pos, edge))
        stacks[c] = {"host": h, "dev": tuple(t.to(dev) for t in h),
                     "out": torch.empty((frames_of[c], S, S, 4), dtype=torch.uint8).pin_memory()}

    def make_pipes(precision):
        return {c: StylizationPipeline(weights[c][0], None if stage1_only else weights[c][1], dev, precision=precision,
                                       batch=args.batch) for c in my_chars}

    last = {}                                             # character -> RGBA frames of the last timed device-resident step

    def measure(pipes, host: bool):
        def fn(keep=False):
            for c in my_chars:
                st = stacks[c]
                if host:
                    pipes[c].run_host(*st["host"], st["out"])
                else:
                    out = pipes[c].run(*st["dev"])
                    if keep:
                        last[c] = out
        for _ in range(args.warmup):
            fn()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(args.steps):
            fn(keep=i == args.steps - 1)
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    peaks, peak_kind = load_peaks()
    peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))

    def layer_roofline(pipe, tensor_factor):
        """Per-launch device times of one batch (CUDA events around every launch on the launching stream) -> the
        roofline entry of the dominant kernel + the whole table."""
        table = []
        gens = (("stage1", pipe.g1),) + ((("stage2", pipe.g2),) if pipe.g2 is not None else ())
        for tag, g in gens:
            for name, ms, fl in g.profile_layers(args.batch, S, S, reps=3):
                table.append({"kernel": tag + "." + name, "ms": ms, "tflops": (fl / (ms * 1e-3) / 1e12) if ms > 0 else 0.0,
                              "gflop": fl / 1e9})
        top = max(table, key=lambda r: r["ms"])
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath) and args.batch == 16 and S == 512:
            with open(tpath) as f:
                ent = json.load(f).get(top["kernel"] + (":x3" if tensor_factor == 3 else ""))
            if ent:
                traffic, traffic_src = ent["bytes"], ent["source"]
        roof = {"bound": "tensor", "kernel": top["kernel"], "achieved": top["tflops"], "peak": peak, "unit": "TFLOP/s",
                "frac": top["tflops"] / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "%s bf16_tflops_sustained (kernel timed inside a long step)" % peak_kind,
                "launch_ms": top["ms"], "launch_gflop": top["gflop"],
                "achieved_definition": "algorithmic conv FLOPs of the launch (SURVEY 8d) / CUDA-event launch time",
                "tensor_work_factor": tensor_factor,
                "executed_tensor_frac": tensor_factor * top["tflops"] / peak}
        return roof, table

    # ---- pipelines: the reported mode first, the other one for config.fast_mode / the parity gate
    main_prec = args.precision
    other_prec = "fp16" if main_prec == "fp16x3" else "fp16x3"
    pipes = make_pipes(main_prec)
    first = pipes[my_chars[0]]

    parity = None
    if rank == 0 and not args.no_parity_gate:
        gate_pipes = {main_prec: first}
        other_first = None
        if not args.no_fast:
            other_first = StylizationPipeline(weights[my_chars[0]][0], None if stage1_only else weights[my_chars[0]][1], dev,
                                              precision=other_prec, batch=args.batch)
            gate_pipes[other_prec] = other_first
        errs = parity_gate(gate_pipes, dev, S if S <= 528 else 512, weights[my_chars[0]][0], weights[my_chars[0]][1], 1234)
        worst = max(errs[main_prec].values())
        parity = {"mode": main_prec, "max_abs_err_512": errs[main_prec], "tol": TOL, "pass": bool(worst <= TOL),
                  "frame": "%dx%d synthetic frame, both stages on identical inputs" % ((S if S <= 528 else 512,) * 2),
                  "checker": "fp32 reference forward (oracle port on cuda, cudnn/matmul TF32 off); the same frame is held to the "
                             "CPU oracle in tests/test_gpu_parity.py::test_benchmark_size_parity"}
        if other_prec in errs:
            parity["other_mode"] = {"mode": other_prec, "max_abs_err_512": errs[other_prec],
                                    "pass": bool(max(errs[other_prec].values()) <= TOL)}
        del gate_pipes, other_first
        torch.cuda.empty_cache()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total = measure(pipes, host=False)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        per_char = DUMP_BYTES // len(my_chars) // (S * S * 4 * 4)
        for c in my_chars:
            idx = np.sort(np.random.default_rng(c).choice(frames_of[c], min(frames_of[c], per_char), replace=False))
            np.save(os.path.join(args.dump_outputs, "rgba_char%d.npy" % c),
                    last[c][torch.from_numpy(idx).to(dev)].float().cpu().numpy())
    last.clear()
    ms_e2e = measure(pipes, host=True)
    fps = all_frames * args.steps / (ms_total / 1e3)
    fps_e2e = all_frames * args.steps / (ms_e2e / 1e3)
    flops_frame = first.flops_per_frame(S, S)
    n_batches = sum((frames_of[c] + args.batch - 1) // args.batch for c in my_chars)
    launches_rank = args.steps * n_batches * first.launches_per_batch(args.batch, S, S)
    workspace = first.workspace_bytes(args.batch, S, S)

    roof, layer_table = (None, [])
    if rank == 0:
        roof, layer_table = layer_roofline(first, 3 if main_prec == "fp16x3" else 1)
        roof["whole_step_frac"] = (flops_frame * fps / world / 1e12) / peak

    fast = None
    if not args.no_fast:
        del pipes, first
        torch.cuda.empty_cache()
        pipes_f = make_pipes(other_prec)
        ms_f = measure(pipes_f, host=False)
        ms_fe = measure(pipes_f, host=True)
        fast = {"dtype": other_prec, "value": all_frames * args.steps / (ms_f / 1e3), "unit": UNIT, "ms_per_step": ms_f / args.steps,
                "e2e": all_frames * args.steps / (ms_fe / 1e3)}
        if rank == 0:
            r_f, t_f = layer_roofline(pipes_f[my_chars[0]], 3 if other_prec == "fp16x3" else 1)
            r_f["whole_step_frac"] = (flops_frame * fast["value"] / world / 1e12) / peak
            fast["roofline"] = {k: r_f[k] for k in ("kernel", "achieved", "frac", "launch_ms", "whole_step_frac")}
            fast["layers_ms"] = {r["kernel"]: round(r["ms"], 4) for r in t_f}
            if parity and "other_mode" in parity:
                fast["max_abs_err_512"] = parity["other_mode"]["max_abs_err_512"]
                fast["parity_pass"] = parity["other_mode"]["pass"]
            fast["note"] = ("single-pass fp16 operands / fp32 accumulate: same operand class as the reference's default GPU "
                            "path (cuDNN TF32, 10-bit mantissa; see gpu_baseline.library_default.max_abs_err_vs_fp32)")
        del pipes_f
        last.clear()
        torch.cuda.empty_cache()

    gpu_base = None
    if rank == 0 and world == 1 and not args.no_gpu_baseline and not stage1_only:
        c0 = my_chars[0]
        color, pos, edge = (t[:16].numpy() for t in stacks[c0]["host"])
        try:
            gpu_base = gpu_reference(dev, S, weights[c0][0], weights[c0][1], color, pos, edge)
        except Exception as exc:      # the comparison arm must never take the engine's own numbers down with it
            gpu_base = {"error": "%s: %s" % (type(exc).__name__, str(exc).splitlines()[0][:200] if str(exc) else "")}

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = usable_cores()
        size, _ = pick_cpu_size(threads, 4, budget_s=100.0, start=args.cpu_size)
        spf, times, threads = cpu_reference(size, 3, 1, threads)
        scale = (size * size) / float(S * S)
        cpu_base = {"value": scale / spf, "unit": UNIT, "cores": threads, "kind": "port",
                    "sample": "1 warm-up + %d timed frames %dx%d through stage1+stage2 on the host CPU (oracle port: torch fp32 conv2d + "
                              "torchvision deform_conv2d), %d threads pinned to the usable physical cores; median %.2f s/frame "
                              "(min %.2f, max %.2f) at the sample size, frames/s scaled by pixel count to %dx%d"
                              % (len(times), size, size, threads, spf, min(times), max(times), S, S)}

    if rank == 0:
        line = {"metric": METRIC if args.config == "c2" else METRIC + " [%s]" % args.config, "value": fps, "unit": UNIT,
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": main_prec + (" (split fp16 hi+lo operands, fp32 accumulate)" if main_prec == "fp16x3" else ""),
                "data": "synthetic",
                "config": {"workload": workload, "frames_total": all_frames, "frames_per_gpu": my_frames, "height": S, "width": S,
                           "batch_per_launch": args.batch, "characters": n_chars, "stages": "stage1" if stage1_only else "stage1+stage2",
                           "parallelism": ("character -> GPU x%d, no weight broadcast" % world) if n_chars > 1 else
                                          ("frame-shard x%d, weights broadcast once" % world),
                           "l2": "inputs+activations per step (>2 GB) exceed the 126 MB L2; no explicit flush",
                           "workspace_bytes_per_handle": workspace,
                           "hbm_fraction_of_180GB": workspace * len(my_chars) / 180e9,
                           "gflop_per_frame": flops_frame / 1e9,
                           "parity": parity, "fast_mode": fast, "gpu_baseline": gpu_base},
                "e2e": {"value": fps_e2e, "unit": UNIT, "h2d_bytes_per_step": int(all_frames * S * S * 9),
                        "d2h_bytes_per_step": int(all_frames * S * S * 4), "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(world * launches_rank), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu_base,
                "layers": layer_table}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and parity is not None and not parity["pass"]:
        sys.stderr.write("bench.py: PARITY GATE FAILED: %s\n" % json.dumps(parity))
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
