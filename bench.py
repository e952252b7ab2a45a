#!/usr/bin/env python
"""bench.py — 10 s-clip waveform -> scores throughput (clips/s) of the B200 path, beside the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--clips C] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (fused log-mel -> VGGish -> multi-level-attention head) over one batch of
C synthetic 10 s / 16 kHz clips per GPU (default 256 = BASELINE.json configs[1]).  For N > 1 the driver launches
one rank per GPU with torchrun; clips are sharded by batch, the path has no collective (SURVEY §8e), so the scaling
is weak (C clips per GPU) and NCCL is used only for the barrier and the max-over-ranks of the timings.

One JSON line is printed by rank 0:
  value      clips/s over all GPUs, inputs resident in HBM (device-timed with CUDA events, max over ranks)
  e2e        the same metric through the host-buffer C-ABI call (vmb_pipeline_forward_host): pinned host input,
             H2D copy, compute, D2H copy of the scores inside the timed region
  roofline   the dominant kernel (tcgen05 implicit GEMM: 5 convs + 3 FCs per step) against the measured 16-bit
             tensor peak: the short timed region against the BURST peak, the >= 3 s back-to-back leg (`sustained`)
             against the SUSTAINED peak
  cpu_baseline  the oracle (numpy front end + torch-CPU VGGish + head = the reference's algorithm) on the host cores
  configs    compact legs for BASELINE.json configs[2..4]: batch8192 (8192 / N clips per rank through the host-buffer
             entry point, micro-batched), stream_1h (1-hour stream, accuracy mode, PCA / uint8), train (head training
             with the NCCL all-reduce of the gradient bucket at N > 1)
  e2e_dropin the reference-named API: per-clip waveform_to_examples + Ensemble.forward, and Ensemble.forward_waveform
--impl reference times the CPU path alone (rank 0 only) on a bounded sample of the same workload.
--dump-outputs DIR writes the scores of the last timed step (the global batch at N > 1; for --impl reference the first
clips of the batch that its sample timed) to DIR/scores.npy.  Inputs and weights are seeded, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "audio-classification-using-a-deep-cnn-combined-with-multi-level-attention_b200")
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

if "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is a CPU measurement on rank 0 alone and must
    # use every host core it can (set before numpy / torch load their thread pools)
    _ncpu = str(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    for _k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[_k] = _ncpu

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "10s-clip audio->logits clips/sec"
UNIT = "clips/s"
MODEL_CONF = (2, 1)
N_CLASSES = 527
CLIP_SAMPLES = 160000

# algorithmic FLOPs per 0.96 s example (SURVEY §8d): 2*M*N*K per GEMM
_CONV = ((96 * 64, 64, 9), (48 * 32, 128, 576), (24 * 16, 256, 1152), (24 * 16, 256, 2304), (12 * 8, 512, 2304),
         (12 * 8, 512, 4608))
_FC = ((12288, 4096), (4096, 4096), (4096, 128))
FLOP_CONV = [2.0 * m * n * k for m, n, k in _CONV]
FLOP_FC = [2.0 * a * b for a, b in _FC]
FLOP_IGEMM_PER_EXAMPLE = sum(FLOP_CONV[1:]) + sum(FLOP_FC)          # what the tcgen05 kernel computes
FLOP_DFT_PER_CLIP = 2.0 * 400 * 514 * 998
FLOP_MEL_PER_CLIP = 2.0 * 257 * 64 * 998
FLOP_HEAD_PER_CLIP = 29.69e6
FLOP_PER_CLIP = FLOP_DFT_PER_CLIP + FLOP_MEL_PER_CLIP + 10 * (sum(FLOP_CONV) + sum(FLOP_FC)) + FLOP_HEAD_PER_CLIP
STAGES = ("logmel", "conv1", "conv2", "conv3_1", "conv3_2", "conv4_1", "conv4_2", "fc1", "fc2", "fc3", "mla",
          "postprocess")



def _json_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to fd 1 when
    the communicator is created), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved
    original stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


_OUT = None


def emit(line):
    (_OUT or sys.stdout).write(json.dumps(line) + "\n")
    (_OUT or sys.stdout).flush()


DUMP_MAX_BYTES = 64 * 10**6


def dump_outputs(out_dir, scores):
    """--dump-outputs: writes the scores (clips x classes) the timed path returned in its last step as
    out_dir/scores.npy, float32, so that two builds run with the same arguments can be compared output for output.
    Scores larger than DUMP_MAX_BYTES are cut to a fixed sample of clips (seed 0, in clip order)."""
    scores = scores.detach().float().cpu().numpy()
    max_rows = (DUMP_MAX_BYTES - 4096) // (4 * scores.shape[1])                   # 4096: room for the .npy header
    if scores.shape[0] > max_rows:
        scores = scores[np.sort(np.random.default_rng(0).choice(scores.shape[0], max_rows, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scores.npy"), np.ascontiguousarray(scores, dtype=np.float32))


def igemm_traffic():
    """(DRAM bytes per launch of the dominant kernel, where the figure comes from): read from the committed ncu
    capture — a profiler figure, not a measurement of this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "igemm_traffic.json")) as fh:
            d = json.load(fh)
        return float(d["dram_bytes_per_launch"]), "ncu --set full, " + str(d.get("source", "profiles/igemm_traffic.json"))
    except Exception:
        return None, None


def tensor_pipe_util():
    """Tensor-pipe utilisation per layer from the committed ncu capture (BASELINE.json's second metric); a profiler
    figure, copied from profiles/, never measured inside the timed run."""
    try:
        with open(os.path.join(ROOT, "profiles", "igemm_traffic.json")) as fh:
            return json.load(fh)["tensor_pipe_active_pct"]
    except Exception:
        return None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        return {"tflops": float(d["bf16_tflops_sustained"]), "tflops_burst": float(d["bf16_tflops"]),
                "hbm_gbs": float(d["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json, sustained bf16)"}
    except Exception:
        return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0,
                "source": "fallback (B200_PROFILING.md: 1.59 PF burst / ~1.4 PF sustained)"}


# ------------------------------------------------------------------------------------------------ CPU arm
def _oracle_modules():
    from b200 import synth
    from oracle import frontend_np, model_torch
    return synth, frontend_np, model_torch


def oracle_pass(waves, vsd, msd):
    """The reference's algorithm on the CPU: numpy float64 front end per clip (vggish_input.py:30-82), torch fp32
    VGGish (vggish.py:21-31), head (model.py:258-269)."""
    _, frontend_np, model_torch = _oracle_modules()
    ex = np.concatenate([frontend_np.waveform_to_examples(w.astype(np.float64)) for w in waves])
    x = torch.from_numpy(ex).float()[:, None]
    with torch.no_grad():
        emb = model_torch.vgg_forward(vsd, x)
        return model_torch.mla_forward(msd, emb.reshape(len(waves), 10, 128), MODEL_CONF)


def time_cpu(vsd, msd, steps, warmup, budget_s):
    """Times `steps` oracle passes (after `warmup`) on a sample sized so that the whole run takes ~budget_s; returns the
    scores of the last pass with the timings."""
    synth, _, _ = _oracle_modules()
    probe = synth.fast_clips(0, 2).numpy()
    oracle_pass(probe[:1], vsd, msd)                         # page-in / thread pools
    t0 = time.perf_counter()
    oracle_pass(probe, vsd, msd)
    per_clip = (time.perf_counter() - t0) / 2
    n = int(max(1, min(16, budget_s / max(1e-3, per_clip * (steps + warmup)))))
    waves = synth.fast_clips(0, n).numpy()
    for _ in range(warmup):
        oracle_pass(waves, vsd, msd)
    t0 = time.perf_counter()
    for _ in range(steps):
        scores = oracle_pass(waves, vsd, msd)
    dt = time.perf_counter() - t0
    return {"clips_per_s": n * steps / dt, "ms_per_step": 1e3 * dt / steps, "sample_clips": n, "steps": steps,
            "threads": torch.get_num_threads(), "scores": scores}


def run_reference(args, rank):
    if rank != 0:
        return
    torch.set_num_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    synth, _, _ = _oracle_modules()
    vsd = synth.vggish_state_dict(0)
    msd = synth.mla_state_dict(MODEL_CONF, 128, 600, N_CLASSES, 10, seed=2)
    # ~90 s of CPU work for the whole run by default (VMB_BENCH_CPU_BUDGET_S overrides, e.g. for the CPU test suite)
    r = time_cpu(vsd, msd, args.steps, args.warmup, budget_s=float(os.environ.get("VMB_BENCH_CPU_BUDGET_S", "90")))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["scores"])
    sample = (f"{r['sample_clips']} of the {args.clips} clips of a step per timed pass, {args.steps} passes after "
              f"{args.warmup} warm-ups; numpy float64 front end + torch {torch.__version__} CPU fp32")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["clips_per_s"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "reference_sample_clips_per_step": r["sample_clips"],
        "note": f"this arm times {r['sample_clips']} of the step's {args.clips} clips per pass (ms_per_step is per "
                "sample, value is clips/s); the reference is pure Python and cannot travel to the GPU box, so this is the "
                "oracle port of its algorithm (kind: port)",
        "cpu_baseline": {"value": r["clips_per_s"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                         "sample": sample},
        "e2e": {"value": r["clips_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "host_cpus": os.cpu_count(),
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""
    REASONS = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
               0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
               0x100: "display_clock_setting"}

    def __init__(self, device_index, period_s=0.01):
        super().__init__(daemon=True)
        self.period_s = period_s
        self.stop_flag = threading.Event()
        self.mhz, self.mask, self.max_mhz, self.power, self.ok = [], 0, None, [], False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.mhz.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    m = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    m = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.mask |= int(m)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(self.period_s)

    def summary(self):
        if not self.ok or not self.mhz:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML sampling unavailable"}
        return {"sm_mhz": float(np.median(self.mhz)), "sm_max_mhz": self.max_mhz,
                "reasons": [n for b, n in self.REASONS.items() if self.mask & b], "samples": len(self.mhz),
                "power_w_max": max(self.power) if self.power else None}


def bind_to_gpu_numa_node(device_index):
    """Pin this rank's threads (and therefore its first-touch pinned host buffers) to the CPUs NVML reports as local
    to its GPU, so that at N > 1 every rank's H2D copies read host memory on the GPU's own socket."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus local to the GPU"
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({type(e).__name__})"
    return "unavailable"


def workload_config(args, world):
    return {"workload": f"batch {args.clips} synthetic 10 s 16 kHz clips per GPU, waveform -> log-mel -> VGGish -> "
                        f"multi-level attention scores ({N_CLASSES} classes, model_conf [2,1]) = BASELINE.json configs[1]",
            "reference_arm": "the CPU reference arm (--impl reference) times a bounded sample of this step — at most 16 "
                             "of its clips per pass, the exact count is in its cpu_baseline.sample — and reports clips/s",
            "clips_per_gpu_per_step": args.clips, "global_clips_per_step": args.clips * world,
            "samples_per_clip": CLIP_SAMPLES, "examples_per_clip": 10, "n_classes": N_CLASSES,
            "parallelism": f"batch-sharded x{world}, no collective on the data path",
            "l2": f"input batch {args.clips * CLIP_SAMPLES * 4 / 1e6:.0f} MB fp32 + >1 GB of activations per step "
                  "(larger than the 126 MB L2)",
            "flop_per_clip": FLOP_PER_CLIP}


# ------------------------------------------------------------------------------------------------ B200 arm
def _timed(fn, steps, barrier, max_over_ranks):
    """Device time of `steps` calls of fn (CUDA events on the current stream), barriers on both sides, max over ranks."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return max_over_ranks(e0.elapsed_time(e1))


def leg_h2d_probe(wave_host, dev, barrier, max_over_ranks, world):
    """Copy-only probe: what the box gives this rank for pinned host -> device copies of one step's input while every
    other rank does the same (one cudaMemcpyAsync per copy on one stream, like csrc/vggish.cu submit_host_any; and the
    same bytes as two halves on two streams)."""
    dst = torch.empty_like(wave_host, device=dev)
    nbytes = wave_host.numel() * 4
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    half = wave_host.shape[0] // 2
    out = {}

    def one():
        dst.copy_(wave_host, non_blocking=True)

    def two():
        cur = torch.cuda.current_stream(dev)
        s1.wait_stream(cur)
        s2.wait_stream(cur)
        with torch.cuda.stream(s1):
            dst[:half].copy_(wave_host[:half], non_blocking=True)
        with torch.cuda.stream(s2):
            dst[half:].copy_(wave_host[half:], non_blocking=True)
        cur.wait_stream(s1)
        cur.wait_stream(s2)

    for name, fn in (("one_stream", one), ("two_streams", two)):
        for _ in range(2):
            fn()
        ms = _timed(fn, 10, barrier, max_over_ranks)          # max over ranks = the slowest rank's rate
        out[name + "_gbs_per_gpu"] = nbytes * 10 / (ms * 1e-3) / 1e9
    out["bytes_per_copy"] = nbytes
    out["aggregate_gbs"] = max(out["one_stream_gbs_per_gpu"], out["two_streams_gbs_per_gpu"]) * world
    return out


def leg_sustained(pipe, wave_dev, clips, world, local_rank, barrier, max_over_ranks, seconds, peaks):
    """The device-resident step back to back for >= `seconds` (independent of --steps): the regime in which the board's
    power limit, not the burst clock, sets the tensor rate.  NVML sampled every ~2 ms."""
    from b200 import _lib
    L = _lib.lib()
    sampler = ClockSampler(local_rank, period_s=0.002)
    L.vmb_profile_collect(None, None, 1)
    for _ in range(3):
        pipe.forward(wave_dev)
    barrier()
    sampler.start()
    chunk = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    n = 0
    # stage timers only on the last chunk: their event pairs would otherwise pile up for thousands of steps
    while True:
        for _ in range(chunk):
            pipe.forward(wave_dev)
        n += chunk
        torch.cuda.current_stream().synchronize() if n % (4 * chunk) == 0 else None
        if time.perf_counter() - t0 >= seconds:
            break
    L.vmb_profile_enable(1)
    for _ in range(chunk):
        pipe.forward(wave_dev)
    n += chunk
    e1.record()
    barrier()
    L.vmb_profile_enable(0)
    sampler.stop_flag.set()
    ms = max_over_ranks(e0.elapsed_time(e1))
    stage_ms = np.zeros(len(STAGES), dtype=np.float64)
    stage_calls = np.zeros(len(STAGES), dtype=np.int64)
    L.vmb_profile_collect(stage_ms.ctypes.data, stage_calls.ctypes.data, 1)
    sampler.join(timeout=1.0)
    n_ex = clips * 10
    per_stage = {STAGES[i]: float(stage_ms[i]) / chunk for i in range(len(STAGES)) if stage_calls[i]}
    stage_flop = dict(zip(STAGES[1:10], [f * n_ex for f in FLOP_CONV + FLOP_FC]))
    ig_ms = sum(per_stage.get(k, 0.0) for k in STAGES[2:10])
    ig_tflops = FLOP_IGEMM_PER_EXAMPLE * n_ex / (ig_ms * 1e-3) / 1e12 if ig_ms > 0 else None
    clk = sampler.summary()
    ms_step = ms / n
    return {"seconds": ms * 1e-3, "steps": n, "value": clips * world / (ms_step * 1e-3), "unit": UNIT,
            "ms_per_step": ms_step, "sm_mhz_median": clk.get("sm_mhz"), "power_w_max": clk.get("power_w_max"),
            "clock_reasons": clk.get("reasons"), "nvml_samples": clk.get("samples"),
            "stage_ms_per_step": {k: round(v, 4) for k, v in per_stage.items()},
            "stage_tflops": {k: round(stage_flop[k] / (per_stage[k] * 1e-3) / 1e12, 1) for k in stage_flop
                             if per_stage.get(k)},
            "igemm_tflops": ig_tflops, "igemm_frac_of_sustained_peak": ig_tflops / peaks["tflops"] if ig_tflops else None,
            "whole_step_tflops": FLOP_PER_CLIP * clips / (ms_step * 1e-3) / 1e12,
            "whole_step_frac_of_sustained_peak": FLOP_PER_CLIP * clips / (ms_step * 1e-3) / 1e12 / peaks["tflops"]}


def leg_batch8192(pipe, wave_host, world, barrier, max_over_ranks):
    """BASELINE.json configs[2]: 8192 clips sharded by batch, 8192 / N per rank, through the host-buffer entry point in
    micro-batches of 256 (H2D of micro-batch i+1 overlaps the compute of micro-batch i); scores land in host memory."""
    per_rank = 8192 // world
    reps = (per_rank + wave_host.shape[0] - 1) // wave_host.shape[0]
    big = wave_host.repeat(reps, 1)[:per_rank].contiguous().pin_memory()     # this rank's shard (the step batch, tiled)
    out = torch.empty(per_rank, N_CLASSES).pin_memory()
    pipe.forward_host(big[:512], out[:512], clips_per_batch=256)
    runs = []
    for _ in range(5):          # five whole passes; the first one also pays the first device touch of the 5 GB shard
        barrier()
        t0 = time.perf_counter()
        pipe.forward_host(big, out, clips_per_batch=256)
        barrier()
        runs.append(max_over_ranks(1e3 * (time.perf_counter() - t0)))
    ms = sorted(runs)[2]        # the median pass
    nb = wave_host.shape[0]
    ok = bool(torch.isfinite(out).all().item())
    if per_rank >= 2 * nb:                       # the shard is the step batch tiled: its blocks must come out identical
        ok = ok and bool(torch.equal(out[:nb], out[nb:2 * nb]))
    return {"value": 8192 / (ms * 1e-3), "unit": UNIT, "ms": ms, "ms_each_pass": runs, "clips_per_rank": per_rank,
            "microbatch_clips": 256,
            "h2d_bytes_per_rank": per_rank * CLIP_SAMPLES * 4, "scores_ok": ok,
            "api": "vmb_pipeline_forward_host (one blocking call per rank; pinned host in, pinned host out)"}


def leg_stream_1h(dev, rank, world, barrier, max_over_ranks, vsd):
    """BASELINE.json configs[3]: one 1-hour 16 kHz stream (230 MB fp32, pinned host) -> 3 749 examples -> VGGish in the
    accuracy mode -> PCA / 8-bit; at N > 1 the stream is sharded by example (sharding.stream_chunks), no collective."""
    import torch.distributed as dist
    from b200 import engine, sharding, stream, synth
    n = 3600 * 16000
    g = torch.Generator().manual_seed(7)
    t = torch.arange(n, dtype=torch.float32) / 16000.0
    wave = (0.3 * torch.sin(2 * np.pi * (110.0 + 40.0 * torch.sin(2 * np.pi * 0.05 * t)) * t)
            + 0.05 * torch.randn(n, generator=g)).pin_memory()
    del t
    eig, means = synth.pca_params(1)
    n_ex = sharding.num_examples(n)
    steps = 3
    res, qs = {}, {}
    for mode in ("split", "fp16"):
        vgg = engine.VggishHandle(vsd, dev, precision=mode)
        for _ in range(2):
            emb, q = stream.embed_stream(vgg, wave, eig, means, 2048, rank, world)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            emb, q = stream.embed_stream(vgg, wave, eig, means, 2048, rank, world)
            checksum = torch.tensor([int(q.sum().item())], device=dev, dtype=torch.int64)   # forces completion, 8 B D2H
        barrier()
        ms = max_over_ranks(1e3 * (time.perf_counter() - t0)) / steps
        if world > 1:
            dist.all_reduce(checksum)
        vgg.check_saturation()
        vgg.close()
        qs[mode] = q
        res[mode] = {"value": n_ex / (ms * 1e-3), "unit": "examples/s", "ms_per_stream": ms,
                     "realtime_factor": 3600.0 / (ms * 1e-3), "uint8_checksum": int(checksum.item())}
    hist = torch.bincount((qs["fp16"].int() - qs["split"].int()).abs().flatten(), minlength=2)    # this rank's share
    out = dict(res["split"])
    out.update({"n_examples": n_ex, "h2d_bytes": n * 4,
                "dtype": "split bf16 (hi + lo planes; uint8 output within +-1 LSB of the fp32 reference, 0.5 % at +-1)",
                "fp16_mode": dict(res["fp16"], uint8_lsb_histogram_vs_split_mode_rank0=hist.tolist()),
                "api": "b200.stream.embed_stream (chunks of 2048 examples, H2D overlapped with compute)"})
    return out


def leg_train(dev, rank, world, barrier, max_over_ranks):
    """BASELINE.json configs[4]: head training on synthetic 10 x 128 embeddings, 4096 / 8 = 512 rows per GPU, one NCCL
    all-reduce of the flat gradient bucket per step at N > 1 (train.py:119-142, :369-372 semantics)."""
    from b200 import _lib, synth, training
    per_gpu, conf = 512, MODEL_CONF
    tr = training.HeadTrainer(conf, 128, 600, N_CLASSES, 10, per_gpu, dev, lr=1e-3, dropout_p=0.4, seed=1234)
    tr.load_state_dict(synth.mla_state_dict(conf, 128, 600, N_CLASSES, 10, seed=2))
    g = torch.Generator().manual_seed(100 + rank)
    x = torch.randn(per_gpu, 10, 128, generator=g).to(dev)
    labels = torch.randint(0, N_CLASSES, (per_gpu,), generator=g).to(dev)
    for _ in range(5):
        tr.step(x, labels)
    steps = 20
    # the two NCCL forms first (A/B in the same run): the whole bucket reduced after the backward pass, and its tail
    # reduced while the backward pass finishes
    ms_serial = ms_overlap = None
    if world > 1:
        ms_serial = _timed(lambda: tr.step(x, labels, overlap=False), steps, barrier, max_over_ranks) / steps
        ms_overlap = _timed(lambda: tr.step(x, labels, overlap=True), steps, barrier, max_over_ranks) / steps
        # the product path: reduce-scatter + Adam + all-gather in one kernel over NVLink peer memory (csrc/dp_adam.cu)
        tr.enable_peer_step()       # False (every rank together) if the arenas cannot be mapped: the NCCL form stays
        for _ in range(5):
            tr.step(x, labels)
    l0 = _lib.lib().vmb_launch_count()
    ms = _timed(lambda: tr.step(x, labels), steps, barrier, max_over_ranks) / steps
    launches = _lib.lib().vmb_launch_count() - l0
    tr.peer_step_status()
    peer = tr._dp is not None
    peer_err = tr.peer_step_error
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    phases = [0.0, 0.0, 0.0]
    loss = float(tr.loss.item())
    tr.close()
    # phase split with the NCCL form (events between the phases): a second trainer, the arena is gone
    tr = training.HeadTrainer(conf, 128, 600, N_CLASSES, 10, per_gpu, dev, lr=1e-3, dropout_p=0.4, seed=1234)
    tr.load_state_dict(synth.mla_state_dict(conf, 128, 600, N_CLASSES, 10, seed=2))
    for it in range(13):
        ev[0].record()
        tr.forward_backward(x, labels)
        ev[1].record()
        w = tr.all_reduce_grads()
        ev[2].record()
        tr.adam(w)
        ev[3].record()
        torch.cuda.synchronize()
        for i in range(3):
            if it >= 3:
                phases[i] += ev[i].elapsed_time(ev[i + 1]) / 10
    tr.close()
    return {"value": per_gpu * world / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "rows_per_gpu": per_gpu,
            "global_batch": per_gpu * world, "allreduce_bytes": tr.n_params * 4 if world > 1 else 0,
            "phase_ms": {"forward_backward": phases[0], "allreduce": phases[1], "adam": phases[2]},
            "gpu_launches_per_step": launches / steps, "final_loss": loss,
            "gradient_exchange": ("vmb_dp_adam_step: reduce-scatter + Adam + parameter all-gather in one kernel over NVLink "
                                  "peer memory (CUDA IPC arenas), two flag barriers") if peer else
                                 ("none (one rank)" if world == 1 else
                                  "NCCL all-reduce, tail overlapped (peer-memory step unavailable: %s)" % peer_err),
            "ms_per_step_nccl_allreduce_then_adam": ms_serial,
            "ms_per_step_nccl_allreduce_tail_overlapped": ms_overlap,
            "dtype": "fp32-equivalent (3-plane split bf16 on tcgen05)"}


def leg_dropin(dev, vsd, msd, wave_host, barrier, max_over_ranks, world):
    """What a user of the reference calls: vggish_input.waveform_to_examples(w, 16000) per clip
    (vggish_input.py:30) then Ensemble.forward (model.py:58-62), with host numpy waveforms in and scores read back; and
    the one-call fast path Ensemble.forward_waveform."""
    import model
    from torchvggish.vggish_input import waveform_to_examples
    old = model.K
    try:
        model.K = N_CLASSES
        conf = dict(cnn_type="vggish", num_classes=N_CLASSES, use_pretrained=False, just_bottlenecks=False,
                    cnn_trainable=False, first_cnn_layer_trainable=False, in_channels=1)
        ens = model.Ensemble("repeat", conf, list(MODEL_CONF), dev)
    finally:
        model.K = old
    ens.cnn.cnn_model.load_state_dict(vsd)
    ens.mla.load_state_dict(msd)
    ens = ens.to(dev).eval()
    n = 64
    waves_np = [wave_host[i].numpy().astype(np.float64) for i in range(n)]

    def per_clip():
        ex = torch.stack([waveform_to_examples(w, 16000) for w in waves_np])     # (n, 10, 1, 96, 64) on the device
        return ens(ex).cpu()

    def one_call():
        return ens.forward_waveform(wave_host[:n].to(dev, non_blocking=True)).cpu()

    out = {}
    for name, fn in (("per_clip_waveform_to_examples_then_forward", per_clip), ("forward_waveform", one_call)):
        fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            y = fn()
        barrier()
        ms = max_over_ranks(1e3 * (time.perf_counter() - t0)) / 3
        out[name] = {"value": n * world / (ms * 1e-3), "unit": UNIT, "ms_per_call": ms, "clips_per_call": n}
    out["scores_agree"] = bool((per_clip() - one_call()).abs().max().item() <= 1e-4)
    return out


def run_b200(args, rank, local_rank, world):
    import torch.distributed as dist
    from b200 import _lib, engine, synth

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    engine.require_b200(dev)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()

    vsd = synth.vggish_state_dict(0)
    msd = synth.mla_state_dict(MODEL_CONF, 128, 600, N_CLASSES, 10, seed=2)
    vgg = engine.VggishHandle(vsd, dev, precision=args.precision)
    head = engine.MlaHandle(msd, MODEL_CONF, 128, 600, N_CLASSES, 10, dev)
    pipe = engine.Pipeline(vgg, head)

    wave_host = synth.fast_clips(rank * args.clips, args.clips).pin_memory()          # this rank's shard
    scores_host = torch.empty(args.clips, N_CLASSES).pin_memory()
    wave_dev = wave_host.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput
    for _ in range(max(3, args.warmup)):
        scores = pipe.forward(wave_dev)
    L.vmb_profile_collect(None, None, 1)
    sampler = ClockSampler(local_rank, period_s=0.002)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    L.vmb_profile_enable(1)
    launches0 = L.vmb_launch_count()
    ev0.record()
    for _ in range(args.steps):
        scores = pipe.forward(wave_dev)
    ev1.record()
    barrier()
    launches = L.vmb_launch_count() - launches0
    L.vmb_profile_enable(0)
    sampler.stop_flag.set()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    ms_step = ms_total / args.steps
    stage_ms = (torch.zeros(len(STAGES), dtype=torch.float64)).numpy()
    stage_calls = np.zeros(len(STAGES), dtype=np.int64)
    L.vmb_profile_collect(stage_ms.ctypes.data, stage_calls.ctypes.data, 1)
    sampler.join(timeout=1.0)
    vgg.check_saturation()
    finite = bool(torch.isfinite(scores).all().item())
    if args.dump_outputs:
        dumped = scores
        if world > 1:                                               # the global batch: every rank's shard in rank order
            parts = [torch.empty_like(scores) for _ in range(world)]
            dist.all_gather(parts, scores)
            dumped = torch.cat(parts)
        if rank == 0:
            dump_outputs(args.dump_outputs, dumped)
    peaks = measured_peaks()

    # ---- the same step back to back for >= 3 s: the sustained regime
    sustained = leg_sustained(pipe, wave_dev, args.clips, world, local_rank, barrier, max_over_ranks,
                              args.sustained_seconds, peaks) if args.sustained_seconds > 0 else None

    # ---- end to end through the host-buffer C-ABI entry points (pinned host in, pinned host out).  Every step's
    # H2D copy of its inputs, its compute and its D2H copy of the scores happen inside the timed region; two steps
    # are kept in flight (submit i+1 before collecting i, as a DataLoader-fed loop would), so the copy of step i+1
    # overlaps the compute of step i.  The strictly serial variant (one blocking call per step) is timed as well.
    if args.e2e_microbatch <= 0:
        args.e2e_microbatch = args.clips
    scores_host2 = torch.empty(args.clips, N_CLASSES).pin_memory()
    outs = (scores_host, scores_host2)
    for _ in range(max(3, args.warmup)):
        pipe.forward_host(wave_host, scores_host, clips_per_batch=args.e2e_microbatch)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    pending = pipe.submit_host(wave_host, outs[0], clips_per_batch=args.e2e_microbatch)
    for i in range(1, args.steps):
        nxt = pipe.submit_host(wave_host, outs[i & 1], clips_per_batch=args.e2e_microbatch)
        pipe.wait_host(pending)
        pending = nxt
    pipe.wait_host(pending)
    e1.record()
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), wall_ms))
    e2e_equal = bool(torch.equal(outs[(args.steps - 1) & 1], scores.cpu()))
    # the same pipelined loop fed with 16-bit PCM (the WAV sample format, vggish_input.py:96-98): half the H2D bytes
    pcm_host = torch.clamp(torch.round(wave_host * 32768.0), -32768, 32767).to(torch.int16).pin_memory()
    pend = pipe.submit_host(pcm_host, outs[0], clips_per_batch=args.e2e_microbatch)
    pipe.wait_host(pend)
    barrier()
    t0 = time.perf_counter()
    pending = pipe.submit_host(pcm_host, outs[0], clips_per_batch=args.e2e_microbatch)
    for i in range(1, args.steps):
        nxt = pipe.submit_host(pcm_host, outs[i & 1], clips_per_batch=args.e2e_microbatch)
        pipe.wait_host(pending)
        pending = nxt
    pipe.wait_host(pending)
    barrier()
    pcm_ms = max_over_ranks(1e3 * (time.perf_counter() - t0))
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pipe.forward_host(wave_host, scores_host, clips_per_batch=args.serial_microbatch)
    barrier()
    serial_ms = max_over_ranks(1e3 * (time.perf_counter() - t0))
    h2d = leg_h2d_probe(wave_host, dev, barrier, max_over_ranks, world)

    # ---- latency of BASELINE.json configs[0]: ONE 10 s clip, host buffer in -> scores on the host (blocking call)
    one_host = wave_host[:1].clone().pin_memory()
    one_out = torch.empty(1, N_CLASSES).pin_memory()
    for _ in range(5):
        pipe.forward_host(one_host, one_out, clips_per_batch=1)
    t0 = time.perf_counter()
    for _ in range(50):
        pipe.forward_host(one_host, one_out, clips_per_batch=1)
    b1_ms = 1e3 * (time.perf_counter() - t0) / 50

    # ---- the same device-resident step in the other two modes of the VGGish body: bf16 (the same kernels on 8 mantissa
    # bits) and split (hi + lo bf16 planes, 3x the tensor work: the mode whose uint8 output matches the fp32 reference)
    other, other_stages = {}, {}
    for mode in ("bf16", "fp16", "split"):
        if mode == args.precision:
            continue
        h2 = engine.VggishHandle(vsd, dev, precision=mode)
        p2 = engine.Pipeline(h2, head)
        for _ in range(3):
            p2.forward(wave_dev)
        k = args.steps if mode != "split" else max(3, min(10, args.steps))   # same region length as the headline
        L.vmb_profile_collect(None, None, 1)
        L.vmb_profile_enable(1)
        other[mode] = _timed(lambda: p2.forward(wave_dev), k, barrier, max_over_ranks) / k
        L.vmb_profile_enable(0)
        sm, sc = np.zeros(len(STAGES), dtype=np.float64), np.zeros(len(STAGES), dtype=np.int64)
        L.vmb_profile_collect(sm.ctypes.data, sc.ctypes.data, 1)
        other_stages[mode] = {STAGES[i]: round(float(sm[i]) / k, 4) for i in range(len(STAGES)) if sc[i]}
        h2.close()
    acc_ms = other["split"]

    # ---- compact legs for BASELINE.json configs[2..4] and the reference-named API.  They run LAST, after the headline
    # line has been assembled, under a watchdog: a leg that hangs (they contain collectives) costs its own entry, not the
    # line — on time-out rank 0 prints the line with what has finished and every rank leaves with exit code 0.
    legs = {}

    def run_legs():
        if args.no_config_legs:
            return
        for name, leg in (("batch8192", lambda: leg_batch8192(pipe, wave_host, world, barrier, max_over_ranks)),
                          ("stream_1h", lambda: leg_stream_1h(dev, rank, world, barrier, max_over_ranks, vsd)),
                          ("train", lambda: leg_train(dev, rank, world, barrier, max_over_ranks)),
                          ("e2e_dropin", lambda: leg_dropin(dev, vsd, msd, wave_host, barrier, max_over_ranks, world))):
            try:
                legs[name] = leg()
            except Exception as e:  # noqa: BLE001 — a leg that fails must not take the headline line with it
                legs[name] = {"error": f"{type(e).__name__}: {e}"[:400]}

    class Watchdog:
        def __init__(self, seconds, on_timeout):
            self.lock, self.done = threading.Lock(), False
            self.timer = threading.Timer(seconds, self._fire)
            self.timer.daemon = True
            self.on_timeout = on_timeout

        def _fire(self):
            with self.lock:
                if self.done:
                    return
                self.done = True
                try:
                    self.on_timeout()
                finally:
                    os._exit(0)

        def __enter__(self):
            self.timer.start()
            return self

        def __exit__(self, *exc):
            with self.lock:
                self.done = True
            self.timer.cancel()
            return False

    if rank != 0:
        with Watchdog(args.legs_timeout + 10.0, lambda: None):
            run_legs()
        if world > 1:
            dist.destroy_process_group()
        return

    n_ex = args.clips * 10
    ig = slice(2, 10)                                                       # conv2 .. fc3 = the tcgen05 kernel
    ig_ms_per_step = float(stage_ms[ig].sum()) / args.steps
    ig_launches_per_step = int(stage_calls[ig].sum()) // args.steps
    ig_flop_per_step = FLOP_IGEMM_PER_EXAMPLE * n_ex
    achieved = ig_flop_per_step / (ig_ms_per_step * 1e-3) / 1e12 if ig_ms_per_step > 0 else None
    per_stage = {STAGES[i]: round(float(stage_ms[i]) / args.steps, 4) for i in range(len(STAGES)) if stage_calls[i]}
    stage_flop = dict(zip(STAGES[1:10], [f * n_ex for f in FLOP_CONV + FLOP_FC]))
    stage_tflops = {k: round(stage_flop[k] / (per_stage[k] * 1e-3) / 1e12, 1) for k in stage_flop if per_stage.get(k)}
    clips_per_s = args.clips * world / (ms_step * 1e-3)
    whole_tflops = FLOP_PER_CLIP * args.clips / (ms_step * 1e-3) / 1e12
    e2e_step_ms = e2e_ms / args.steps
    traffic, traffic_src = igemm_traffic()
    line = {
        "metric": METRIC, "value": clips_per_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": args.clips * world / (e2e_step_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": args.clips * CLIP_SAMPLES * 4, "d2h_bytes_per_step": args.clips * N_CLASSES * 4,
                "ms_per_step": e2e_step_ms, "wall_ms_per_step": wall_ms / args.steps,
                "microbatch_clips": args.e2e_microbatch, "matches_device_path": e2e_equal, "steps_in_flight": 2,
                "serial_value": args.clips * world / (serial_ms / args.steps * 1e-3),
                "serial_ms_per_step": serial_ms / args.steps, "serial_microbatch_clips": args.serial_microbatch,
                "pcm16_value": args.clips * world / (pcm_ms / args.steps * 1e-3),
                "pcm16_h2d_bytes_per_step": args.clips * CLIP_SAMPLES * 2,
                # achieved H2D rate of this leg per GPU, beside what a copy-only loop of the same shape gets on this
                # box with all ranks copying at once: when the two agree the leg is bound by the host -> device link
                "h2d_gbs_per_gpu": args.clips * CLIP_SAMPLES * 4 / (e2e_step_ms * 1e-3) / 1e9,
                "h2d_ceiling_gbs": max(h2d["one_stream_gbs_per_gpu"], h2d["two_streams_gbs_per_gpu"]),
                "h2d_probe": h2d,
                "compute_bound_value": clips_per_s,
                "api": "vmb_pipeline_submit_host / vmb_pipeline_wait_host via b200.engine.Pipeline (serial_*: one "
                       "blocking vmb_pipeline_forward_host call per step)"},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        # the timed region is short (steps x ~3.5 ms): the GPU runs at its burst clock, so the matching peak is the
        # measured BURST 16-bit tensor rate; the >= 3 s leg below is compared with the SUSTAINED one
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
                     "frac": (achieved / peaks["tflops_burst"]) if achieved else None,
                     "regime": f"burst ({ms_total * 1e-3:.3f} s timed region)", "traffic": traffic,
                     "traffic_source": traffic_src,
                     "tensor_pipe_active_pct_ncu": tensor_pipe_util(),
                     "kernel": "igemm_pair_kernel (tcgen05 cta_group::2 implicit GEMM: conv3_1..conv4_2, fc1, fc2) + "
                               "igemm_bf16_kernel (cta_group::1: conv2, fc3)",
                     "launches_per_step": ig_launches_per_step, "algorithmic_flop_per_launch":
                         ig_flop_per_step / max(1, ig_launches_per_step),
                     "avg_launch_ms": ig_ms_per_step / max(1, ig_launches_per_step), "peak_source": peaks["source"],
                     "whole_step_tflops": whole_tflops, "whole_step_frac": whole_tflops / peaks["tflops_burst"],
                     "sustained": None if sustained is None else {
                         "achieved": sustained["igemm_tflops"], "peak": peaks["tflops"],
                         "frac": sustained["igemm_frac_of_sustained_peak"],
                         "whole_step_frac": sustained["whole_step_frac_of_sustained_peak"],
                         "regime": f"sustained ({sustained['seconds']:.1f} s back to back)"}},
        "sustained": sustained,
        "stage_ms_per_step": per_stage, "stage_tflops": stage_tflops,
        "single_clip_latency_ms": b1_ms, "host_affinity": numa,
        "modes": {m: {"value": args.clips * world / (v * 1e-3), "unit": UNIT, "ms_per_step": v,
                      "stage_ms_per_step": other_stages.get(m)} for m, v in other.items()},
        "accuracy_mode": {"value": args.clips * world / (acc_ms * 1e-3), "unit": UNIT, "ms_per_step": acc_ms,
                          "dtype": "split bf16 (hi + lo planes, fp32-class body)"},
        "configs": legs,
        "scores_finite": finite,
    }
    if world == 1 and not args.no_cpu_baseline:
        r = time_cpu(vsd, msd, steps=3, warmup=1, budget_s=20.0)
        line["cpu_baseline"] = {
            "value": r["clips_per_s"], "unit": UNIT, "cores": r["threads"], "kind": "port",
            "sample": f"{r['sample_clips']} of the {args.clips} clips per pass, 3 timed passes after 1 warm-up "
                      f"(numpy float64 front end + torch CPU fp32 VGGish + head); host has {os.cpu_count()} CPUs"}

    def emit_without_the_rest():
        for name in ("batch8192", "stream_1h", "train", "e2e_dropin"):
            legs.setdefault(name, {"error": f"not finished within {args.legs_timeout:.0f} s (leg watchdog)"})
        emit(line)

    with Watchdog(args.legs_timeout, emit_without_the_rest):
        run_legs()
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    global _OUT
    _OUT = _json_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--clips", type=int, default=256, help="clips per GPU per step")
    ap.add_argument("--e2e-microbatch", type=int, default=0,
                    help="clips per H2D/compute micro-batch in the pipelined e2e leg (0 = the whole step)")
    ap.add_argument("--serial-microbatch", type=int, default=64,
                    help="clips per micro-batch in the serial (one blocking call per step) e2e variant")
    ap.add_argument("--impl", choices=("b200", "reference"), default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--precision", choices=("fp16", "bf16", "split"), default="fp16",
                    help="arithmetic of the VGGish body for the headline legs (fp16 and bf16 run at the same tensor rate)")
    ap.add_argument("--sustained-seconds", type=float, default=3.0,
                    help="length of the back-to-back leg that measures the sustained regime (0 = skip)")
    ap.add_argument("--legs-timeout", type=float, default=300.0,
                    help="seconds the configs[2..4] / drop-in legs may take before the line is printed without them")
    ap.add_argument("--no-config-legs", action="store_true",
                    help="skip the batch8192 / stream_1h / train / e2e_dropin legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the scores of the last timed step to DIR/scores.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world > 1:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
