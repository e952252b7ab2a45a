#!/usr/bin/env python
"""bench_train.py — BASELINE.json configs[4]: multi-level attention head training on synthetic 10x128 embeddings,
global batch 4096 split over the GPUs of one box (512 rows per GPU at 8 GPUs), data parallel with ONE NCCL
all-reduce of the flat gradient bucket per step (1.99 M fp32 = 7.96 MB at K = 527).

    python bench_train.py [--steps K] [--warmup W] [--per-gpu 512]            # 1 GPU
    torchrun --nproc-per-node N bench_train.py --gpus N ...                   # N GPUs
    python bench_train.py --emb-in 12288 ...          # the just_bottlenecks head: 12 288-d conv features per step

With --emb-in wider than the hidden width the line also carries the device time and executed TFLOP/s of the two GEMMs
over the input width (forward and weight gradient of the first Linear) and the device-to-device copies of a step (the
staging copy of x dominates), from a separate torch.profiler pass after the timed window.

One step = library forward + backward (vmb_mla_train_step: CE on the sigmoid outputs, dropout 0.4, batch-statistics
BatchNorm), dist.all_reduce(SUM) of the bucket, library Adam (vmb_adam_step, lr 1e-3).  Prints one JSON line
(rank 0): samples/s over all GPUs, ms per step (device-timed, max over ranks) and the per-phase split.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "audio-classification-using-a-deep-cnn-combined-with-multi-level-attention_b200")
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402



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

def _wide_profile(tr, x, labels, per_gpu, emb_in, steps=5):
    """Device time per step of the two GEMMs over the input width and of the device-to-device copies, from
    torch.profiler over `steps` extra steps; executed TFLOP/s counts the padded shapes and all six plane products."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(2):
        tr.forward_backward(x, labels)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            tr.forward_backward(x, labels)
        torch.cuda.synchronize()
    fwd = cp = 0.0
    n_fwd = 0
    mn = []
    from torch.autograd import DeviceType
    for e in prof.events():
        if e.device_type != DeviceType.CUDA:
            continue
        name, us = e.name, e.time_range.elapsed_us()
        if "planes_gemm_kernel<3, true, 0, 128, false>" in name:      # split-K forward GEMM of the wide layer
            fwd += us
            n_fwd += 1
        elif "128, true>" in name:                                     # MN-major dW GEMMs: the wide one is the longest
            mn.append(us)
        elif "Memcpy DtoD" in name:
            cp += us
    mn.sort()
    dw, n_dw = sum(mn[-steps:]), min(len(mn), steps)
    if not (n_fwd and n_dw):
        sys.stderr.write("wide-layer GEMMs not found in the trace; planes GEMM kernels seen: %s\n"
                         % sorted({e.name for e in prof.events() if "planes_gemm" in e.name}))
    rows = per_gpu * 10
    rows_pad = (rows + 63) // 64 * 64
    inpad = (emb_in + 127) // 128 * 128
    flop_fwd = 6 * 2.0 * ((rows + 127) // 128 * 128) * 640 * inpad
    flop_dw = 6 * 2.0 * 640 * inpad * rows_pad
    out = {"forward_gemm_ms": fwd / steps / 1e3, "dw_gemm_ms": dw / steps / 1e3,
           "forward_gemm_launches_per_step": n_fwd / steps,
           "memcpy_dtod_ms_per_step": cp / steps / 1e3, "x_bytes": per_gpu * 10 * emb_in * 4}
    if fwd > 0 and dw > 0:
        out["forward_gemm_tflops_executed"] = flop_fwd / (fwd / steps * 1e-6) / 1e12
        out["dw_gemm_tflops_executed"] = flop_dw / (dw / steps * 1e-6) / 1e12
    return out


def main():
    global _OUT
    _OUT = _json_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--per-gpu", type=int, default=512)
    ap.add_argument("--emb-in", type=int, default=128, help="embedding width fed to the head (12288: just_bottlenecks)")
    ap.add_argument("--cpu-baseline", action="store_true", help="also time the CPU oracle step on a 64-row sample")
    ap.add_argument("--exchange", choices=("peer", "nccl-overlap", "nccl"), default="peer",
                    help="gradient exchange at N > 1: 'peer' = reduce-scatter + Adam + all-gather in one kernel over NVLink "
                         "peer memory (csrc/dp_adam.cu, the default); 'nccl' = one NCCL all-reduce after the backward pass "
                         "+ Adam on every rank; 'nccl-overlap' = the tail of the bucket reduced while the backward pass "
                         "finishes")
    args = ap.parse_args()
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    from b200 import _lib, synth, training
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    conf, K, E = (2, 1), 527, args.emb_in
    tr = training.HeadTrainer(conf, E, 600, K, 10, args.per_gpu, dev, lr=1e-3, dropout_p=0.4, seed=1234)
    tr.load_state_dict(synth.mla_state_dict(conf, E, 600, K, 10, seed=2))
    g = torch.Generator().manual_seed(100 + rank)
    x = torch.randn(args.per_gpu, 10, E, generator=g).to(dev)
    labels = torch.randint(0, K, (args.per_gpu,), generator=g).to(dev)

    if world > 1 and args.exchange == "peer":
        tr.enable_peer_step()

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        tr.step(x, labels, overlap=args.exchange != 'nccl')
    sync()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    phases = [0.0, 0.0, 0.0]
    launches0 = _lib.lib().vmb_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    import time
    t0.record()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        tr.step(x, labels, overlap=args.exchange != 'nccl')
    host_ms = (time.perf_counter() - w0) * 1e3 / args.steps      # host time to ENQUEUE a step (no synchronisation inside)
    t1.record()
    sync()
    launches = _lib.lib().vmb_launch_count() - launches0
    ms = t0.elapsed_time(t1) / args.steps
    loss_end = float(tr.loss.item())
    tr.peer_step_status()
    if tr._dp is not None:     # phase split below uses the NCCL form on a fresh trainer
        tr.close()
        tr = training.HeadTrainer(conf, E, 600, K, 10, args.per_gpu, dev, lr=1e-3, dropout_p=0.4, seed=1234)
        tr.load_state_dict(synth.mla_state_dict(conf, E, 600, K, 10, seed=2))
    # phase split on a few extra steps (events between phases serialise nothing: same stream)
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
            if it >= 3:     # the first passes of a fresh trainer warm NCCL and the graph up
                phases[i] += ev[i].elapsed_time(ev[i + 1]) / 10
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if rank == 0:
        line = {"metric": f"MLA head training samples/sec (synthetic 10x{E} embeddings, K=527, model_conf [2,1])",
                "value": args.per_gpu * world / (ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "dtype": "fp32-equivalent (3-plane split bf16 on tcgen05)", "data": "synthetic",
                "config": {"workload": f"global batch {args.per_gpu * world} = {args.per_gpu} per GPU, Adam lr 1e-3, "
                                       "dropout 0.4, CE on sigmoid outputs", "allreduce_bytes": tr.n_params * 4,
                           "gradient_exchange": args.exchange if world > 1 else "none (one rank)"},
                "phase_ms": {"forward_backward": phases[0], "allreduce": phases[1], "adam": phases[2]},
                "gpu_launches": int(launches), "final_loss": loss_end, "host_enqueue_ms_per_step": host_ms,
                "cuda_graph": os.environ.get("VMB_TRAIN_GRAPH", "1") != "0"}
        if E > 640:
            line["wide_layer"] = _wide_profile(tr, x, labels, args.per_gpu, E)
        if args.cpu_baseline and world == 1:
            import time
            from oracle import train_torch
            sd = synth.mla_state_dict(conf, E, 600, K, 10, seed=2)
            xs, ls = x[:64].cpu(), labels[:64].cpu()
            train_torch.head_step(sd, xs, ls, conf, dropout_p=0.4)
            t = time.perf_counter()
            for _ in range(5):
                train_torch.head_step(sd, xs, ls, conf, dropout_p=0.4)
            dt = (time.perf_counter() - t) / 5
            line["cpu_baseline"] = {"value": 64 / dt, "unit": "samples/s", "cores": torch.get_num_threads(),
                                    "kind": "port", "sample": "forward+backward of 64 rows (no optimiser), 5 passes"}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
