#!/usr/bin/env python
"""bench_finetune.py — one fine-tuning step of VGGish's FC stack (fc1-fc3) together with the attention head, convs
frozen: 512 clips (5 120 examples), K = 527, model_conf (2, 1), dropout 0.4, on one GPU.

    python bench_finetune.py [--steps K] [--warmup W] [--clips 512] [--train-conv4-2]

A step is what `loss.backward(); opt.step()` of the reference-style loop runs on the library, timed phase by phase with
CUDA events on one stream:
  conv_fwd   conv stack of vmb_vggish_forward_train (run on its own through vmb_vggish_forward with the FC stack
             skipped: the same kernels)
  fc_fwd     vmb_vggish_forward_train minus conv_fwd
  fc_bwd     vmb_vggish_fc_backward (dW1-dW3, db1-db3, the dgrad of fc3 and fc2)
  head_step  the head's train-mode forward and backward with the input gradient (vmb_mla_train_forward +
             vmb_mla_train_backward_dx)
  refresh    vmb_vggish_refresh_fc after the optimiser step (the FC weights' inference copy and training planes)
The optimiser itself (Adam over 69.6 M parameters) is not part of any phase.  Prints one JSON line.

Arithmetic, not measured: the FC forward and backward are 1.6 TFLOP of algorithmic work per step at 512 clips
(0.69 forward, 0.69 for the three dW, 0.18 for the dgrad of fc3 and fc2); with three-plane operands (six products) that
is ~9.4 TFLOP of tensor work.

--train-conv4-2 times the step with conv4_2 (features.13) trainable as well, on the same data:
  fwd        vmb_vggish_forward_train_conv4_2 (conv1 .. conv4_1, conv4_2's im2col + GEMM + pool pass, fc1-fc3)
  head_step  as above
  bwd        vmb_vggish_conv4_2_backward (the FC backward with fc1's dgrad, conv4_2's pool backward, dW and db)
  refresh    vmb_vggish_refresh_fc + vmb_vggish_refresh_conv4_2
and, from one extra step under torch.profiler, the device time of every kernel of the step by name (kernels_ms).
Arithmetic, not measured: at 512 clips conv4_2's forward and its dW are 2.32 TFLOP each and fc1's dgrad 0.52.
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


def fc_flops(n):
    fwd = 2 * n * (12288 * 4096 + 4096 * 4096 + 4096 * 128)
    dw = fwd
    dgrad = 2 * n * (4096 * 4096 + 4096 * 128)
    return fwd, dw, dgrad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--clips", type=int, default=512)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--train-conv4-2", action="store_true")
    args = ap.parse_args()
    if args.gpus != 1:
        raise SystemExit("bench_finetune.py measures one GPU")
    if args.train_conv4_2:
        return conv4_2_main(args)
    from b200 import _lib, engine, synth, training
    from b200._lib import check, ptr, stream_ptr
    dev = torch.device("cuda:0")
    engine.require_b200(dev)
    conf, T, K, H, B = (2, 1), 10, 527, 600, args.clips
    n = B * T
    vsd = synth.vggish_state_dict(0)
    vgg = engine.VggishHandle(vsd, dev)
    fc_w = [vsd[f"embeddings.{i}.weight"].to(dev) for i in (0, 2, 4)]
    fc_b = [vsd[f"embeddings.{i}.bias"].to(dev) for i in (0, 2, 4)]
    vgg.refresh_fc(fc_w, fc_b)
    tr = training.HeadTrainer(conf, 128, H, K, T, B, dev, dropout_p=0.4)
    tr.load_state_dict(synth.mla_state_dict(conf, 128, H, K, T, seed=2))
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n, 96, 64, generator=g).to(dev)
    labels = torch.randint(0, K, (B,), generator=g).to(dev)
    L = _lib.lib()
    scores = torch.empty(B, K, device=dev)
    names = ("conv_fwd", "fc_fwd", "fc_bwd", "head_step", "refresh")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
    sums = dict.fromkeys(names, 0.0)
    totals = 0.0
    for it in range(args.warmup + args.steps):
        ev[0].record()
        vgg.forward(x, want_bottleneck=True, want_embeddings=False)         # the conv stack alone
        ev[1].record()
        emb = vgg.forward_train(x)
        ev[2].record()
        with torch.cuda.device(dev):
            check(L.vmb_mla_train_forward(tr._h, ptr(tr.params), ptr(tr.running), ptr(emb), B, 0.4, it, ptr(scores),
                                          stream_ptr()), "vmb_mla_train_forward")
            dscores = torch.nn.functional.softmax(scores, dim=1)
            dscores[torch.arange(B, device=dev), labels] -= 1.0
            dscores /= B
            dx = torch.empty_like(emb)
            check(L.vmb_mla_train_backward_dx(tr._h, ptr(tr.params), ptr(emb), ptr(dscores), B, 0.4, it,
                                              ptr(tr.grads), ptr(dx), stream_ptr()), "vmb_mla_train_backward_dx")
        ev[3].record()
        grads = vgg.fc_backward(dx)
        ev[4].record()
        views = engine.fc_grad_views(grads)
        with torch.no_grad():                                                 # stand-in for the optimiser's update
            for w, key in zip(fc_w + fc_b, ("0.weight", "2.weight", "4.weight", "0.bias", "2.bias", "4.bias")):
                w.add_(views[key], alpha=-1e-9)
        ev[5].record()
        vgg.refresh_fc(fc_w, fc_b)
        ev[6].record()
        torch.cuda.synchronize()
        if it >= args.warmup:
            conv = ev[0].elapsed_time(ev[1])
            t = {"conv_fwd": conv, "fc_fwd": ev[1].elapsed_time(ev[2]) - conv, "fc_bwd": ev[3].elapsed_time(ev[4]),
                 "head_step": ev[2].elapsed_time(ev[3]), "refresh": ev[5].elapsed_time(ev[6])}
            for k in names:
                sums[k] += t[k]
            totals += sum(t.values())
    ms = {k: round(v / args.steps, 3) for k, v in sums.items()}
    fwd, dw, dgrad = fc_flops(n)
    props = torch.cuda.get_device_properties(dev)
    out = {"metric": "fc_finetune_step_ms", "value": round(totals / args.steps, 3), "clips": B, "examples": n,
           "K": K, "model_conf": list(conf), "dropout": 0.4, "phases_ms": ms,
           "fc_algorithmic_tflop": round((fwd + dw + dgrad) / 1e12, 3),
           "fc_fwd_tflops_algorithmic": round(fwd / (ms["fc_fwd"] * 1e-3) / 1e12, 1) if ms["fc_fwd"] > 0 else None,
           "fc_bwd_tflops_algorithmic": round((dw + dgrad) / (ms["fc_bwd"] * 1e-3) / 1e12, 1)
           if ms["fc_bwd"] > 0 else None,
           "gpu": props.name, "steps": args.steps, "warmup": args.warmup}
    print(json.dumps(out))
    tr.close()
    vgg.close()


def conv4_2_flops(n):
    conv = 2 * n * 96 * 512 * 4608
    return conv, conv, 2 * n * 4096 * 12288      # forward, dW, fc1's dgrad


def gpu_identity():
    import subprocess
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_properties(0).name


def conv4_2_main(args):
    from b200 import engine, synth, training
    from b200._lib import check, ptr, stream_ptr
    from b200 import _lib
    dev = torch.device("cuda:0")
    engine.require_b200(dev)
    conf, T, K, H, B = (2, 1), 10, 527, 600, args.clips
    n = B * T
    vsd = synth.vggish_state_dict(0)
    vgg = engine.VggishHandle(vsd, dev)
    fc_w = [vsd[f"embeddings.{i}.weight"].to(dev) for i in (0, 2, 4)]
    fc_b = [vsd[f"embeddings.{i}.bias"].to(dev) for i in (0, 2, 4)]
    cw, cb = vsd["features.13.weight"].to(dev), vsd["features.13.bias"].to(dev)
    vgg.refresh_fc(fc_w, fc_b)
    vgg.refresh_conv4_2(cw, cb, fc_w[0])
    tr = training.HeadTrainer(conf, 128, H, K, T, B, dev, dropout_p=0.4)
    tr.load_state_dict(synth.mla_state_dict(conf, 128, H, K, T, seed=2))
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n, 96, 64, generator=g).to(dev)
    labels = torch.randint(0, K, (B,), generator=g).to(dev)
    L = _lib.lib()
    scores = torch.empty(B, K, device=dev)
    names = ("fwd", "head_step", "bwd", "refresh")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]

    def step(it):
        ev[0].record()
        emb = vgg.forward_train_conv4_2(x)
        ev[1].record()
        with torch.cuda.device(dev):
            check(L.vmb_mla_train_forward(tr._h, ptr(tr.params), ptr(tr.running), ptr(emb), B, 0.4, it, ptr(scores),
                                          stream_ptr()), "vmb_mla_train_forward")
            dscores = torch.nn.functional.softmax(scores, dim=1)
            dscores[torch.arange(B, device=dev), labels] -= 1.0
            dscores /= B
            dx = torch.empty_like(emb)
            check(L.vmb_mla_train_backward_dx(tr._h, ptr(tr.params), ptr(emb), ptr(dscores), B, 0.4, it,
                                              ptr(tr.grads), ptr(dx), stream_ptr()), "vmb_mla_train_backward_dx")
        ev[2].record()
        conv, fc = vgg.conv4_2_backward(dx, want_fc=True)
        ev[3].record()
        with torch.no_grad():                                                 # stand-in for the optimiser's update
            cw.add_(engine.conv4_2_grad_views(conv)["weight"], alpha=-1e-9)
            fc_w[0].add_(engine.fc_grad_views(fc)["0.weight"], alpha=-1e-9)
        ev[4].record()
        vgg.refresh_fc(fc_w, fc_b)
        vgg.refresh_conv4_2(cw, cb, fc_w[0])
        ev[5].record()
        torch.cuda.synchronize()
        return {"fwd": ev[0].elapsed_time(ev[1]), "head_step": ev[1].elapsed_time(ev[2]),
                "bwd": ev[2].elapsed_time(ev[3]), "refresh": ev[4].elapsed_time(ev[5])}

    sums = dict.fromkeys(names, 0.0)
    for it in range(args.warmup + args.steps):
        t = step(it)
        if it >= args.warmup:
            for k in names:
                sums[k] += t[k]
    ms = {k: round(v / args.steps, 3) for k, v in sums.items()}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(args.warmup + args.steps)
    kernels = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.device_time_total > 0:
            kernels[e.key[:80]] = round(e.device_time_total / 1e3, 3)
    kernels = dict(sorted(kernels.items(), key=lambda kv: -kv[1])[:16])
    fwd, dw, dgrad = conv4_2_flops(n)
    ffwd, fdw, fdgrad = fc_flops(n)
    out = {"metric": "conv4_2_finetune_step_ms", "value": round(sum(ms.values()), 3), "clips": B, "examples": n,
           "K": K, "model_conf": list(conf), "dropout": 0.4, "phases_ms": ms, "kernels_ms": kernels,
           "conv4_2_algorithmic_tflop": {"fwd": round(fwd / 1e12, 3), "dw": round(dw / 1e12, 3),
                                         "fc1_dgrad": round(dgrad / 1e12, 3)},
           "step_algorithmic_tflop_conv4_2_and_fc": round((fwd + dw + dgrad + ffwd + fdw + fdgrad) / 1e12, 3),
           "gpu": gpu_identity(), "steps": args.steps, "warmup": args.warmup}
    print(json.dumps(out))
    tr.close()
    vgg.close()


if __name__ == "__main__":
    main()
