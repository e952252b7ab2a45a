"""Times the log-mel front end alone (CUDA events, 256 clips of 10 s) and compares it with the fp32 CUDA-core kernel.
Aligned input takes the centred kernel; VMB_LIB=<path> times another build of the library."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "audio-classification-using-a-deep-cnn-combined-with-multi-level-attention_b200"))
from b200 import engine, synth  # noqa: E402

dev = torch.device("cuda:0")
waves = synth.fast_clips(0, 256).to(dev)
pcm = (waves * 32767).round().clamp(-32768, 32767).to(torch.int16)
ref = engine.logmel_cudacore(waves)
for name, fn, x in (("fp32", engine.logmel, waves), ("pcm16", engine.logmel_pcm16, pcm)):
    out = fn(x)
    torch.cuda.synchronize()
    if name == "fp32":
        print("max-abs diff vs CUDA-core kernel:", (out - ref).abs().max().item(), "finite:", bool(torch.isfinite(out).all()))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(5):
        fn(x)
    torch.cuda.synchronize()
    a.record()
    for _ in range(50):
        fn(x)
    b.record()
    torch.cuda.synchronize()
    print(f"{name}: {a.elapsed_time(b) / 50:.4f} ms per 256 clips")
