"""Times the eval-mode attention head alone (CUDA events, batch 256 x 10 x 128, K = 527, model_conf [2, 1]).
VMB_LIB=<path> times another build of the library."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "audio-classification-using-a-deep-cnn-combined-with-multi-level-attention_b200"))
from b200 import engine, synth  # noqa: E402

dev = torch.device("cuda:0")
batch = int(sys.argv[1]) if len(sys.argv) > 1 else 256
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 200
conf = tuple(int(c) for c in sys.argv[3].split(",")) if len(sys.argv) > 3 else (2, 1)
sd = synth.mla_state_dict(conf, 128, 600, 527, 10, seed=2)
h = engine.MlaHandle(sd, conf, 128, 600, 527, 10, dev)
x = torch.randn(batch, 10, 128, device=dev)
for _ in range(5):
    h.forward(x)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(reps):
    h.forward(x)
b.record()
torch.cuda.synchronize()
sw = {k[4:]: os.environ[k] for k in os.environ if k.startswith("VMB_")}
print(f"head {conf} batch {batch}: {a.elapsed_time(b) / reps * 1000:.1f} us per forward  {sw}")
