"""Compare the head-training step of two builds on identical seeded inputs, in one process.
usage: python tools/cmp_train_libs.py ref.so new.so

For every case (model_conf (2, 1) and (1, 2, 1), K = 527 and 10, dropout 0 and 0.4, emb_in 128) each build runs one
seeded vmb_mla_train_step twice from the same parameters and running statistics.  Printed per output: whether the
two builds agree bit for bit, and the largest difference between them next to the largest difference between two runs
of the reference build (the split-K weight-gradient GEMMs and the bias column sums add with fp32 atomics, so a
gradient may differ in the last bits from run to run of one build)."""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "audio-classification-using-a-deep-cnn-combined-with-multi-level-attention_b200"))
from b200 import synth, training  # noqa: E402

dev = torch.device("cuda:0")
vp, ll, ci, cf = C.c_void_p, C.c_longlong, C.c_int, C.c_float


def load(path):
    L = C.CDLL(path)
    L.vmb_mla_trainer_create.argtypes = [C.POINTER(vp), ci, C.POINTER(ci), ci, ci, ci, ci, ll, vp]
    L.vmb_mla_trainer_destroy.argtypes = [vp]
    L.vmb_mla_train_step.argtypes = [vp, vp, vp, vp, vp, ll, cf, C.c_ulonglong, vp, vp, vp, vp]
    L.vmb_last_error.restype = C.c_char_p
    return L


def run(L, conf, emb_in, K, batch, p, x, labels, params0, running0, steps=2):
    arr = (ci * len(conf))(*conf)
    h = vp()
    st = torch.cuda.current_stream().cuda_stream
    assert L.vmb_mla_trainer_create(C.byref(h), len(conf), arr, emb_in, 600, K, 10, batch, st) == 0, L.vmb_last_error()
    outs = []
    for s in range(steps):      # the first step runs eagerly, the second replays a captured graph
        params, running = params0.clone(), running0.clone()
        grads = torch.zeros_like(params)
        loss = torch.zeros(1, device=dev)
        scores = torch.empty(batch, K, device=dev)
        assert L.vmb_mla_train_step(h, params.data_ptr(), running.data_ptr(), x.data_ptr(), labels.data_ptr(), batch, p,
                                    99, grads.data_ptr(), loss.data_ptr(), scores.data_ptr(), st) == 0, L.vmb_last_error()
        torch.cuda.synchronize()
        outs.append({"loss": loss.clone(), "scores": scores.clone(), "grads": grads.clone(), "running": running.clone()})
    L.vmb_mla_trainer_destroy(h)
    return outs


def main():
    ref, new = load(sys.argv[1]), load(sys.argv[2])
    worst_gap = 0.0
    not_bitwise = []
    for conf in ((2, 1), (1, 2, 1)):
        for K in (527, 10):
            for p in (0.0, 0.4):
                emb_in, batch = 128, 512
                sd = synth.mla_state_dict(conf, emb_in, 600, K, 10, seed=2)
                lay = training.train_layout(conf, emb_in, 600, K, 10)
                params0 = torch.cat([sd[k].reshape(-1).float() for k, _, _ in lay[0]]).to(dev)
                running0 = torch.cat([sd[k].reshape(-1).float() for k, _, _ in lay[1]]).to(dev)
                g = torch.Generator().manual_seed(5)
                x = torch.randn(batch, 10, emb_in, generator=g).to(dev)
                labels = torch.randint(0, K, (batch,), generator=g).to(dev)
                a = run(ref, conf, emb_in, K, batch, p, x, labels, params0, running0)
                b = run(new, conf, emb_in, K, batch, p, x, labels, params0, running0)
                for step in range(2):
                    for key in ("loss", "scores", "grads", "running"):
                        same = torch.equal(a[step][key], b[step][key])
                        d = float((a[step][key] - b[step][key]).abs().max())
                        noise = float((a[0][key] - a[1][key]).abs().max())
                        scale = float(a[step][key].abs().max()) or 1.0
                        print(f"conf {conf} K {K} p {p} step {step} {key:8s}: bitwise={same} maxdiff={d:.3g} "
                              f"ref run-to-run={noise:.3g}", flush=True)
                        if not same:
                            not_bitwise.append((conf, K, p, step, key))
                            worst_gap = max(worst_gap, (d - noise) / scale)
    print("NOT BITWISE", not_bitwise)
    print("WORST (new-vs-ref minus ref run-to-run) / max|ref|", worst_gap)


if __name__ == "__main__":
    main()
