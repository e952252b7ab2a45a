"""Generates the golden vectors under tests/golden/ by running the REFERENCE's own Python
(/root/reference, read-only) on seeded synthetic inputs.  Run in the build container only:

    python tests/golden/make_golden.py

The reference ships no tests, fixtures or checkpoints (SURVEY.md §4, F8), so these vectors — outputs of the
reference itself — are the pin for oracle/ and, through it, for the CUDA path.  The GPU box has no
/root/reference; tests read only the .npz files written here.

resampy / soundfile are imported at module top by the reference (vggish_input.py:22,27) but never touched for
16 kHz ndarray input; they are absent in this image, so empty stub modules stand in for them (SURVEY F9).
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PKG = os.path.join(ROOT, "audio-classification-using-a-deep-cnn-combined-with-multi-level-attention_b200")
REF = "/root/reference"

# synth.py has no dependency on the CUDA library; load it by path so the package's torchvggish/params names
# cannot shadow the reference's.
import importlib.util

_spec = importlib.util.spec_from_file_location("vmb_synth", os.path.join(PKG, "b200", "synth.py"))
synth = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(synth)

sys.path.insert(0, REF)
for name in ("resampy", "soundfile", "librosa", "librosa.display", "h5py", "matplotlib", "matplotlib.pyplot"):
    sys.modules.setdefault(name, types.ModuleType(name))     # imported at module top by the reference, never used here
sys.modules["librosa"].display = sys.modules["librosa.display"]
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
from torchvggish import mel_features as ref_mel  # noqa: E402
from torchvggish import vggish_input as ref_input  # noqa: E402
from torchvggish import vggish as ref_vggish  # noqa: E402
import model as ref_model  # noqa: E402
import dataset as ref_dataset  # noqa: E402

torch.manual_seed(0)
torch.set_num_threads(8)      # fp32 sums depend on the thread count: tests/test_oracle_golden.py runs the oracle with 8

SHORT = 19200  # 1.2 s -> 118 frames -> 1 example


def front_end():
    """4 short clips (one per signal family) + a stereo case + edge cases."""
    waves = synth.make_clips(0, 4, SHORT, dtype=np.float32)          # stored: the exact fp32 samples used
    out = {"waves_f32": waves}
    logmels, examples = [], []
    for i in range(4):
        w = waves[i].astype(np.float64)
        logmels.append(ref_mel.log_mel_spectrogram(w, audio_sample_rate=16000, log_offset=0.01,
                                                   window_length_secs=0.025, hop_length_secs=0.010,
                                                   num_mel_bins=64, lower_edge_hertz=125, upper_edge_hertz=7500))
        examples.append(ref_input.waveform_to_examples(w, 16000, return_tensor=False))
    out["logmel_f64"] = np.stack(logmels)                           # (4, 118, 64)
    out["examples_f64"] = np.stack(examples)                        # (4, 1, 96, 64)
    # tensor flavour of the API (F7): float32, (N, 1, 96, 64)
    t = ref_input.waveform_to_examples(waves[0].astype(np.float64), 16000)
    out["examples_tensor_f32"] = t.detach().numpy()
    # stereo (samples, channels) input, averaged over axis 1 (vggish_input.py:49-50)
    stereo = np.stack([waves[0], waves[2]], axis=1).astype(np.float64)
    out["stereo_examples_f64"] = ref_input.waveform_to_examples(stereo, 16000, return_tensor=False)
    # constant tables
    out["hann400"] = ref_mel.periodic_hann(400)
    out["mel257x64"] = ref_mel.spectrogram_to_mel_matrix(num_mel_bins=64, num_spectrogram_bins=257,
                                                          audio_sample_rate=16000, lower_edge_hertz=125,
                                                          upper_edge_hertz=7500)
    out["stft_mag_clip1"] = ref_mel.stft_magnitude(waves[1].astype(np.float64), 512, 160, 400)[:8]
    # frame counts for a sweep of lengths (F10): examples per length, -1 where the reference raises
    lengths = np.array([0, 1, 399, 400, 401, 559, 560, 15599, 15600, 15601, 30959, 30960, 160000, 57600000],
                       dtype=np.int64)
    frames, n_examples = [], []
    for n in lengths:
        nf = 1 + int(np.floor((int(n) - 400) / 160))
        frames.append(nf)
        if n > 200000:  # do not run a 1-hour stream through numpy here; the count follows from frame()
            n_examples.append(1 + (nf - 96) // 96)
            continue
        try:
            n_examples.append(ref_input.waveform_to_examples(np.zeros(int(n)), 16000, return_tensor=False).shape[0])
        except ValueError:
            n_examples.append(-1)
    out["lengths"], out["frames"], out["n_examples"] = lengths, np.array(frames), np.array(n_examples)
    np.savez_compressed(os.path.join(HERE, "front_end.npz"), **out)
    return out


def vggish(front):
    sd = synth.vggish_state_dict(0)
    net = ref_vggish.VGGish(urls={}, pretrained=False, preprocess=False, postprocess=False)
    net.load_state_dict(sd)
    net.eval()
    x = torch.from_numpy(front["examples_f64"][:, 0]).float()[:, None]      # (4, 1, 96, 64)
    acts = []
    with torch.no_grad():
        h = x
        for layer in net.features:
            h = layer(h)
            if isinstance(layer, torch.nn.MaxPool2d) or (isinstance(layer, torch.nn.ReLU)):
                acts.append(h.clone())
        emb = net(x)
    # per-layer fingerprints of the post-ReLU / post-pool activations: (mean, abs-max, value at a fixed index)
    finger = np.array([[a.mean().item(), a.abs().max().item(), a.flatten()[a.numel() // 3].item()] for a in acts])
    eig, means = synth.pca_params(1)
    pp = ref_vggish.Postprocessor()
    pp.load_state_dict({"pca_eigen_vectors": eig, "pca_means": means})
    with torch.no_grad():
        post = pp(emb)
        post1 = pp(emb[:1])                                                  # squeeze -> (128,)
    full = ref_vggish.VGGish(urls={}, pretrained=False, preprocess=True, postprocess=True)
    full.load_state_dict({**sd, "pproc.pca_eigen_vectors": eig, "pproc.pca_means": means})
    full.eval()
    with torch.no_grad():
        e2e = full(front["waves_f32"][2].astype(np.float64), 16000)          # ndarray -> postprocessed (128,)
    np.savez_compressed(os.path.join(HERE, "vggish.npz"), embeddings=emb.numpy(), layer_fingerprints=finger,
                        postprocessed=post.numpy(), postprocessed_single=post1.numpy(),
                        preprocess_postprocess=e2e.numpy(),
                        state_dict_keys=np.array(sorted(full.state_dict().keys())))
    return emb


def head():
    out = {}
    for K, tag in ((527, "k527"), (10, "k10")):
        ref_model.K = K
        conf = [2, 1]
        m = ref_model.MultiLevelAttention(conf, 128)
        sd = synth.mla_state_dict(conf, 128, 600, K, 10, seed=2)
        m.load_state_dict(sd)
        m.eval()
        g = torch.Generator().manual_seed(11)
        x = torch.randn(6, 10, 128, generator=g).abs() * 2.0               # post-ReLU-like embeddings
        with torch.no_grad():
            out[f"x_{tag}"] = x.numpy()
            out[f"y_{tag}"] = m(x).numpy()
        out[f"keys_{tag}"] = np.array(sorted(m.state_dict().keys()))
        out[f"nparams_{tag}"] = np.array(sum(p.numel() for p in m.parameters()))
    # a 3-level configuration too
    ref_model.K = 10
    conf = [1, 2, 1]
    m = ref_model.MultiLevelAttention(conf, 128)
    m.load_state_dict(synth.mla_state_dict(conf, 128, 600, 10, 10, seed=5))
    m.eval()
    x = torch.randn(3, 10, 128, generator=torch.Generator().manual_seed(12)).abs()
    with torch.no_grad():
        out["x_c121"], out["y_c121"] = x.numpy(), m(x).numpy()

    # one training step of the head (train.py:124-138, :369-372): CE on the sigmoid outputs, Adam lr 1e-3,
    # dropout disabled (DR = 0) so the step is deterministic; K = 527.
    ref_model.K, ref_model.DR = 527, 0.0
    m = ref_model.MultiLevelAttention([2, 1], 128)
    m.load_state_dict(synth.mla_state_dict([2, 1], 128, 600, 527, 10, seed=2))
    m.train()
    g = torch.Generator().manual_seed(21)
    x = torch.randn(16, 10, 128, generator=g)
    labels = torch.randint(0, 527, (16,), generator=g)
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=0.001)
    opt.zero_grad()
    y = m(x)
    loss = torch.nn.CrossEntropyLoss()(y, labels)
    loss.backward()
    grads = {n: (None if p.grad is None else p.grad.clone()) for n, p in m.named_parameters()}
    opt.step()
    out["train_x"], out["train_labels"] = x.numpy(), labels.numpy()
    out["train_y"], out["train_loss"] = y.detach().numpy(), np.array(loss.item())
    out["train_no_grad_params"] = np.array(sorted(n for n, gr in grads.items() if gr is None))
    for n in ("fc.weight", "norm.weight", "attention_modules.0.fcv.bias", "attention_modules.1.normv.weight",
              "embedded_mappings.0.fc.0.bias", "embedded_mappings.0.norm0.weight", "embedded_mappings.1.norms.0.bias"):
        # big matrices: keep the first 4 rows only (fixtures stay small); the norm of every gradient is kept below
        cut = (lambda a: a[:4] if a.size > 20000 else a)
        out["grad::" + n] = cut(grads[n].numpy())
        out["after::" + n] = cut(dict(m.named_parameters())[n].detach().numpy())
    out["grad_norms"] = np.array([0.0 if gr is None else gr.norm().item() for gr in grads.values()])
    out["grad_names"] = np.array(list(grads.keys()))
    out["running_mean_after::embedded_mappings.0.norm0"] = m.embedded_mappings[0].norm0.running_mean.numpy()
    out["running_var_after::norm"] = m.norm.running_var.numpy()
    ref_model.DR = 0.4
    np.savez_compressed(os.path.join(HERE, "head.npz"), **out)


def levels():
    """Standalone EmbeddedMapping.forward / AttentionModule.forward (model.py:217-222, :235-242) of the K = 527 head, and the
    state_dict key set of Ensemble(just_bottlenecks=True), whose CNN is re-wrapped as nn.Sequential (model.py:161-166)."""
    ref_model.K = 527
    m = ref_model.MultiLevelAttention([2, 1], 128)
    m.load_state_dict(synth.mla_state_dict([2, 1], 128, 600, 527, 10, seed=2))
    m.eval()
    x = torch.randn(6, 10, 128, generator=torch.Generator().manual_seed(11)).abs() * 2.0      # == head.npz x_k527
    with torch.no_grad():
        e0 = m.embedded_mappings[0](x)
        e1 = m.embedded_mappings[1](e0)
        y0 = m.attention_modules[0](e0)
        y1 = m.attention_modules[1](e1)
    ref_model.K = 10
    conf = dict(cnn_type="vggish", num_classes=10, use_pretrained=False, just_bottlenecks=True, cnn_trainable=False,
                first_cnn_layer_trainable=False, in_channels=1)
    ens = ref_model.Ensemble("repeat", conf, [1], torch.device("cpu"))
    sd = ens.state_dict()
    np.savez_compressed(os.path.join(HERE, "levels.npz"), x=x.numpy(), emb0=e0.numpy(), emb1=e1.numpy(), y0=y0.numpy(),
                        y1=y1.numpy(), jb_keys=np.array(sorted(sd.keys())),
                        jb_shapes=np.array([",".join(map(str, sd[k].shape)) for k in sorted(sd.keys())]))


def ensemble(front):
    """Ensemble.forward for the vggish branch (model.py:58-62): 2 clips x T = 10 examples, K = 527."""
    ref_model.K = 527
    conf = dict(cnn_type="vggish", num_classes=527, use_pretrained=False, just_bottlenecks=False, cnn_trainable=False,
                first_cnn_layer_trainable=False, in_channels=1)
    ens = ref_model.Ensemble("repeat", conf, [2, 1], torch.device("cpu"))
    ens.cnn.cnn_model.load_state_dict(synth.vggish_state_dict(0))
    ens.mla.load_state_dict(synth.mla_state_dict([2, 1], 128, 600, 527, 10, seed=2))
    ens.eval()
    waves = synth.make_clips(4, 2, 160000, dtype=np.float32)                 # clips 4 and 5 (families 0, 1)
    ex = torch.stack([ref_input.waveform_to_examples(w.astype(np.float64), 16000).detach() for w in waves])
    with torch.no_grad():
        scores = ens(ex)                                                     # (2, 527)
        emb = ens.cnn(ens.input(ex))
    np.savez_compressed(os.path.join(HERE, "ensemble.npz"), clip_indices=np.array([4, 5]), scores=scores.numpy(),
                        embeddings=emb.numpy(), examples_f32_checksum=np.array([ex.double().sum().item(),
                                                                                ex.double().abs().sum().item()]),
                        keys=np.array(sorted(ens.state_dict().keys())))


def dataset_tiling():
    """dataset.create_spec (torchvggish branch) + dataset.split for a full 4 s clip and a 2.5 s one (2 examples)."""
    out = {}
    for tag, n in (("4s", 64000), ("2s5", 40000)):
        w = synth.make_clips(20, 1, n, dtype=np.float32)[0]
        spec = ref_dataset.create_spec(w.astype(np.float64), "vggish", 16000, 64000, 96, 64, False, True)
        # inputs are synth.make_clips(20, 1, n) (reproducible, see test_synth_clips_reproduce_golden_inputs)
        out[f"spec_checksum_{tag}"] = np.array([spec.sum(), np.abs(spec).sum()])
        out[f"frames_{tag}"] = ref_dataset.split(spec, 10, 96, 64, True).astype(np.float32)
    w = synth.make_clips(20, 1, 64000, dtype=np.float32)[0]
    spec = ref_dataset.create_spec(w.astype(np.float64), "vggish", 16000, 64000, 96, 64, False, False)
    out["frames_contig_4s"] = ref_dataset.split(spec, 4, 96, 64, False).astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "dataset.npz"), **out)


if __name__ == "__main__":
    dataset_tiling()
    f = front_end()
    vggish(f)
    head()
    levels()
    ensemble(f)
    for fn in sorted(os.listdir(HERE)):
        if fn.endswith(".npz"):
            print(fn, os.path.getsize(os.path.join(HERE, fn)))
