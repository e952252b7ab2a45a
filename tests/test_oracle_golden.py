"""The oracle (oracle/) against the golden vectors produced by the reference's own Python
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from b200 import synth
from oracle import frontend_np, model_torch

GOLDEN_THREADS = 8      # the CPU thread count make_golden.py ran the reference with


@pytest.fixture(autouse=True)
def _golden_thread_count():
    """torch splits fp32 reductions by thread count, so the last bits of the oracle's outputs depend on it: the oracle
    runs with the thread count the golden vectors were made with, whatever the host has."""
    threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(threads)


def test_tables_bit_exact(golden_front):
    assert np.array_equal(frontend_np.periodic_hann(400), golden_front["hann400"])
    assert np.array_equal(frontend_np.mel_matrix(), golden_front["mel257x64"])
    mel = golden_front["mel257x64"]
    nz = np.nonzero(mel.any(axis=1))[0]
    assert nz.min() == 5 and nz.max() == 239            # the kernel evaluates bins 4..239 only (SURVEY H1)


def test_logmel_and_examples(golden_front):
    waves = golden_front["waves_f32"]
    for i in range(4):
        w = waves[i].astype(np.float64)
        lm = frontend_np.log_mel_spectrogram(w)
        np.testing.assert_allclose(lm, golden_front["logmel_f64"][i], rtol=0, atol=1e-9)
        ex = frontend_np.waveform_to_examples(w)
        assert ex.shape == (1, 96, 64)
        np.testing.assert_allclose(ex, golden_front["examples_f64"][i], rtol=0, atol=1e-9)
    np.testing.assert_allclose(frontend_np.waveform_to_examples(waves[0].astype(np.float64)).astype(np.float32),
                               golden_front["examples_tensor_f32"][:, 0], rtol=0, atol=1e-6)


def test_stft_and_stereo(golden_front):
    waves = golden_front["waves_f32"]
    mag = frontend_np.stft_magnitude(waves[1].astype(np.float64), 512, 160, 400)[:8]
    np.testing.assert_allclose(mag, golden_front["stft_mag_clip1"], rtol=1e-12, atol=1e-12)
    stereo = np.stack([waves[0], waves[2]], axis=1).astype(np.float64)
    np.testing.assert_allclose(frontend_np.waveform_to_examples(stereo), golden_front["stereo_examples_f64"],
                               rtol=0, atol=1e-9)


def test_frame_counts(golden_front):
    for n, nf, ne in zip(golden_front["lengths"], golden_front["frames"], golden_front["n_examples"]):
        assert frontend_np.num_frames(int(n), 400, 160) == nf
        if n > 200000:
            continue
        if ne < 0:
            with pytest.raises(ValueError):
                frontend_np.waveform_to_examples(np.zeros(int(n)))
        else:
            assert frontend_np.waveform_to_examples(np.zeros(int(n))).shape[0] == ne


def test_synth_clips_reproduce_golden_inputs(golden_front):
    # the golden inputs are make_clips(0, 4, 19200): the generator must be stable across numpy versions
    np.testing.assert_array_equal(synth.make_clips(0, 4, 19200), golden_front["waves_f32"])


def test_vggish_and_postprocessor(golden_front, golden_vggish, vgg_sd):
    x = torch.from_numpy(golden_front["examples_f64"][:, 0]).float()[:, None]
    acts = []
    with torch.no_grad():
        emb = model_torch.vgg_forward(vgg_sd, x, acts)
    ref = golden_vggish["embeddings"]
    np.testing.assert_allclose(emb.numpy(), ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())
    eig, means = synth.pca_params(1)
    post = model_torch.postprocess(eig, means, torch.from_numpy(ref))
    assert post.dtype == torch.float32 and post.shape == (4, 128)                      # F6: float values 0..255
    assert np.array_equal(post.numpy(), golden_vggish["postprocessed"])
    assert model_torch.postprocess(eig, means, torch.from_numpy(ref[:1])).shape == (128,)   # squeeze quirk
    assert np.array_equal(model_torch.postprocess(eig, means, torch.from_numpy(ref[:1])).numpy(),
                          golden_vggish["postprocessed_single"])
    assert 0 < (post > 0).float().mean() < 1 and post.min() >= 0 and post.max() <= 255


@pytest.mark.parametrize("tag,K,conf,seed", [("k527", 527, (2, 1), 2), ("k10", 10, (2, 1), 2), ("c121", 10, (1, 2, 1), 5)])
def test_head_forward(golden_head, tag, K, conf, seed):
    sd = synth.mla_state_dict(conf, 128, 600, K, 10, seed=seed)
    x = torch.from_numpy(golden_head[f"x_{tag}"])
    with torch.no_grad():
        y = model_torch.mla_forward(sd, x, conf)
    np.testing.assert_allclose(y.numpy(), golden_head[f"y_{tag}"], rtol=0, atol=2e-6)
    assert y.shape[1] == K and float(y.min()) >= 0 and float(y.max()) <= 1                # sigmoid outputs (F2)


def test_head_param_inventory(golden_head):
    sd = synth.mla_state_dict((2, 1), 128, 600, 527, 10, seed=2)
    assert sorted(sd.keys()) == list(golden_head["keys_k527"])                            # 66 state_dict entries
    n_param = sum(v.numel() for k, v in sd.items() if "running_" not in k and "num_batches" not in k)
    assert n_param == int(golden_head["nparams_k527"]) == 2622727


def test_ensemble(golden_ensemble, vgg_sd, head_sd):
    waves = synth.make_clips(4, 2)
    ex = np.stack([frontend_np.waveform_to_examples(w.astype(np.float64)) for w in waves]).astype(np.float32)
    chk = golden_ensemble["examples_f32_checksum"]
    assert abs(ex.astype(np.float64).sum() - chk[0]) < 1e-3 * abs(chk[1]) * 1e-4
    with torch.no_grad():
        scores = model_torch.ensemble_forward(vgg_sd, head_sd, torch.from_numpy(ex)[:, :, None], (2, 1))
    np.testing.assert_allclose(scores.numpy(), golden_ensemble["scores"], rtol=0, atol=1e-4)


def test_head_training_step(golden_head):
    """One reference training step (train.py:124-138 semantics, dropout off): loss, outputs, gradients, Adam update
    and BatchNorm running statistics of the oracle against the reference module's."""
    from oracle import train_torch
    sd = synth.mla_state_dict((2, 1), 128, 600, 527, 10, seed=2)
    x = torch.from_numpy(golden_head["train_x"])
    labels = torch.from_numpy(golden_head["train_labels"])
    loss, scores, grads = train_torch.head_step(sd, x, labels, (2, 1))
    assert abs(loss.item() - float(golden_head["train_loss"])) < 1e-5
    np.testing.assert_allclose(scores.numpy(), golden_head["train_y"], rtol=0, atol=2e-6)
    assert sorted(k for k, g in grads.items() if g is None) == list(golden_head["train_no_grad_params"])
    for key in golden_head.files:
        if key.startswith("grad::"):
            name = key[len("grad::"):]
            g = grads[name].numpy()
            ref = golden_head[key]
            g = g[:ref.shape[0]] if g.shape != ref.shape else g
            np.testing.assert_allclose(g, ref, rtol=1e-3, atol=1e-7 + 1e-4 * np.abs(ref).max())
            after = train_torch.adam_update(sd[name], grads[name]).numpy()
            ref_after = golden_head["after::" + name]
            after = after[:ref_after.shape[0]] if after.shape != ref_after.shape else after
            np.testing.assert_allclose(after, ref_after, rtol=0, atol=2e-5)     # lr = 1e-3: sign errors would show as 2e-3
    names = list(golden_head["grad_names"])
    for name, ref_norm in zip(names, golden_head["grad_norms"]):
        got = 0.0 if grads[name] is None else grads[name].norm().item()
        assert abs(got - ref_norm) <= 1e-3 * ref_norm + 1e-9, name
    run = train_torch.updated_running_stats(sd, x, (2, 1))
    np.testing.assert_allclose(run["embedded_mappings.0.norm0.running_mean"].numpy(),
                               golden_head["running_mean_after::embedded_mappings.0.norm0"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(run["norm.running_var"].numpy(), golden_head["running_var_after::norm"], rtol=1e-4,
                               atol=1e-7)


def test_dataset_tiling_restatement():
    """The (64, 384) spectrogram + 10 overlapping (64, 96) windows of dataset.py:318-326, :355-359, restated with the
    oracle front end, against the reference's output."""
    from conftest import load_golden
    g = load_golden("dataset.npz")
    for tag, n in (("4s", 64000), ("2s5", 40000)):
        w = synth.make_clips(20, 1, n)[0].astype(np.float64)
        slots = frontend_np.waveform_to_examples(w)
        padded = np.zeros((4, 96, 64))
        padded[:slots.shape[0]] = slots
        spec = np.concatenate(np.swapaxes(padded, 1, 2), axis=1)
        chk = g[f"spec_checksum_{tag}"]
        assert abs(spec.sum() - chk[0]) < 1e-6 * chk[1]
        frames = np.stack([spec[:, i:i + 96] for i in range(0, 384, 288 // 9)][:10])
        np.testing.assert_allclose(frames, g[f"frames_{tag}"], rtol=0, atol=1e-5)
