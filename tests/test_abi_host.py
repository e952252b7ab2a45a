"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares, its host-only helpers
agree with the reference's frame arithmetic and tables, the reference-name shims expose the documented surface
and fail loudly without a GPU, and the sharding arithmetic keeps frame indices (SURVEY §8b, §8e, H5)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT

from b200 import _lib, sharding
from b200._lib import B200Error


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "vggish_mla_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vmb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    names = _declared_symbols()
    assert len(names) >= 25
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} is declared in include/vggish_mla_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == names          # the ctypes table mirrors the header one to one
    assert _lib.lib().vmb_abi_version() == 2


def test_frame_arithmetic_matches_reference(golden_front):
    L = _lib.lib()
    for n, nf, ne in zip(golden_front["lengths"], golden_front["frames"], golden_front["n_examples"]):
        assert L.vmb_num_frames(int(n)) == nf
        assert L.vmb_num_examples(int(n)) == ne
        if ne >= 0:
            assert sharding.num_examples(int(n)) == ne
        else:
            with pytest.raises(ValueError):
                sharding.num_examples(int(n))
    assert L.vmb_num_examples(160000) == 10 and L.vmb_num_examples(57600000) == 3749     # F10


def test_tables_built_by_the_library_are_bit_exact(golden_front):
    hann = np.empty(400)
    mel = np.empty((257, 64))
    assert _lib.lib().vmb_front_end_tables(hann.ctypes.data, mel.ctypes.data) == 0
    assert np.array_equal(hann, golden_front["hann400"])
    assert np.array_equal(mel, golden_front["mel257x64"])


def test_compiled_mel_band_layout_matches_the_reference_matrix(golden_front):
    """The log-mel kernel's epilogue has the band interval of every evaluated DFT bin compiled in (kBandOfBin in
    csrc/logmel_tc.cu; the library re-checks it against its own float64 tables on the device box).  Here it is derived
    again from the reference's own spectrogram_to_mel_matrix output (mel_features.py:114-189, golden vector)."""
    src = open(os.path.join(ROOT, "audio-classification-using-a-deep-cnn-combined-with-multi-level-attention_b200",
                            "csrc", "logmel_tc.cu")).read()
    body = re.search(r"kBandOfBin\[kEvalBins\]\s*=\s*\{([^}]*)\}", src).group(1)
    compiled = [int(v) for v in body.replace("\n", " ").split(",") if v.strip()]
    mel = golden_front["mel257x64"]                            # (257, 64)
    assert mel.shape == (257, 64)
    lo, n = 4, 240                                             # kBinLo, kEvalBins
    assert not mel[:lo].any() and not mel[lo + n:].any()       # nothing outside the evaluated bins
    derived, prev = [], 0
    for k in range(lo, lo + n):
        nz = np.nonzero(mel[k])[0]
        assert len(nz) <= 2 and (len(nz) < 2 or nz[1] == nz[0] + 1)   # every bin feeds at most two adjacent bands
        e = prev
        if len(nz) == 2:
            e = int(nz[1])
        elif len(nz) == 1:
            e = int(nz[0]) if nz[0] >= prev else int(nz[0]) + 1
        assert prev <= e <= prev + 1 and all(m in (e - 1, e) for m in nz)
        derived.append(e)
        prev = e
    assert compiled == derived


def test_compute_entry_points_fail_loudly_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = _lib.lib()
    assert L.vmb_device_arch(0) < 0
    assert b"no CUDA device" in L.vmb_last_error()
    buf = np.zeros(16000, dtype=np.float32)
    out = np.zeros((98, 64), dtype=np.float32)
    assert L.vmb_logmel(buf.ctypes.data, 1, 16000, 16000, 98, out.ctypes.data, None) != 0
    assert not out.any()                                   # nothing was computed on the host
    from b200 import engine
    with pytest.raises(B200Error):
        engine.require_b200()
    import torchvggish.vggish_input as vi
    with pytest.raises((B200Error, RuntimeError, AssertionError)):
        vi.waveform_to_examples(np.zeros(16000), 16000)


def test_argument_validation_without_touching_the_device():
    L = _lib.lib()
    assert L.vmb_logmel(None, 1, 300, 300, 1, None, None) != 0
    assert b"shorter than one 400-sample window" in L.vmb_last_error()
    assert L.vmb_logmel(None, 1, 16000, 16000, 99, None, None) != 0           # only 98 frames exist
    assert L.vmb_mla_param_count(2, (ctypes.c_int * 2)(2, 1), 128, 600, 527, 10) == 2622727 - 2 * (527 * 600 + 527) + 2 * 10 * 9 + 2 * 527  # params - fcf + running stats
    assert L.vmb_launch_count() == 0


def test_constants_match_reference_values():
    import params
    from torchvggish import vggish_params as vp
    assert (vp.NUM_FRAMES, vp.NUM_BANDS, vp.EMBEDDING_SIZE, vp.SAMPLE_RATE) == (96, 64, 128, 16000)
    assert (vp.STFT_WINDOW_LENGTH_SECONDS, vp.STFT_HOP_LENGTH_SECONDS) == (0.025, 0.010)
    assert (vp.NUM_MEL_BINS, vp.MEL_MIN_HZ, vp.MEL_MAX_HZ, vp.LOG_OFFSET) == (64, 125, 7500, 0.01)
    assert (vp.EXAMPLE_WINDOW_SECONDS, vp.EXAMPLE_HOP_SECONDS) == (0.96, 0.96)
    assert (vp.QUANTIZE_MIN_VAL, vp.QUANTIZE_MAX_VAL) == (-2.0, 2.0)
    assert (vp.PCA_EIGEN_VECTORS_NAME, vp.PCA_MEANS_NAME) == ("pca_eigen_vectors", "pca_means")
    assert (params.T, params.M_VGGISH, params.M_VGGISH_JB, params.H, params.DR, params.K) == (10, 128, 12288, 600, 0.4, 10)
    assert params.S_VGGISH_SHAPE == (96, 64)


def test_shim_state_dict_keys_match_reference(golden_vggish, golden_head, golden_ensemble):
    import model
    from torchvggish.vggish import VGGish
    net = VGGish(urls={}, pretrained=False, preprocess=True, postprocess=True)
    assert sorted(net.state_dict().keys()) == list(golden_vggish["state_dict_keys"])
    old = model.K
    try:
        model.K = 527
        head = model.MultiLevelAttention([2, 1], 128)
        assert sorted(head.state_dict().keys()) == list(golden_head["keys_k527"])
        assert sum(p.numel() for p in head.parameters()) == int(golden_head["nparams_k527"])
        conf = dict(cnn_type="vggish", num_classes=527, use_pretrained=False, just_bottlenecks=False,
                    cnn_trainable=False, first_cnn_layer_trainable=False, in_channels=1)
        ens = model.Ensemble("repeat", conf, [2, 1], torch.device("cpu"))
        assert sorted(ens.state_dict().keys()) == list(golden_ensemble["keys"])
        assert not any(p.requires_grad for p in ens.cnn.parameters())          # frozen CNN (model.py:159-160)
        assert all(p.requires_grad for p in ens.mla.parameters())
        with pytest.raises(B200Error):
            ens(torch.zeros(1, 10, 1, 96, 64))                                 # CPU module: no fallback
        with pytest.raises(NotImplementedError):
            model.Ensemble("repeat", dict(conf, cnn_type="resnet"), [2, 1], torch.device("cpu"))
        with pytest.raises(Exception, match="CNN type is not valid"):
            model.Ensemble("repeat", dict(conf, cnn_type="alexnet"), [2, 1], torch.device("cpu"))
    finally:
        model.K = old
    assert model.MultiLevelAttention([2], 128).fc.out_features == old         # K is bound at construction (F1)


def test_just_bottlenecks_keys_pickling_and_host_side_guards():
    """CPU-side halves of the boundary checks: the just_bottlenecks Ensemble has the reference's re-wrapped key layout
    (model.py:161-166, tests/golden/levels.npz), modules pickle / deep-copy (the reference checkpoints whole objects,
    train.py:259-268), sub-modules raise instead of falling back without a GPU."""
    import copy
    import io
    import model
    from conftest import load_golden
    lv = load_golden("levels.npz")
    old = model.K
    try:
        model.K = 10
        conf = dict(cnn_type="vggish", num_classes=10, use_pretrained=False, just_bottlenecks=True, cnn_trainable=False,
                    first_cnn_layer_trainable=False, in_channels=1)
        ens = model.Ensemble("repeat", conf, [1], torch.device("cpu"))
    finally:
        model.K = old
    sd = ens.state_dict()
    assert sorted(sd.keys()) == list(lv["jb_keys"])
    assert [",".join(map(str, sd[k].shape)) for k in lv["jb_keys"]] == list(lv["jb_shapes"])
    assert not any(k.startswith("cnn.cnn_model.embeddings") for k in sd)
    clone = copy.deepcopy(ens)
    assert sorted(clone.state_dict().keys()) == sorted(sd.keys())
    buf = io.BytesIO()
    torch.save({"model": ens}, buf)
    buf.seek(0)
    back = torch.load(buf, weights_only=False)["model"]
    assert all(torch.equal(a, b) for a, b in zip(back.state_dict().values(), sd.values()))
    state = ens.mla.__getstate__()
    assert state["_handle"] is None and state["_train_state"] is None
    with pytest.raises(B200Error):
        ens.mla.embedded_mappings[0].eval()(torch.zeros(1, 10, 12288))         # CPU module: no fallback
    with pytest.raises(B200Error):
        ens.mla.attention_modules[0].eval()(torch.zeros(1, 10, 600))
    with pytest.raises(NotImplementedError):
        ens.mla.attention_modules[0].train()(torch.zeros(1, 10, 600))
    from torchvggish import mel_features as mf
    with pytest.raises(NotImplementedError):
        mf.stft_magnitude(np.zeros(1000), 1024, 160, 400)


def test_shim_error_behaviour():
    from torchvggish import mel_features as mf
    from torchvggish.vggish import Postprocessor, VGGish
    with pytest.raises(ValueError, match="must be >= 0"):
        mf.spectrogram_to_mel_matrix(lower_edge_hertz=-1.0)
    with pytest.raises(ValueError, match=">= upper_edge_hertz"):
        mf.spectrogram_to_mel_matrix(lower_edge_hertz=4000.0, upper_edge_hertz=3800.0)
    with pytest.raises(ValueError, match="greater than Nyquist"):
        mf.spectrogram_to_mel_matrix(upper_edge_hertz=5000.0)
    with pytest.raises(ValueError):
        mf.frame(np.zeros(10), 400, 160)                                      # negative frame count (F10)
    assert mf.frame(np.arange(1000.0), 400, 160).shape == (4, 400)
    assert mf.frame(np.arange(1000.0), 400, 160)[3, 0] == 480.0
    assert tuple(mf.frame(torch.arange(1000.0), 400, 160).shape) == (4, 400)
    with pytest.raises(AssertionError, match="Expected 2-d batch"):
        Postprocessor().postprocess(torch.zeros(128))
    with pytest.raises(AssertionError, match="Bad batch shape"):
        Postprocessor().postprocess(torch.zeros(2, 64))
    with pytest.raises(AttributeError):
        VGGish(urls={}, pretrained=False)(torch.zeros(3), 16000)              # vggish.py:175-180


def test_dp_slices_partition_the_padded_bucket():
    """vmb_dp_slice (csrc/dp_adam.cu): the slices of the ranks are disjoint, 16-byte aligned, in rank order, and cover
    the bucket padded to a multiple of four floats — host arithmetic, no device."""
    import ctypes as C
    L = _lib.lib()
    for n in (1, 3, 4, 5, 1023, 1989273, 823050):
        for world in range(1, 9):
            prev_end = 0
            for rank in range(world):
                b, e = C.c_longlong(-1), C.c_longlong(-1)
                L.vmb_dp_slice(n, world, rank, C.byref(b), C.byref(e))
                assert b.value == prev_end and e.value >= b.value and b.value % 4 == 0 and e.value % 4 == 0
                prev_end = e.value
            assert prev_end == (n + 3) // 4 * 4


def test_shard_bounds_partition():
    for n in (0, 1, 7, 256, 8192, 3749):
        for world in (1, 2, 3, 4, 8):
            cuts = [sharding.shard_bounds(n, r, world) for r in range(world)]
            assert cuts[0][0] == 0 and cuts[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
            sizes = [b - a for a, b in cuts]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        sharding.shard_bounds(4, 4, 4)


def test_stream_chunks_keep_frame_indices():
    n = 57_600_000                                                             # 1 hour at 16 kHz
    assert sharding.num_examples(n) == 3749
    seen = []
    for world in (1, 8):
        covered = []
        for r in range(world):
            for e0, e1, s0, s1 in sharding.stream_chunks(n, 500, r, world):
                assert s0 == e0 * 15360 and s1 - s0 == (e1 - e0 - 1) * 15360 + 15600 and s1 <= n
                assert sharding.num_examples(s1 - s0) == e1 - e0               # the chunk alone yields its examples
                covered.append((e0, e1))
        assert covered[0][0] == 0 and covered[-1][1] == 3749
        assert all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
        seen.append(covered)
    # frame 96*j of the stream starts at sample 15360*j: identical in every chunking
    from oracle import frontend_np
    sig = np.random.default_rng(0).standard_normal(15360 * 5 + 15600)
    whole = frontend_np.waveform_to_examples(sig)
    e0, e1, s0, s1 = 2, 5, *sharding.stream_sample_range(2, 5)
    part = frontend_np.waveform_to_examples(sig[s0:s1])
    assert np.array_equal(part, whole[e0:e1])


def test_pack_mla_params_layout(head_sd):
    from b200 import engine
    flat = engine.pack_mla_params(head_sd, (2, 1), torch.device("cpu"))
    conf = (ctypes.c_int * 2)(2, 1)
    assert flat.numel() == _lib.lib().vmb_mla_param_count(2, conf, 128, 600, 527, 10)
    # level 0: norm0 (4*T) then fc.0 weight
    assert torch.equal(flat[:10], head_sd["embedded_mappings.0.norm0.weight"])
    assert torch.equal(flat[40:40 + 600 * 128], head_sd["embedded_mappings.0.fc.0.weight"].reshape(-1))
    assert torch.equal(flat[-527:], head_sd["norm.running_var"])


def test_bench_reference_arm_prints_exactly_one_json_line():
    """bench.py contract: ONE JSON line on stdout (everything else, including what libraries print to fd 1, goes to
    stderr).  The reference arm runs on the CPU, so it can be exercised here with a tiny time budget."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, VMB_BENCH_CPU_BUDGET_S="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup",
                        "0"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "clips/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_reference_arm_dumps_the_scores_of_its_last_step(tmp_path):
    """--dump-outputs DIR: the reference arm writes the scores of its last timed pass, which are the oracle's scores of
    the first clips of the benchmark batch."""
    import json
    import subprocess
    import sys
    import bench
    from b200 import synth
    env = dict(os.environ, VMB_BENCH_CPU_BUDGET_S="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup",
                        "0", "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    n = json.loads(r.stdout)["reference_sample_clips_per_step"]
    got = np.load(tmp_path / "out" / "scores.npy")
    assert got.dtype == np.float32 and got.shape == (n, 527)
    want = bench.oracle_pass(synth.fast_clips(0, n).numpy(), synth.vggish_state_dict(0),
                             synth.mla_state_dict((2, 1), 128, 600, 527, 10, seed=2)).numpy()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-5)


def test_bench_dump_is_capped_to_a_fixed_sample(tmp_path):
    """Scores above bench.DUMP_MAX_BYTES are cut to the same sample of clips on every run, kept in clip order."""
    import bench
    scores = torch.rand(40000, 527, generator=torch.Generator().manual_seed(0))
    scores[:, 0] = torch.arange(40000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), scores)
    a, b = np.load(tmp_path / "a" / "scores.npy"), np.load(tmp_path / "b" / "scores.npy")
    assert os.path.getsize(tmp_path / "a" / "scores.npy") <= bench.DUMP_MAX_BYTES and np.array_equal(a, b)
    rows = a[:, 0].astype(np.int64)
    assert a.shape[0] > 30000 and np.all(np.diff(rows) > 0) and np.array_equal(a, scores.numpy()[rows])
