"""GPU parity tests: the CUDA path (through the C-ABI library) against the oracle and the golden vectors.

Tolerances (BASELINE.json north_star):
  * frame indexing, tables: bit-exact
  * log-mel: <= 1e-4 absolute against the float64 reference
  * conv / FC layers (16-bit operands, fp32 accumulation): per layer max-abs <= 0.5 % of the layer's max activation
    and cosine >= 0.9999 against fp32 math on the same operands; embeddings of the default fp16 body <= 0.3 %
    (measured 0.12 %), of the bf16 body <= 1.5 % (0.9 %), of the split body <= 0.05 % (0.016 %)
  * head (fp32 CUDA cores): <= 2e-5 absolute on the sigmoid scores given identical embeddings
  * postprocessor: bit-exact on identical fp32 embeddings except where fp32 summation order straddles a
    quantisation boundary (+-1 LSB, counted and bounded)
  * mAP on the fixed synthetic label set (SURVEY 8d's recipe): identical to 3 decimals for the benchmarked (fp16) mode
"""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from b200 import _lib, engine, sharding, synth
from oracle import frontend_np, model_torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def vgg_handle(vgg_sd):
    h = engine.VggishHandle(vgg_sd, DEV)
    yield h
    h.close()


@pytest.fixture(scope="module")
def head_handle(head_sd):
    h = engine.MlaHandle(head_sd, (2, 1), 128, 600, 527, 10, DEV)
    yield h
    h.close()


def test_library_is_the_thing_that_runs():
    engine.require_b200(DEV)
    before = _lib.lib().vmb_launch_count()
    engine.logmel(torch.zeros(1, 16000, device=DEV))
    torch.cuda.synchronize()
    # one fused kernel (framing + tcgen05 DFT + mel + log) + the float64 kernel that redoes the frames it flagged
    assert _lib.lib().vmb_launch_count() == before + 2


# ------------------------------------------------------------------------------------------------ front end
def test_logmel_golden(golden_front):
    waves = torch.from_numpy(golden_front["waves_f32"]).to(DEV)
    lm = engine.logmel(waves).cpu().numpy().astype(np.float64)
    ref = golden_front["logmel_f64"]
    assert lm.shape == ref.shape == (4, 118, 64)
    err = np.abs(lm - ref).max(axis=(1, 2))
    print("log-mel max-abs error per signal family:", err)
    assert err.max() <= 1e-4


@pytest.mark.parametrize("first", [0, 4])
def test_logmel_full_clips_vs_oracle(first):
    waves = synth.make_clips(first, 4)                                   # 10 s clips, all four families
    got = engine.logmel(torch.from_numpy(waves).to(DEV)).cpu().numpy().astype(np.float64)
    assert got.shape == (4, 998, 64)
    for i in range(4):
        ref = frontend_np.log_mel_spectrogram(waves[i].astype(np.float64))
        assert np.abs(got[i] - ref).max() <= 1e-4


def test_logmel_full_batch_tensor_core_vs_cuda_core():
    """Full bench size (256 clips): the tcgen05 kernel against the independent fp32 CUDA-core kernel on the device
    (both are within 1e-4 of the float64 reference, so they must agree within 2e-4), plus row independence."""
    waves = synth.fast_clips(0, 256).to(DEV)
    a = engine.logmel(waves)
    b = engine.logmel_cudacore(waves)
    assert a.shape == b.shape == (256, 998, 64)
    d = (a - b).abs().max().item()
    print(f"log-mel tensor-core vs CUDA-core over 256 clips: max-abs diff {d:.3e}")
    assert d <= 2e-4 and torch.isfinite(a).all()
    assert torch.equal(engine.logmel(waves[200:203]), a[200:203])


def test_logmel_unaligned_input_takes_the_plane_kernel():
    """The centred kernel reads the waveform through TMA (16-byte aligned base / clip stride); anything else is served
    by the first tensor-core kernel (bf16 planes + straight DFT).  Both stay within the 1e-4 bound, and one launch
    more (the split pass) shows which path ran; both are followed by the float64 kernel for flagged frames."""
    waves = synth.make_clips(0, 2)
    w = torch.from_numpy(waves).to(DEV)
    lib = _lib.lib()
    for sl, launches in ((slice(0, 32000), 2), (slice(1, 32001), 3), (slice(3, 32003), 3)):
        x = w[0, sl]
        before = lib.vmb_launch_count()
        got = engine.logmel(x)[0].cpu().numpy().astype(np.float64)
        assert lib.vmb_launch_count() == before + launches
        ref = frontend_np.log_mel_spectrogram(waves[0, sl].astype(np.float64))
        assert np.abs(got - ref).max() <= 1e-4
    # the same for 16-bit PCM: an odd sample offset is served by the plane kernel, and both paths agree with the float
    # path of the same alignment class bit for bit
    pcm = torch.from_numpy((waves[0, :32001] * 20000).astype(np.int16)).to(DEV)
    for sl in (slice(0, 32000), slice(1, 32001)):
        before = lib.vmb_launch_count()
        a = engine.logmel_pcm16(pcm[sl])
        assert lib.vmb_launch_count() == before + (2 if sl.start == 0 else 3)
        ref = frontend_np.log_mel_spectrogram(pcm[sl].cpu().numpy() / 32768.0)
        assert np.abs(a[0].cpu().numpy() - ref).max() <= 1e-4
    # two clips whose stride is not a multiple of four samples
    odd = torch.zeros(2, 32001, device=DEV)
    odd[:, :32000] = w[:, :32000]
    got = engine.logmel(odd[:, :32000]).cpu().numpy().astype(np.float64)
    for i in range(2):
        assert np.abs(got[i] - frontend_np.log_mel_spectrogram(waves[i, :32000].astype(np.float64))).max() <= 1e-4


def test_logmel_ill_conditioned_frames_take_the_float64_kernel():
    """north_star: log-mel within 1e-4 of the float64 reference.  Loud tonal / band-limited signals over digitally
    silent bands are where a 22-bit tensor-core DFT cannot get there (log(x + 0.01) has slope 100 at an empty band):
    the epilogue flags those frames (energy / quietest band > 3500) and logmel_exact_kernel redoes them in float64.
    Every case must meet the bound, on the aligned (centred kernel) and the unaligned (plane kernel) path."""
    n = 16000
    t = np.arange(n + 8)
    rng = np.random.default_rng(0)
    lp = np.fft.rfft(rng.standard_normal(n + 8))
    lp[len(lp) // 4:] = 0
    cases = {
        "fp32 tone": np.sin(t * 1.3) * 0.9,
        "two int16 tones": ((np.sin(t * 0.31) + np.sin(t * 1.9)) * 16000).astype(np.int16) / 32768.0,
        "tone + 3e-4 noise": np.sin(t * 0.4) * 0.5 + 3e-4 * rng.standard_normal(n + 8),
        "tone + 1e-3 noise": np.sin(t * 0.4) * 0.5 + 1e-3 * rng.standard_normal(n + 8),
        "quiet tone": np.sin(t * 0.4) * 0.1,
        "low-passed noise": np.fft.irfft(lp, n + 8) * 0.5,
        "harmonic stack": sum(np.sin(t * 0.08 * h) / h for h in range(1, 12)) * 0.3,
        "decaying tone": np.sin(t * 0.2) * np.exp(-t / 800.0),
        "square wave": np.sign(np.sin(t * 0.1)) * 0.8,
    }
    worst = 0.0
    for name, x in cases.items():
        x = x.astype(np.float32)
        w = torch.from_numpy(x).to(DEV)
        for off in (0, 1):                                   # 0: centred TMA kernel, 1: plane kernel
            got = engine.logmel(w[off:off + n])[0].cpu().numpy().astype(np.float64)
            ref = frontend_np.log_mel_spectrogram(x[off:off + n].astype(np.float64))
            err = np.abs(got - ref).max()
            worst = max(worst, err)
            print(f"log-mel {name:18s} {'plane' if off else 'centred'} kernel: max-abs error {err:.2e}")
            assert err <= 1e-4, (name, off)
    # a batch that mixes flagged and clean clips (and rows past the end of the last tile) stays row-independent
    mix = torch.stack([torch.from_numpy(cases["fp32 tone"][:n].astype(np.float32)),
                       torch.from_numpy(synth.make_clips(0, 1, n)[0]),
                       torch.from_numpy(cases["harmonic stack"][:n].astype(np.float32))]).to(DEV)
    out = engine.logmel(mix)
    for i in range(3):
        assert torch.equal(out[i], engine.logmel(mix[i])[0])


def test_examples_shape_indexing_and_edges():
    waves = synth.make_clips(0, 2)
    ex = engine.examples_from_wave(torch.from_numpy(waves).to(DEV))
    assert tuple(ex.shape) == (20, 96, 64) and ex.dtype == torch.float32
    ref = frontend_np.waveform_to_examples(waves[1].astype(np.float64))
    assert np.abs(ex[10:].cpu().numpy() - ref).max() <= 1e-4
    # frame i of the log-mel starts at sample 160 i: computing a shifted slice reproduces shifted frames exactly
    w = torch.from_numpy(waves[0]).to(DEV)
    whole = engine.logmel(w)[0]
    part = engine.logmel(w[160 * 37:160 * 37 + 16000])[0]
    assert torch.equal(part, whole[37:37 + part.shape[0]])
    # lengths around the edges (F10)
    assert engine.logmel(torch.zeros(400, device=DEV)).shape == (1, 1, 64)
    assert engine.logmel(torch.zeros(559, device=DEV)).shape == (1, 1, 64)
    assert engine.logmel(torch.zeros(560, device=DEV)).shape == (1, 2, 64)
    assert engine.examples_from_wave(torch.zeros(15599, device=DEV)).shape[0] == 0
    assert engine.examples_from_wave(torch.zeros(15600, device=DEV)).shape[0] == 1
    with pytest.raises(ValueError):
        engine.logmel(torch.zeros(100, device=DEV))
    # silence: log(0 + 0.01)
    z = engine.logmel(torch.zeros(1, 4000, device=DEV))
    assert torch.allclose(z, torch.full_like(z, float(np.log(0.01))), atol=1e-6)
    # strided rows (clip_stride > samples_per_clip) are honoured
    big = torch.from_numpy(waves).to(DEV)
    assert torch.equal(engine.logmel(big[:, :32000]), engine.logmel(big[:, :32000].contiguous()))


def test_reference_named_front_end_api(golden_front):
    from torchvggish import mel_features, vggish_input
    w = golden_front["waves_f32"][0].astype(np.float64)
    t = vggish_input.waveform_to_examples(w, 16000)
    assert tuple(t.shape) == (1, 1, 96, 64) and t.dtype == torch.float32 and t.is_cuda
    assert np.abs(t.cpu().numpy() - golden_front["examples_tensor_f32"]).max() <= 1e-4
    a = vggish_input.waveform_to_examples(w, 16000, return_tensor=False)
    assert a.dtype == np.float64 and a.shape == (1, 96, 64)
    stereo = np.stack([golden_front["waves_f32"][0], golden_front["waves_f32"][2]], axis=1).astype(np.float64)
    s = vggish_input.waveform_to_examples(stereo, 16000, return_tensor=False)
    assert np.abs(s - golden_front["stereo_examples_f64"]).max() <= 1e-4
    lm = mel_features.log_mel_spectrogram(w, audio_sample_rate=16000, log_offset=0.01, window_length_secs=0.025,
                                          hop_length_secs=0.010, num_mel_bins=64, lower_edge_hertz=125,
                                          upper_edge_hertz=7500)
    assert np.abs(lm - golden_front["logmel_f64"][0]).max() <= 1e-4
    with pytest.raises(NotImplementedError):
        vggish_input.waveform_to_examples(w, 22050)
    with pytest.raises(ValueError):
        vggish_input.waveform_to_examples(np.zeros(100), 16000)


# ------------------------------------------------------------------------------------------------ VGGish layers
def _layer_check(got, ref, name, rel_tol=0.015, cos_tol=0.9999):
    got, ref = got.float().cpu(), ref.float().cpu()
    rel = (got - ref).abs().max().item() / (ref.abs().max().item() + 1e-12)
    cos = F.cosine_similarity(got.flatten(), ref.flatten(), dim=0).item()
    print(f"{name}: rel-max-err {rel:.3e} cos {cos:.6f}")
    assert not torch.isnan(got).any()
    assert rel <= rel_tol and cos >= cos_tol, name


DTYPES = [(0, torch.bfloat16, 0.005), (1, torch.float16, 0.0007)]       # (C-ABI dtype code, torch dtype, output rounding bound)


@pytest.mark.parametrize("dt", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("n,H,W,Cin,Cout,pool", [(3, 48, 32, 64, 128, 1), (3, 24, 16, 128, 256, 0),
                                                 (3, 24, 16, 256, 256, 1), (5, 12, 8, 256, 512, 0),
                                                 (5, 12, 8, 512, 512, 1), (1, 12, 8, 256, 512, 0)])
def test_conv3x3_layer(n, H, W, Cin, Cout, pool, dt):
    code, tdt, tol = dt
    g = torch.Generator().manual_seed(H * 7 + Cin + n)
    x = torch.randn(n, Cin, H, W, generator=g).to(DEV).to(tdt)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) * (2.0 / (9 * Cin)) ** 0.5).to(DEV).to(tdt)
    b = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    w_k = w.permute(0, 2, 3, 1).contiguous().reshape(Cout, 9 * Cin)
    Ho, Wo = (H // 2, W // 2) if pool else (H, W)
    out = torch.full((n, Ho, Wo, Cout), float("nan"), device=DEV, dtype=tdt)
    engine.check(_lib.lib().vmb_conv3x3_relu_ex(x_nhwc.data_ptr(), w_k.data_ptr(), b.data_ptr(), out.data_ptr(), n, H, W,
                                                Cin, Cout, pool, code, engine.stream_ptr()), "vmb_conv3x3_relu_ex")
    ref = F.relu(F.conv2d(x.float(), w.float(), b, padding=1))           # same 16-bit-rounded operands, fp32 math
    if pool:
        ref = F.max_pool2d(ref, 2, 2)
    _layer_check(out.permute(0, 3, 1, 2), ref, f"conv {H}x{W} {Cin}->{Cout} pool={pool} {tdt}", rel_tol=tol)


@pytest.mark.parametrize("dt", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("n", [1, 3, 77])
def test_pair_kernel_bit_identical_to_single_cta(n, dt):
    """The CTA-pair (tcgen05 cta_group::2) kernel and the single-CTA kernel run the same K order into fp32 TMEM
    accumulators: their outputs must be bit-identical, including odd tile counts (the partner CTA of the last pair then
    works on an out-of-range tile that TMA zero-fills and the epilogue masks)."""
    L = _lib.lib()
    code, tdt, _ = dt
    g = torch.Generator().manual_seed(n)
    cases = []
    for (H, W, Cin, Cout, pool) in [(24, 16, 128, 256, 0), (24, 16, 256, 256, 1), (12, 8, 256, 512, 0), (12, 8, 512, 512, 1)]:
        x = torch.randn(n, H, W, Cin, generator=g).to(DEV).to(tdt)
        w = (torch.randn(Cout, 9 * Cin, generator=g) * 0.03).to(DEV).to(tdt)
        b = torch.randn(Cout, generator=g).to(DEV)
        shape = (n, H // 2, W // 2, Cout) if pool else (n, H, W, Cout)
        cases.append((f"conv {H}x{W} {Cin}->{Cout} p{pool}", shape,
                      lambda o, x=x, w=w, b=b, H=H, W=W, Cin=Cin, Cout=Cout, pool=pool: L.vmb_conv3x3_relu_ex(
                          x.data_ptr(), w.data_ptr(), b.data_ptr(), o.data_ptr(), n, H, W, Cin, Cout, pool, code,
                          engine.stream_ptr())))
    # the last shape leaves 12 of 160 pair tiles for an incomplete third round: they go to the single-CTA kernel
    for (M, N, K) in [(n, 4096, 4096), (256 + n, 256, 12288), (130 * n, 512, 128), (2560 - n, 4096, 512)]:
        a = torch.randn(M, K, generator=g).to(DEV).to(tdt)
        w = (torch.randn(N, K, generator=g) * 0.02).to(DEV).to(tdt)
        b = torch.randn(N, generator=g).to(DEV)
        cases.append((f"linear {M}x{N}x{K}", (M, N),
                      lambda o, a=a, w=w, b=b, M=M, N=N, K=K: L.vmb_linear_ex(a.data_ptr(), w.data_ptr(), b.data_ptr(),
                                                                              o.data_ptr(), 0, 1, M, N, K, code,
                                                                              engine.stream_ptr())))
    prev = L.vmb_igemm_pair_enable(1)
    try:
        for name, shape, fn in cases:
            outs = []
            for pair in (1, 0):
                L.vmb_igemm_pair_enable(pair)
                o = torch.full(shape, float("nan"), device=DEV, dtype=tdt)
                engine.check(fn(o), name)
                torch.cuda.synchronize()
                outs.append(o)
            assert not torch.isnan(outs[0].float()).any(), name
            assert torch.equal(outs[0], outs[1]), name
    finally:
        L.vmb_igemm_pair_enable(-1)
    assert prev in (0, 1)


@pytest.mark.parametrize("H,W,Cin,Cout", [(48, 32, 64, 128), (24, 16, 128, 256), (24, 16, 256, 256)])
def test_halo_boxes_bit_identical_to_per_tap_boxes(H, W, Cin, Cout):
    """conv2 (256 x 128 single-CTA tiles) and conv3_x (CTA-pair tiles): the haloed-box kernels (one activation box per
    dx feeding the three dy taps) against the one-box-per-tap kernels, and against the small-batch path on a slice of
    the batch — every bf16 conv kernel adds the partial products in the same (channel block, dx, dy) order."""
    L = _lib.lib()
    g = torch.Generator().manual_seed(11 + Cin)
    n = 77
    x = torch.randn(n, H, W, Cin, generator=g).to(DEV).bfloat16()
    w = (torch.randn(Cout, 9 * Cin, generator=g) * 0.04).to(DEV).bfloat16()
    b = torch.randn(Cout, generator=g).to(DEV)

    def run(xx, pool):
        m = xx.shape[0]
        o = torch.full((m, H // 2, W // 2, Cout) if pool else (m, H, W, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
        engine.check(L.vmb_conv3x3_relu(xx.data_ptr(), w.data_ptr(), b.data_ptr(), o.data_ptr(), m, H, W, Cin, Cout, pool,
                                        engine.stream_ptr()), "vmb_conv3x3_relu")
        torch.cuda.synchronize()
        return o

    try:
        for pool in (1, 0):
            L.vmb_igemm_halo_enable(1)
            a = run(x, pool)
            small = run(x[:5].contiguous(), pool)          # 5 images: for conv2 the 128 x 128 tile path
            L.vmb_igemm_halo_enable(0)
            c = run(x, pool)
            L.vmb_igemm_pair_enable(0)                     # and the single-CTA per-tap kernel
            d = run(x, pool)
            L.vmb_igemm_pair_enable(-1)
            assert not torch.isnan(a.float()).any()
            assert torch.equal(a, c) and torch.equal(a, d) and torch.equal(a[:5], small)
    finally:
        L.vmb_igemm_halo_enable(-1)
        L.vmb_igemm_pair_enable(-1)


@pytest.mark.parametrize("dt", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("M,N,K,f32", [(1, 128, 64, 1), (10, 4096, 12288, 0), (130, 256, 512, 0), (257, 128, 4096, 1)])
def test_linear_layer(M, N, K, f32, dt):
    code, tdt, tol = dt
    g = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).to(DEV).to(tdt)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(DEV).to(tdt)
    b = torch.randn(N, generator=g).to(DEV)
    out = torch.full((M, N), float("nan"), device=DEV, dtype=torch.float32 if f32 else tdt)
    engine.check(_lib.lib().vmb_linear_ex(a.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(), f32, 1, M, N, K, code,
                                          engine.stream_ptr()), "vmb_linear_ex")
    ref = F.relu(a.float() @ w.float().t() + b)
    _layer_check(out, ref, f"linear {M}x{N}x{K} {tdt}", rel_tol=1e-5 if f32 else tol)


def test_conv1_layer(vgg_sd):
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(7, 96, 64, generator=g) * 2 - 3).to(DEV)
    w, b = vgg_sd["features.0.weight"].to(DEV), vgg_sd["features.0.bias"].to(DEV)
    out = torch.empty(7, 48, 32, 64, device=DEV, dtype=torch.bfloat16)
    engine.check(_lib.lib().vmb_conv1_relu_pool(x.data_ptr(), w.contiguous().data_ptr(), b.data_ptr(), out.data_ptr(), 7,
                                                engine.stream_ptr()), "vmb_conv1_relu_pool")
    ref = F.max_pool2d(F.relu(F.conv2d(x[:, None], w, b, padding=1)), 2, 2)
    _layer_check(out.permute(0, 3, 1, 2), ref, "conv1 (tensor cores)", rel_tol=0.005)
    out16 = torch.empty(7, 48, 32, 64, device=DEV, dtype=torch.float16)
    engine.check(_lib.lib().vmb_conv1_relu_pool_ex(x.data_ptr(), w.contiguous().data_ptr(), b.data_ptr(), out16.data_ptr(),
                                                   7, 1, engine.stream_ptr()), "vmb_conv1_relu_pool_ex")
    _layer_check(out16.permute(0, 3, 1, 2), ref, "conv1 (tensor cores, fp16 output)", rel_tol=0.0007)
    out2 = torch.empty_like(out)
    engine.check(_lib.lib().vmb_conv1_relu_pool_cudacore(x.data_ptr(), w.contiguous().data_ptr(), b.data_ptr(),
                                                         out2.data_ptr(), 7, engine.stream_ptr()), "conv1 cudacore")
    _layer_check(out2.permute(0, 3, 1, 2), ref, "conv1 (CUDA-core cross-check)", rel_tol=0.005)
    # large batch: the two kernels agree to bf16 rounding (weights are bf16 on the tensor-core path)
    xb = (torch.randn(300, 96, 64, generator=g) * 3).to(DEV)
    o1 = torch.empty(300, 48, 32, 64, device=DEV, dtype=torch.bfloat16)
    o2 = torch.empty_like(o1)
    engine.check(_lib.lib().vmb_conv1_relu_pool(xb.data_ptr(), w.contiguous().data_ptr(), b.data_ptr(), o1.data_ptr(), 300,
                                                engine.stream_ptr()), "conv1")
    engine.check(_lib.lib().vmb_conv1_relu_pool_cudacore(xb.data_ptr(), w.contiguous().data_ptr(), b.data_ptr(),
                                                         o2.data_ptr(), 300, engine.stream_ptr()), "conv1 cudacore")
    _layer_check(o1, o2, "conv1 tensor cores vs CUDA cores, 300 examples", rel_tol=0.01)


def test_vggish_embeddings_vs_golden_and_oracle(golden_front, golden_vggish, vgg_handle, vgg_sd):
    x = torch.from_numpy(golden_front["examples_f64"][:, 0]).float().to(DEV)
    emb, bott = vgg_handle.forward(x, want_bottleneck=True)
    _layer_check(emb, torch.from_numpy(golden_vggish["embeddings"]), "embeddings vs reference golden", rel_tol=0.003)
    with torch.no_grad():
        feats = model_torch.vgg_flatten(model_torch.vgg_features(vgg_sd, x.cpu()[:, None]))
    _layer_check(bott, feats, "conv features (h,w,c) flatten order")
    assert tuple(vgg_handle.forward(x[:, None]).shape) == (4, 128)
    assert vgg_handle.forward(torch.empty(0, 96, 64, device=DEV)).shape == (0, 128)
    with pytest.raises(ValueError):
        vgg_handle.forward(torch.zeros(2, 64, 96, device=DEV))


def test_vggish_batch_invariance(vgg_handle):
    """An example's embedding must not depend on its position in the batch or on the batch size (sharding relies
    on it): bit-identical."""
    ex = engine.examples_from_wave(torch.from_numpy(synth.make_clips(0, 3)).to(DEV))      # 30 examples
    full = vgg_handle.forward(ex)
    assert torch.equal(vgg_handle.forward(ex[7:19]), full[7:19])
    assert torch.equal(vgg_handle.forward(ex[29:30]), full[29:30])


def test_postprocessor(golden_vggish):
    eig, means = synth.pca_params(1)
    emb = torch.from_numpy(golden_vggish["embeddings"])
    out, u8 = engine.postprocess(emb.to(DEV), eig.to(DEV), means.to(DEV), want_u8=True)
    ref = golden_vggish["postprocessed"]
    diff = np.abs(out.cpu().numpy() - ref)
    print("postprocess: LSB histogram on identical fp32 embeddings:", np.bincount(diff.astype(np.int64).ravel()))
    assert diff.max() <= 1 and (diff > 0).mean() <= 0.01
    assert u8.dtype == torch.uint8 and np.array_equal(u8.cpu().numpy().astype(np.float32), out.cpu().numpy())
    # larger random batch against the oracle, incl. values that clamp at both ends
    g = torch.Generator().manual_seed(9)
    big = torch.randn(1001, 128, generator=g).abs() * 6
    got = engine.postprocess(big.to(DEV), eig.to(DEV), means.to(DEV)).cpu()
    want = model_torch.postprocess(eig, means, big)
    d = (got - want).abs()
    assert d.max() <= 1 and (d > 0).float().mean() <= 0.01
    assert got.min() >= 0 and got.max() <= 255 and (got == 0).any() and (got == 255).any()


def test_reference_named_vggish_module(golden_front, golden_vggish, vgg_sd):
    from torchvggish.vggish import VGGish
    eig, means = synth.pca_params(1)
    net = VGGish(urls={}, pretrained=False, preprocess=True, postprocess=True)
    net.load_state_dict({**vgg_sd, "pproc.pca_eigen_vectors": eig, "pproc.pca_means": means})
    net = net.to(DEV).eval()
    out = net(golden_front["waves_f32"][2].astype(np.float64), 16000)
    assert tuple(out.shape) == (128,) and out.dtype == torch.float32                  # squeeze + float 0..255 (F6)
    ref = golden_vggish["preprocess_postprocess"]
    d = np.abs(out.cpu().numpy() - ref)
    print("VGGish(preprocess, postprocess) vs reference: LSB histogram", np.bincount(d.astype(np.int64)))
    assert d.max() <= 1 and (d == 0).mean() >= 0.9        # default fp16 body: measured 127 exact + 1 at +-1 LSB of 128
    plain = VGGish(urls={}, pretrained=False, preprocess=False, postprocess=False)
    plain.load_state_dict(vgg_sd)
    plain = plain.to(DEV).eval()
    x = torch.from_numpy(golden_front["examples_tensor_f32"]).to(DEV)
    _layer_check(plain(x), torch.from_numpy(golden_vggish["embeddings"][:1]), "VGGish module")
    # in-place weight update invalidates the cached library handle
    with torch.no_grad():
        plain.embeddings[4].bias.add_(1.0)
    ref1 = torch.from_numpy(golden_vggish["embeddings"][:1]).to(DEV)
    moved = plain(x) - ref1
    assert (moved[ref1 > 0] > 0.9).all() and (moved >= 0).all()


# ------------------------------------------------------------------------------------------------ head
@pytest.mark.parametrize("tag,K,conf,seed", [("k527", 527, (2, 1), 2), ("k10", 10, (2, 1), 2), ("c121", 10, (1, 2, 1), 5)])
def test_head_vs_golden(golden_head, tag, K, conf, seed):
    sd = synth.mla_state_dict(conf, 128, 600, K, 10, seed=seed)
    h = engine.MlaHandle(sd, conf, 128, 600, K, 10, DEV)
    x = torch.from_numpy(golden_head[f"x_{tag}"]).to(DEV)
    y = h.forward(x).cpu().numpy()
    ref = golden_head[f"y_{tag}"]
    y32 = h.forward(x, fp32_crosscheck=True).cpu().numpy()
    print(f"head {tag}: max-abs-err tensor-core path {np.abs(y - ref).max():.3e}, fused fp32 kernel "
          f"{np.abs(y32 - ref).max():.3e}")
    assert np.abs(y - ref).max() <= 2e-5 and np.abs(y32 - ref).max() <= 2e-5
    # odd batch sizes and both CTA shapes
    xb = x.repeat(120, 1, 1)[:601]
    yb = h.forward(xb).cpu().numpy()
    assert np.abs(yb - np.tile(ref, (120, 1))[:601]).max() <= 2e-5
    assert h.forward(x[:1]).shape == (1, K)
    h.close()


@pytest.mark.parametrize("K,conf,emb_in,seed", [(527, (2, 1), 128, 2), (10, (1, 2, 1), 128, 5), (527, (1,), 128, 6),
                                                (33, (3,), 12288, 4)])
def test_head_fused_epilogues_are_bit_identical(K, conf, emb_in, seed):
    """The glue of the eval-mode head (model.py:219-221 BatchNorm1d(T) + ReLU, :268 BatchNorm1d(K) + sigmoid) runs in
    the GEMM epilogues by default; with vmb_mla_fuse_enable(0) it runs as separate kernels.  Both evaluate the same
    expressions in the same order: the scores must be equal bit for bit, at full and ragged tile sizes."""
    L = _lib.lib()
    sd = synth.mla_state_dict(conf, emb_in, 600, K, 10, seed=seed)
    h = engine.MlaHandle(sd, conf, emb_in, 600, K, 10, DEV)
    g = torch.Generator().manual_seed(seed)
    try:
        for batch in (1, 13, 256, 300):
            x = (torch.randn(batch, 10, emb_in, generator=g) * 1.5).to(DEV)
            L.vmb_mla_fuse_enable(1)
            n0 = L.vmb_launch_count()
            fused = h.forward(x)
            n_fused = L.vmb_launch_count() - n0
            L.vmb_mla_fuse_enable(0)
            n0 = L.vmb_launch_count()
            plain = h.forward(x)
            n_plain = L.vmb_launch_count() - n0
            torch.cuda.synchronize()
            assert torch.equal(fused, plain), f"K={K} conf={conf} batch={batch}"
            # (with VMB_PLANES_GEMM=0 the fused epilogues do not exist and both runs take the separate kernels)
            assert n_fused < n_plain or (os.environ.get("VMB_PLANES_GEMM") == "0" and n_fused == n_plain)
        print(f"head {conf} K={K}: {n_fused} launches fused, {n_plain} as separate kernels")
    finally:
        L.vmb_mla_fuse_enable(-1)
        h.close()


def test_reference_named_head_module(golden_head):
    import model
    old = model.K
    try:
        model.K = 527
        m = model.MultiLevelAttention([2, 1], 128)
    finally:
        model.K = old
    m.load_state_dict(synth.mla_state_dict((2, 1), 128, 600, 527, 10, seed=2))
    m = m.to(DEV).eval()
    y = m(torch.from_numpy(golden_head["x_k527"]).to(DEV))
    assert np.abs(y.cpu().numpy() - golden_head["y_k527"]).max() <= 2e-5


def test_standalone_embedded_mapping_and_attention_module():
    """EmbeddedMapping.forward / AttentionModule.forward on their own (model.py:217-222, :235-242) against the outputs
    of the reference's own sub-modules (tests/golden/levels.npz), and consistency with the whole head."""
    import model
    from conftest import load_golden
    lv = load_golden("levels.npz")
    old = model.K
    try:
        model.K = 527
        m = model.MultiLevelAttention([2, 1], 128)
    finally:
        model.K = old
    m.load_state_dict(synth.mla_state_dict((2, 1), 128, 600, 527, 10, seed=2))
    m = m.to(DEV).eval()
    x = torch.from_numpy(lv["x"]).to(DEV)
    e0 = m.embedded_mappings[0](x)
    e1 = m.embedded_mappings[1](e0)
    y0 = m.attention_modules[0](e0)
    y1 = m.attention_modules[1](e1)
    for name, got, ref, tol in (("emb0", e0, lv["emb0"], 5e-5), ("emb1", e1, lv["emb1"], 5e-5), ("y0", y0, lv["y0"], 2e-5),
                                ("y1", y1, lv["y1"], 2e-5)):
        err = np.abs(got.cpu().numpy() - ref).max()
        print(f"standalone {name}: max-abs-err {err:.2e} (max |ref| {np.abs(ref).max():.2f})")
        assert got.shape == ref.shape and err <= tol * max(1.0, np.abs(ref).max()), name
    # the same sub-modules composed by hand like MultiLevelAttention.forward does (model.py:258-269)
    out = torch.sigmoid(torch.nn.functional.batch_norm(
        torch.nn.functional.linear(torch.cat([y0, y1], dim=1), m.fc.weight, m.fc.bias), m.norm.running_mean,
        m.norm.running_var, m.norm.weight, m.norm.bias, False, 0.0, 1e-5))
    assert (out - m(x)).abs().max().item() <= 2e-5
    m.train()
    with pytest.raises(NotImplementedError):
        m.embedded_mappings[0](x)


def test_stft_magnitude_vs_reference_golden(golden_front):
    """mel_features.stft_magnitude (mel_features.py:71-92) on its own: float64 on the device, all 257 bins."""
    from torchvggish import mel_features
    w = golden_front["waves_f32"][1].astype(np.float64)
    got = mel_features.stft_magnitude(w, 512, 160, 400)
    ref = golden_front["stft_mag_clip1"]
    assert got.dtype == np.float64 and got.shape == (118, 257)
    err = np.abs(got[:8] - ref).max() / np.abs(ref).max()
    full = np.abs(np.fft.rfft(mel_features.frame(w, 400, 160) * mel_features.periodic_hann(400), 512))
    err_full = np.abs(got - full).max() / np.abs(full).max()
    print(f"stft_magnitude vs reference golden: rel-max-err {err:.2e}; vs numpy on all frames {err_full:.2e}")
    assert err <= 1e-12 and err_full <= 1e-12
    t = mel_features.stft_magnitude(torch.from_numpy(w).to(DEV), 512, 160, 400)
    assert t.is_cuda and t.dtype == torch.float64 and np.array_equal(t.cpu().numpy(), got)
    with pytest.raises(NotImplementedError):
        mel_features.stft_magnitude(w, 1024, 160, 400)
    with pytest.raises(ValueError):
        mel_features.stft_magnitude(np.zeros(100), 512, 160, 400)


def test_modules_pickle_and_deepcopy_after_forward(tmp_path, vgg_sd, head_sd):
    """The reference checkpoints WHOLE objects (torch.save({'model': model, ...}), train.py:259-268) and deep-copies
    state (train.py:150-158): the cached library handles must not travel with the module."""
    import copy
    import model
    old = model.K
    try:
        model.K = 527
        conf = dict(cnn_type="vggish", num_classes=527, use_pretrained=False, just_bottlenecks=False,
                    cnn_trainable=False, first_cnn_layer_trainable=False, in_channels=1)
        ens = model.Ensemble("repeat", conf, [2, 1], DEV)
    finally:
        model.K = old
    ens.cnn.cnn_model.load_state_dict(vgg_sd)
    ens.mla.load_state_dict(head_sd)
    ens = ens.to(DEV).eval()
    x = engine.examples_from_wave(torch.from_numpy(synth.make_clips(4, 2)).to(DEV)).reshape(2, 10, 1, 96, 64)
    y = ens(x)
    clone = copy.deepcopy(ens)                               # after an eval forward
    assert torch.equal(clone(x), y)
    path = str(tmp_path / "ckpt.pt")
    ens.train()
    ens.cnn.eval()
    loss = torch.nn.CrossEntropyLoss()(ens(x), torch.tensor([3, 5], device=DEV))
    loss.backward()                                          # after a train forward + backward
    torch.save({"model": ens, "epoch": 1}, path)             # _save_checkpoint, train.py:259-268
    back = torch.load(path, map_location=DEV, weights_only=False)["model"]      # _resume_from_checkpoint
    back.eval()
    ens.eval()
    assert torch.equal(back(x), ens(x))
    # edits through .data bypass the version counters: invalidate() is the documented way to refresh the library copy
    before = ens(x).clone()
    ens.mla.fc.bias.data.add_(3.0)
    ens.mla.invalidate()
    assert not torch.equal(ens(x), before)


def test_vggish_module_precision_knob(golden_front, golden_vggish, vgg_sd):
    """VGGish(postprocess=True) in the accuracy mode meets the +-1 LSB bar of north_star; the default (fp16) mode is
    reported next to it."""
    from torchvggish.vggish import VGGish
    eig, means = synth.pca_params(1)
    ref = golden_vggish["preprocess_postprocess"]
    hist = {}
    for prec in ("fp16", "bf16", "split"):
        net = VGGish(urls={}, pretrained=False, preprocess=True, postprocess=True)
        net.load_state_dict({**vgg_sd, "pproc.pca_eigen_vectors": eig, "pproc.pca_means": means})
        net = net.to(DEV).eval().set_precision(prec)
        d = np.abs(net(golden_front["waves_f32"][2].astype(np.float64), 16000).cpu().numpy() - ref).astype(np.int64)
        hist[prec] = np.bincount(d).tolist()
    print("VGGish(preprocess, postprocess) uint8 LSB histograms vs reference:", hist)
    assert len(hist["split"]) <= 2 and len(hist["fp16"]) <= 2                   # nothing further than 1 LSB
    assert hist["split"][0] >= 126 and hist["fp16"][0] >= 120


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_devices_in_one_process(vgg_sd, head_sd):
    """Kernel attributes (dynamic shared memory opt-in), SM counts and constant tables are per DEVICE: a process that
    ran on cuda:0 must be able to run on cuda:1 afterwards, with identical results."""
    waves = torch.from_numpy(synth.make_clips(0, 3))
    outs = []
    for i in (0, 1):
        dev = torch.device("cuda", i)
        with torch.cuda.device(dev):
            v = engine.VggishHandle(vgg_sd, dev)
            h = engine.MlaHandle(head_sd, (2, 1), 128, 600, 527, 10, dev)
            outs.append(engine.Pipeline(v, h).forward(waves.to(dev)).cpu())
            y32 = h.forward(torch.zeros(2, 10, 128, device=dev), fp32_crosscheck=True)
            assert torch.isfinite(y32).all()
            v.close()
            h.close()
    assert torch.equal(outs[0], outs[1])


def test_fp16_saturation_is_reported(vgg_sd):
    """fp16 ends at 65504: the epilogues convert with saturation and raise a flag that the host API turns into an error
    (weights scaled so that conv2's outputs overflow)."""
    sd = {k: v.clone() for k, v in vgg_sd.items()}
    sd["features.3.weight"] *= 3.0e4
    h = engine.VggishHandle(sd, DEV, precision="fp16")
    x = engine.examples_from_wave(torch.from_numpy(synth.make_clips(0, 1)).to(DEV))
    emb = h.forward(x)
    assert torch.isfinite(emb).all()                          # saturated, not inf / nan
    with pytest.raises(engine.B200Error, match="saturated"):
        h.check_saturation()
    h.check_saturation()                                      # the flags were cleared by the failed check
    h.close()
    ok = engine.VggishHandle(vgg_sd, DEV, precision="fp16")
    ok.forward(x)
    ok.check_saturation()
    ok.close()


# ------------------------------------------------------------------------------------------------ whole path
def test_pipeline_vs_reference_golden(golden_ensemble, vgg_handle, head_handle):
    pipe = engine.Pipeline(vgg_handle, head_handle)
    waves = torch.from_numpy(synth.make_clips(4, 2)).to(DEV)
    scores, emb = pipe.forward(waves, want_embeddings=True)
    _layer_check(emb, torch.from_numpy(golden_ensemble["embeddings"]), "pipeline embeddings vs reference", rel_tol=0.003)
    d = np.abs(scores.cpu().numpy() - golden_ensemble["scores"]).max()
    print(f"pipeline scores vs reference Ensemble: max-abs-err {d:.3e}")
    assert d <= 2e-2
    # host-buffer entry point gives the same bits as the device-resident one
    host = pipe.forward_host(torch.from_numpy(synth.make_clips(4, 2)).pin_memory(), clips_per_batch=1)
    assert torch.equal(host, scores.cpu())


def test_ensemble_module_matches_pipeline(golden_ensemble, vgg_sd, head_sd):
    import model
    old = model.K
    try:
        model.K = 527
        conf = dict(cnn_type="vggish", num_classes=527, use_pretrained=False, just_bottlenecks=False,
                    cnn_trainable=False, first_cnn_layer_trainable=False, in_channels=1)
        ens = model.Ensemble("repeat", conf, [2, 1], DEV)
    finally:
        model.K = old
    ens.cnn.cnn_model.load_state_dict(vgg_sd)
    ens.mla.load_state_dict(head_sd)
    ens = ens.to(DEV).eval()
    from torchvggish.vggish_input import waveform_to_examples
    waves = synth.make_clips(4, 2)
    ex = torch.stack([waveform_to_examples(w.astype(np.float64), 16000) for w in waves])     # (2, 10, 1, 96, 64)
    y = ens(ex)
    assert tuple(y.shape) == (2, 527)
    assert np.abs(y.cpu().numpy() - golden_ensemble["scores"]).max() <= 2e-2
    assert torch.equal(ens.forward_waveform(torch.from_numpy(waves).to(DEV)), y)


def test_map_identical_to_three_decimals(head_handle, vgg_sd, head_sd):
    """north_star: mAP on a fixed synthetic label set identical to 3 decimals, for the mode bench.py reports as `value`
    (engine.DEFAULT_PRECISION = fp16 body).  B200 scores vs the fp32 CPU oracle on the same 256 clips; label sets:
      * SURVEY 8d's recipe — seeded Bernoulli(0.05) multi-hot (B, 527), every class >= 1 positive (the defaults of
        synth.multihot_labels) — and labels that follow the oracle's own ranking (what a trained classifier looks like):
        the 3-decimal strings must be EQUAL;
      * round 1's set (first 128 clips, p = 0.2): random labels are the worst case — mAP sits at the base rate and moves
        with every swap of two nearly tied scores — and there the oracle's 0.22865 is 1.5e-4 from a rounding boundary:
        fp16 (|delta| 1.6e-4) lands on the other side of it, only the split mode matches as a string.  Bound there:
        |delta| < 2.5e-4;
      * 20 more seeds of the SURVEY recipe for the spread: printed per mode (fp16 18/20 equal strings, mean |delta| 6.5e-5;
        bf16 15/20, 2.2e-4; split 20/20, 1.2e-5 — DESIGN 3)."""
    n = 256
    waves = synth.make_clips(100, n)
    ex = np.concatenate([frontend_np.waveform_to_examples(w.astype(np.float64)) for w in waves]).astype(np.float32)
    with torch.no_grad():
        emb = model_torch.vgg_forward(vgg_sd, torch.from_numpy(ex)[:, None])
        want = model_torch.mla_forward(head_sd, emb.reshape(n, 10, 128), (2, 1)).numpy()
    sets = {"survey_8d": (slice(0, n), synth.multihot_labels(n, 527)),
            "oracle_ranked": (slice(0, n), (want >= np.quantile(want, 0.8, axis=0, keepdims=True)).astype(np.int64)),
            "round1_p02_128": (slice(0, 128), synth.multihot_labels(128, 527, p=0.2, seed=3))}
    for sd_ in range(20):
        sets[f"seed{100 + sd_}"] = (slice(0, n), synth.multihot_labels(n, 527, seed=100 + sd_))
    ref = {k: synth.mean_average_precision(lab, want[sl]) for k, (sl, lab) in sets.items()}
    wave_dev = torch.from_numpy(waves).to(DEV)
    got = {}
    for mode in ("fp16", "bf16", "split"):
        h = engine.VggishHandle(vgg_sd, DEV, precision=mode)
        try:
            sc = engine.Pipeline(h, head_handle).forward(wave_dev).cpu().numpy()
            h.check_saturation()
        finally:
            h.close()
        got[mode] = {k: synth.mean_average_precision(lab, sc[sl]) for k, (sl, lab) in sets.items()}
        d = np.array([got[mode][k] - ref[k] for k in ref if k.startswith("seed")])
        eq = sum(f"{got[mode][k]:.3f}" == f"{ref[k]:.3f}" for k in ref if k.startswith("seed"))
        print(f"mAP {mode:5s}: " + "  ".join(f"{k} {got[mode][k]:.5f} (oracle {ref[k]:.5f})" for k in
                                             ("survey_8d", "oracle_ranked", "round1_p02_128")) +
              f"; 20 seeds: |delta| mean {np.abs(d).mean():.2e} max {np.abs(d).max():.2e}, equal to 3 decimals {eq}/20; "
              f"scores max-abs-err {np.abs(sc - want).max():.2e}")
    head = engine.DEFAULT_PRECISION
    assert head == "fp16"
    for k in ("survey_8d", "oracle_ranked"):
        assert f"{got[head][k]:.3f}" == f"{ref[k]:.3f}", (k, got[head][k], ref[k])
        assert f"{got['split'][k]:.3f}" == f"{ref[k]:.3f}", (k, got["split"][k], ref[k])
    assert f"{got['split']['round1_p02_128']:.3f}" == f"{ref['round1_p02_128']:.3f}"
    assert abs(got[head]["round1_p02_128"] - ref["round1_p02_128"]) < 2.5e-4
    seeds = [k for k in ref if k.startswith("seed")]
    assert np.mean([abs(got[head][k] - ref[k]) for k in seeds]) < 1.5e-4
    assert np.mean([abs(got["split"][k] - ref[k]) for k in seeds]) < 5e-5


def test_shard_invariance(vgg_handle, head_handle):
    """Results must be bit-identical however the batch is cut (1/2/4/8-way contiguous shards)."""
    pipe = engine.Pipeline(vgg_handle, head_handle)
    waves = torch.from_numpy(synth.make_clips(200, 8)).to(DEV)
    whole = pipe.forward(waves)
    for world in (2, 4, 8):
        parts = [pipe.forward(waves[slice(*sharding.shard_bounds(8, r, world))]).clone() for r in range(world)]
        assert torch.equal(torch.cat(parts), whole)


def test_batch_size_invariance_across_kernel_variants(vgg_handle, head_handle):
    """Small and large batches select different kernels (128 x 128 or 256 x 128 tiles and haloed boxes for conv2, CTA
    pairs, the single-CTA tail of fc1 / fc2): a 300-clip batch must still equal its pieces bit for bit."""
    pipe = engine.Pipeline(vgg_handle, head_handle)
    waves = synth.fast_clips(900, 300).to(DEV)
    whole = pipe.forward(waves).clone()
    parts, i = [], 0
    for m in (1, 3, 5, 41, 250):
        parts.append(pipe.forward(waves[i:i + m]).clone())
        i += m
    assert i == 300 and torch.equal(torch.cat(parts), whole)


def test_stream_embeddings_chunking_is_exact(vgg_handle):
    """Long-stream path (config 4 shape, shortened): chunked at multiples of 15 360 samples == unchunked."""
    n_ex = 41
    rng = np.random.default_rng(7)
    stream = (rng.standard_normal(15360 * (n_ex - 1) + 15600 + 777) * 0.1).astype(np.float32)
    assert sharding.num_examples(len(stream)) == n_ex
    w = torch.from_numpy(stream).to(DEV)
    whole = vgg_handle.forward(engine.examples_from_wave(w))
    eig, means = synth.pca_params(1)
    q_whole = engine.postprocess(whole, eig.to(DEV), means.to(DEV), want_u8=True)[1]
    parts = []
    for rank in range(3):
        for e0, e1, s0, s1 in sharding.stream_chunks(len(stream), 6, rank, 3):
            parts.append(vgg_handle.forward(engine.examples_from_wave(w[s0:s1])))
    emb = torch.cat(parts)
    assert torch.equal(emb, whole)
    assert torch.equal(engine.postprocess(emb, eig.to(DEV), means.to(DEV), want_u8=True)[1], q_whole)


def test_async_host_pipeline_matches_blocking_call(vgg_handle, head_handle):
    """submit/wait with two calls in flight returns the same bits as the blocking call, in submission order."""
    pipe = engine.Pipeline(vgg_handle, head_handle)
    a = torch.from_numpy(synth.make_clips(300, 5)).pin_memory()
    b = torch.from_numpy(synth.make_clips(305, 3)).pin_memory()
    ra = torch.empty(5, 527).pin_memory()
    rb = torch.empty(3, 527).pin_memory()
    ta = pipe.submit_host(a, ra, clips_per_batch=2)
    tb = pipe.submit_host(b, rb, clips_per_batch=2)
    with pytest.raises(engine.B200Error):
        pipe.submit_host(a, ra, clips_per_batch=2)                       # only two calls may be in flight
    pipe.wait_host(ta)
    pipe.wait_host(tb)
    assert torch.equal(ra, pipe.forward_host(a, clips_per_batch=5))
    assert torch.equal(rb, pipe.forward(b.to(DEV)).cpu())
    with pytest.raises(engine.B200Error):
        pipe.wait_host(ta)                                               # ticket already collected


# ------------------------------------------------------------------------------------------------ accuracy mode
@pytest.fixture(scope="module")
def vgg_split(vgg_sd):
    h = engine.VggishHandle(vgg_sd, DEV, precision="split")
    yield h
    h.close()


def test_accuracy_mode_embeddings_and_uint8(golden_front, golden_vggish, vgg_split, vgg_sd):
    """precision='split' (hi + lo bf16 activations and weights): embeddings within 5e-4 (relative to the max) of the fp32 reference and the
    8-bit quantised output bit-exact except where rounding straddles a quantisation boundary (north_star)."""
    x = torch.from_numpy(golden_front["examples_f64"][:, 0]).float().to(DEV)
    emb, bott = vgg_split.forward(x, want_bottleneck=True)
    ref = torch.from_numpy(golden_vggish["embeddings"])
    rel = ((emb.cpu() - ref).abs().max() / ref.abs().max()).item()
    print(f"accuracy mode: embeddings rel-max-err {rel:.3e}")
    assert rel < 5e-4
    eig, means = synth.pca_params(1)
    q = engine.postprocess(emb, eig.to(DEV), means.to(DEV)).cpu().numpy()
    d = np.abs(q - golden_vggish["postprocessed"]).astype(np.int64)
    print("accuracy mode: uint8 LSB histogram vs reference:", np.bincount(d.ravel()).tolist())
    assert d.max() <= 1 and (d > 0).mean() <= 0.02
    # larger sample against the oracle: 3 clips = 30 examples
    waves = synth.make_clips(0, 3)
    ex = engine.examples_from_wave(torch.from_numpy(waves).to(DEV))
    got = vgg_split.forward(ex)
    exo = np.concatenate([frontend_np.waveform_to_examples(w.astype(np.float64)) for w in waves]).astype(np.float32)
    with torch.no_grad():
        want = model_torch.vgg_forward(vgg_sd, torch.from_numpy(exo)[:, None])
    rel = ((got.cpu() - want).abs().max() / want.abs().max()).item()
    qd = (engine.postprocess(got, eig.to(DEV), means.to(DEV)).cpu() - model_torch.postprocess(eig, means, want)).abs()
    print(f"accuracy mode, 30 examples: embeddings rel-max-err {rel:.3e}; uint8 LSB histogram "
          f"{np.bincount(qd.numpy().astype(np.int64).ravel()).tolist()}")
    assert rel < 1e-3 and qd.max() <= 1 and (qd > 0).float().mean() <= 0.02
    # batch invariance holds in this mode too
    assert torch.equal(vgg_split.forward(ex[7:19]), got[7:19])


def test_just_bottlenecks_variant(vgg_sd):
    """SURVEY §8(f)-2: Ensemble(just_bottlenecks=True) feeds the 12 288-d conv features straight into the head
    (model.py:43-44, :162-167): the tensor-core head takes emb_in = 12288."""
    import model
    old = model.K
    try:
        model.K = 10
        conf = dict(cnn_type="vggish", num_classes=10, use_pretrained=False, just_bottlenecks=True,
                    cnn_trainable=False, first_cnn_layer_trainable=False, in_channels=1)
        ens = model.Ensemble("repeat", conf, [1], DEV)
    finally:
        model.K = old
    assert ens.emb_input_size == 12288
    head_sd = synth.mla_state_dict((1,), 12288, 600, 10, 10, seed=4)
    # the reference re-wraps the conv stack as nn.Sequential(features, CnnFlatten) (model.py:161-166): keys 0.N.*, no FCs
    from conftest import load_golden
    lv = load_golden("levels.npz")
    assert sorted(ens.state_dict().keys()) == list(lv["jb_keys"])
    assert [",".join(map(str, ens.state_dict()[k].shape)) for k in lv["jb_keys"]] == list(lv["jb_shapes"])
    ens.cnn.cnn_model.load_state_dict({k.replace("features.", "0."): v for k, v in vgg_sd.items()
                                       if k.startswith("features.")})
    ens.mla.load_state_dict(head_sd)
    ens = ens.to(DEV).eval()
    waves = synth.make_clips(8, 2)
    ex = np.stack([frontend_np.waveform_to_examples(w.astype(np.float64)) for w in waves]).astype(np.float32)
    x = torch.from_numpy(ex)[:, :, None]                                   # (2, 10, 1, 96, 64)
    y = ens(x.to(DEV))
    with torch.no_grad():
        feats = model_torch.vgg_flatten(model_torch.vgg_features(vgg_sd, x.reshape(-1, 1, 96, 64)))
        want = model_torch.mla_forward(head_sd, feats.reshape(2, 10, 12288), (1,))
    d = (y.cpu() - want).abs().max().item()
    print(f"just_bottlenecks: scores max-abs-err {d:.3e}")
    assert tuple(y.shape) == (2, 10) and d < 2e-2


def test_pcm16_ingestion_is_bit_identical():
    """SURVEY §8(f)-3: int16 PCM goes straight to the device; pcm / 32768 is exact in fp32, so the log-mel equals the
    float path bit for bit (and the wavfile convention of vggish_input.py:96-98 is kept)."""
    rng = np.random.default_rng(11)
    pcm = torch.from_numpy(rng.integers(-32768, 32768, size=(3, 48000), dtype=np.int16))
    pcm[1] = torch.from_numpy((np.sin(np.arange(48000) * 0.05) * 20000).astype(np.int16))
    pcm[2, 1000:] = 0
    a = engine.logmel_pcm16(pcm.to(DEV))
    b = engine.logmel((pcm.float() / 32768.0).to(DEV))
    assert a.shape == (3, 298, 64) and torch.equal(a, b)
    # row 1 is a noiseless full-scale tone: mel bands far from it hold ~2e-4, where log(x + 0.01) has slope ~100 and the
    # 22-bit operand planes + truncating fp32 accumulation of the tensor-core DFT leave 1.7e-4.  Its frames have > 70 dB
    # between the spectrum's energy and the quietest band, so the epilogue flags them and the float64 kernel redoes
    # them: the 1e-4 bound of north_star holds here too.
    ref = frontend_np.log_mel_spectrogram(pcm[1].numpy() / 32768.0)
    tone_err = np.abs(a[1].cpu().numpy() - ref).max()
    print(f"log-mel max-abs error, noiseless full-scale tone: {tone_err:.3e}")
    assert tone_err <= 1e-4
    for i in (0, 2):
        ref = frontend_np.log_mel_spectrogram(pcm[i].numpy() / 32768.0)
        assert np.abs(a[i].cpu().numpy() - ref).max() <= 1e-4


def test_wavfile_to_examples_pcm16(tmp_path):
    """wavfile_to_examples (vggish_input.py:85-99) on a 16-bit mono WAV: int16 samples straight to the device."""
    import wave as wav
    from torchvggish import vggish_input
    pcm = (np.random.default_rng(3).standard_normal(32000) * 3000).astype("<i2")
    path = str(tmp_path / "clip.wav")
    with wav.open(path, "wb") as f:
        f.setnchannels(1)
        f.setsampwidth(2)
        f.setframerate(16000)
        f.writeframes(pcm.tobytes())
    t = vggish_input.wavfile_to_examples(path)
    assert tuple(t.shape) == (2, 1, 96, 64) and t.is_cuda
    ref = frontend_np.waveform_to_examples(pcm / 32768.0)
    assert np.abs(t[:, 0].cpu().numpy() - ref).max() <= 1e-4
    assert vggish_input.wavfile_to_examples(path, return_tensor=False).shape == (2, 96, 64)


def test_dataset_tiling_vs_reference():
    """SURVEY §8(f)-1: dataset.create_spec (torchvggish branch) + dataset.split against the reference's own output
    (tests/golden/dataset.npz), through the numpy-compatible drop-in functions and the batched device path."""
    import dataset
    from conftest import load_golden
    g = load_golden("dataset.npz")
    for tag, n in (("4s", 64000), ("2s5", 40000)):
        w = synth.make_clips(20, 1, n)[0]
        spec = dataset.create_spec(w.astype(np.float64), "vggish", 16000, 64000, 96, 64, False, True)
        assert spec.shape == (64, 384)
        frames = dataset.split(spec, 10, 96, 64, True)
        assert frames.shape == (10, 64, 96)
        assert np.abs(frames - g[f"frames_{tag}"]).max() <= 1e-4
        dev = dataset.clips_to_frames(torch.from_numpy(w)[None].to(DEV))
        assert tuple(dev.shape) == (1, 10, 1, 64, 96)
        assert np.abs(dev[0, :, 0].cpu().numpy() - g[f"frames_{tag}"]).max() <= 1e-4
        assert np.array_equal(dev[0, :, 0].cpu().numpy(), frames.astype(np.float32))      # same kernel output, tiled
    w = synth.make_clips(20, 1, 64000)[0]
    spec = dataset.create_spec(w.astype(np.float64), "vggish", 16000, 64000, 96, 64, False, False)
    assert np.abs(dataset.split(spec, 4, 96, 64, False) - g["frames_contig_4s"]).max() <= 1e-4
    dev = dataset.clips_to_frames(torch.from_numpy(w)[None].to(DEV), num_frames=4, overlap=False)
    assert np.abs(dev[0, :, 0].cpu().numpy() - g["frames_contig_4s"]).max() <= 1e-4
    with pytest.raises(NotImplementedError):
        dataset.create_spec(w, "vggish", 16000, 64000, 96, 64, True, True)
    # the frames feed Ensemble exactly like the reference's loader does: (B, T, 1, 64, 96) reshaped by Input
    batch = dataset.clips_to_frames(torch.from_numpy(synth.make_clips(20, 3, 64000)).to(DEV))
    assert tuple(batch.shape) == (3, 10, 1, 64, 96) and torch.isfinite(batch).all()


def test_reference_eval_loop_and_checkpoint_roundtrip(tmp_path, vgg_sd):
    """SURVEY §8(f)-4: the reference's test_model / save_model / load_model flow (train.py:182-240, :275-281) on the
    drop-in Ensemble: state_dict round trip through torch.save, DataLoader batches, argmax accuracy == the oracle's."""
    import dataset
    import model
    old = model.K
    conf = dict(cnn_type="vggish", num_classes=10, use_pretrained=False, just_bottlenecks=False, cnn_trainable=False,
                first_cnn_layer_trainable=False, in_channels=1)
    args = dict(input_conf="repeat", cnn_conf=conf, model_conf=[2, 1], device=DEV)
    try:
        model.K = 10
        clf = model.Ensemble(**args)
        head_sd = synth.mla_state_dict((2, 1), 128, 600, 10, 10, seed=6)
        clf.cnn.cnn_model.load_state_dict(vgg_sd)
        clf.mla.load_state_dict(head_sd)
        path = str(tmp_path / "wts.h5")
        torch.save(clf.state_dict(), path)                                   # save_model, train.py:275-276
        clf2 = model.Ensemble(**args)                                        # load_model, train.py:278-281
        clf2.load_state_dict(torch.load(path, map_location=DEV))
    finally:
        model.K = old
    clf2 = clf2.to(DEV).eval()
    waves = synth.make_clips(40, 12, 64000)                                   # 4 s clips like UrbanSound8K
    frames = dataset.clips_to_frames(torch.from_numpy(waves).to(DEV)).cpu()   # (12, 10, 1, 64, 96)
    labels = torch.arange(12) % 10
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(frames, labels), batch_size=5)
    criterion = torch.nn.CrossEntropyLoss()
    preds, loss_sum = [], 0.0
    for inputs, lab in loader:                                               # test_model, train.py:208-229
        inputs, lab = inputs.to(DEV).float(), lab.to(DEV).long()
        with torch.set_grad_enabled(False):
            outputs = clf2(inputs)
            loss_sum += criterion(outputs, lab).item() * inputs.size(0)
            preds.append(torch.max(outputs, 1)[1])
    preds = torch.cat(preds).cpu()
    # oracle on the same frames (Input only reshapes (64, 96) -> (96, 64), model.py:98-99)
    with torch.no_grad():
        want = model_torch.ensemble_forward(vgg_sd, head_sd, frames.reshape(12, 10, 1, 96, 64), (2, 1))
    agree = (preds == want.argmax(1)).float().mean().item()
    print(f"eval loop: argmax agreement with the oracle {agree:.3f}, mean loss {loss_sum / 12:.4f}")
    assert agree >= 11 / 12
    assert abs(loss_sum / 12 - criterion(want, labels).item()) < 5e-3


def test_pcm16_host_pipeline(vgg_handle, head_handle):
    """int16 PCM host buffers through submit/wait == the float pipeline on pcm / 32768 (bit-identical)."""
    pipe = engine.Pipeline(vgg_handle, head_handle)
    w = torch.from_numpy(synth.make_clips(60, 3))
    pcm = torch.clamp(torch.round(w * 32768.0), -32768, 32767).to(torch.int16).pin_memory()
    out = torch.empty(3, 527).pin_memory()
    pipe.wait_host(pipe.submit_host(pcm, out, clips_per_batch=2))
    want = pipe.forward((pcm.float() / 32768.0).to(DEV)).cpu()
    assert torch.equal(out, want)


def test_bench_dumps_the_scores_of_its_last_timed_step(tmp_path, vgg_sd, head_handle):
    """bench.py --dump-outputs DIR: DIR/scores.npy holds what the timed device-resident step returned, bit for bit."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1", "--clips", "64",
                        "--sustained-seconds", "0", "--no-config-legs", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.load(tmp_path / "scores.npy")
    vgg = engine.VggishHandle(vgg_sd, DEV, precision="fp16")
    want = engine.Pipeline(vgg, head_handle).forward(synth.fast_clips(0, 64).to(DEV)).cpu().numpy()
    vgg.close()
    assert got.dtype == np.float32 and np.array_equal(got, want)
