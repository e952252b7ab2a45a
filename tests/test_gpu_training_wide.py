"""GPU parity of head training with a wide first layer: emb_in = 12288, the just_bottlenecks configuration
(model.py:43-44, :162-167), where the first Linear reads the planes of the normalised input xhat and its GEMM epilogue
applies norm0's affine (csrc/mla_train.cu, FNormalize / wide_grad_tile_kernel).  Same oracle and tolerances as
tests/test_gpu_training.py: loss 1e-5, scores 2e-5, every gradient tensor |err| <= 3e-4 * max|ref| + 5e-7, parameters
after one Adam step 2e-5 (compared where the reference gradient is resolved, |g| > 1e-6: Adam's first step moves a
parameter by ~lr * g / (|g| + eps), which is ill-conditioned for gradients that are rounding noise in both runs)."""
import ctypes as C

import numpy as np
import pytest
import torch

from b200 import _lib, engine, synth, training
from b200._lib import check, ptr, stream_ptr
from oracle import train_torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
JB = 12288


def _ok(a, b):
    return float(np.abs(a - b).max()) <= 3e-4 * float(np.abs(b).max()) + 5e-7


# Zero in exact arithmetic: the output Linear's bias before BatchNorm1d(K) and normv.bias before the class softmax.  Both
# runs hold only rounding noise there, which on the conv features (larger activations than randn) reaches the 5e-7 floor
# of _ok (measured: 5.6e-7 here against 3.6e-7 in the reference itself); they are checked to stay at noise level.
_ZERO_BY_SYMMETRY = ("fc.bias", ".normv.bias")
_NOISE = 2e-6


def _trainer(conf, K, max_batch, sd):
    tr = training.HeadTrainer(conf, JB, 600, K, 10, max_batch, DEV, dropout_p=0.0)
    tr.load_state_dict(sd)
    return tr


def _check_grads(tr, ref_grads, keys=None):
    keys = keys or [k for k, _, _ in tr.p_layout]
    bad = []
    for k in keys:
        got, ref = tr.view(tr.grads, k).cpu().numpy(), ref_grads[k].numpy()
        if k.endswith(_ZERO_BY_SYMMETRY) and float(np.abs(ref).max()) < _NOISE:
            if float(np.abs(got).max()) >= _NOISE:
                bad.append((k, float(np.abs(got).max()), float(np.abs(ref).max())))
        elif not _ok(got, ref):
            bad.append((k, float(np.abs(got - ref).max()), float(np.abs(ref).max())))
    assert not bad, bad


def _check_step(tr, sd, x, labels, conf):
    loss, scores = tr.forward_backward(x, labels, want_scores=True)
    ref_loss, ref_scores, ref_grads = train_torch.head_step(sd, x, labels, conf)
    assert abs(loss.item() - ref_loss.item()) < 1e-5
    assert float((scores.cpu() - ref_scores).abs().max()) < 2e-5
    _check_grads(tr, ref_grads)
    return ref_grads


def _check_adam(tr, sd, ref_grads):
    tr.adam(1)
    for key, _, _ in tr.p_layout:
        g = ref_grads[key]
        want = train_torch.adam_update(sd[key].float(), g)
        got = tr.view(tr.params, key).cpu()
        resolved = g.abs() > 1e-6
        if resolved.any():
            assert float((got - want)[resolved].abs().max()) < 2e-5, key


def _check_running(tr, sd, x, conf):
    want = train_torch.updated_running_stats(sd, x, conf)
    out = tr.state_dict()
    np.testing.assert_allclose(out["embedded_mappings.0.norm0.running_mean"].cpu().numpy(),
                               want["embedded_mappings.0.norm0.running_mean"].numpy(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(out["embedded_mappings.0.norms.0.running_var"].cpu().numpy(),
                               want["embedded_mappings.0.norms.0.running_var"].numpy(), rtol=1e-3, atol=1e-7)
    np.testing.assert_allclose(out["norm.running_var"].cpu().numpy(), want["norm.running_var"].numpy(), rtol=1e-3,
                               atol=1e-7)


def _bottleneck_features(n_clips, first=0):
    """Non-negative conv4_2 features of the library's own VGGish conv stack on synthetic clips: (n_clips, 10, 12288)."""
    h = engine.VggishHandle(synth.vggish_state_dict(0), DEV)
    wave = torch.from_numpy(synth.make_clips(first, n_clips)).to(DEV)
    _, bott = h.forward(engine.examples_from_wave(wave), want_bottleneck=True, want_embeddings=False)
    h.close()
    return bott.float().reshape(n_clips, 10, JB).cpu()


def test_tiny_wide_step_runs_every_new_kernel():
    """Smallest shapes first: two clips, one level, K = 10 (one row tile of every new kernel).  BatchNorm1d(K) over two
    rows amplifies rounding in the scores, so only the wide layer's own gradients are compared here."""
    conf = (1,)
    sd = synth.mla_state_dict(conf, JB, 600, 10, 10, seed=3)
    tr = _trainer(conf, 10, 2, sd)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 10, JB, generator=g)
    labels = torch.randint(0, 10, (2,), generator=g)
    tr.forward_backward(x, labels)
    _, _, ref = train_torch.head_step(sd, x, labels, conf)
    _check_grads(tr, ref, ["embedded_mappings.0.norm0.weight", "embedded_mappings.0.norm0.bias",
                           "embedded_mappings.0.fc.0.weight", "embedded_mappings.0.fc.0.bias"])
    tr.close()


@pytest.mark.parametrize("conf,K,batch", [((2, 1), 527, 33), ((2, 1), 527, 96), ((1,), 10, 33), ((1,), 10, 96)])
def test_wide_step_vs_oracle(conf, K, batch):
    sd = synth.mla_state_dict(conf, JB, 600, K, 10, seed=7)
    tr = _trainer(conf, K, 128, sd)
    g = torch.Generator().manual_seed(batch)
    x = torch.randn(batch, 10, JB, generator=g)
    labels = torch.randint(0, K, (batch,), generator=g)
    ref_grads = _check_step(tr, sd, x, labels, conf)
    _check_running(tr, sd, x, conf)
    # a second, smaller batch on the same handle: padded rows of the wide planes must not leak
    x2, l2 = x[:5], labels[:5]
    tr.forward_backward(x2, l2)
    _, _, ref2 = train_torch.head_step(sd, x2, l2, conf)
    _check_grads(tr, ref2, ["fc.weight", "embedded_mappings.0.fc.0.weight", "attention_modules.0.fcv.weight",
                            "embedded_mappings.0.norm0.weight", "embedded_mappings.0.norm0.bias"])
    # and the first batch again: captured into a graph (the first step of a handle runs eagerly), then replayed
    _check_step(tr, sd, x, labels, conf)
    ref_grads = _check_step(tr, sd, x, labels, conf)
    _check_adam(tr, sd, ref_grads)
    tr.close()


@pytest.mark.parametrize("conf,K,batch", [((2, 1), 527, 33), ((1,), 10, 96)])
def test_wide_step_on_bottleneck_features(conf, K, batch):
    x = _bottleneck_features(batch)
    assert float(x.min()) >= 0 and float(x.max()) > 0
    sd = synth.mla_state_dict(conf, JB, 600, K, 10, seed=5)
    tr = _trainer(conf, K, batch, sd)
    labels = torch.randint(0, K, (batch,), generator=torch.Generator().manual_seed(1))
    for _ in range(3):                      # eager step, graph capture, graph replay
        ref_grads = _check_step(tr, sd, x, labels, conf)
    _check_adam(tr, sd, ref_grads)
    tr.close()


def test_small_norm0_weight_has_no_division():
    """A norm0 weight of 1e-3: the wide layer's formulas never divide by gamma, so nothing is amplified."""
    conf = (2, 1)
    sd = synth.mla_state_dict(conf, JB, 600, 527, 10, seed=9)
    sd["embedded_mappings.0.norm0.weight"][3] = 1e-3
    tr = _trainer(conf, 527, 64, sd)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(48, 10, JB, generator=g) * 2 + 0.5
    labels = torch.randint(0, 527, (48,), generator=g)
    for _ in range(2):
        _check_step(tr, sd, x, labels, conf)
    tr.close()


def _gemm_launches(tr, x, labels):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tr.forward_backward(x, labels)
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and "gemm" in e.name]


def test_wide_step_launches_two_gemms_over_the_input_width():
    """One wide step (eager, first of its handle; 640 rows): the split-K forward GEMM and the no-split MN-major dW GEMM
    run once each, and they are the only GEMMs over the input width: the step launches one GEMM fewer than the 128-wide
    one (no dX GEMM)."""
    conf = (2, 1)
    counts = {}
    for emb_in in (128, JB):
        tr = training.HeadTrainer(conf, emb_in, 600, 527, 10, 64, DEV, dropout_p=0.4)
        tr.load_state_dict(synth.mla_state_dict(conf, emb_in, 600, 527, 10, seed=2))
        g = torch.Generator().manual_seed(2)
        x = torch.randn(64, 10, emb_in, generator=g).to(DEV)
        labels = torch.randint(0, 527, (64,), generator=g).to(DEV)
        counts[emb_in] = _gemm_launches(tr, x, labels)
        tr.close()
    wide = counts[JB]
    fwd, dw = "planes_gemm_kernel<3, true, 0, 128, false>", "planes_gemm_kernel<3, false, 0, 128, true>"
    assert sum(fwd in n for n in wide) == 1 and sum(dw in n for n in wide) == 1
    assert not any(fwd in n or dw in n for n in counts[128])
    assert len(wide) == len(counts[128]) - 1


def test_reference_loop_on_the_bottleneck_ensemble():
    """Ensemble(just_bottlenecks=True) with synthetic weights driven like train.py:124-138: .train(), CrossEntropyLoss
    on the outputs, backward(), torch.optim.Adam(lr=1e-3).step(); the head's parameters after the step match the oracle
    run on the same conv features."""
    import model
    old_k, old_dr = model.K, model.DR
    try:
        model.K, model.DR = 10, 0.0
        cnn_conf = dict(cnn_type="vggish", num_classes=10, use_pretrained=False, just_bottlenecks=True,
                        cnn_trainable=False, first_cnn_layer_trainable=False, in_channels=1)
        ens = model.Ensemble("repeat", cnn_conf, [2, 1], DEV)
    finally:
        model.K, model.DR = old_k, old_dr
    vgg_sd = synth.vggish_state_dict(0)
    ens.cnn.cnn_model.load_state_dict({k.replace("features.", "0."): v for k, v in vgg_sd.items()
                                       if k.startswith("features.")})
    head_sd = synth.mla_state_dict((2, 1), JB, 600, 10, 10, seed=4)
    ens.mla.load_state_dict(head_sd)
    ens = ens.to(DEV).train()
    n = 12
    wave = torch.from_numpy(synth.make_clips(0, n)).to(DEV)
    x = engine.examples_from_wave(wave).reshape(n, 10, 1, 96, 64)
    labels = torch.randint(0, 10, (n,), generator=torch.Generator().manual_seed(6)).to(DEV)
    with torch.no_grad():
        feats = ens.cnn(ens.input(x)).reshape(n, 10, JB).cpu()
    opt = torch.optim.Adam([p for p in ens.parameters() if p.requires_grad], lr=1e-3)
    opt.zero_grad()
    out = ens(x)
    loss = torch.nn.CrossEntropyLoss()(out, labels)
    loss.backward()
    opt.step()
    ref_loss, ref_scores, ref_grads = train_torch.head_step(head_sd, feats, labels.cpu(), (2, 1))
    assert abs(loss.item() - ref_loss.item()) < 1e-5
    assert float((out.detach().cpu() - ref_scores).abs().max()) < 2e-5
    params = dict(ens.mla.named_parameters())
    for key, g in ref_grads.items():
        if g is None:
            assert params[key].grad is None, key
            continue
        want = train_torch.adam_update(head_sd[key].float(), g)
        resolved = g.abs() > 1e-6
        if resolved.any():
            got = params[key].detach().cpu()
            assert float((got - want)[resolved].abs().max()) < 2e-5, key


def test_peer_memory_optimizer_step_single_rank_arithmetic_wide_bucket():
    """vmb_dp_adam_step with world = 1 on the 9.3 M-float bucket of the wide head, conf (2, 1), K = 527: against
    torch.optim.Adam over three steps with alternating gradient buffers."""
    L = _lib.lib()
    n = training.train_layout((2, 1), JB, 600, 527, 10)[2]
    assert n == 9285273
    handle = (C.c_char * 64)()
    dp = C.c_void_p()
    check(L.vmb_dp_create(C.byref(dp), n, 0, 1, C.cast(handle, C.c_void_p)), "vmb_dp_create")
    params = grads = None
    try:
        params = torch.as_tensor(training._DeviceArray(L.vmb_dp_params(dp), n), device=DEV)
        grads = [torch.as_tensor(training._DeviceArray(L.vmb_dp_grads(dp, i), n), device=DEV) for i in (0, 1)]
        g = torch.Generator().manual_seed(3)
        p0 = torch.randn(n, generator=g)
        params.copy_(p0)
        npad = (n + 3) // 4 * 4
        m, v = torch.zeros(npad, device=DEV), torch.zeros(npad, device=DEV)
        ref = p0.clone().requires_grad_(True)
        opt = torch.optim.Adam([ref], lr=1e-3)
        for step in range(1, 4):
            gr = torch.randn(n, generator=g) * 0.02
            grads[(step - 1) & 1].copy_(gr)
            check(L.vmb_dp_adam_step(dp, (step - 1) & 1, ptr(m), ptr(v), 1e-3, 0.9, 0.999, 1e-8, 0.0, step, stream_ptr()),
                  "vmb_dp_adam_step")
            ref.grad = gr.clone()
            opt.step()
            torch.cuda.synchronize()
            check(L.vmb_dp_status(dp), "vmb_dp_status")
            assert float((params.cpu() - ref.detach()).abs().max()) < 5e-7, f"step {step}"
        assert float(m[n:].abs().max()) == 0.0 and float(v[n:].abs().max()) == 0.0
    finally:
        del params, grads
        L.vmb_dp_destroy(dp)


def _two_rank_worker(rank, world, port, out):
    import os
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    conf = (2, 1)
    sd = synth.mla_state_dict(conf, JB, 600, 527, 10, seed=2)
    g = torch.Generator().manual_seed(40 + rank)
    x = torch.randn(128, 10, JB, generator=g).to(dev)
    labels = torch.randint(0, 527, (128,), generator=g).to(dev)
    tr = training.HeadTrainer(conf, JB, 600, 527, 10, 128, dev, dropout_p=0.4, seed=77)
    tr.load_state_dict(sd)
    peer = tr.enable_peer_step()
    ref = training.HeadTrainer(conf, JB, 600, 527, 10, 128, dev, dropout_p=0.4, seed=77)     # NCCL all-reduce + Adam
    ref.load_state_dict(sd)
    losses, ref_losses = [], []
    for _ in range(4):
        losses.append(float(tr.step(x, labels).item()))
        ref_losses.append(float(ref.step(x, labels).item()))
    torch.cuda.synchronize()
    tr.peer_step_status()
    every = [torch.empty_like(tr.params) for _ in range(world)]
    dist.all_gather(every, tr.params)
    same = all(torch.equal(every[0], e) for e in every)
    cos = float(torch.nn.functional.cosine_similarity(tr.params, ref.params, dim=0))
    if rank == 0:
        out.put((peer, losses, ref_losses, same, cos))
    ref.close()
    tr.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_wide_data_parallel_two_ranks():
    """Two ranks on the wide head: the peer-memory step (when the GPUs can map each other) next to the overlapped NCCL
    all-reduce + Adam; replicas stay bit-identical and the two exchange forms agree."""
    import socket
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    peer, losses, ref_losses, same, cos = q.get(timeout=600)
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    print("wide head, two ranks: peer step" if peer else "wide head, two ranks: NCCL (no peer access)", losses, ref_losses)
    assert same
    assert losses[-1] < losses[0]
    assert all(abs(a - b) <= 1e-4 * abs(b) for a, b in zip(losses, ref_losses))
    assert cos > 0.99999
