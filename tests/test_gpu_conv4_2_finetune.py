"""GPU parity of VGGish conv4_2 fine-tuning: features.13 trainable (conv1 .. conv4_1 frozen), with fc1-fc3 trainable or
frozen, driven through the reference-named Ensemble like train.py:124-138.

Oracle: float64 torch autograd (on the device) from conv4_1's output read back from the train workspace — so the
frozen stack's 16-bit precision is out of the comparison — through conv4_2 (F.conv2d, padding 1), ReLU, the 2x2 max-pool,
the (h, w, c) flatten, fc1-fc3, the head step (oracle.model_torch with the step's dropout masks from oracle.dropout_np),
the loss and every gradient.  Tolerances are the suite's: loss 1e-5, scores 2e-5, every gradient tensor and the running
statistics |err| <= 3e-4 * max|ref| + 5e-7.

The device's z (conv4_2's fp32 pre-activation) is compared with float64 z against the bound of the arithmetic: the
operands are exact three-plane splits (conv4_1's outputs are 16-bit values, the weights fp32), the three dropped plane
products are below 3 u |a||w| each, and every one of the at most 6 * 768 / 16 = 288 accumulator steps per K slice, the
6 slice reductions and the bias add rounds by at most u = 2^-23 times the partial sum, so |z - z64| <= 300 u (S + |b|)
with S = sum |a||w| (computed in float64 as conv2d(|a|, |w|)).

Margins: every comparison asserts that the smallest ReLU margin of conv4_2, fc1-fc3 and the head is at least 10x the
measured error of z (BAND), and likewise the smallest max-pool gap (best minus runner-up in windows whose maximum is
positive).  conv4_2 has 2.4 M pre-activations at 5 clips and every data seed puts a few of them, and a few pool gaps,
within 1e-5 of zero, so:
  * conv4_2's and fc1-fc3's biases are saturated in every case (each unit on, or off, for every row of the batch by at
    least a quarter of its spread, as test_gpu_fc_finetune.py does for fc1-fc3);
  * pool windows cannot be saturated: in windows whose float64 gap is under BAND the oracle's backward takes the
    device's routing (derived from the device's own z); the test asserts that the routing agrees with float64 in every
    other window and prints how many windows took the device's;
  * the head is saturated (tests/_head_step_oracle.saturate) and the data seed chosen for a margin >= 1e-2: z's
    measured error is ~1e-5, and at 5 clips no seed among the first gives the ordinary head a margin of 1e-4.
    Hence no case at dropout 0: with the saturated head and no dropout, BatchNorm1d(K) normalises columns of almost
    no spread and fp32 scores differ from float64 by 4-5e-5 at 5 clips whatever the body does (test_gpu_fc_finetune.py
    leaves out 512 clips at dropout 0 for the same reason)."""
import pytest
import torch
import torch.nn.functional as F

from b200 import synth
from oracle import dropout_np, model_torch, train_torch
from test_gpu_fc_finetune import CONF, DEV, F64, FC_KEYS, TORCH_SEED, _bridge_seed, _data, _device_step, _ok, _saturate_fc

pytestmark = pytest.mark.gpu
U = 2.0 ** -23


def _ensemble(p, precision="fp16", fc_trainable=True):
    import model
    old = model.K, model.DR
    model.K, model.DR = 527, p
    try:
        conf = dict(cnn_type="vggish", num_classes=527, use_pretrained=False, just_bottlenecks=False,
                    cnn_trainable=False, first_cnn_layer_trainable=False, in_channels=1)
        clf = model.Ensemble("repeat", conf, list(CONF), DEV)
    finally:
        model.K, model.DR = old
    clf.cnn.cnn_model.load_state_dict(synth.vggish_state_dict(0))
    clf.mla.load_state_dict(synth.mla_state_dict(CONF, 128, 600, 527, 10, seed=2))
    clf = clf.to(DEV)
    clf.cnn.cnn_model.set_precision(precision)
    model.set_requires_grad(clf.cnn.cnn_model.features[13], True)
    if fc_trainable:
        model.set_requires_grad(clf.cnn.cnn_model.embeddings, True)
    return clf


def _windows(z_nchw):
    """(n, C, 12, 8) -> (n, C, 6, 4, 4): the 2x2 pool windows, element q = dh * 2 + dw (PyTorch's scan order)."""
    n, c = z_nchw.shape[:2]
    return z_nchw.reshape(n, c, 6, 2, 4, 2).permute(0, 1, 2, 4, 3, 5).reshape(n, c, 6, 4, 4)


def _conv41(vgg, x):
    h = vgg._b200_handle(train=True, conv4_2=True)
    h.forward_train_conv4_2(x.reshape(-1, 1, 96, 64).to(DEV))
    return h.train_conv4_1_output()


def _oracle(A41, c42_sd, fc_sd, head_sd, labels, masks, route=None):
    """float64 step from conv4_1's output A41 (n, 12, 8, 512).  route (n, 512, 6, 4): the window element each pooled
    value comes from (None: the float64 first maximum).  Returns a dict."""
    a = A41.permute(0, 3, 1, 2)
    cw = {k: c42_sd[k].to(DEV, F64).requires_grad_(True) for k in ("weight", "bias")}
    fc = {k: fc_sd[k].to(DEV, F64).requires_grad_(True) for k in FC_KEYS}
    leaves, work = {}, {}
    for k, v in head_sd.items():
        v = v.to(DEV)
        if v.is_floating_point() and "running_" not in k:
            leaves[k] = work[k] = v.to(F64).requires_grad_(True)
        else:
            work[k] = v.to(F64) if v.is_floating_point() else v
    z = F.conv2d(a, cw["weight"], cw["bias"], padding=1)
    zw = _windows(z.detach())
    if route is None:
        route = zw.argmax(dim=-1)
    pooled = _windows(F.relu(z)).gather(-1, route.unsqueeze(-1)).squeeze(-1)
    n = a.shape[0]
    h = pooled.permute(0, 2, 3, 1).reshape(n, 12288)
    pre = [z.detach()]
    for i in (0, 2, 4):
        zi = F.linear(h, fc[f"{i}.weight"], fc[f"{i}.bias"])
        pre.append(zi.detach())
        h = F.relu(zi)
    xh = h.reshape(labels.shape[0], 10, 128)
    scores = model_torch.mla_forward(work, xh, CONF, training=True, masks=masks, relu_pre=pre)
    loss = F.cross_entropy(scores, labels.to(DEV))
    loss.backward()
    running = train_torch.updated_running_stats({k: v.to(DEV) for k, v in head_sd.items()}, xh.detach(), CONF,
                                                masks=masks, dtype=F64)
    top = zw.topk(2, dim=-1).values
    gaps = (top[..., 0] - top[..., 1])[top[..., 0] > 0]
    S = F.conv2d(a.abs(), cw["weight"].detach().abs(), None, padding=1)
    return dict(loss=float(loss.detach()), scores=scores.detach(), conv={k: t.grad for k, t in cw.items()},
                fc={k: t.grad for k, t in fc.items()}, head={k: t.grad for k, t in leaves.items()}, running=running,
                margin=train_torch.relu_margin(pre), z=z.detach(), zw=zw, gaps=gaps, S=S)


def _saturate_conv(c42_sd, A41, on_share=0.7, seed=7):
    """Move each conv4_2 channel's bias so that the channel is on (share on_share) or off at every pixel of this batch,
    by at least a quarter of its spread."""
    sd = dict(c42_sd)
    w = sd["weight"].to(DEV, F64)
    z = F.conv2d(A41.permute(0, 3, 1, 2), w, None, padding=1).transpose(0, 1).reshape(512, -1)
    g = torch.Generator().manual_seed(seed)
    on = (torch.rand(512, generator=g) < on_share).to(DEV)
    lo, hi = z.min(1).values, z.max(1).values
    delta = 0.25 * (hi - lo) + 1e-2
    sd["bias"] = torch.where(on, -lo + delta, -hi - delta).float().cpu()
    return sd


def _choose(clf, clips, p, sat_head, min_margin, seeds=range(40)):
    """First data seed whose oracle step (conv4_2 and FC biases saturated for it) has a ReLU margin >= min_margin."""
    vgg = clf.cnn.cnn_model
    head_sd = {k: v.detach().cpu() for k, v in clf.mla.state_dict().items()}
    if sat_head:
        from _head_step_oracle import saturate
        head_sd = saturate(head_sd, CONF)
    masks = dropout_np.step_masks(_bridge_seed(TORCH_SEED), CONF, clips, 10, 600, p)
    for seed in seeds:
        x, labels = _data(seed, clips)
        A41 = _conv41(vgg, x)
        c42_sd = _saturate_conv({k: v.detach().cpu() for k, v in vgg.features[13].state_dict().items()}, A41)
        with torch.no_grad():
            a = A41.permute(0, 3, 1, 2)
            z = F.conv2d(a, c42_sd["weight"].to(DEV, F64), c42_sd["bias"].to(DEV, F64), padding=1)
            X = _windows(F.relu(z)).amax(-1).permute(0, 2, 3, 1).reshape(a.shape[0], 12288)
        fc_sd = _saturate_fc({k: v.detach().cpu() for k, v in vgg.embeddings.state_dict().items()}, X)
        ref = _oracle(A41, c42_sd, fc_sd, head_sd, labels, masks)
        if ref["margin"] >= min_margin:
            return x, labels, c42_sd, fc_sd, head_sd, masks, seed
    pytest.fail(f"no data seed with a ReLU margin >= {min_margin}")


def _check(clf, x, labels, c42_sd, fc_sd, head_sd, masks, fc_trainable=True, tag=""):
    """One device step against the oracle at the given parameters (loaded by the caller).  Returns the report."""
    vgg = clf.cnn.cnn_model
    loss, scores, _ = _device_step(clf, x, labels)
    h = vgg._handle
    A41 = h.train_conv4_1_output()
    z_dev = h.train_conv4_2_z().double().permute(0, 3, 1, 2)
    route_dev = _windows(z_dev).argmax(-1)
    ref0 = _oracle(A41, c42_sd, fc_sd, head_sd, labels, masks)
    z_err = float((z_dev - ref0["z"]).abs().max())
    bias = c42_sd["bias"].to(DEV, F64).view(1, -1, 1, 1).abs()
    bound_ratio = float(((z_dev - ref0["z"]).abs() / (300 * U * (ref0["S"] + bias))).max())
    assert bound_ratio <= 1.0, bound_ratio
    band = 10 * z_err
    zw = ref0["zw"]
    top = zw.topk(2, dim=-1).values
    close = (top[..., 0] > 0) & (top[..., 0] - top[..., 1] < band)
    route64 = zw.argmax(-1)
    live = top[..., 0] > 0
    assert torch.equal(route_dev[live & ~close], route64[live & ~close])     # float64 routing everywhere else
    ref = _oracle(A41, c42_sd, fc_sd, head_sd, labels, masks, route=torch.where(close, route_dev, route64))
    assert ref["margin"] >= band, (ref["margin"], band)
    assert abs(loss.item() - ref["loss"]) < 1e-5, (loss.item(), ref["loss"])
    assert float((scores.double() - ref["scores"]).abs().max()) < 2e-5
    worst, bad = 0.0, []

    def cmp(name, got, want):
        nonlocal worst
        got, want = got.double(), want.double()
        worst = max(worst, float((got - want).abs().max()) / (3e-4 * float(want.abs().max()) + 5e-7))
        if not _ok(got, want):
            bad.append((name, float((got - want).abs().max()), float(want.abs().max())))

    for k, p_ in vgg.features[13].named_parameters():
        cmp("features.13." + k, p_.grad, ref["conv"][k])
    for k, p_ in vgg.embeddings.named_parameters():
        if fc_trainable:
            cmp("embeddings." + k, p_.grad, ref["fc"][k])
        else:
            assert p_.grad is None, k
    params = dict(clf.mla.named_parameters())
    for k, g in ref["head"].items():
        if ".fcf." in k:
            assert params[k].grad is None
            continue
        if k.endswith(("fc.bias", ".normv.bias")) and float(g.abs().max()) < 2e-6:
            assert float(params[k].grad.abs().max()) < 2e-6, k
            continue
        cmp("mla." + k, params[k].grad, g)
    assert not bad, f"{tag}: {bad}"
    sd = clf.mla.state_dict()
    for k, want in ref["running"].items():
        err = float((sd[k].double() - want).abs().max())
        assert err <= 3e-4 * float(want.abs().max()) + 5e-7, (k, err)
    rep = dict(z_err=z_err, bound_ratio=bound_ratio, margin=ref["margin"], gap=float(ref["gaps"][~close[live]].min()),
               routed=int(close.sum()), worst=worst)
    print(f"{tag}: |z - z64| {z_err:.2e} ({bound_ratio:.2e} of the bound), ReLU margin {rep['margin']:.2e}, pool gap "
          f"{rep['gap']:.2e}, {rep['routed']} of {int(live.sum())} windows took the device's routing, worst gradient "
          f"error {worst:.2f} of its tolerance")
    assert rep["gap"] >= band
    return rep


def _frozen_snapshot(vgg):
    return {k: v.detach().clone() for k, v in vgg.features.named_parameters() if not k.startswith("13.")}


def _assert_frozen(vgg, before):
    for k, v in vgg.features.named_parameters():
        if k in before:
            assert v.grad is None and torch.equal(v.detach(), before[k]), k


CASES = [(5, 0.4, "fp16", True, 1e-2), (5, 0.4, "bf16", True, 1e-2), (5, 0.4, "split", True, 1e-2),
         (96, 0.4, "fp16", True, 1e-2), (512, 0.4, "fp16", True, 1e-2)]


@pytest.mark.parametrize("clips,p,precision,sat_head,min_margin", CASES)
def test_conv4_2_fc_and_head_gradients_vs_float64_oracle(clips, p, precision, sat_head, min_margin):
    clf = _ensemble(p, precision)
    clf.train()
    x, labels, c42_sd, fc_sd, head_sd, masks, seed = _choose(clf, clips, p, sat_head, min_margin)
    vgg = clf.cnn.cnn_model
    vgg.features[13].load_state_dict(c42_sd)
    vgg.embeddings.load_state_dict(fc_sd)
    clf.mla.load_state_dict(head_sd)
    before = _frozen_snapshot(vgg)
    _check(clf, x, labels, c42_sd, fc_sd, head_sd, masks, tag=f"{clips} clips, p {p}, {precision}, seed {seed}")
    _assert_frozen(vgg, before)


def test_conv4_2_with_frozen_fc():
    """conv4_2 trainable, fc1-fc3 frozen: the gradient flows through the frozen FCs, their grads stay None and their
    weights are bit-unchanged after an optimiser step."""
    clf = _ensemble(0.4, fc_trainable=False)
    clf.train()
    x, labels, c42_sd, fc_sd, head_sd, masks, seed = _choose(clf, 5, 0.4, True, 1e-2)
    vgg = clf.cnn.cnn_model
    vgg.features[13].load_state_dict(c42_sd)
    vgg.embeddings.load_state_dict(fc_sd)
    clf.mla.load_state_dict(head_sd)
    fc_before = {k: v.detach().clone() for k, v in vgg.embeddings.state_dict().items()}
    opt = torch.optim.Adam([p for p in clf.parameters() if p.requires_grad], lr=1e-4)
    _check(clf, x, labels, c42_sd, fc_sd, head_sd, masks, fc_trainable=False, tag=f"frozen FCs, seed {seed}")
    w_before = vgg.features[13].weight.detach().clone()
    opt.step()
    assert not torch.equal(vgg.features[13].weight.detach(), w_before)
    for k, v in vgg.embeddings.state_dict().items():
        assert torch.equal(v, fc_before[k]), k
    for p_ in vgg.embeddings.parameters():
        assert p_.grad is None


def test_reference_loop_three_adam_steps():
    """Three steps of the reference-style loop (one torch Adam at lr 1e-6 over every trainable parameter: Adam moves
    every weight by about lr, and at 1e-4 the 12 288 inputs of an fc1 unit move it by more than its saturation), each checked
    against the oracle at the module's current parameters; then eval-mode embeddings equal those of a freshly built
    handle bit for bit, the handle was refreshed in place, and the frozen convs are bit-unchanged with grad None."""
    from torchvggish import vggish
    clf = _ensemble(0.4)
    clf.train()
    x, labels, c42_sd, fc_sd, head_sd, masks, seed = _choose(clf, 5, 0.4, True, 1e-2)
    vgg = clf.cnn.cnn_model
    vgg.features[13].load_state_dict(c42_sd)
    vgg.embeddings.load_state_dict(fc_sd)
    clf.mla.load_state_dict(head_sd)
    before = _frozen_snapshot(vgg)
    opt = torch.optim.Adam([p for p in clf.parameters() if p.requires_grad], lr=1e-6)
    handle = None
    for step in range(3):
        now = lambda m: {k: v.detach().cpu() for k, v in m.state_dict().items()}   # noqa: E731
        opt.zero_grad()
        _check(clf, x, labels, now(vgg.features[13]), now(vgg.embeddings), now(clf.mla), masks,
               tag=f"reference loop step {step}, seed {seed}")
        handle = handle or vgg._handle
        assert vgg._handle is handle                              # refreshed in place, not rebuilt
        opt.step()
        _assert_frozen(vgg, before)
    ex = x.reshape(-1, 1, 96, 64).to(DEV)
    with torch.no_grad():
        vgg.eval()
        emb = vgg(ex)
        assert vgg._handle is handle
        fresh = vggish.VGG(vggish.make_layers())
        fresh.load_state_dict(vgg.state_dict())
        fresh = fresh.to(DEV).set_precision(vgg.b200_precision).eval()
        want = fresh(ex)
    assert torch.equal(emb, want)
    fresh.invalidate()


def test_stale_backward_raises():
    from b200._lib import B200Error
    clf = _ensemble(0.0)
    clf.train()
    vgg = clf.cnn.cnn_model
    x, _ = _data(0, 2)
    ex = x.reshape(-1, 1, 96, 64).to(DEV)
    e1 = vgg(ex)
    vgg(ex)
    with pytest.raises(B200Error, match="stale"):
        e1.sum().backward()
