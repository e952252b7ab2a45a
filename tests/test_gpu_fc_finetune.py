"""GPU parity of VGGish FC fine-tuning: embeddings.{0,2,4} (fc1-fc3) trainable, convs frozen, driven through the
reference-named Ensemble like train.py:124-138 with the CNN's FC parameters given to Adam (train.py:370).

Oracle: float64 torch autograd (on the device) from the conv features the library saved in its train workspace — so
the conv stack's 16-bit precision is out of the comparison — through fc1-fc3, the head step (oracle.model_torch with the
step's dropout masks from oracle.dropout_np), the loss, and every FC and head gradient.  The chain frozen convs -> FC
autograd -> head autograd is checked end to end: the gradient reaching the embeddings (the head's dx) is compared too.

Tolerances are the suite's: loss 1e-5, scores 2e-5, every gradient tensor |err| <= 3e-4 * max|ref| + 5e-7 (dx too).
Every comparison asserts the ReLU margin (smallest |pre-activation|) of every FC and head ReLU site:
  * 5 clips: ordinary parameters, data seed chosen for a margin >= 1e-6;
  * 96 clips: "saturated" FC parameters (each unit's bias moved so that the unit is on, or off, for every row of the
    batch by at least a quarter of its spread: the masks still zero three units in ten) with ordinary head parameters
    and a data seed chosen for a margin >= 1e-6 — at 96 clips fc1 and fc2 have 7.9 M pre-activations, and an
    fp32-level margin over all of them does not occur with ordinary parameters;
  * 512 clips, dropout 0.4 (the benchmark step): saturated FC and head parameters (tests/_head_step_oracle.saturate),
    margin >= 1e-2.  Not at dropout 0: with the saturated head and no dropout the 512 clips' attention outputs are
    nearly equal, BatchNorm1d(K) normalises columns of almost no spread, and fp32 scores differ from float64 by ~7e-5
    whatever the FC stack does."""
import pytest
import torch
import torch.nn.functional as F

from b200 import engine, synth
from oracle import dropout_np, model_torch, train_torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CONF = (2, 1)
F64 = torch.float64
TORCH_SEED = 1234            # torch.manual_seed before each forward: the head bridge draws its dropout seed from it
FC_KEYS = ("0.weight", "0.bias", "2.weight", "2.bias", "4.weight", "4.bias")


def _ok(a, b):
    return float((a - b).abs().max()) <= 3e-4 * float(b.abs().max()) + 5e-7


def _bridge_seed(torch_seed):
    torch.manual_seed(torch_seed)
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def _ensemble(p, precision="fp16"):
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
    model.set_requires_grad(clf.cnn.cnn_model.embeddings, True)
    return clf


LEVEL_STD, CONTRAST = 0.5, (0.75, 1.25)


def _data(seed, clips):
    """Synthetic log-mel examples whose clips differ somewhat in level and contrast, as recordings do.  Clips drawn
    from one distribution give nearly the same attention outputs: the output Linear's BatchNorm1d(K) then normalises
    columns whose batch spread is a small fraction of their mean, any fp32 evaluation loses digits there, and the
    gradients that are zero by symmetry show it as noise above the suite's noise floor."""
    g = torch.Generator().manual_seed(seed)
    level = torch.randn(clips, 1, 1, 1, 1, generator=g) * LEVEL_STD
    contrast = torch.rand(clips, 1, 1, 1, 1, generator=g) * (CONTRAST[1] - CONTRAST[0]) + CONTRAST[0]
    x = torch.randn(clips, 10, 1, 96, 64, generator=g) * contrast + level
    return x, torch.randint(0, 527, (clips,), generator=g)


def _saturate_fc(fc_sd, X, on_share=0.7, seed=5):
    """Move each FC unit's bias so that the unit is on (share on_share) or off for every row of this batch, by at
    least a quarter of its spread over the batch."""
    sd, h = dict(fc_sd), X
    g = torch.Generator().manual_seed(seed)
    for i in (0, 2, 4):
        w = sd[f"{i}.weight"].to(DEV, F64)
        z = h @ w.T
        on = (torch.rand(w.shape[0], generator=g) < on_share).to(DEV)
        lo, hi = z.min(0).values, z.max(0).values
        delta = 0.25 * (hi - lo) + 1e-2
        b = torch.where(on, -lo + delta, -hi - delta)
        sd[f"{i}.bias"] = b.float().cpu()
        h = F.relu(z + sd[f"{i}.bias"].to(DEV, F64))
    return sd


def _oracle(X, fc_sd, head_sd, labels, masks):
    """float64 step from the conv features X (n, 12288): (loss, scores, fc grads, head grads, dE, running, margin)."""
    fc = {k: fc_sd[k].to(DEV, F64).requires_grad_(True) for k in FC_KEYS}
    leaves, work = {}, {}
    for k, v in head_sd.items():
        v = v.to(DEV)
        if v.is_floating_point() and "running_" not in k:
            leaves[k] = work[k] = v.to(F64).requires_grad_(True)
        else:
            work[k] = v.to(F64) if v.is_floating_point() else v
    pre = []
    h = X
    for i in (0, 2, 4):
        z = F.linear(h, fc[f"{i}.weight"], fc[f"{i}.bias"])
        pre.append(z.detach())
        h = F.relu(z)
    e = h
    e.retain_grad()
    B = labels.shape[0]
    xh = e.reshape(B, 10, 128)
    scores = model_torch.mla_forward(work, xh, CONF, training=True, masks=masks, relu_pre=pre)
    loss = F.cross_entropy(scores, labels.to(DEV))
    loss.backward()
    running = train_torch.updated_running_stats({k: v.to(DEV) for k, v in head_sd.items()}, xh.detach(), CONF,
                                                 masks=masks, dtype=F64)
    return (float(loss.detach()), scores.detach(), {k: t.grad for k, t in fc.items()}, {k: t.grad for k, t in leaves.items()},
            e.grad.detach(), running, train_torch.relu_margin(pre))


def _device_step(clf, x, labels):
    """clf(x), CE, backward with the gradient reaching the embeddings captured; returns (loss, scores, dE)."""
    got = {}

    def hook(mod, inp, out):
        out.register_hook(lambda g: got.__setitem__("dE", g.detach().clone()))

    hnd = clf.cnn.register_forward_hook(hook)
    try:
        torch.manual_seed(TORCH_SEED)
        out = clf(x.to(DEV))
        loss = torch.nn.CrossEntropyLoss()(out, labels.to(DEV))
        loss.backward()
    finally:
        hnd.remove()
    return loss.detach(), out.detach(), got["dE"]


def _choose(clf, clips, p, sat_fc, sat_head, min_margin, seeds=range(40)):
    """First data seed whose oracle step has ReLU margin >= min_margin; returns (x, labels, fc_sd, head_sd, masks)."""
    vgg = clf.cnn.cnn_model
    head_sd = {k: v.detach().cpu() for k, v in clf.mla.state_dict().items()}
    if sat_head:
        from _head_step_oracle import saturate
        head_sd = saturate(head_sd, CONF)
    masks = dropout_np.step_masks(_bridge_seed(TORCH_SEED), CONF, clips, 10, 600, p)
    for seed in seeds:
        x, labels = _data(seed, clips)
        with torch.no_grad():
            X = vgg.bottlenecks(x.reshape(-1, 1, 96, 64).to(DEV)).to(F64)
        fc_sd = {k: v.detach().cpu() for k, v in vgg.embeddings.state_dict().items()}
        if sat_fc:
            fc_sd = _saturate_fc(fc_sd, X)
        margin = _oracle(X, fc_sd, head_sd, labels, masks)[-1]
        if margin >= min_margin:
            return x, labels, fc_sd, head_sd, masks, seed
    pytest.fail(f"no data seed with a ReLU margin >= {min_margin}")


CASES = [(5, 0.0, False, False, 1e-6), (5, 0.4, False, False, 1e-6), (96, 0.0, True, False, 1e-6),
         (96, 0.4, True, False, 1e-6), (512, 0.4, True, True, 1e-2)]


@pytest.mark.parametrize("clips,p,sat_fc,sat_head,min_margin", CASES)
def test_fc_and_head_gradients_vs_float64_oracle(clips, p, sat_fc, sat_head, min_margin):
    clf = _ensemble(p)
    clf.train()
    x, labels, fc_sd, head_sd, masks, seed = _choose(clf, clips, p, sat_fc, sat_head, min_margin)
    vgg = clf.cnn.cnn_model
    vgg.embeddings.load_state_dict(fc_sd)
    clf.mla.load_state_dict(head_sd)
    conv_before = {k: v.detach().clone() for k, v in vgg.features.state_dict().items()}
    loss, scores, dE = _device_step(clf, x, labels)
    X = vgg._handle.train_features()                    # the conv features the FC stack saw
    with torch.no_grad():
        X_eval = vgg.bottlenecks(x.reshape(-1, 1, 96, 64).to(DEV)).to(F64)
    assert torch.equal(X, X_eval)                       # the conv stack ran exactly as in inference
    ref_loss, ref_scores, ref_fc, ref_head, ref_dE, ref_running, margin = _oracle(X, fc_sd, head_sd, labels, masks)
    assert margin >= min_margin, margin
    assert abs(loss.item() - ref_loss) < 1e-5, (loss.item(), ref_loss)
    assert float((scores.double() - ref_scores).abs().max()) < 2e-5
    worst, bad = 0.0, []

    def cmp(name, got, ref):
        nonlocal worst
        got, ref = got.double(), ref.double()
        worst = max(worst, float((got - ref).abs().max()) / (3e-4 * float(ref.abs().max()) + 5e-7))
        if not _ok(got, ref):
            bad.append((name, float((got - ref).abs().max()), float(ref.abs().max())))

    cmp("dE", dE, ref_dE)
    for k, p_ in vgg.embeddings.named_parameters():
        cmp("embeddings." + k, p_.grad, ref_fc[k])
    params = dict(clf.mla.named_parameters())
    for k, g in ref_head.items():
        if ".fcf." in k:
            assert params[k].grad is None
            continue
        if k.endswith(("fc.bias", ".normv.bias")) and float(g.abs().max()) < 2e-6:
            assert float(params[k].grad.abs().max()) < 2e-6, k        # zero by symmetry: rounding noise only
            continue
        cmp("mla." + k, params[k].grad, g)
    assert not bad, f"data seed {seed}: {bad}"
    for k, v in vgg.features.named_parameters():
        assert v.grad is None, k
        assert torch.equal(v.detach(), conv_before[k]), k
    sd = clf.mla.state_dict()
    for k, want in ref_running.items():
        err = float((sd[k].double() - want).abs().max())
        assert err <= 1e-4 * float(want.abs().max()) + 1e-6, (k, err)
    print(f"{clips} clips, p {p}: data seed {seed}, ReLU margin {margin:.2e}, worst gradient error {worst:.2f} of "
          f"its tolerance")


def test_reference_loop_three_adam_steps():
    """Three steps of the reference-style loop (one torch Adam at lr 1e-4 over every trainable parameter).  Each step is
    checked as tests/_head_step_oracle.py checks a trainer step: the float64 oracle evaluated at the device's current
    FC and head parameters (errors cannot compound over steps), every gradient within the suite's bound, the ReLU
    margin >= 1e-6 at every step; the update against train_torch.adam_update in float64 from the same gradients and
    moments (5e-7 absolute, as test_gpu_training.py's Adam test); the BatchNorm running statistics chained through the
    oracle over the three steps; conv parameters bit-identical with grad None."""
    lr = 1e-4
    clf = _ensemble(0.4)
    clf.train()
    x, labels, fc_sd, head_sd, masks, seed = _choose(clf, 5, 0.4, False, False, 1e-6)
    vgg = clf.cnn.cnn_model
    conv_before = {k: v.detach().clone() for k, v in vgg.features.state_dict().items()}
    opt = torch.optim.Adam([p for p in clf.parameters() if p.requires_grad], lr=lr)
    named = {**{"embeddings." + k: p for k, p in vgg.embeddings.named_parameters()},
             **{"mla." + k: p for k, p in clf.mla.named_parameters()}}
    running = None
    for step in range(3):
        fc_now = {k: v.detach().cpu() for k, v in vgg.embeddings.state_dict().items()}
        head_now = {k: v.detach().cpu() for k, v in clf.mla.state_dict().items()}
        if running is not None:
            head_now.update({k: v.float().cpu() for k, v in running.items()})
        opt.zero_grad()
        _device_step(clf, x, labels)
        X = vgg._handle.train_features()
        ref_loss, _, ref_fc, ref_head, ref_dE, ref_running, margin = _oracle(X, fc_now, head_now, labels, masks)
        assert margin >= 1e-6, (step, margin)
        bad = []
        refs = {**{"embeddings." + k: g for k, g in ref_fc.items()}, **{"mla." + k: g for k, g in ref_head.items()}}
        for k, g in refs.items():
            if ".fcf." in k:
                continue
            got = named[k].grad.double()
            if k.endswith(("fc.bias", ".normv.bias")) and float(g.abs().max()) < 2e-6:
                if float(got.abs().max()) >= 2e-6:
                    bad.append((k, "noise", float(got.abs().max())))
            elif not _ok(got, g):
                bad.append((k, float((got - g).abs().max()), float(g.abs().max())))
        assert not bad, (step, seed, bad)
        before = {k: p.detach().double().clone() for k, p in named.items() if p.grad is not None}
        grads = {k: named[k].grad.double().clone() for k in before}
        moments = {k: (opt.state[named[k]]["exp_avg"].double().clone(), opt.state[named[k]]["exp_avg_sq"].double().clone())
                   if named[k] in opt.state and opt.state[named[k]] else (None, None) for k in before}
        opt.step()
        for k, p0 in before.items():
            want = train_torch.adam_update(p0, grads[k], lr, (0.9, 0.999), 1e-8, step + 1, *moments[k])
            err = float((named[k].detach().double() - want).abs().max())
            assert err <= 5e-7, (step, k, err)
        sd = clf.mla.state_dict()
        for k, want in ref_running.items():
            err = float((sd[k].double() - want).abs().max())
            assert err <= 1e-4 * float(want.abs().max()) + 1e-6, (step, k, err)
        running = ref_running                                  # chained: the next step starts from the oracle's
        for k, v in vgg.features.named_parameters():
            assert v.grad is None and torch.equal(v.detach(), conv_before[k]), k
        print(f"reference loop step {step}: data seed {seed}, ReLU margin {margin:.2e}")


@pytest.mark.parametrize("precision", ["fp16", "bf16", "split"])
def test_refresh_after_step_matches_a_fresh_handle(precision, monkeypatch):
    """After opt.step() the eval-mode forward uses the new FC weights without rebuilding the handle, and equals the
    forward of a freshly built handle bit for bit."""
    from torchvggish import vggish
    clf = _ensemble(0.0, precision)
    clf.train()
    x, labels = _data(0, 5)
    opt = torch.optim.Adam([p for p in clf.parameters() if p.requires_grad], lr=1e-4)
    _device_step(clf, x, labels)
    vgg = clf.cnn.cnn_model
    handle = vgg._handle
    builds = []
    orig = engine.VggishHandle.__init__

    def counting(self, *a, **kw):
        builds.append(1)
        orig(self, *a, **kw)

    monkeypatch.setattr(engine.VggishHandle, "__init__", counting)
    opt.step()
    ex = x.reshape(-1, 1, 96, 64).to(DEV)
    with torch.no_grad():
        vgg.eval()
        emb = vgg(ex)
        assert vgg._handle is handle and not builds              # refreshed in place, not rebuilt
        vgg.train()
        opt.zero_grad()
        torch.manual_seed(TORCH_SEED)
    _device_step(clf, x, labels)                                   # a second step after the refresh
    assert vgg._handle is handle and not builds
    opt.step()
    with torch.no_grad():
        vgg.eval()
        emb2 = vgg(ex)
        fresh = vggish.VGG(vggish.make_layers())
        fresh.load_state_dict(vgg.state_dict())
        fresh = fresh.to(DEV).set_precision(precision).eval()
        want2 = fresh(ex)
    monkeypatch.undo()
    assert torch.equal(emb2, want2)
    assert not torch.equal(emb, emb2)                              # the step changed the embeddings
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
