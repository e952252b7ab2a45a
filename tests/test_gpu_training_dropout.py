"""Head training with dropout on, against the float64 oracle with the step's own dropout masks
(tests/_head_step_oracle.py): the configuration bench_train.py times (conf (2, 1), K = 527, T = 10, 512 clips per GPU,
dropout 0.4, a CUDA-graph replay of vmb_mla_train_step with a new seed every step), small batches where the ReLUs
really zero elements, the reference-named module under the reference's loop, and the wide first layer's benchmark
line (emb_in 12288)."""
import numpy as np
import pytest
import torch

from _head_step_oracle import DEV, SATURATED_MARGIN, check_step, ok, reference, saturate
from b200 import synth, training
from oracle import dropout_np, train_torch

pytestmark = pytest.mark.gpu
CONF = (2, 1)


def _bench_trainer(emb_in, sd):
    tr = training.HeadTrainer(CONF, emb_in, 600, 527, 10, 512, DEV, dropout_p=0.4, seed=1234)
    tr.load_state_dict(sd)
    return tr


def _bench_inputs(emb_in, data_seed):
    sd = saturate(synth.mla_state_dict(CONF, emb_in, 600, 527, 10, seed=2), CONF)
    g = torch.Generator().manual_seed(data_seed)
    return sd, torch.randn(512, 10, emb_in, generator=g), torch.randint(0, 527, (512,), generator=g)


def test_benchmark_step_repeated():
    """Five forward_backward + adam steps of the benchmark's configuration: one eager step, the capture and three
    replays, each with its own seed (seed + step_count), checked at the device's current parameters; the running
    statistics against the chained oracle update."""
    sd, x, labels = _bench_inputs(128, 0)
    tr = _bench_trainer(128, sd)
    running = {k: v.double() for k, v in sd.items() if "running_" in k}
    try:
        for step in range(5):
            margin, worst, running = check_step(tr, x, labels, min_margin=SATURATED_MARGIN, running=running)
            print(f"benchmark step {step}: ReLU margin {margin:.2e}, "
                  f"worst gradient error {worst:.2f} of its tolerance")
        assert tr.step_count == 5
    finally:
        tr.close()


# (batch, p) -> data seed whose float64 ReLU margin is >= 1e-6 at both dropout seeds below
SMALL_SEEDS = {(33, 0.1): 3, (33, 0.4): 4, (33, 0.9): 2, (96, 0.1): 49, (96, 0.4): 10, (96, 0.9): 2}
SMALL_DROPOUT_SEEDS = (2 ** 32 + 7, 2 ** 40 + 3)      # eager step, replayed step: upper 32 bits in use


def small_inputs(batch, data_seed):
    sd = synth.mla_state_dict(CONF, 128, 600, 527, 10, seed=7)
    g = torch.Generator().manual_seed(data_seed)
    return sd, torch.randn(batch, 10, 128, generator=g), torch.randint(0, 527, (batch,), generator=g)


@pytest.mark.parametrize("batch,p", list(SMALL_SEEDS))
def test_small_batch_with_relu_zeros(batch, p):
    sd, x, labels = small_inputs(batch, SMALL_SEEDS[(batch, p)])
    tr = training.HeadTrainer(CONF, 128, 600, 527, 10, 128, DEV, dropout_p=p)
    tr.load_state_dict(sd)
    try:
        for step, seed in enumerate(SMALL_DROPOUT_SEEDS):
            tr.seed = seed
            margin, worst, _ = check_step(tr, x, labels, adam=False)
            print(f"batch {batch} p {p} {'eager' if step == 0 else 'replay'}: ReLU margin {margin:.2e}, "
                  f"worst gradient error {worst:.2f} of its tolerance")
    finally:
        tr.close()


BRIDGE_TORCH_SEED = 0        # torch.manual_seed before the forward: the bridge draws its dropout seed from it


def bridge_seed(torch_seed):
    """The dropout seed the module bridge draws (b200/training.py, _HeadTrainFn.forward) after manual_seed."""
    torch.manual_seed(torch_seed)
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def test_reference_loop_on_the_module_with_dropout(golden_head):
    """model.MultiLevelAttention with DR = 0.4 driven like train.py:124-138: loss, outputs, every parameter gradient
    and torch.optim.Adam's step against the oracle with the masks of the seed the bridge drew."""
    import model
    old_k, old_dr = model.K, model.DR
    try:
        model.K, model.DR = 527, 0.4
        m = model.MultiLevelAttention([2, 1], 128)
    finally:
        model.K, model.DR = old_k, old_dr
    sd = synth.mla_state_dict(CONF, 128, 600, 527, 10, seed=2)
    m.load_state_dict(sd)
    m = m.to(DEV).train()
    x = torch.from_numpy(golden_head["train_x"])
    labels = torch.from_numpy(golden_head["train_labels"])
    seed = bridge_seed(BRIDGE_TORCH_SEED)
    masks = dropout_np.step_masks(seed, CONF, x.shape[0], 10, 600, 0.4)
    ref_loss, ref_scores, ref_grads, ref_running, margin = reference(sd, x, labels, CONF, masks)
    assert margin >= 1e-6, margin
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=0.001)
    opt.zero_grad()
    torch.manual_seed(BRIDGE_TORCH_SEED)
    out = m(x.to(DEV))
    loss = torch.nn.CrossEntropyLoss()(out, labels.to(DEV))
    loss.backward()
    assert abs(loss.item() - ref_loss) < 1e-5
    assert float((out.detach().double().cpu() - ref_scores).abs().max()) < 2e-5
    params = dict(m.named_parameters())
    bad = []
    for key, g in ref_grads.items():
        if g is None:
            assert params[key].grad is None, key
            continue
        got, ref = params[key].grad.double().cpu().numpy(), g.numpy()
        if key.endswith(("fc.bias", ".normv.bias")) and float(np.abs(ref).max()) < 2e-6:
            ok_ = float(np.abs(got).max()) < 2e-6
        else:
            ok_ = ok(got, ref)
        if not ok_:
            bad.append(key)
    assert not bad, bad
    before = {k: p.detach().clone() for k, p in params.items()}
    grads = {k: p.grad.detach().clone() for k, p in params.items() if p.grad is not None}
    opt.step()
    for key, g in grads.items():
        want = train_torch.adam_update(before[key], g)
        assert float((params[key].detach() - want).abs().max()) <= 5e-7, key
    for key, want in ref_running.items():
        got = m.state_dict()[key].double().cpu()
        assert float((got - want).abs().max()) <= 1e-4 * float(want.abs().max()) + 1e-6, key


def test_wide_benchmark_line():
    """bench_train.py --emb-in 12288: 512 clips, dropout 0.4, the eager step and a replayed one."""
    sd, x, labels = _bench_inputs(12288, 1)
    tr = _bench_trainer(12288, sd)
    try:
        for step in range(2):
            margin, worst, _ = check_step(tr, x, labels, min_margin=SATURATED_MARGIN, oracle_dev=DEV)
            print(f"wide benchmark step {step}: ReLU margin {margin:.2e}, "
                  f"worst gradient error {worst:.2f} of its tolerance")
    finally:
        tr.close()
