"""One training step of a HeadTrainer checked against the float64 oracle with the step's own dropout masks (used by
tests/test_gpu_training_dropout.py and tests/test_gpu_training_shapes.py).

The reference is evaluated at the device's current parameters and running statistics, copied back before the step,
with the masks oracle.dropout_np reconstructs from the step's seed: errors cannot compound over steps, and a step that
used another mask than the one its seed names (a stale seed in a graph replay, a backward pass recomputing another mask)
moves whole gradient rows.

An fp32 run can take the other side of a ReLU than the reference where a pre-activation lies within its rounding error
of zero, and one such flip moves a weight-gradient row by about a per cent.  So every comparison asserts the smallest
|pre-activation| of the step (the ReLU margin): >= 1e-6 for ordinary parameters, whose data seeds are chosen for it,
and >= 1e-2 for "saturated" parameters (every norms.j weight 0.25, bias 3: every ReLU site active by many sigma), which
the larger batches use.  The tolerances are the suite's: loss 1e-5, scores 2e-5, every gradient tensor
|err| <= 3e-4 * max|ref| + 5e-7; the two gradients that are zero by symmetry are checked to stay at rounding noise."""
import numpy as np
import torch

from oracle import dropout_np, train_torch

DEV = torch.device("cuda:0")
ZERO_BY_SYMMETRY = ("fc.bias", ".normv.bias")     # the output Linear's bias before BatchNorm1d(K), normv.bias
NOISE = 2e-6
MARGIN = 1e-6
SATURATED_MARGIN = 1e-2


def saturate(sd: dict, conf) -> dict:
    sd = dict(sd)
    for l, n_fc in enumerate(conf):
        for j in range(n_fc):
            p = f"embedded_mappings.{l}.norms.{j}"
            sd[p + ".weight"] = torch.full_like(sd[p + ".weight"], 0.25)
            sd[p + ".bias"] = torch.full_like(sd[p + ".bias"], 3.0)
    return sd


def ok(a: np.ndarray, b: np.ndarray) -> bool:
    return float(np.abs(a - b).max()) <= 3e-4 * float(np.abs(b).max()) + 5e-7


def reference(sd: dict, x: torch.Tensor, labels: torch.Tensor, conf, masks: dict, oracle_dev=None):
    """(loss, scores, grads, running stats after the step, ReLU margin) in float64."""
    dev = oracle_dev or torch.device("cpu")
    sd = {k: v.to(dev) for k, v in sd.items()}
    x, labels = x.to(dev), labels.to(dev)
    pre = []
    loss, scores, grads = train_torch.head_step(sd, x, labels, conf, masks=masks, dtype=torch.float64, relu_pre=pre)
    running = train_torch.updated_running_stats(sd, x, conf, masks=masks, dtype=torch.float64)
    return (float(loss), scores.cpu(), {k: (None if g is None else g.cpu()) for k, g in grads.items()},
            {k: v.cpu() for k, v in running.items()}, train_torch.relu_margin(pre))


def check_step(tr, x: torch.Tensor, labels: torch.Tensor, *, min_margin: float = MARGIN, running=None,
               keys=None, all_noise: bool = False, adam: bool = True, oracle_dev=None):
    """One tr.forward_backward (+ tr.adam) against the oracle.  `running`: the chained oracle running statistics
    (None: start from the device's).  keys: compare only these gradient tensors, and neither the loss, the scores nor
    the running statistics (at two clips BatchNorm1d(K) amplifies rounding there); all_noise: every gradient
    and the loss are zero in exact arithmetic (K = 1) and are checked to stay at rounding noise.  Returns
    (margin, largest gradient error as a fraction of its tolerance, chained running statistics)."""
    conf = tr.model_conf
    emb_in, hidden, K, T = tr.dims
    B = x.shape[0]
    sd = {k: v.cpu() for k, v in tr.state_dict().items()}
    if running is not None:
        sd.update(running)
    seed = tr.seed + tr.step_count
    masks = dropout_np.step_masks(seed, conf, B, T, hidden, tr.dropout_p)
    loss, scores = tr.forward_backward(x, labels, want_scores=True)
    ref_loss, ref_scores, ref_grads, ref_running, margin = reference(sd, x, labels, conf, masks, oracle_dev)
    assert margin >= min_margin, f"ReLU margin {margin:.3e} < {min_margin:.0e}: choose other data"
    full = keys is None
    keys = keys or [k for k, _, _ in tr.p_layout]
    worst, bad = 0.0, []
    for k in keys:
        got, ref = tr.view(tr.grads, k).double().cpu().numpy(), ref_grads[k].numpy()
        ref_max = float(np.abs(ref).max())
        if all_noise or (k.endswith(ZERO_BY_SYMMETRY) and ref_max < NOISE):
            if float(np.abs(got).max()) >= NOISE:
                bad.append((k, float(np.abs(got).max()), ref_max))
            continue
        worst = max(worst, float(np.abs(got - ref).max()) / (3e-4 * ref_max + 5e-7))
        if not ok(got, ref):
            bad.append((k, float(np.abs(got - ref).max()), ref_max))
    assert not bad, f"seed {seed}: {bad}"
    if all_noise:
        assert abs(loss.item()) <= NOISE and abs(ref_loss) <= NOISE
    elif full:
        assert abs(loss.item() - ref_loss) < 1e-5, (loss.item(), ref_loss)
        assert float((scores.double().cpu() - ref_scores).abs().max()) < 2e-5
    if full:
        out = tr.state_dict()
        for k, want in ref_running.items():
            got = out[k].double().cpu()
            err = float((got - want).abs().max())
            assert err <= 1e-4 * float(want.abs().max()) + 1e-6, (k, err)
    if adam:
        g, m0, v0, p0 = tr.grads.clone(), tr.exp_avg.clone(), tr.exp_avg_sq.clone(), tr.params.clone()
        tr.adam(1)
        want_p, want_m, want_v = train_torch.adam_update(p0, g, tr.lr, tr.betas, tr.eps, tr.step_count, m0, v0,
                                                         moments=True)
        for name, got, want in (("exp_avg", tr.exp_avg, want_m), ("exp_avg_sq", tr.exp_avg_sq, want_v),
                                ("params", tr.params, want_p)):
            err = float((got[:tr.n_params] - want[:tr.n_params]).abs().max())
            assert err <= 5e-7, (name, err)
    return margin, worst, ref_running
