"""ORACLE (test infrastructure, never shipped or timed as the product): one training step of the multi-level
attention head on the CPU with torch autograd, restating what the reference's loop does to the head
(train.py:124-138 with criterion = nn.CrossEntropyLoss() applied to the sigmoid outputs, train.py:372, and
optim.Adam(lr=0.001), train.py:369; the CNN is frozen, model.py:159-160).

Parity pin: tests/golden/head.npz holds the loss, outputs, gradients, updated parameters and updated running
statistics of ONE such step run through the reference's own MultiLevelAttention module
(tests/golden/make_golden.py); tests/test_oracle_golden.py checks this restatement against them.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import model_torch

BN_MOMENTUM = 0.1


def cast(sd: dict, x: torch.Tensor, dtype):
    """(sd, x) with x and every floating-point tensor of sd in `dtype` (None: unchanged)."""
    if dtype is None:
        return sd, x
    return {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}, x.to(dtype)


def relu_margin(relu_pre: list) -> float:
    """Smallest |input| over every ReLU site collected by mla_forward(relu_pre=...): an fp32 run can only take the
    other side of a ReLU than this reference where its rounding error reaches this margin."""
    return min(float(t.abs().min()) for t in relu_pre)


def head_step(sd: dict, x: torch.Tensor, labels: torch.Tensor, model_conf, dropout_p: float = 0.0,
              masks: dict | None = None, dtype=None, relu_pre: list | None = None):
    """Returns (loss, scores, grads) for the mean CE-on-sigmoid loss; `grads` maps state_dict keys of trainable
    tensors to gradients (None for fcf, which the forward never touches — SURVEY F3).  `masks`: explicit dropout
    scales (model_torch.mla_forward); dtype=torch.float64 evaluates the step in double precision."""
    sd, x = cast(sd, x, dtype)
    leaves = {}
    work = {}
    for k, v in sd.items():
        if v.is_floating_point() and "running_" not in k:
            leaves[k] = v.detach().clone().requires_grad_(True)
            work[k] = leaves[k]
        else:
            work[k] = v
    scores = model_torch.mla_forward(work, x, model_conf, training=True, dropout_p=dropout_p, masks=masks,
                                     relu_pre=relu_pre)
    loss = F.cross_entropy(scores, labels)
    loss.backward()
    return loss.detach(), scores.detach(), {k: t.grad for k, t in leaves.items()}


def updated_running_stats(sd: dict, x: torch.Tensor, model_conf, masks: dict | None = None, dtype=None) -> dict:
    """running_mean / running_var of every BatchNorm after one train-mode forward (momentum 0.1, unbiased variance),
    computed by replaying the forward with F.batch_norm writing into copies of the buffers.  With dropout the
    statistics of every later BatchNorm depend on the step's `masks` (model_torch.mla_forward)."""
    sd, x = cast(sd, x, dtype)
    work = {k: (v.clone() if "running_" in k else v) for k, v in sd.items()}

    def bn(prefix, t):
        return F.batch_norm(t, work[prefix + ".running_mean"], work[prefix + ".running_var"], work[prefix + ".weight"],
                            work[prefix + ".bias"], True, BN_MOMENTUM, model_torch.BN_EPS)

    with torch.no_grad():
        embs, h = [], x
        for lvl, n_fc in enumerate(model_conf):
            p = f"embedded_mappings.{lvl}"
            h = bn(p + ".norm0", h)
            for j in range(n_fc):
                h = F.relu(bn(f"{p}.norms.{j}", F.linear(h, work[f"{p}.fc.{j}.weight"], work[f"{p}.fc.{j}.bias"])))
                if masks is not None:
                    h = h * torch.as_tensor(masks[(lvl, j)], dtype=h.dtype, device=h.device)
            embs.append(h)
        ys = []
        for lvl in range(len(model_conf)):
            p = f"attention_modules.{lvl}"
            z = F.linear(embs[lvl], work[p + ".fcv.weight"], work[p + ".fcv.bias"])
            att = F.softmax(bn(p + ".normv", z), dim=2)
            cla = torch.sigmoid(bn(p + ".normf", z))
            ys.append(torch.sum(cla * (att / att.sum(dim=1)[:, None, :]), dim=1))
        bn("norm", F.linear(torch.cat(ys, dim=1), work["fc.weight"], work["fc.bias"]))
    return {k: v for k, v in work.items() if "running_" in k}


def adam_update(param: torch.Tensor, grad: torch.Tensor, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, step=1,
                exp_avg=None, exp_avg_sq=None, moments: bool = False):
    """torch.optim.Adam's single-tensor update (amsgrad False, weight_decay 0): the new parameter, or with
    moments=True (parameter, exp_avg, exp_avg_sq)."""
    m = torch.zeros_like(param) if exp_avg is None else exp_avg
    v = torch.zeros_like(param) if exp_avg_sq is None else exp_avg_sq
    m = m.lerp(grad, 1 - betas[0])
    v = v * betas[1] + (1 - betas[1]) * grad * grad
    bc1, bc2 = 1 - betas[0] ** step, 1 - betas[1] ** step
    new = param - (lr / bc1) * m / (v.sqrt() / bc2 ** 0.5 + eps)
    return (new, m, v) if moments else new
