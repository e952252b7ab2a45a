"""ORACLE (test infrastructure, never shipped or timed as the product): fp32 CPU restatement of the
reference's VGGish network, PCA postprocessor and multi-level-attention head as pure functions of a
reference-format state_dict (key names of SURVEY.md §8b).

Follows
  torchvggish/vggish.py:108-118  make_layers  (conv3x3 pad 1 + ReLU, MaxPool2d(2,2) after convs 1, 2, 4, 6)
  torchvggish/vggish.py:21-31    VGG.forward  (NCHW -> (h,w,c) flatten -> 3x Linear+ReLU)
  torchvggish/vggish.py:62-102   Postprocessor.postprocess
  model.py:217-222               EmbeddedMapping.forward
  model.py:236-242               AttentionModule.forward  (uses fcv twice; softmax over the class axis)
  model.py:258-269               MultiLevelAttention.forward
The arithmetic third parties (torch CPU conv/linear/batch_norm kernels) are whatever torch is installed
(2.11.0 here); the reference pins none.

Parity pin: checked bit-for-bit / to 1e-6 against the reference's own nn.Modules executed in the build
container (tests/golden/make_golden.py), see tests/test_oracle_golden.py.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

CONV_KEYS = (0, 3, 6, 8, 11, 13)          # indices of the Conv2d modules inside VGG.features
POOL_AFTER = (0, 3, 8, 13)                # convs followed by MaxPool2d
FC_KEYS = (0, 2, 4)                       # indices of the Linear modules inside VGG.embeddings
BN_EPS = 1e-5                             # nn.BatchNorm1d default


def vgg_features(sd: dict, x: torch.Tensor, collect: list | None = None) -> torch.Tensor:
    for k in CONV_KEYS:
        x = F.relu(F.conv2d(x, sd[f"features.{k}.weight"], sd[f"features.{k}.bias"], padding=1))
        if k in POOL_AFTER:
            x = F.max_pool2d(x, kernel_size=2, stride=2)
        if collect is not None:
            collect.append(x)
    return x


def vgg_flatten(x: torch.Tensor) -> torch.Tensor:
    """NCHW -> (N, H*W*C) in (h, w, c) order (vggish.py:26-29)."""
    return x.permute(0, 2, 3, 1).contiguous().view(x.size(0), -1)


def vgg_embeddings(sd: dict, x: torch.Tensor, collect: list | None = None) -> torch.Tensor:
    for k in FC_KEYS:
        x = F.relu(F.linear(x, sd[f"embeddings.{k}.weight"], sd[f"embeddings.{k}.bias"]))
        if collect is not None:
            collect.append(x)
    return x


def vgg_forward(sd: dict, x: torch.Tensor, collect: list | None = None) -> torch.Tensor:
    """x (N,1,96,64) fp32 -> (N,128) post-ReLU embeddings."""
    return vgg_embeddings(sd, vgg_flatten(vgg_features(sd, x, collect)), collect)


def postprocess(eigen: torch.Tensor, means: torch.Tensor, emb: torch.Tensor) -> torch.Tensor:
    """PCA + clamp + 8-bit quantise; float32 values in 0..255, squeezed like the reference (F6)."""
    assert emb.dim() == 2, "Expected 2-d batch, got %r" % (emb.shape,)
    assert emb.shape[1] == 128, "Bad batch shape: %r" % (emb.shape,)
    pca = torch.mm(eigen, (emb.t() - means.reshape(-1, 1))).t()
    clipped = torch.clamp(pca, -2.0, 2.0)
    q = torch.round((clipped - (-2.0)) * (255.0 / (2.0 - (-2.0))))
    return torch.squeeze(q)


def _bn_time(sd: dict, prefix: str, x: torch.Tensor, training: bool) -> torch.Tensor:
    """BatchNorm1d(T) on (B, T, F): the 'channel' is the time step (model.py:205; SURVEY F5)."""
    return F.batch_norm(x, None if training else sd[prefix + ".running_mean"],
                        None if training else sd[prefix + ".running_var"],
                        sd[prefix + ".weight"], sd[prefix + ".bias"], training, 0.1, BN_EPS)


def attention_module(sd: dict, lvl: int, h: torch.Tensor, training: bool = False) -> torch.Tensor:
    """AttentionModule.forward of level `lvl` (model.py:235-242): (B, T, H) -> (B, K)."""
    p = f"attention_modules.{lvl}"
    z = F.linear(h, sd[p + ".fcv.weight"], sd[p + ".fcv.bias"])
    att = F.softmax(_bn_time(sd, p + ".normv", z, training), dim=2)
    cla = torch.sigmoid(_bn_time(sd, p + ".normf", z, training))
    norm_att = att / torch.sum(att, dim=1)[:, None, :]
    return torch.sum(cla * norm_att, dim=1)


def mla_forward(sd: dict, x: torch.Tensor, model_conf, training: bool = False, dropout_p: float = 0.0,
                masks: dict | None = None, relu_pre: list | None = None):
    """x (B, T, M) -> (B, K) sigmoid scores.  training=True uses batch statistics (running stats are not
    updated here) and dropout_p (the reference's DR = 0.4) if non-zero.  `masks` {(level, j): (B, T, H) scale}
    replaces F.dropout with given inverted-dropout scales (oracle.dropout_np.step_masks); `relu_pre` collects the
    input of every ReLU."""
    embs = []
    h = x
    for lvl, n_fc in enumerate(model_conf):
        p = f"embedded_mappings.{lvl}"
        h = _bn_time(sd, p + ".norm0", h, training)
        for j in range(n_fc):
            h = F.linear(h, sd[f"{p}.fc.{j}.weight"], sd[f"{p}.fc.{j}.bias"])
            h = _bn_time(sd, f"{p}.norms.{j}", h, training)
            if relu_pre is not None:
                relu_pre.append(h.detach())
            h = F.relu(h)
            if masks is not None:
                h = h * torch.as_tensor(masks[(lvl, j)], dtype=h.dtype, device=h.device)
            elif training and dropout_p > 0:
                h = F.dropout(h, dropout_p, True)
        embs.append(h)
    conc = torch.cat([attention_module(sd, lvl, embs[lvl], training) for lvl in range(len(model_conf))], dim=1)
    out = F.linear(conc, sd["fc.weight"], sd["fc.bias"])
    out = F.batch_norm(out, None if training else sd["norm.running_mean"], None if training else sd["norm.running_var"],
                       sd["norm.weight"], sd["norm.bias"], training, 0.1, BN_EPS)
    return torch.sigmoid(out)


def ensemble_forward(vgg_sd: dict, mla_sd: dict, x: torch.Tensor, model_conf, t_steps: int = 10) -> torch.Tensor:
    """Ensemble.forward for cnn_type='vggish', just_bottlenecks=False (model.py:58-62): x (B,T,1,96,64)."""
    feats = vgg_forward(vgg_sd, x.reshape(-1, 1, 96, 64))
    return mla_forward(mla_sd, feats.reshape(-1, t_steps, 128), model_conf)
