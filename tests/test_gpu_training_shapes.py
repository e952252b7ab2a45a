"""Head training at the limits of the shapes vmb_mla_trainer_create accepts (T 1..16, hidden and K 1..1024, emb_in
1..16384, 1..4 levels of 1..4 Linears, batch 2..max_batch), with dropout 0.4: every case runs an eager step and a
CUDA-graph replay (under another seed) against the float64 oracle with the step's own dropout masks
(tests/_head_step_oracle.py).  Up to 128 clips the parameters are ordinary and the data seed is one whose ReLU margin
is >= 1e-6; above that the parameters are saturated."""
import pytest
import torch

from _head_step_oracle import DEV, SATURATED_MARGIN, check_step, saturate
from b200 import synth, training

pytestmark = pytest.mark.gpu
SEEDS = (2 ** 32 + 11, 2 ** 41 + 7)     # eager step, replayed step

# id: (model_conf, emb_in, hidden, K, T, batch, data seed)
CASES = {
    "T1": ((1,), 128, 64, 3, 1, 33, 0),                  # BatchNorm1d(T) over one time step
    "T16_K1024": ((2, 1), 128, 600, 1024, 16, 33, 5),    # attention-backward shared memory; fused-statistics limit
    "T13_K1024": ((1,), 128, 64, 1024, 13, 33, 0),       # smallest T whose attention backward needs > 100 KB
    "hidden1024": ((2, 1), 128, 1024, 10, 10, 33, 6),    # largest accepted width
    "hidden40_K130": ((2, 1), 128, 40, 130, 10, 33, 0),  # K > hidden: the padded width comes from K
    "emb131": ((2, 1), 131, 64, 10, 10, 33, 2),          # row stride not a multiple of 4
    "emb640": ((2, 1), 640, 600, 10, 10, 33, 1),         # last narrow first layer
    "emb641": ((2, 1), 641, 600, 10, 10, 33, 13),        # first wide first layer (inpad 768, one split-K slice)
    "conf4444": ((4, 4, 4, 4), 128, 128, 10, 10, 33, 2), # every weight-job and BatchNorm slot limit
    "K1": ((2, 1), 128, 64, 1, 10, 33, 0),               # loss and every gradient zero in exact arithmetic
    "batch2": ((2, 1), 128, 64, 10, 10, 2, 0),           # smallest batch
    "batch77": ((2, 1), 128, 64, 10, 10, 77, 0),         # ragged row tiles (770 rows)
    "batch513": ((2, 1), 128, 600, 527, 10, 513, 0),     # out_bn_backward past its register path
    "batch1000": ((2, 1), 128, 600, 527, 10, 1000, 0),   # weight-gradient contraction of 10 000 rows
    "batch4096": ((2, 1), 128, 600, 527, 10, 4096, 0),   # the module bridge's capacity
}


def case_inputs(conf, emb_in, hidden, K, T, batch, data_seed):
    sd = synth.mla_state_dict(conf, emb_in, hidden, K, T, seed=3)
    if batch > 128:
        sd = saturate(sd, conf)
    g = torch.Generator().manual_seed(data_seed)
    x = torch.randn(batch, T, emb_in, generator=g)
    labels = torch.randint(0, K, (batch,), generator=g)
    return sd, x, labels


@pytest.mark.parametrize("case", list(CASES))
def test_shape_limits_vs_float64_oracle(case):
    conf, emb_in, hidden, K, T, batch, data_seed = CASES[case]
    sd, x, labels = case_inputs(conf, emb_in, hidden, K, T, batch, data_seed)
    tr = training.HeadTrainer(conf, emb_in, hidden, K, T, batch, DEV, dropout_p=0.4)
    tr.load_state_dict(sd)
    kw = dict(adam=False, oracle_dev=DEV if batch >= 1000 else None)
    if batch > 128:
        kw["min_margin"] = SATURATED_MARGIN
    if K == 1:
        kw["all_noise"] = True
    if batch == 2:
        # BatchNorm1d(K) over two rows amplifies rounding in the scores: compare the first Linear's block
        kw["keys"] = ["embedded_mappings.0.norm0.weight", "embedded_mappings.0.norm0.bias",
                      "embedded_mappings.0.fc.0.weight", "embedded_mappings.0.fc.0.bias"]
    try:
        for step, seed in enumerate(SEEDS):
            tr.seed = seed
            margin, worst, _ = check_step(tr, x, labels, **kw)
            print(f"{case} {'eager' if step == 0 else 'replay'}: ReLU margin {margin:.2e}, "
                  f"worst gradient error {worst:.2f} of its tolerance")
    finally:
        tr.close()
