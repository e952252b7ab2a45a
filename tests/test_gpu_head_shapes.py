"""The eval-mode head (vmb_mla_forward, csrc/mla_tc.cu: what MultiLevelAttention.eval(), Ensemble, the pipeline and
bench.py run) across the shapes vmb_mla_create accepts: 1..4 levels of 1..4 Linears, emb_in 1..16384, hidden and K
1..608, T = 10.  Each case sits on a boundary of the code: the padded operand widths (multiples of 64 against the
640-column activation pitch), the fp32 cross-check kernel's input limit and its transposed-weight limit, the rotating
plane buffers of deep configurations, and GEMMs of more than one wave of tiles.

Every case is checked against the float64 oracle evaluated from the same fp32 parameters and inputs, at the head's
bound of 2e-5 absolute on the scores (test_gpu_parity.py).  Every case also asserts that at least 30 % of the scores
lie in [0.02, 0.98]: saturated scores would meet the bound whatever the kernels computed (if one stops doing so, scale
its inputs, not the tolerance)."""
import pytest
import torch

from b200 import _lib, engine, synth
from oracle import model_torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
T = 10
TOL = 2e-5
MIN_UNSATURATED = 0.3

# id: (model_conf, emb_in, hidden, K, batch)
CASES = {
    "hidden1": ((2, 1), 128, 1, 10, 33),                   # smallest width
    "hidden40_K130": ((2, 1), 128, 40, 130, 33),           # K > hidden
    "hidden64": ((1, 2, 1), 128, 64, 10, 77),              # operands of hidden width padded to 64 < 640; ragged row tiles
    "hidden576": ((2, 1), 128, 576, 527, 33),              # largest width padded to less than 640
    "hidden577": ((2, 1), 128, 577, 527, 33),              # smallest width padded to 640
    "limits608": ((2, 1), 128, 608, 608, 33),              # both limits; pooling at 48 640 B of shared memory
    "K1": ((2, 1), 128, 64, 1, 33),                        # BatchNorm1d(1), softmax over one class
    "emb1": ((1,), 1, 64, 10, 13),                         # narrowest input
    "emb131": ((2, 1), 131, 600, 10, 33),                  # input rows not a multiple of 4
    "emb641": ((2, 1), 641, 600, 10, 33),                  # first input past the fp32 cross-check's limit
    "emb4097": ((1,), 4097, 600, 10, 33),                  # no transposed fp32 copy of the first Linear above 4 096
    "emb12288": ((1,), 12288, 600, 527, 77),               # just_bottlenecks in eval mode
    "emb16384": ((2, 1), 16384, 600, 10, 13),              # widest accepted input
    "conf111": ((1, 1, 1), 128, 600, 527, 400),            # middle level of one Linear, more than one wave of tiles
    "conf212": ((2, 1, 2), 128, 64, 10, 1000),             # the same at hidden 64
    "conf1111": ((1, 1, 1, 1), 128, 600, 527, 4096),       # three rotating buffers, side stream, two middle levels
    "conf4444": ((4, 4, 4, 4), 128, 128, 10, 300),         # every level and Linear slot
    "batch1": ((2, 1), 128, 600, 527, 1),                  # one clip
    "batch4096": ((2, 1), 128, 600, 527, 4096),            # the module bridge's capacity
}


def oracle_scores(sd: dict, x: torch.Tensor, conf, dev) -> torch.Tensor:
    """Scores of the head in float64 from the fp32 parameters and inputs, on `dev`, returned on the CPU."""
    sd64 = {k: v.to(device=dev, dtype=torch.float64) for k, v in sd.items() if v.is_floating_point()}
    with torch.no_grad():
        return model_torch.mla_forward(sd64, x.to(device=dev, dtype=torch.float64), conf).cpu()


def case_inputs(conf, emb_in, hidden, K, batch, seed=0):
    sd = synth.mla_state_dict(conf, emb_in, hidden, K, T, seed=seed + 2)
    g = torch.Generator().manual_seed(seed)
    return sd, torch.randn(batch, T, emb_in, generator=g) * 1.5


def unsaturated(ref: torch.Tensor) -> float:
    return float(((ref >= 0.02) & (ref <= 0.98)).double().mean())


@pytest.mark.parametrize("case", list(CASES))
def test_eval_head_vs_float64_oracle(case):
    conf, emb_in, hidden, K, batch = CASES[case]
    sd, x = case_inputs(conf, emb_in, hidden, K, batch)
    ref = oracle_scores(sd, x, conf, DEV if batch >= 1000 else torch.device("cpu"))
    assert unsaturated(ref) >= MIN_UNSATURATED, f"{case}: only {unsaturated(ref):.0%} of the scores are unsaturated"
    L = _lib.lib()
    h = engine.MlaHandle(sd, conf, emb_in, hidden, K, T, DEV)
    xd = x.to(DEV)
    L.vmb_mla_fuse_enable(1)
    try:
        first = h.forward(xd)
        second = h.forward(xd)
        y32 = h.forward(xd, fp32_crosscheck=True) if emb_in <= 608 else None
        torch.cuda.synchronize()
    finally:
        L.vmb_mla_fuse_enable(-1)
        h.close()
    assert first.shape == (batch, K)
    err = float((first.double().cpu() - ref).abs().max())
    msg = f"{case}: worst error {err / TOL:.3f} of {TOL:.0e} ({unsaturated(ref):.0%} of the scores unsaturated)"
    if y32 is not None:
        err32 = float((y32.double().cpu() - ref).abs().max())
        msg += f"; fp32 CUDA-core kernel {err32 / TOL:.3f}"
    print(msg)
    assert torch.equal(first, second), f"{case}: two calls on the same input differ"
    assert err <= TOL, msg
    if y32 is not None:
        assert err32 <= TOL, msg


def _reference_head(conf, hidden, K):
    """model.MultiLevelAttention built the way INTEGRATION.md tells users to: the module globals set first."""
    import model
    old = model.H, model.K
    try:
        model.H, model.K = hidden, K
        return model.MultiLevelAttention(list(conf), 128)
    finally:
        model.H, model.K = old


def test_standalone_modules_at_hidden_64():
    """EmbeddedMapping.forward and AttentionModule.forward on their own (model.py:217-222, :235-242) at H = 64, K = 10,
    against the float64 oracle: level 0 and a later level, each with two Linears, so that the second Linear and fcv read
    operands of hidden width.  Tolerances of test_standalone_embedded_mapping_and_attention_module."""
    conf = (2, 2)
    m = _reference_head(conf, 64, 10)
    sd = synth.mla_state_dict(conf, 128, 64, 10, T, seed=7)
    m.load_state_dict(sd)
    m = m.to(DEV).eval()
    x = torch.randn(33, T, 128, generator=torch.Generator().manual_seed(1)) * 1.5
    e0 = m.embedded_mappings[0](x.to(DEV))
    e1 = m.embedded_mappings[1](e0)
    y0 = m.attention_modules[0](e0)
    y1 = m.attention_modules[1](e1)
    sd64 = {k: v.double() for k, v in sd.items() if v.is_floating_point()}
    pre = []
    with torch.no_grad():
        model_torch.mla_forward(sd64, x.double(), conf, relu_pre=pre)
        refs = {"emb0": (e0, torch.relu(pre[1]), 5e-5), "emb1": (e1, torch.relu(pre[3]), 5e-5),
                "y0": (y0, model_torch.attention_module(sd64, 0, e0.double().cpu()), 2e-5),
                "y1": (y1, model_torch.attention_module(sd64, 1, e1.double().cpu()), 2e-5)}
    for name, (got, ref, tol) in refs.items():
        err = float((got.double().cpu() - ref).abs().max())
        bound = tol * max(1.0, float(ref.abs().max()))
        print(f"standalone {name} at H=64: worst error {err / bound:.3f} of its tolerance")
        assert got.shape == ref.shape and err <= bound, name


def test_train_step_then_eval_at_hidden_64():
    """conf [1, 1, 1] at H = 64, K = 10: one train-mode step of the reference's loop (train.py:124-138), then .eval():
    the eval-mode head must compute the float64 oracle's scores at the module's updated parameters and running
    statistics, at a batch whose middle-level GEMM takes more than one wave of tiles."""
    conf = (1, 1, 1)
    m = _reference_head(conf, 64, 10)
    m.load_state_dict(synth.mla_state_dict(conf, 128, 64, 10, T, seed=8))
    m = m.to(DEV).train()
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(64, T, 128, generator=g) * 1.5).to(DEV)
    labels = torch.randint(0, 10, (64,), generator=g).to(DEV)
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=0.001)
    opt.zero_grad()
    loss = torch.nn.CrossEntropyLoss()(m(x), labels)
    loss.backward()
    opt.step()
    assert int(m.norm.num_batches_tracked) == 1
    m.eval()
    xe = torch.randn(400, T, 128, generator=g) * 1.5
    y = m(xe.to(DEV))
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    ref = oracle_scores(sd, xe, conf, torch.device("cpu"))
    assert unsaturated(ref) >= MIN_UNSATURATED
    err = float((y.double().cpu() - ref).abs().max())
    print(f"train step then eval at H=64: worst error {err / TOL:.3f} of {TOL:.0e}")
    assert err <= TOL
