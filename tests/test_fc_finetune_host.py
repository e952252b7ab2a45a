"""CPU-side checks of VGGish FC fine-tuning (fc1-fc3 trainable, convs frozen): argument checks of the new entry points,
the train-mode workspace arithmetic, the flat FC gradient layout against state_dict order, the split handle key, and
the configurations that still raise before anything reaches a device."""
import ctypes as C

import pytest
import torch

from b200 import _lib, engine, training
from b200._lib import B200Error


def _pad64(n):
    return (n + 63) // 64 * 64


def _up(v):
    return (v + 1023) // 1024 * 1024


def _train_ws_bytes(n):
    """fc_train_layout (csrc/fc_train.cu): X, A1, A2 planes, Z1, Z2, Z3, G planes, dA, column sums, conv scratch."""
    np_ = _pad64(n)
    regions = [np_ * 3 * 12288 * 2, np_ * 3 * 4096 * 2, np_ * 3 * 4096 * 2, np_ * 4096 * 4, np_ * 4096 * 4,
               np_ * 128 * 4, np_ * 3 * 4096 * 2, np_ * 4096 * 4, (4096 + 4096 + 128) * 8,
               int(_lib.lib().vmb_vggish_workspace_bytes(n)) * 2]
    return sum(_up(r) for r in regions)


@pytest.mark.parametrize("n", [1, 50, 63, 64, 65, 960, 5120])
def test_train_workspace_arithmetic(n):
    assert int(_lib.lib().vmb_vggish_fc_train_workspace_bytes(n)) == _train_ws_bytes(n)


def test_train_workspace_of_no_examples_is_zero():
    L = _lib.lib()
    assert L.vmb_vggish_fc_train_workspace_bytes(0) == 0 and L.vmb_vggish_fc_train_workspace_bytes(-3) == 0


def test_flat_gradient_layout_matches_state_dict_order():
    from torchvggish import vggish
    vgg = vggish.VGG(vggish.make_layers())
    sd = vgg.embeddings.state_dict()
    assert [k for k, _ in engine.FC_GRAD_LAYOUT] == list(sd.keys())
    assert [tuple(s) for _, s in engine.FC_GRAD_LAYOUT] == [tuple(v.shape) for v in sd.values()]
    total = sum(v.numel() for v in sd.values())
    assert int(_lib.lib().vmb_vggish_fc_grad_count()) == total == 67_641_472
    flat = torch.arange(total, dtype=torch.float32)
    views = engine.fc_grad_views(flat)
    off = 0
    for k, v in sd.items():                         # consecutive, in order, no gaps
        assert views[k].shape == v.shape and float(views[k].reshape(-1)[0]) == off
        off += v.numel()


def test_entry_points_check_their_arguments():
    L = _lib.lib()
    null3 = (C.c_void_p * 3)()
    assert L.vmb_vggish_refresh_fc(None, null3, null3, None) != 0
    assert "null handle" in _lib.last_error()
    assert L.vmb_vggish_forward_train(None, None, 10, None, None, 0, None) != 0
    assert "vmb_vggish_forward_train: null handle" in _lib.last_error()
    assert L.vmb_vggish_fc_backward(None, None, 0, None, 10, None, None) != 0
    assert "vmb_vggish_fc_backward: null handle" in _lib.last_error()
    assert L.vmb_mla_train_backward_dx(None, None, None, None, 2, 0.0, 0, None, None, None) != 0
    assert "null d(scores)" in _lib.last_error()
    assert L.vmb_mla_train_backward_dx(None, None, None, C.c_void_p(16), 2, 0.0, 0, None, None, None) != 0
    assert "null dx" in _lib.last_error()


@pytest.mark.parametrize("emb_in,hidden,K,ok", [(128, 600, 527, True), (640, 600, 527, True), (641, 600, 527, False),
                                                (12288, 600, 527, False), (131, 40, 1, False), (131, 40, 200, True)])
def test_input_gradient_needs_the_narrow_path(emb_in, hidden, K, ok):
    assert training.input_grad_supported(emb_in, hidden, K) is ok


def test_split_handle_key():
    from torchvggish.vggish import handle_action
    conv, fc = ("conv", 1, "fp16"), ("fc", 1)
    assert handle_action(None, (conv, fc), False) == "rebuild"
    assert handle_action((conv, fc), (conv, fc), True) == "keep"
    assert handle_action((conv, fc), (conv, ("fc", 2)), True) == "refresh"       # an optimiser step of fc1-fc3
    assert handle_action((conv, fc), (conv, ("fc", 2)), False) == "rebuild"      # eval-only handle: as before
    assert handle_action((conv, fc), (("conv", 2, "fp16"), fc), True) == "rebuild"
    assert handle_action((conv, fc), (("conv", 1, "bf16"), fc), True) == "rebuild"   # precision is in the conv part


def _ensemble(**kw):
    import model
    conf = dict(cnn_type="vggish", num_classes=10, use_pretrained=False, just_bottlenecks=False, cnn_trainable=False,
                first_cnn_layer_trainable=False, in_channels=1)
    conf.update(kw)
    return model.Ensemble("repeat", conf, [2, 1], torch.device("cpu"))


def test_conv_training_still_raises():
    import model
    x = torch.zeros(1, 10, 1, 96, 64)
    ens = _ensemble(cnn_trainable=True).train()
    with pytest.raises(NotImplementedError, match="conv stack"):
        ens.cnn(ens.input(x))
    ens = _ensemble().train()
    model.set_requires_grad(ens.cnn.cnn_model.features[0], True)               # one trainable conv layer
    with pytest.raises(NotImplementedError, match="conv stack"):
        ens.cnn(ens.input(x))
    model.set_requires_grad(ens.cnn.cnn_model.features[0], False)
    model.set_requires_grad(ens.cnn.cnn_model.embeddings, True)                # fc1-fc3 only: reaches the device
    with pytest.raises(B200Error):
        ens.cnn(ens.input(x))                                                   # CPU module: no fallback


def test_wide_head_refuses_an_input_gradient():
    ens = _ensemble(just_bottlenecks=True).train()
    x = torch.zeros(2, 10, 12288, requires_grad=True)
    with pytest.raises(NotImplementedError, match="wide first layer"):
        ens.mla(x)
