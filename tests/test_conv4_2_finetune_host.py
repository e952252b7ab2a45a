"""CPU-side checks of VGGish conv4_2 fine-tuning (features.13 trainable, conv1 .. conv4_1 frozen): argument checks of
the new entry points, the conv4_2 train workspace arithmetic, the conv4_2 gradient layout against state_dict order,
the three-part handle key, and the configurations that raise before anything reaches a device."""
import ctypes as C

import pytest
import torch

from b200 import _lib, engine
from b200._lib import B200Error


def _up(v):
    return (v + 1023) // 1024 * 1024


def _conv4_2_ws_bytes(n):
    """conv4_2_layout (csrc/conv_train.cu): the FC train layout, then z, dz planes, dX1, dW, bias sums, im2col chunk."""
    L = _lib.lib()
    rows = n * 96
    regions = [rows * 512 * 4, rows * 3 * 512 * 2, n * 12288 * 4, 512 * 4608 * 4, 512 * 8,
               min(n, 256) * 96 * 3 * 4608 * 2]
    return int(L.vmb_vggish_fc_train_workspace_bytes(n)) + sum(_up(r) for r in regions)


@pytest.mark.parametrize("n", [1, 63, 64, 65, 960, 5120])
def test_conv4_2_workspace_arithmetic(n):
    assert int(_lib.lib().vmb_vggish_conv4_2_train_workspace_bytes(n)) == _conv4_2_ws_bytes(n)


def test_conv4_2_workspace_of_no_examples_is_zero():
    L = _lib.lib()
    assert L.vmb_vggish_conv4_2_train_workspace_bytes(0) == 0
    assert L.vmb_vggish_conv4_2_train_workspace_bytes(-3) == 0


def test_conv4_2_gradient_layout_matches_state_dict_order():
    from torchvggish import vggish
    vgg = vggish.VGG(vggish.make_layers())
    sd = vgg.features[13].state_dict()
    assert [k for k, _ in engine.CONV4_2_GRAD_LAYOUT] == list(sd.keys())
    assert [tuple(s) for _, s in engine.CONV4_2_GRAD_LAYOUT] == [tuple(v.shape) for v in sd.values()]
    total = sum(v.numel() for v in sd.values())
    assert engine.CONV4_2_GRAD_COUNT == total == 2_359_808
    views = engine.conv4_2_grad_views(torch.arange(total, dtype=torch.float32))
    off = 0
    for k, v in sd.items():
        assert views[k].shape == v.shape and float(views[k].reshape(-1)[0]) == off
        off += v.numel()
    # OIHW like nn.Conv2d: element [o][c][kh][kw] at ((o * 512 + c) * 3 + kh) * 3 + kw
    assert float(views["weight"][2, 5, 1, 2]) == ((2 * 512 + 5) * 3 + 1) * 3 + 2


def test_conv4_2_entry_points_check_their_arguments():
    L = _lib.lib()
    assert L.vmb_vggish_refresh_conv4_2(None, None, None, None, None) != 0
    assert "vmb_vggish_refresh_conv4_2: null handle" in _lib.last_error()
    assert L.vmb_vggish_forward_train_conv4_2(None, None, 10, None, None, 0, None) != 0
    assert "vmb_vggish_forward_train_conv4_2: null handle" in _lib.last_error()
    assert L.vmb_vggish_conv4_2_backward(None, None, 0, None, 10, None, None, None) != 0
    assert "vmb_vggish_conv4_2_backward: null handle" in _lib.last_error()


def test_three_part_handle_key():
    from torchvggish.vggish import handle_action
    frozen, c42, fc = ("convs", 1, "fp16"), ("c42", 1), ("fc", 1)
    key = (frozen, c42, fc)
    assert handle_action(None, key, False, False) == "rebuild"
    assert handle_action(key, key, True, True) == "keep"
    assert handle_action(key, (frozen, ("c42", 2), fc), True, True) == "refresh"      # an optimiser step of conv4_2
    assert handle_action(key, (frozen, ("c42", 2), ("fc", 2)), True, True) == "refresh"
    assert handle_action(key, (frozen, ("c42", 2), fc), True, False) == "rebuild"     # no conv training copy
    assert handle_action(key, (frozen, ("c42", 2), fc), False, False) == "rebuild"
    assert handle_action(key, (frozen, c42, ("fc", 2)), True, False) == "refresh"     # FC fine-tuning as before
    assert handle_action(key, (frozen, c42, ("fc", 2)), False, True) == "rebuild"
    assert handle_action(key, (("convs", 2, "fp16"), c42, fc), True, True) == "rebuild"
    assert handle_action(key, (("convs", 1, "bf16"), c42, fc), True, True) == "rebuild"


def _ensemble(**kw):
    import model
    conf = dict(cnn_type="vggish", num_classes=10, use_pretrained=False, just_bottlenecks=False, cnn_trainable=False,
                first_cnn_layer_trainable=False, in_channels=1)
    conf.update(kw)
    return model.Ensemble("repeat", conf, [2, 1], torch.device("cpu"))


X = torch.zeros(1, 10, 1, 96, 64)


@pytest.mark.parametrize("layers", [(11,), (11, 13)])
def test_conv_below_conv4_2_still_raises(layers):
    import model
    ens = _ensemble().train()
    for i in layers:
        model.set_requires_grad(ens.cnn.cnn_model.features[i], True)
    with pytest.raises(NotImplementedError, match="conv stack"):
        ens.cnn(ens.input(X))


def test_whole_body_still_raises():
    ens = _ensemble(cnn_trainable=True).train()
    with pytest.raises(NotImplementedError, match="conv stack"):
        ens.cnn(ens.input(X))


def test_conv4_2_alone_reaches_the_library():
    import model
    ens = _ensemble().train()
    model.set_requires_grad(ens.cnn.cnn_model.features[13], True)
    with pytest.raises(B200Error):
        ens.cnn(ens.input(X))                                                    # CPU module: no fallback
    model.set_requires_grad(ens.cnn.cnn_model.embeddings, True)
    with pytest.raises(B200Error):
        ens.cnn(ens.input(X))


def test_just_bottlenecks_with_conv4_2_trainable_raises():
    import model
    ens = _ensemble(just_bottlenecks=True).train()
    model.set_requires_grad(ens.cnn.cnn_model[0][13], True)
    with pytest.raises(NotImplementedError, match="just_bottlenecks"):
        ens.cnn(ens.input(X))


def test_just_bottlenecks_with_cnn_trainable_raises_in_train_mode():
    """It used to train nothing: the features came back detached and Adam skipped every conv parameter."""
    ens = _ensemble(just_bottlenecks=True, cnn_trainable=True).train()
    with pytest.raises(NotImplementedError, match="just_bottlenecks"):
        ens.cnn(ens.input(X))
    with torch.no_grad(), pytest.raises(B200Error):                              # inference still reaches the library
        ens.cnn(ens.input(X))
