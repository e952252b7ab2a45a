"""Host-side checks of head training with a wide first layer (emb_in = 12288, the just_bottlenecks configuration,
model.py:43-44): the flat parameter layout the Python side and the library agree on, and the capacity bound that
vmb_mla_trainer_create validates before it allocates anything."""
import ctypes as C

import pytest
import torch

from b200 import _lib, training

JB = 12288


@pytest.mark.parametrize("conf,K,want", [((2, 1), 527, 9285273), ((1,), 10, None)])
def test_wide_layout_matches_the_library(conf, K, want):
    _, _, n_p, n_r = training.train_layout(conf, JB, 600, K, 10)
    arr = (C.c_int * len(conf))(*conf)
    n_run = C.c_longlong(0)
    assert _lib.lib().vmb_mla_train_param_count(len(conf), arr, JB, 600, K, 10, C.byref(n_run)) == n_p
    assert n_run.value == n_r
    if want is not None:
        assert n_p == want
        assert training.train_layout(conf, 128, 600, K, 10)[2] == 1989273
        assert n_p - 1989273 == 600 * (JB - 128)


def _create(conf, emb_in, max_batch, t_steps=10):
    arr = (C.c_int * len(conf))(*conf)
    h = C.c_void_p()
    rc = _lib.lib().vmb_mla_trainer_create(C.byref(h), len(conf), arr, emb_in, 600, 527, t_steps, max_batch, None)
    if rc == 0:
        _lib.lib().vmb_mla_trainer_destroy(h)
    return rc, _lib.lib().vmb_last_error().decode()


def test_wide_trainer_capacity_bound_is_checked_before_allocation():
    # the operand planes of xhat, [pad64(batch * T)][3 * 12288] bf16, stay within a signed 32-bit element index:
    # 58240 rows, 5824 clips at T = 10
    rc, msg = _create((2, 1), JB, 5825)
    assert rc != 0 and "too large for emb_in 12288" in msg and "at most 5824 clips" in msg
    rc, msg = _create((1,), JB, 100000, t_steps=4)
    assert rc != 0 and "at most 14560 clips" in msg
    # within the bound (the module bridge's 4096 included) validation passes: without a GPU only the workspace
    # allocation can fail, never the argument checks
    for mb in (4096, 5824):
        rc, msg = _create((2, 1), JB, mb)
        if rc != 0:
            assert not torch.cuda.is_available()
            assert "not supported" not in msg and "too large" not in msg and "bad max_batch" not in msg
            assert "workspace allocation failed" in msg
    # the narrow configuration keeps its bound
    rc, msg = _create((2, 1), 128, 0x7FFFFFFF // 2048 // 10 + 1)
    assert rc != 0 and "bad max_batch" in msg
