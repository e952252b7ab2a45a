"""Host-side checks of head training that need no GPU: the numpy port of the trainer's dropout masks
(oracle/dropout_np.py, which the float64 reference steps of tests/test_gpu_training_dropout.py use), the flat parameter
layout at the edges of the accepted shapes, and the argument checks of vmb_mla_trainer_create."""
import ctypes as C

import numpy as np
import pytest
import torch

from b200 import _lib, training
from oracle import dropout_np

N = 3 * 1024 * 1024


def _sigma(q, n):
    return (q * (1 - q) / n) ** 0.5


@pytest.mark.parametrize("p", [0.1, 0.4, 0.9])
def test_keep_rate_and_inverted_scale(p):
    s = dropout_np.dropout_scale(2 ** 33 + 5, dropout_np.layer_id(1, 2), np.arange(N, dtype=np.uint64), p)
    assert s.dtype == np.float32
    kept = s != 0
    assert abs(kept.mean() - (1 - p)) <= 5 * _sigma(1 - p, N)
    # the kept value is the float32 quotient 1 / (1 - p), exactly
    assert np.all(s[kept] == np.float32(1) / (np.float32(1) - np.float32(p)))


@pytest.mark.parametrize("p", [0.1, 0.4, 0.9])
def test_layers_and_seeds_draw_independent_masks(p):
    idx = np.arange(N, dtype=np.uint64)
    a = dropout_np.dropout_scale(1234, dropout_np.layer_id(0, 0), idx, p) != 0
    agree = p * p + (1 - p) ** 2
    for b in (dropout_np.dropout_scale(1234, dropout_np.layer_id(0, 1), idx, p) != 0,     # next Linear
              dropout_np.dropout_scale(1235, dropout_np.layer_id(0, 0), idx, p) != 0):    # next step
        assert abs((a == b).mean() - agree) <= 5 * _sigma(agree, N)


def test_upper_seed_bits_change_the_mask():
    idx = np.arange(1 << 16, dtype=np.uint64)
    lo = 0x12345678
    base = dropout_np.dropout_scale(lo, 1, idx, 0.4)
    for hi in (1, 2, 0x80000000):
        other = dropout_np.dropout_scale((hi << 32) | lo, 1, idx, 0.4)
        assert (base != other).mean() > 0.4


def test_step_masks_layout():
    """One array per (level, Linear), element (b, t, c) at index (b * T + t) * H + c of layer 1 + 4 * level + j."""
    m = dropout_np.step_masks(99, (2, 1), 3, 10, 7, 0.4)
    assert sorted(m) == [(0, 0), (0, 1), (1, 0)]
    idx = np.arange(3 * 10 * 7, dtype=np.uint64)
    np.testing.assert_array_equal(m[(1, 0)].reshape(-1), dropout_np.dropout_scale(99, 5, idx, 0.4))
    assert m[(0, 1)][2, 9, 6] == dropout_np.dropout_scale(99, 2, np.array([(2 * 10 + 9) * 7 + 6], np.uint64), 0.4)[0]
    assert all(np.all(v == 1) for v in dropout_np.step_masks(99, (1,), 2, 3, 4, 0.0).values())


def _param_count(conf, emb_in, hidden, K, T):
    arr = (C.c_int * len(conf))(*conf)
    n_run = C.c_longlong(0)
    n = _lib.lib().vmb_mla_train_param_count(len(conf), arr, emb_in, hidden, K, T, C.byref(n_run))
    return n, n_run.value


@pytest.mark.parametrize("conf,emb_in,hidden,K,T", [
    ((4, 4, 4, 4), 128, 128, 10, 10),      # 16 Linears + 4 fcv + fc: 21 weight jobs, the library's limit
    ((1,), 64, 64, 3, 1),
    ((2, 1), 128, 600, 1024, 16),
    ((1,), 128, 40, 130, 10),              # K > hidden
    ((2, 1), 640, 600, 527, 10),           # last narrow first layer
    ((2, 1), 641, 600, 527, 10),           # first wide first layer
    ((1,), 131, 1024, 1, 13),
])
def test_layout_matches_the_library_at_the_edges(conf, emb_in, hidden, K, T):
    _, _, n_p, n_r = training.train_layout(conf, emb_in, hidden, K, T)
    assert _param_count(conf, emb_in, hidden, K, T) == (n_p, n_r)


def _create(conf, emb_in=128, hidden=600, K=527, T=10, max_batch=64):
    arr = (C.c_int * len(conf))(*conf)
    h = C.c_void_p()
    rc = _lib.lib().vmb_mla_trainer_create(C.byref(h), len(conf), arr, emb_in, hidden, K, T, max_batch, None)
    if rc == 0:
        _lib.lib().vmb_mla_trainer_destroy(h)
    return rc, _lib.lib().vmb_last_error().decode()


@pytest.mark.parametrize("kw,msg", [
    (dict(T=17), "1 <= T <= 16"),
    (dict(T=0), "1 <= T <= 16"),
    (dict(hidden=1025), "hidden and n_classes must be in 1..1024"),
    (dict(K=1025), "hidden and n_classes must be in 1..1024"),
    (dict(emb_in=16385), "emb_in in 1..16384"),
    (dict(conf=(1, 1, 1, 1, 1)), "1..4 levels"),
    (dict(conf=(2, 5)), "1..4 fully connected layers per level"),
    (dict(max_batch=1), "bad max_batch"),
])
def test_trainer_create_rejects_shapes_outside_the_range(kw, msg):
    kw = dict(kw)
    rc, err = _create(kw.pop("conf", (2, 1)), **kw)
    assert rc != 0 and msg in err, err


@pytest.mark.parametrize("kw", [dict(T=16, K=1024), dict(T=1, hidden=64, K=3), dict(hidden=1024, K=1),
                                dict(conf=(4, 4, 4, 4), hidden=128, K=10), dict(emb_in=16384), dict(max_batch=2),
                                dict(max_batch=4096)])
def test_trainer_create_accepts_the_edges_of_the_range(kw):
    kw = dict(kw)
    rc, err = _create(kw.pop("conf", (2, 1)), **kw)
    if rc != 0:                 # without a GPU only the workspace allocation can fail, never an argument check
        assert not torch.cuda.is_available()
        assert "workspace allocation failed" in err, err
