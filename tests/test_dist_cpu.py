"""world_size-2 gloo tests (CPU): the host-side logic of the multi-GPU paths.
   * inference: contiguous batch shards, results gathered in rank order == unsharded result (no collective on the
     data path; the gather here is only the test's way of comparing)
   * head training: flat gradient bucket layout + ONE all-reduce(SUM) / world == average of per-shard gradients; the
     sharded optimiser step (reduce-scatter + Adam + all-gather over the library's slice partition) == all-reduce + Adam
The arithmetic on each rank is the CPU oracle (this container has no GPU); what is under test is the sharding,
packing and collective plumbing that the GPU ranks use unchanged."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import PKG, ROOT

THREADS = 2             # torch splits fp32 reductions by thread count: the ranks and the check below use the same one


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    import sys
    for p in (PKG, ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.set_num_threads(THREADS)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from b200 import sharding, synth, training
    from oracle import model_torch, train_torch
    assert sharding.dist_env() == (rank, rank, world)
    conf, K = (2, 1), 10
    sd = synth.mla_state_dict(conf, 128, 600, K, 10, seed=2)
    g = torch.Generator().manual_seed(0)
    emb = torch.randn(7, 10, 128, generator=g).abs()
    # ---- inference shard
    lo, hi = sharding.shard_bounds(emb.shape[0], rank, world)
    with torch.no_grad():
        part = model_torch.mla_forward(sd, emb[lo:hi], conf)
    parts = [None] * world
    dist.all_gather_object(parts, part)
    # ---- training shard: flat bucket, one all-reduce
    x = torch.randn(12, 10, 128, generator=g)
    labels = torch.randint(0, K, (12,), generator=g)
    lo, hi = sharding.shard_bounds(12, rank, world)
    _, _, grads = train_torch.head_step(sd, x[lo:hi], labels[lo:hi], conf)
    p_layout, _, n_p, _ = training.train_layout(conf, 128, 600, K, 10)
    bucket = torch.zeros(n_p)
    for key, shape, off in p_layout:
        bucket[off:off + grads[key].numel()] = grads[key].reshape(-1)
    assert all(".fcf." not in key for key, _, _ in p_layout)
    local = bucket.clone()
    dist.all_reduce(bucket, op=dist.ReduceOp.SUM)
    bucket /= world
    # ---- the sharded optimiser step (csrc/dp_adam.cu) in the library's own partition (vmb_dp_slice): every rank sums ITS
    # slice of all ranks' gradients in rank order, applies Adam to the slice, and the slices are gathered into every
    # replica — the same parameters as all-reduce + Adam on every rank
    import ctypes as C
    from b200 import _lib
    b, e = C.c_longlong(0), C.c_longlong(0)
    _lib.lib().vmb_dp_slice(n_p, world, rank, C.byref(b), C.byref(e))
    npad = (n_p + 3) // 4 * 4
    everyone = [torch.zeros(npad) for _ in range(world)]
    padded = torch.zeros(npad)
    padded[:n_p] = local
    dist.all_gather(everyone, padded)                       # stands in for the peer loads
    params0 = torch.cat([sd[key].reshape(-1) for key, _, _ in p_layout] + [torch.zeros(npad - n_p)])
    mine = torch.zeros(e.value - b.value)
    for r in range(world):
        mine += everyone[r][b.value:e.value]
    new_slice = train_torch.adam_update(params0[b.value:e.value], mine / world)
    slices = [None] * world
    dist.all_gather_object(slices, (b.value, e.value, new_slice))      # stands in for the peer stores
    sharded = torch.zeros(npad)
    for lo_, hi_, sl in slices:
        sharded[lo_:hi_] = sl
    replicated = train_torch.adam_update(params0[:n_p], bucket)
    if rank == 0:
        torch.save({"scores": torch.cat(parts), "bucket": bucket, "sharded": sharded[:n_p], "replicated": replicated,
                    "slices": [(lo_, hi_) for lo_, hi_, _ in slices], "npad": npad},
                   os.path.join(out_dir, "rank0.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.fixture
def rank_thread_count():
    threads = torch.get_num_threads()
    torch.set_num_threads(THREADS)
    yield
    torch.set_num_threads(threads)


def test_two_rank_gloo(tmp_path, rank_thread_count):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    got = torch.load(os.path.join(tmp_path, "rank0.pt"))
    from b200 import sharding, synth, training
    from oracle import model_torch, train_torch
    conf, K = (2, 1), 10
    sd = synth.mla_state_dict(conf, 128, 600, K, 10, seed=2)
    g = torch.Generator().manual_seed(0)
    emb = torch.randn(7, 10, 128, generator=g).abs()
    with torch.no_grad():
        whole = model_torch.mla_forward(sd, emb, conf)
    assert torch.allclose(got["scores"], whole, atol=1e-6)          # eval mode: rows are independent
    x = torch.randn(12, 10, 128, generator=g)
    labels = torch.randint(0, K, (12,), generator=g)
    p_layout, _, n_p, _ = training.train_layout(conf, 128, 600, K, 10)
    want = torch.zeros(n_p)
    for r in range(world):
        lo, hi = sharding.shard_bounds(12, r, world)
        _, _, grads = train_torch.head_step(sd, x[lo:hi], labels[lo:hi], conf)
        for key, shape, off in p_layout:
            want[off:off + grads[key].numel()] += grads[key].reshape(-1) / world
    assert torch.allclose(got["bucket"], want, rtol=1e-4, atol=1e-6)      # the all-reduce sums in another order
    # sharded optimiser step == all-reduce + Adam on every rank; the slices tile the padded bucket in rank order
    assert got["slices"][0][0] == 0 and got["slices"][-1][1] == got["npad"]
    assert all(a[1] == b[0] for a, b in zip(got["slices"], got["slices"][1:]))
    assert torch.allclose(got["sharded"], got["replicated"], rtol=0, atol=1e-7)
    # local BatchNorm statistics: the data-parallel average is NOT the single-process full-batch gradient (H6)
    _, _, full = train_torch.head_step(sd, x, labels, conf)
    key, shape, off = p_layout[2]
    assert not torch.allclose(want[off:off + full[key].numel()], full[key].reshape(-1), rtol=1e-3, atol=1e-6)
