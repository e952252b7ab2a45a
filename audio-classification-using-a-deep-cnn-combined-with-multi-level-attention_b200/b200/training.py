"""Head training on the B200 (SURVEY §8 a21, config 5): the multi-level attention head's train-mode forward,
backward and Adam update run in the library (csrc/mla_train.cu); across GPUs the only communication is ONE NCCL
all-reduce of the flat gradient bucket per step (data parallel, BatchNorm statistics stay local to each rank, which
is what stock DistributedDataParallel computes — SURVEY §7 H6).

Two entry levels:
  * `HeadTrainer` — flat fp32 parameter / gradient / Adam-moment buffers, `step(x, labels)` = one library call for
    forward+backward, one `dist.all_reduce`, one Adam kernel.  Used by bench_train.py and the tests.
  * `head_train_forward(module, x)` — autograd bridge for the reference-named `model.MultiLevelAttention` in
    train mode, so the reference's own loop (`criterion(outputs, labels); loss.backward(); optimizer.step()`,
    train.py:130-138) keeps working on top of the library kernels.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import B200Error, check, ptr, stream_ptr


def train_layout(model_conf: Sequence[int], emb_in: int, hidden: int, n_classes: int, t_steps: int):
    """(params, running): lists of (state_dict key, shape, offset) in the library's flat order — the reference
    module's named_parameters() order with `fcf` left out (it never receives a gradient, SURVEY F3)."""
    params: List[Tuple[str, Tuple[int, ...], int]] = []
    running: List[Tuple[str, Tuple[int, ...], int]] = []
    po = ro = 0

    def add_p(key, shape):
        nonlocal po
        n = 1
        for s in shape:
            n *= s
        params.append((key, tuple(shape), po))
        po += n

    def add_bn(prefix, n):
        nonlocal ro
        add_p(prefix + ".weight", (n,))
        add_p(prefix + ".bias", (n,))
        running.append((prefix + ".running_mean", (n,), ro))
        running.append((prefix + ".running_var", (n,), ro + n))
        ro += 2 * n

    for lvl, n_fc in enumerate(model_conf):
        p = f"embedded_mappings.{lvl}"
        add_bn(p + ".norm0", t_steps)
        for j in range(n_fc):
            fin = emb_in if (lvl == 0 and j == 0) else hidden
            add_p(f"{p}.fc.{j}.weight", (hidden, fin))
            add_p(f"{p}.fc.{j}.bias", (hidden,))
        for j in range(n_fc):
            add_bn(f"{p}.norms.{j}", t_steps)
    for lvl in range(len(model_conf)):
        p = f"attention_modules.{lvl}"
        add_p(p + ".fcv.weight", (n_classes, hidden))
        add_p(p + ".fcv.bias", (n_classes,))
        add_bn(p + ".normv", t_steps)
        add_bn(p + ".normf", t_steps)
    add_p("fc.weight", (n_classes, len(model_conf) * n_classes))
    add_p("fc.bias", (n_classes,))
    add_bn("norm", n_classes)
    return params, running, po, ro


class _DeviceArray:
    """A float32 device array the library owns, presented to torch through __cuda_array_interface__."""

    def __init__(self, address: int, n: int):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<f4", "data": (int(address), False),
                                         "version": 2}


class HeadTrainer:
    """Owns the library trainer handle and the flat buffers of one data-parallel rank."""

    def __init__(self, model_conf: Sequence[int], emb_in: int, hidden: int, n_classes: int, t_steps: int,
                 max_batch: int, device: torch.device, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 dropout_p: float = 0.4, seed: int = 0, process_group=None):
        from . import engine
        engine.require_b200(device)
        self.device, self.model_conf = device, tuple(int(v) for v in model_conf)
        self.dims = (emb_in, hidden, n_classes, t_steps)
        self.lr, self.betas, self.eps, self.dropout_p, self.seed = lr, betas, eps, dropout_p, seed
        self.group = process_group
        self.p_layout, self.r_layout, n_p, n_r = train_layout(self.model_conf, emb_in, hidden, n_classes, t_steps)
        conf = (C.c_int * len(self.model_conf))(*self.model_conf)
        n_run = C.c_longlong(0)
        expect = _lib.lib().vmb_mla_train_param_count(len(self.model_conf), conf, emb_in, hidden, n_classes, t_steps,
                                                      C.byref(n_run))
        if expect != n_p or n_run.value != n_r:
            raise B200Error(f"flat layout mismatch: python {n_p}/{n_r} vs library {expect}/{n_run.value}")
        self.n_params = n_p
        with torch.cuda.device(device):
            self.params = torch.zeros(n_p, device=device)
            self.grads = torch.zeros(n_p, device=device)
            self.exp_avg = torch.zeros(n_p, device=device)
            self.exp_avg_sq = torch.zeros(n_p, device=device)
            self.running = torch.zeros(n_r, device=device)
            self.loss = torch.zeros(1, device=device)
            self._h = C.c_void_p()
            check(_lib.lib().vmb_mla_trainer_create(C.byref(self._h), len(self.model_conf), conf, emb_in, hidden,
                                                    n_classes, t_steps, int(max_batch), stream_ptr()),
                  "vmb_mla_trainer_create")
        self.max_batch = int(max_batch)
        self._dp = None              # vmb_dp handle once enable_peer_step() has run
        self.peer_step_error = None
        self._parity = 0
        self._comm_stream = None     # created by the first overlapped all-reduce
        self._tail = 0
        self.step_count = 0
        self.num_batches_tracked = 0
        self.generation = 0      # bumped by every train-mode forward through the autograd bridge (one step in flight)
        self.fcf: Dict[str, torch.Tensor] = {}      # carried through state_dict round trips untouched

    def close(self, _collective: bool = True) -> None:
        if _lib is None:                                                         # interpreter exit
            return
        if getattr(self, "_dp", None):
            # the arena is mapped by the other ranks: everybody unmaps, then everybody frees
            import torch.distributed as dist
            dp, self._dp = self._dp, None
            self.params = self.params.clone()
            self.grads = self.grads.clone()
            self._grads2 = None
            _lib.lib().vmb_dp_disconnect(dp)
            if _collective and dist.is_available() and dist.is_initialized():
                try:
                    dist.barrier(group=self.group)
                except Exception:                                                # a peer is already gone
                    pass
            _lib.lib().vmb_dp_destroy(dp)
        if getattr(self, "_h", None) and self._h.value:
            _lib.lib().vmb_mla_trainer_destroy(self._h)
            self._h = C.c_void_p()

    # -- data parallel over the GPUs of one box without NCCL on the step
    def enable_peer_step(self) -> bool:
        """Move params / grads into a library-owned arena that every rank of the process group maps through CUDA IPC,
        so that step() can use vmb_dp_adam_step: ONE kernel per rank that reduce-scatters the gradients over NVLink peer
        loads, applies Adam to the rank's slice and all-gathers the new parameters with peer stores (csrc/dp_adam.cu),
        instead of an NCCL all-reduce followed by the Adam kernel on every rank.  The Adam moments become sharded: each
        rank keeps its slice.  Collective over the group; returns False (and changes nothing) for a single rank, or when
        any rank cannot create / map the arenas (no peer access between the GPUs, IPC not permitted): then every rank
        stays on the NCCL path together and `peer_step_error` says why."""
        import torch.distributed as dist
        if self._dp is not None:
            return True
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.group) == 1:
            return False
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        L = _lib.lib()
        handle = (C.c_char * 64)()
        dp = C.c_void_p()
        error = None
        with torch.cuda.device(self.device):
            # every rank takes part in every collective below whatever happens locally: a rank that fails reports it and
            # ALL ranks fall back together (a half-connected group would hang in the first cross-GPU barrier)
            try:
                check(L.vmb_dp_create(C.byref(dp), self.n_params, rank, world, C.cast(handle, C.c_void_p)), "vmb_dp_create")
            except B200Error as e:
                error, dp = str(e), C.c_void_p()
            every = [None] * world
            dist.all_gather_object(every, bytes(handle.raw) if dp.value else None, group=self.group)
            if error is None and all(h is not None for h in every):
                try:
                    check(L.vmb_dp_connect(dp, C.cast(C.c_char_p(b"".join(every)), C.c_void_p)), "vmb_dp_connect")
                except B200Error as e:
                    error = str(e)
            elif error is None:
                error = "another rank could not create its arena"
            ok = torch.tensor([0 if error else 1], device=self.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if int(ok.item()) == 0:
                if dp.value:
                    L.vmb_dp_disconnect(dp)
                dist.barrier(group=self.group)
                if dp.value:
                    L.vmb_dp_destroy(dp)
                self.peer_step_error = error or "another rank could not map the arenas"
                return False
            npad = (self.n_params + 3) // 4 * 4
            params = torch.as_tensor(_DeviceArray(L.vmb_dp_params(dp), self.n_params), device=self.device)
            params.copy_(self.params)
            self._grads2 = [torch.as_tensor(_DeviceArray(L.vmb_dp_grads(dp, i), self.n_params), device=self.device)
                            for i in (0, 1)]
            for name in ("exp_avg", "exp_avg_sq"):
                full = torch.zeros(npad, device=self.device)
                full[:self.n_params].copy_(getattr(self, name))
                setattr(self, name, full)
            self.params, self.grads, self._parity, self._dp = params, self._grads2[0], 0, dp
            b, e = C.c_longlong(0), C.c_longlong(0)
            L.vmb_dp_slice(self.n_params, world, rank, C.byref(b), C.byref(e))
            self.slice = (b.value, e.value)
            torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        return True

    def peer_step_status(self) -> None:
        """Raises if a cross-GPU barrier of vmb_dp_adam_step gave up waiting for a rank (synchronises the device)."""
        if self._dp is not None:
            with torch.cuda.device(self.device):
                check(_lib.lib().vmb_dp_status(self._dp), "vmb_dp_status")

    def __del__(self):
        self.close(_collective=False)      # no collective from the garbage collector

    # -- reference-format state_dict in / out
    def load_state_dict(self, sd: dict) -> None:
        for key, shape, off in self.p_layout:
            self.view(self.params, key).copy_(sd[key].detach().to(self.device, torch.float32))
        for key, shape, off in self.r_layout:
            self.running[off:off + shape[0]].copy_(sd[key].detach().to(self.device, torch.float32))
        self.fcf = {k: v.detach().clone() for k, v in sd.items() if ".fcf." in k}

    def view(self, flat: torch.Tensor, key: str) -> torch.Tensor:
        for k, shape, off in self.p_layout:
            if k == key:
                n = 1
                for s in shape:
                    n *= s
                return flat[off:off + n].view(shape)
        raise KeyError(key)

    def state_dict(self) -> dict:
        out = {}
        for key, shape, off in self.p_layout:
            out[key] = self.view(self.params, key).clone()
        for key, shape, off in self.r_layout:
            out[key] = self.running[off:off + shape[0]].clone()
            if key.endswith("running_var"):
                out[key[:-len("running_var")] + "num_batches_tracked"] = torch.tensor(self.num_batches_tracked)
        out.update(self.fcf)
        return out

    # -- one optimisation step
    def forward_backward(self, x: torch.Tensor, labels: torch.Tensor, want_scores: bool = False):
        """grads <- d(mean CE-on-sigmoid loss)/d(params) of THIS rank's batch; returns (loss tensor, scores|None)."""
        if x.dim() != 3 or x.shape[1] != self.dims[3] or x.shape[2] != self.dims[0]:
            raise ValueError(f"expected (B, {self.dims[3]}, {self.dims[0]}), got {tuple(x.shape)}")
        x = x.to(self.device, torch.float32).contiguous()
        labels = labels.to(self.device, torch.int64).contiguous()
        b = x.shape[0]
        scores = torch.empty(b, self.dims[2], device=self.device) if want_scores else None
        with torch.cuda.device(self.device):
            check(_lib.lib().vmb_mla_train_step(self._h, ptr(self.params), ptr(self.running), ptr(x), ptr(labels), b,
                                                float(self.dropout_p), int(self.seed + self.step_count) & (2 ** 63 - 1),
                                                ptr(self.grads), ptr(self.loss), ptr(scores), stream_ptr()),
                  "vmb_mla_train_step")
        self.num_batches_tracked += 1
        return self.loss, scores

    def all_reduce_grads(self) -> int:
        """One SUM all-reduce of the flat gradient bucket; returns the world size (the Adam kernel divides)."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return 1
        world = dist.get_world_size(self.group)
        if world > 1:
            dist.all_reduce(self.grads, op=dist.ReduceOp.SUM, group=self.group)
        return world

    def adam(self, world: int = 1) -> None:
        self.step_count += 1
        with torch.cuda.device(self.device):
            check(_lib.lib().vmb_adam_step(ptr(self.params), ptr(self.grads), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                                           self.n_params, float(self.lr), float(self.betas[0]), float(self.betas[1]),
                                           float(self.eps), 0.0, self.step_count, 1.0 / world, stream_ptr()),
                  "vmb_adam_step")

    def all_reduce_grads_overlapped(self) -> int:
        """The same SUM all-reduce in two pieces, the first one overlapped with the rest of the backward pass: the
        library computes level 0's embedding chain last, and its parameters come first in the flat order, so
        grads[tail:] are final while that chain still runs (vmb_mla_train_wait_tail).  The tail (78 % of the bucket for
        model_conf [2, 1]) is reduced from a communication stream that waits for that point only; the head follows
        when the step is complete.  Call right after forward_backward(); returns the world size."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return 1
        world = dist.get_world_size(self.group)
        if world == 1:
            return 1
        if self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream(device=self.device)
            self._tail = int(_lib.lib().vmb_mla_train_tail_offset(self._h))
        main = torch.cuda.current_stream(self.device)
        check(_lib.lib().vmb_mla_train_wait_tail(self._h, C.c_void_p(self._comm_stream.cuda_stream)),
              "vmb_mla_train_wait_tail")
        with torch.cuda.stream(self._comm_stream):
            work = dist.all_reduce(self.grads[self._tail:], op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        dist.all_reduce(self.grads[:self._tail], op=dist.ReduceOp.SUM, group=self.group)
        work.wait()                                   # the current stream waits for the tail's reduction
        main.wait_stream(self._comm_stream)
        return world

    def step(self, x: torch.Tensor, labels: torch.Tensor, overlap: bool = True) -> torch.Tensor:
        """forward + backward, gradient averaging over the ranks, Adam.  After enable_peer_step(): the fused
        reduce-scatter + Adam + all-gather kernel over NVLink peer memory.  Otherwise an NCCL all-reduce (overlapped
        with the end of the backward pass unless overlap=False — the same sums either way) and the Adam kernel."""
        if self._dp is not None:
            # gradients alternate between the arena's two buffers (a slower rank may still be reading the previous one)
            self.grads = self._grads2[self._parity]
            loss, _ = self.forward_backward(x, labels)
            self.step_count += 1
            with torch.cuda.device(self.device):
                check(_lib.lib().vmb_dp_adam_step(self._dp, self._parity, ptr(self.exp_avg), ptr(self.exp_avg_sq),
                                                  float(self.lr), float(self.betas[0]), float(self.betas[1]),
                                                  float(self.eps), 0.0, self.step_count, stream_ptr()),
                      "vmb_dp_adam_step")
            self._parity ^= 1
            return loss
        loss, _ = self.forward_backward(x, labels)
        self.adam(self.all_reduce_grads_overlapped() if overlap else self.all_reduce_grads())
        return loss


# ---------------------------------------------------------------------------------------------- nn.Module bridge
class _HeadTrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, x, *params):
        st = module._b200_train_state()
        tr: HeadTrainer = st["trainer"]
        ctx.x_dtype = x.dtype
        x = x.detach().to(tr.device, torch.float32).contiguous()
        if x.shape[0] > tr.max_batch:
            raise B200Error(f"batch {x.shape[0]} > trainer capacity {tr.max_batch}")
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())        # follows torch's global RNG like nn.Dropout does
        scores = torch.empty(x.shape[0], tr.dims[2], device=tr.device)
        with torch.cuda.device(tr.device):
            check(_lib.lib().vmb_mla_train_forward(tr._h, ptr(tr.params), ptr(tr.running), ptr(x), x.shape[0],
                                                   float(tr.dropout_p), seed, ptr(scores), stream_ptr()),
                  "vmb_mla_train_forward")
        # the activations, BatchNorm statistics and dropout masks the backward pass needs live in the trainer handle,
        # which holds ONE step: remember which forward this graph belongs to
        tr.generation += 1
        ctx.module, ctx.seed, ctx.x, ctx.generation = module, seed, x, tr.generation
        ctx.param_key = tuple((p.data_ptr(), p._version) for p in params)
        return scores

    @staticmethod
    def backward(ctx, dscores):
        st = ctx.module._b200_train_state()
        tr: HeadTrainer = st["trainer"]
        if ctx.generation != tr.generation:
            raise B200Error("backward of a stale head forward: the library trainer keeps the activations of ONE train-mode "
                            "forward per module, and another train-mode forward ran before this backward (e.g. two "
                            "micro-batches summed into one loss); call backward() before the next forward")
        if ctx.param_key != tuple((p.data_ptr(), p._version) for _, p in ctx.module.named_parameters()):
            raise B200Error("the head's parameters changed between forward and backward")
        d = dscores.to(tr.device, torch.float32).contiguous()
        dx = None
        with torch.cuda.device(tr.device):
            if ctx.needs_input_grad[1]:
                # the embeddings come from a trainable module (VGGish fc1-fc3): norm0's backward pass to its input too
                dx = torch.empty_like(ctx.x)
                check(_lib.lib().vmb_mla_train_backward_dx(tr._h, ptr(tr.params), ptr(ctx.x), ptr(d), ctx.x.shape[0],
                                                           float(tr.dropout_p), ctx.seed, ptr(tr.grads), ptr(dx),
                                                           stream_ptr()),
                      "vmb_mla_train_backward_dx")
            else:
                check(_lib.lib().vmb_mla_train_backward(tr._h, ptr(tr.params), ptr(ctx.x), ptr(d), ctx.x.shape[0],
                                                        float(tr.dropout_p), ctx.seed, ptr(tr.grads), stream_ptr()),
                      "vmb_mla_train_backward")
        grads = []
        for name in st["param_names"]:
            grads.append(None if ".fcf." in name else tr.view(tr.grads, name).clone())
        if dx is not None and ctx.x_dtype != dx.dtype:
            dx = dx.to(ctx.x_dtype)
        return (None, dx, *grads)


def input_grad_supported(emb_in: int, hidden: int, n_classes: int) -> bool:
    """The head forms d(loss)/d(embeddings) only when the padded input width does not exceed the padded hidden width:
    the wide first layer (just_bottlenecks, emb_in 12288) runs no dX GEMM."""
    def pad(v):
        return (v + 127) // 128 * 128
    return pad(emb_in) <= max(pad(hidden), pad(n_classes))


def head_train_forward(module, x: torch.Tensor) -> torch.Tensor:
    """Train-mode forward of the reference-named head through the library (autograd-aware).  When x requires grad
    (a trainable module in front of the head, e.g. VGGish's fc1-fc3), backward also returns d(loss)/dx."""
    if (isinstance(x, torch.Tensor) and x.requires_grad and torch.is_grad_enabled()
            and not input_grad_supported(module.emb_input_size, module._h, module._k)):
        raise NotImplementedError("the gradient with respect to the embeddings is formed only when the input width "
                                  "is not wider than the hidden width; the wide first layer (just_bottlenecks, 12288-d "
                                  "conv features) has no input gradient, and the VGGish conv stack cannot be trained "
                                  "on this path (model.py:159-160); pass x.detach()")
    st = module._b200_train_state()
    st["sync_in"]()
    params = [p for _, p in module.named_parameters()]
    out = _HeadTrainFn.apply(module, x, *params)
    st["sync_out"]()
    return out
