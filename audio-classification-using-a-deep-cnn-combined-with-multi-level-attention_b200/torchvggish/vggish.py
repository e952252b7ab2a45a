"""Drop-in for torchvggish/vggish.py: `VGG`, `Postprocessor`, `make_layers`, `VGGish` with the reference's
constructor signatures and state_dict keys (vggish.py:9-184), computing on the B200 library.

The nn.Conv2d / nn.Linear children exist only to own the parameters under the reference's key names
(`features.{0,3,6,8,11,13}.*`, `embeddings.{0,2,4}.*`, `pproc.pca_*`): forward never runs them.  On the first
call (and whenever the parameters change) the weights are handed to the library, which keeps bf16 copies in its
implicit-GEMM layout; the forward pass is conv1 -> 5 tcgen05 implicit-GEMM convs with fused ReLU / max-pool ->
3 tcgen05 FC layers (csrc/vggish.cu).  There is no CPU path: a module that is not on a CUDA device raises.
"""
import numpy as np
import torch
import torch.nn as nn

from b200 import engine as _engine
from b200._lib import B200Error

from . import vggish_input, vggish_params

_CONV_PLAN = (64, "M", 128, "M", 256, 256, "M", 512, 512, "M")   # vggish.py:111


def make_layers():
    """Parameter holders for the conv stack, laid out so the state_dict keys match vggish.py:108-118."""
    mods, c_in = [], 1
    for item in _CONV_PLAN:
        if item == "M":
            mods.append(nn.MaxPool2d(kernel_size=2, stride=2))
        else:
            mods.extend((nn.Conv2d(c_in, item, kernel_size=3, padding=1), nn.ReLU(inplace=True)))
            c_in = item
    return nn.Sequential(*mods)


class B200HandleMixin:
    """Caches the library-side copy of a module's weights (a ctypes handle) next to the nn.Module that owns them.

    The copy is rebuilt when a parameter or buffer was replaced, moved, or modified in place through torch (tensor
    version counters); edits that bypass the counters (`p.data.copy_()`, `p.data.mul_()`, EMA / clipping code) need an
    explicit `invalidate()`.  The handle never travels with the module: pickling, `torch.save(model)` and
    `copy.deepcopy` (the reference checkpoints whole objects, train.py:259-268) drop it and the copy rebuilds it on its
    first forward."""
    _B200_TRANSIENT = ("_handle", "_handle_key", "_train_state", "_sub_handle", "_sub_handle_key")

    def invalidate(self):
        """Forget the cached library copy of the weights (call after editing parameters through `.data`)."""
        for name in self._B200_TRANSIENT:
            h = self.__dict__.get(name)
            if hasattr(h, "close"):
                h.close()
            if name in self.__dict__:
                self.__dict__[name] = None

    def __getstate__(self):
        state = self.__dict__.copy()
        for name in self._B200_TRANSIENT:
            if name in state:
                state[name] = None
        return state

    @staticmethod
    def _tensor_key(tensors, dev):
        return tuple((t.data_ptr(), t._version) for t in tensors) + (str(dev),)


def handle_action(old_key, new_key, fc_trainable: bool) -> str:
    """What a change of the VGGish parameters does to the library handle.  A key is (conv part, FC part): the conv
    part covers the conv tensors and the precision, the FC part the embeddings.* tensors.  "rebuild" (a new handle:
    vmb_vggish_create_ex re-lays every weight and synchronises), "refresh" (only the FC weights changed and the handle
    already holds a training copy of them: vmb_vggish_refresh_fc, stream-ordered), or "keep"."""
    if old_key is None or old_key[0] != new_key[0]:
        return "rebuild"
    if old_key[1] != new_key[1]:
        return "refresh" if fc_trainable else "rebuild"
    return "keep"


class _FcTrainFn(torch.autograd.Function):
    """Train-mode VGGish with the conv stack frozen and fc1-fc3 trainable: the conv features and the FC stack's
    activations stay in the handle's train workspace, which holds ONE forward: backward checks it is still this one."""

    @staticmethod
    def forward(ctx, module, x, *params):
        h = module._b200_handle(train=True)
        emb = h.forward_train(x.detach().to(device=h.device, dtype=torch.float32))
        module._fc_generation = getattr(module, "_fc_generation", 0) + 1
        ctx.module, ctx.handle, ctx.generation = module, h, module._fc_generation
        ctx.param_key = tuple((p.data_ptr(), p._version) for p in params)
        return emb

    @staticmethod
    def backward(ctx, d_emb):
        m = ctx.module
        if ctx.generation != getattr(m, "_fc_generation", 0) or m._handle is not ctx.handle:
            raise B200Error("backward of a stale VGGish forward: the library keeps the activations of ONE train-mode "
                            "forward per module, and another train-mode forward ran before this backward; call "
                            "backward() before the next forward")
        if ctx.param_key != tuple((p.data_ptr(), p._version) for p in m.embeddings.parameters()):
            raise B200Error("the VGGish FC parameters changed between forward and backward")
        views = _engine.fc_grad_views(ctx.handle.fc_backward(d_emb))
        names = [k for k, _ in m.embeddings.named_parameters()]
        grads = [views[k] if ctx.needs_input_grad[2 + i] else None for i, k in enumerate(names)]
        return (None, None, *grads)


def _body_tensors(features, embeddings):
    named = [(f"features.{k}", v) for k, v in features.named_parameters()]
    if embeddings is not None:
        named += [(f"embeddings.{k}", v) for k, v in embeddings.named_parameters()]
    return named


class VGG(B200HandleMixin, nn.Module):
    """VGGish body: (N, 1, 96, 64) log-mel examples -> (N, 128) post-ReLU embeddings (vggish.py:9-31).

    `b200_precision` selects the arithmetic of the library copy: "fp16" (default; fp16 operands, fp32 accumulation),
    "bf16" (same kernels and speed, 8 mantissa bits) or "split" (hi + lo bf16 pairs, 3x the tensor work — the mode in
    which `postprocess=True` reproduces the reference's 8-bit output up to +-1 LSB at quantisation boundaries).  The
    reference's constructor has no such argument; set the attribute (or pass it to `set_precision`) before forward."""
    b200_precision = _engine.DEFAULT_PRECISION

    def __init__(self, features):
        super().__init__()
        self.features = features
        fc_dims = ((512 * 4 * 6, 4096), (4096, 4096), (4096, vggish_params.EMBEDDING_SIZE))
        mods = []
        for fin, fout in fc_dims:
            mods.extend((nn.Linear(fin, fout), nn.ReLU(True)))
        self.embeddings = nn.Sequential(*mods)
        self._handle = None
        self._handle_key = None

    def set_precision(self, precision):
        if precision not in _engine.PRECISIONS:
            raise ValueError("precision must be 'fp16', 'bf16' or 'split'")
        self.b200_precision = precision
        return self

    # -- library handle: rebuilt when a conv parameter was modified in place, replaced or moved; a change of the FC
    # parameters alone (an optimiser step of FC fine-tuning) refreshes the FC weights of the existing handle
    def _b200_handle(self, train: bool = False):
        named = _body_tensors(self.features, self.embeddings)
        dev = named[0][1].device
        if dev.type != "cuda":
            raise B200Error("VGGish parameters are on %s: move the module to a CUDA device (.to('cuda')); this build "
                            "has no CPU path" % dev)
        fc = [v for _, v in self.embeddings.named_parameters()]
        key = (self._tensor_key(self.features.parameters(), dev) + (self.b200_precision,), self._tensor_key(fc, dev))
        action = handle_action(self._handle_key if self._handle is not None else None, key,
                               self._handle is not None and self._handle.fc_trainable)
        if action == "rebuild":
            if self._handle is not None:
                self._handle.close()
            self._handle = _engine.VggishHandle(dict(named), dev, precision=self.b200_precision)
        if action == "refresh" or (train and not self._handle.fc_trainable):
            self._handle.refresh_fc(fc[0::2], fc[1::2])
        self._handle_key = key
        return self._handle

    def forward(self, x):
        if torch.is_grad_enabled() and self.training:
            if any(p.requires_grad for p in self.features.parameters()):
                raise NotImplementedError("training the VGGish conv stack is outside the B200 path (the reference "
                                          "freezes it, model.py:159-160); fine-tuning the FC stack alone "
                                          "(set_requires_grad(vgg.embeddings, True)) is supported; otherwise call "
                                          "set_requires_grad(module, False) or .eval()")
            fc = list(self.embeddings.parameters())
            if any(p.requires_grad for p in fc):
                if not isinstance(x, torch.Tensor):
                    raise TypeError("expected a (N, 1, 96, 64) tensor")
                return _FcTrainFn.apply(self, x, *fc)
        h = self._b200_handle()
        if not isinstance(x, torch.Tensor):
            raise TypeError("expected a (N, 1, 96, 64) tensor")
        x = x.detach().to(device=h.device, dtype=torch.float32)
        return h.forward(x)

    def bottlenecks(self, x):
        """(N, 12288) 16-bit conv features in (h, w, c) order (the flatten of vggish.py:26-29)."""
        h = self._b200_handle()
        return h.forward(x.detach().to(device=h.device, dtype=torch.float32), want_bottleneck=True,
                         want_embeddings=False)[1]


class VGGishFeatures(B200HandleMixin, nn.Sequential):
    """The reference's just_bottlenecks re-wrap of VGGish: nn.Sequential(features, CnnFlatten) (model.py:161-166), so
    that its state_dict keys are `0.{0,3,6,8,11,13}.{weight,bias}` and the FC stack is gone.  forward runs the library's
    conv stack and returns the (N, 12288) features in (h, w, c) order as float32."""
    b200_precision = _engine.DEFAULT_PRECISION

    def __init__(self, features, flatten):
        super().__init__(features, flatten)
        self._handle = None
        self._handle_key = None

    def _b200_handle(self):
        named = _body_tensors(self[0], None)
        dev = named[0][1].device
        if dev.type != "cuda":
            raise B200Error("VGGish parameters are on %s: move the module to a CUDA device; this build has no CPU "
                            "path" % dev)
        key = self._tensor_key((v for _, v in named), dev) + (self.b200_precision,)
        if self._handle is None or key != self._handle_key:
            if self._handle is not None:
                self._handle.close()
            self._handle = _engine.VggishHandle(dict(named), dev, precision=self.b200_precision)
            self._handle_key = key
        return self._handle

    def forward(self, x):
        h = self._b200_handle()
        x = x.detach().to(device=h.device, dtype=torch.float32)
        return h.forward(x, want_bottleneck=True, want_embeddings=False)[1].float()


class Postprocessor(nn.Module):
    """PCA (+ whitening) and 8-bit quantisation of the embeddings (vggish.py:34-105): returns FLOAT32 values in
    0..255, squeezed, like the reference."""

    def __init__(self):
        super().__init__()
        n = vggish_params.EMBEDDING_SIZE
        self.pca_eigen_vectors = nn.Parameter(torch.empty((n, n), dtype=torch.float), requires_grad=False)
        self.pca_means = nn.Parameter(torch.empty((n, 1), dtype=torch.float), requires_grad=False)

    def postprocess(self, embeddings_batch):
        assert len(embeddings_batch.shape) == 2, "Expected 2-d batch, got %r" % (embeddings_batch.shape,)
        assert embeddings_batch.shape[1] == vggish_params.EMBEDDING_SIZE, "Bad batch shape: %r" % (
            embeddings_batch.shape,)
        dev = self.pca_eigen_vectors.device
        if dev.type != "cuda":
            raise B200Error("Postprocessor parameters are on %s: this build has no CPU path" % dev)
        q = _engine.postprocess(embeddings_batch.detach().to(device=dev, dtype=torch.float32),
                                self.pca_eigen_vectors.data, self.pca_means.data)
        return torch.squeeze(q)

    def quantized_uint8(self, embeddings_batch):
        """Same values as postprocess() but as a uint8 tensor (N, 128) — the AudioSet release format."""
        dev = self.pca_eigen_vectors.device
        return _engine.postprocess(embeddings_batch.detach().to(device=dev, dtype=torch.float32),
                                   self.pca_eigen_vectors.data, self.pca_means.data, want_u8=True)[1]

    def forward(self, x):
        return self.postprocess(x)


def _vgg():
    return VGG(make_layers())


class VGGish(VGG):
    """VGGish with optional waveform pre-processing and PCA post-processing (vggish.py:143-184).

    `pretrained=True` needs network access to the URLs in `urls` exactly like the reference
    (torch.hub.load_state_dict_from_url); offline, build with pretrained=False and load_state_dict()."""

    def __init__(self, urls, pretrained=True, preprocess=True, postprocess=True, progress=True):
        super().__init__(make_layers())
        if pretrained:
            from torch import hub
            super().load_state_dict(hub.load_state_dict_from_url(urls["vggish"], progress=progress))
        self.preprocess = preprocess
        self.postprocess = postprocess
        if self.postprocess:
            self.pproc = Postprocessor()
            if pretrained:
                from torch import hub
                sd = hub.load_state_dict_from_url(urls["pca"], progress=progress)
                self.pproc.load_state_dict({
                    vggish_params.PCA_EIGEN_VECTORS_NAME: torch.as_tensor(
                        sd[vggish_params.PCA_EIGEN_VECTORS_NAME], dtype=torch.float),
                    vggish_params.PCA_MEANS_NAME: torch.as_tensor(
                        sd[vggish_params.PCA_MEANS_NAME].reshape(-1, 1), dtype=torch.float)})

    def forward(self, x, fs=None):
        if self.preprocess:
            x = self._preprocess(x, fs)
        x = VGG.forward(self, x)
        if self.postprocess:
            x = self._postprocess(x)
        return x

    def _preprocess(self, x, fs):
        if isinstance(x, np.ndarray):
            return vggish_input.waveform_to_examples(x, fs)
        if isinstance(x, str):
            return vggish_input.wavfile_to_examples(x)
        raise AttributeError

    def _postprocess(self, x):
        return self.pproc(x)
