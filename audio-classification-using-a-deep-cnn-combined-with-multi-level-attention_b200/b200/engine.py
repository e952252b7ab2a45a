"""Host side of the B200 path: thin, typed wrappers that hand torch CUDA tensors to the C-ABI library.

torch is plumbing here (device memory, streams); all arithmetic happens in libvggish_mla_b200.so.  Every wrapper
validates shapes / dtypes / devices in Python and raises; nothing falls back to torch ops or the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import B200Error, check, ptr, stream_ptr

CONV_KEYS = (0, 3, 6, 8, 11, 13)
FC_KEYS = (0, 2, 4)
WIN, HOP, FRAMES_PER_EXAMPLE, MEL = 400, 160, 96, 64


def _need_cuda(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise B200Error(f"{name} must live on a CUDA device (no CPU path exists)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def require_b200(device: Optional[torch.device] = None) -> None:
    """Fail loudly unless a sm_100 device is present and the library loads."""
    if not torch.cuda.is_available():
        raise B200Error("no CUDA device: the B200 path has no CPU fallback")
    idx = torch.cuda.current_device() if device is None or device.index is None else device.index
    arch = _lib.lib().vmb_device_arch(idx)
    if arch != 100:
        raise B200Error(f"device {idx} has compute capability {arch}; the kernels are built for sm_100a only")


def num_frames(n_samples: int) -> int:
    return int(_lib.lib().vmb_num_frames(int(n_samples)))


def num_examples(n_samples: int) -> int:
    return int(_lib.lib().vmb_num_examples(int(n_samples)))


def logmel(wave: torch.Tensor, frames_out: Optional[int] = None) -> torch.Tensor:
    """wave (n_clips, n_samples) or (n_samples,) fp32 CUDA -> (n_clips, frames_out, 64) fp32 log-mel."""
    wave = _need_cuda(wave, "wave")
    if wave.dim() == 1:
        wave = wave[None]
    if wave.dim() != 2:
        raise ValueError("wave must be (n_clips, n_samples)")
    n_clips, n_samples = wave.shape
    nf = num_frames(n_samples)
    if nf < 0:
        raise ValueError("negative dimensions are not allowed")  # what the reference's frame() raises (F10)
    if frames_out is None:
        frames_out = nf
    out = torch.empty((n_clips, frames_out, MEL), device=wave.device, dtype=torch.float32)
    with torch.cuda.device(wave.device):
        for c0 in range(0, n_clips, 32768):
            nc = min(32768, n_clips - c0)
            check(_lib.lib().vmb_logmel(ptr(wave[c0:]), nc, n_samples, wave.stride(0), frames_out, ptr(out[c0:]),
                                        stream_ptr()), "vmb_logmel")
    return out


def logmel_pcm16(pcm: torch.Tensor, frames_out: Optional[int] = None) -> torch.Tensor:
    """pcm (n_clips, n_samples) or (n_samples,) int16 CUDA -> (n_clips, frames_out, 64) fp32 log-mel of pcm / 32768
    (the int16 WAV convention of vggish_input.py:96-98), without a float copy of the waveform."""
    pcm = _need_cuda(pcm, "pcm", torch.int16)
    if pcm.dim() == 1:
        pcm = pcm[None]
    n_clips, n_samples = pcm.shape
    nf = num_frames(n_samples)
    if nf < 0:
        raise ValueError("negative dimensions are not allowed")
    if frames_out is None:
        frames_out = nf
    out = torch.empty((n_clips, frames_out, MEL), device=pcm.device, dtype=torch.float32)
    with torch.cuda.device(pcm.device):
        for c0 in range(0, n_clips, 32768):
            nc = min(32768, n_clips - c0)
            check(_lib.lib().vmb_logmel_pcm16(ptr(pcm[c0:]), nc, n_samples, pcm.stride(0), frames_out, ptr(out[c0:]),
                                              stream_ptr()), "vmb_logmel_pcm16")
    return out


def logmel_cudacore(wave: torch.Tensor) -> torch.Tensor:
    """Diagnostic: the fp32 CUDA-core log-mel kernel (vmb_logmel_cudacore), same contract as logmel()."""
    wave = _need_cuda(wave, "wave")
    if wave.dim() == 1:
        wave = wave[None]
    n_clips, n_samples = wave.shape
    nf = num_frames(n_samples)
    if nf < 0:
        raise ValueError("negative dimensions are not allowed")
    out = torch.empty((n_clips, nf, MEL), device=wave.device, dtype=torch.float32)
    with torch.cuda.device(wave.device):
        for c0 in range(0, n_clips, 32768):
            nc = min(32768, n_clips - c0)
            check(_lib.lib().vmb_logmel_cudacore(ptr(wave[c0:]), nc, n_samples, wave.stride(0), nf, ptr(out[c0:]),
                                                 stream_ptr()), "vmb_logmel_cudacore")
    return out


def stft_magnitude(signal: torch.Tensor) -> torch.Tensor:
    """signal (n_samples,) float64 CUDA -> (n_frames, 257) float64 |rfft(frame * hann, 512)| (mel_features.py:71-92 with
    the VGGish framing: window 400, hop 160), computed in float64 on the device."""
    signal = _need_cuda(signal, "signal", torch.float64)
    if signal.dim() != 1:
        raise ValueError("signal must be 1-D")
    nf = num_frames(signal.shape[0])
    if nf < 0:
        raise ValueError("negative dimensions are not allowed")
    out = torch.empty((nf, 257), device=signal.device, dtype=torch.float64)
    if nf > 0:
        with torch.cuda.device(signal.device):
            check(_lib.lib().vmb_stft_magnitude(ptr(signal), signal.shape[0], ptr(out), stream_ptr()), "vmb_stft_magnitude")
    return out


def examples_from_wave(wave: torch.Tensor) -> torch.Tensor:
    """(n_clips, n_samples) fp32 CUDA -> (n_clips * examples_per_clip, 96, 64) fp32 (vggish_input.py:66-76)."""
    if wave.dim() == 1:
        wave = wave[None]
    per = num_examples(wave.shape[-1])
    if per < 0:
        raise ValueError("negative dimensions are not allowed")
    lm = logmel(wave, per * FRAMES_PER_EXAMPLE)
    return lm.view(wave.shape[0] * per, FRAMES_PER_EXAMPLE, MEL)


def front_end_tables():
    """(hann[400], mel[257, 64]) float64 numpy arrays as built inside the library."""
    import numpy as np
    hann = np.empty(400, dtype=np.float64)
    mel = np.empty((257, 64), dtype=np.float64)
    check(_lib.lib().vmb_front_end_tables(hann.ctypes.data, mel.ctypes.data), "vmb_front_end_tables")
    return hann, mel


def postprocess(emb: torch.Tensor, eigen: torch.Tensor, means: torch.Tensor, want_u8: bool = False):
    emb = _need_cuda(emb, "embeddings")
    eigen = _need_cuda(eigen, "pca_eigen_vectors")
    means = _need_cuda(means.reshape(-1), "pca_means")
    n = emb.shape[0]
    out = torch.empty((n, 128), device=emb.device, dtype=torch.float32)
    u8 = torch.empty((n, 128), device=emb.device, dtype=torch.uint8) if want_u8 else None
    with torch.cuda.device(emb.device):
        check(_lib.lib().vmb_postprocess(ptr(emb), ptr(eigen), ptr(means), ptr(out), ptr(u8), n, stream_ptr()),
              "vmb_postprocess")
    return (out, u8) if want_u8 else out


PRECISIONS = {"bf16": 0, "split": 1, "fp16": 2}
DEFAULT_PRECISION = "fp16"
SAT_LAYERS = ("conv1", "conv2", "conv3_1", "conv3_2", "conv4_1", "conv4_2", "fc1", "fc2")


class VggishHandle:
    """Owns the library-side VGGish weights (16-bit, implicit-GEMM layout) built from a reference state_dict."""

    def __init__(self, state_dict: dict, device: torch.device, precision: str = DEFAULT_PRECISION):
        """precision: "fp16" (default: fp16 activations and weights, fp32 accumulation — the same tensor rate as bf16
        with 11 instead of 8 mantissa bits; outputs saturate at 65504 and raise, see check_saturation), "bf16" (the
        same kernels on bf16), or "split" (accuracy mode: hi + lo bf16 activations and weights, 3x the tensor work,
        embeddings within ~1e-4 of fp32 — for 8-bit quantised long-form extraction)."""
        require_b200(device)
        if precision not in PRECISIONS:
            raise ValueError("precision must be 'fp16', 'bf16' or 'split'")
        self.device = device
        self.precision = precision
        self._h = C.c_void_p()
        self._ws: Optional[torch.Tensor] = None
        with torch.cuda.device(device):
            keep = []

            def dev(key):
                t = state_dict[key].detach().to(device=device, dtype=torch.float32).contiguous()
                keep.append(t)
                return t.data_ptr()

            cw = (C.c_void_p * 6)(*[dev(f"features.{k}.weight") for k in CONV_KEYS])
            cb = (C.c_void_p * 6)(*[dev(f"features.{k}.bias") for k in CONV_KEYS])
            # a state_dict without the FC stack (the reference's just_bottlenecks re-wrap, model.py:161-166) gives a
            # handle that serves the conv features only
            self.has_fc = all(f"embeddings.{k}.weight" in state_dict for k in FC_KEYS)
            fw = (C.c_void_p * 3)(*[dev(f"embeddings.{k}.weight") for k in FC_KEYS]) if self.has_fc else None
            fb = (C.c_void_p * 3)(*[dev(f"embeddings.{k}.bias") for k in FC_KEYS]) if self.has_fc else None
            check(_lib.lib().vmb_vggish_create_ex(C.byref(self._h), cw, cb, fw, fb, PRECISIONS[precision],
                                                  stream_ptr()), "vmb_vggish_create_ex")
            del keep

    @property
    def raw(self) -> C.c_void_p:
        return self._h

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value and _lib is not None:     # _lib is None at interpreter exit
            _lib.lib().vmb_vggish_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def _workspace(self, nbytes: int) -> torch.Tensor:
        if self._ws is None or self._ws.numel() < nbytes + 1024:
            self._ws = None
            self._ws = torch.empty(nbytes + 1024, device=self.device, dtype=torch.uint8)
        return self._ws

    @property
    def act_dtype(self) -> torch.dtype:
        """Element type of the 16-bit activations (and of the bottleneck features forward() can return)."""
        return torch.float16 if self.precision == "fp16" else torch.bfloat16

    def check_saturation(self, synchronize: bool = True) -> None:
        """fp16 mode: raise if any layer's output reached the fp16 maximum since the last check.  The flags are written
        by the kernels into mapped host memory; with synchronize=False only work that already finished is seen
        (forward() does that on entry, so a saturated batch is reported by the next call at the latest)."""
        if self.precision != "fp16":
            return
        if synchronize:
            torch.cuda.synchronize(self.device)
        mask = int(_lib.lib().vmb_vggish_saturation(self._h, 1))
        if mask:
            layers = [n for i, n in enumerate(SAT_LAYERS) if mask >> i & 1]
            raise B200Error(f"fp16 activations saturated (65504) in {layers}: the results are invalid; build the handle "
                            "with precision='bf16' or 'split'")

    def forward(self, examples: torch.Tensor, want_bottleneck: bool = False, want_embeddings: bool = True):
        """examples (n, 96, 64) or (n, 1, 96, 64) fp32 CUDA -> (n, 128) fp32 post-ReLU embeddings
        [, (n, 12288) 16-bit conv features in (h, w, c) order].  want_embeddings=False skips the FC stack."""
        self.check_saturation(synchronize=False)
        if want_embeddings and not self.has_fc:
            raise B200Error("this handle was built without the FC stack: only the bottleneck features are available")
        if not want_embeddings and not want_bottleneck:
            raise ValueError("nothing to compute")
        examples = _need_cuda(examples, "examples")
        if examples.dim() == 4 and examples.shape[1] == 1:
            examples = examples[:, 0]
        if examples.dim() != 3 or tuple(examples.shape[1:]) != (96, 64):
            raise ValueError(f"examples must be (n, 1, 96, 64) or (n, 96, 64), got {tuple(examples.shape)}")
        examples = examples.contiguous()
        n = examples.shape[0]
        emb = torch.empty((n, 128), device=self.device, dtype=torch.float32) if want_embeddings else None
        bott = torch.empty((n, 12288), device=self.device, dtype=self.act_dtype) if want_bottleneck else None
        if n == 0:
            return (emb, bott) if want_bottleneck else emb
        with torch.cuda.device(self.device):
            need = int(_lib.lib().vmb_vggish_handle_workspace_bytes(self._h, n))
            ws = self._workspace(need)
            base = (ws.data_ptr() + 1023) // 1024 * 1024
            check(_lib.lib().vmb_vggish_forward(self._h, ptr(examples), n, ptr(emb), ptr(bott), base, need, stream_ptr()),
                  "vmb_vggish_forward")
        return (emb, bott) if want_bottleneck else emb

    # -- train-mode FC stack (fc1-fc3 trainable, convs frozen): csrc/fc_train.cu
    @property
    def fc_trainable(self) -> bool:
        """True once refresh_fc() has derived the training copy of the FC weights."""
        return bool(getattr(self, "_fc_refreshed", False))

    def refresh_fc(self, weights, biases) -> None:
        """Re-derive every device copy of the FC weights (inference copy and training planes) from fp32 masters
        [embeddings.0/2/4.weight], [embeddings.0/2/4.bias] — stream-ordered, the conv weights are not touched."""
        if not self.has_fc:
            raise B200Error("this handle was built without the FC stack")
        with torch.cuda.device(self.device):
            keep = [t.detach().to(device=self.device, dtype=torch.float32).contiguous() for t in (*weights, *biases)]
            fw = (C.c_void_p * 3)(*[t.data_ptr() for t in keep[:3]])
            fb = (C.c_void_p * 3)(*[t.data_ptr() for t in keep[3:]])
            check(_lib.lib().vmb_vggish_refresh_fc(self._h, fw, fb, stream_ptr()), "vmb_vggish_refresh_fc")
            self._fc_keep = keep        # the masters' copies must outlive the enqueued kernels that read them
        self._fc_refreshed = True

    def _train_workspace(self, n: int):
        need = int(_lib.lib().vmb_vggish_fc_train_workspace_bytes(n))
        ws = getattr(self, "_train_ws", None)
        if ws is None or ws.numel() < need + 1024:
            self._train_ws = None
            ws = self._train_ws = torch.empty(need + 1024, device=self.device, dtype=torch.uint8)
        return (ws.data_ptr() + 1023) // 1024 * 1024, need

    def forward_train(self, examples: torch.Tensor) -> torch.Tensor:
        """(n, 96, 64) / (n, 1, 96, 64) fp32 CUDA -> (n, 128) fp32 embeddings, keeping what fc_backward() needs."""
        self.check_saturation(synchronize=False)
        examples = _need_cuda(examples, "examples")
        if examples.dim() == 4 and examples.shape[1] == 1:
            examples = examples[:, 0]
        if examples.dim() != 3 or tuple(examples.shape[1:]) != (96, 64):
            raise ValueError(f"examples must be (n, 1, 96, 64) or (n, 96, 64), got {tuple(examples.shape)}")
        examples = examples.contiguous()
        n = examples.shape[0]
        emb = torch.empty((n, 128), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            base, need = self._train_workspace(n)
            check(_lib.lib().vmb_vggish_forward_train(self._h, ptr(examples), n, ptr(emb), base, need, stream_ptr()),
                  "vmb_vggish_forward_train")
        self._train_n = n
        return emb

    def fc_backward(self, d_emb: torch.Tensor) -> torch.Tensor:
        """d(loss)/d(emb) (n, 128) of the last forward_train -> flat fp32 FC gradients in state_dict order."""
        n = getattr(self, "_train_n", None)
        if n is None:
            raise B200Error("fc_backward without a forward_train")
        d = d_emb.to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(d.shape) != (n, 128):
            raise ValueError(f"d_emb must be ({n}, 128), got {tuple(d.shape)}")
        grads = torch.empty(int(_lib.lib().vmb_vggish_fc_grad_count()), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            base, need = self._train_workspace(n)
            check(_lib.lib().vmb_vggish_fc_backward(self._h, base, need, ptr(d), n, ptr(grads), stream_ptr()),
                  "vmb_vggish_fc_backward")
        return grads

    def train_features(self) -> torch.Tensor:
        """(n, 12288) float64 conv features of the last forward_train, as its FC stack saw them (sum of the three
        operand planes at the start of the workspace)."""
        n = self._train_n
        base, _ = self._train_workspace(n)
        off = base - self._train_ws.data_ptr()
        planes = self._train_ws[off:off + n * 3 * 12288 * 2].view(torch.bfloat16).view(n, 3, 12288)
        return planes.double().sum(dim=1)


FC_GRAD_LAYOUT = (("0.weight", (4096, 12288)), ("0.bias", (4096,)), ("2.weight", (4096, 4096)), ("2.bias", (4096,)),
                  ("4.weight", (128, 4096)), ("4.bias", (128,)))


def fc_grad_views(flat: torch.Tensor) -> dict:
    """The flat FC gradient buffer as {embeddings key suffix: tensor view} in state_dict order."""
    out, off = {}, 0
    for key, shape in FC_GRAD_LAYOUT:
        n = 1
        for s in shape:
            n *= s
        out[key] = flat[off:off + n].view(shape)
        off += n
    return out


def pack_mla_params(sd: dict, model_conf: Sequence[int], device: torch.device) -> torch.Tensor:
    """Flatten a MultiLevelAttention state_dict into the layout documented in vggish_mla_b200.h."""
    parts = []

    def add(key):
        parts.append(sd[key].detach().to(device=device, dtype=torch.float32).reshape(-1))

    def add_bn(prefix):
        for s in ("weight", "bias", "running_mean", "running_var"):
            add(f"{prefix}.{s}")

    for lvl, n_fc in enumerate(model_conf):
        p = f"embedded_mappings.{lvl}"
        add_bn(p + ".norm0")
        for j in range(n_fc):
            add(f"{p}.fc.{j}.weight")
            add(f"{p}.fc.{j}.bias")
            add_bn(f"{p}.norms.{j}")
    for lvl in range(len(model_conf)):
        p = f"attention_modules.{lvl}"
        add(p + ".fcv.weight")
        add(p + ".fcv.bias")
        add_bn(p + ".normv")
        add_bn(p + ".normf")
    add("fc.weight")
    add("fc.bias")
    add_bn("norm")
    return torch.cat(parts).contiguous()


class MlaHandle:
    """Library-side multi-level attention head (eval mode) built from a reference state_dict."""

    def __init__(self, state_dict: dict, model_conf: Sequence[int], emb_in: int, hidden: int, n_classes: int,
                 t_steps: int, device: torch.device):
        require_b200(device)
        self.device = device
        self.n_classes = n_classes
        self.t_steps = t_steps
        self.emb_in = emb_in
        self.hidden = hidden
        self._h = C.c_void_p()
        conf = (C.c_int * len(model_conf))(*[int(v) for v in model_conf])
        with torch.cuda.device(device):
            flat = pack_mla_params(state_dict, model_conf, device)
            expect = _lib.lib().vmb_mla_param_count(len(model_conf), conf, emb_in, hidden, n_classes, t_steps)
            if expect != flat.numel():
                raise B200Error(f"head parameter count {flat.numel()} != expected {expect} for this configuration")
            check(_lib.lib().vmb_mla_create(C.byref(self._h), len(model_conf), conf, emb_in, hidden, n_classes, t_steps,
                                            ptr(flat), flat.numel(), stream_ptr()), "vmb_mla_create")

    @property
    def raw(self) -> C.c_void_p:
        return self._h

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value and _lib is not None:     # _lib is None at interpreter exit
            _lib.lib().vmb_mla_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def embedded_mapping(self, level: int, x: torch.Tensor) -> torch.Tensor:
        """EmbeddedMapping.forward of one level (eval mode, model.py:217-222): (B, T, in) -> (B, T, hidden)."""
        x = _need_cuda(x, "x")
        if x.dim() != 3 or x.shape[1] != self.t_steps:
            raise ValueError(f"expected (B, {self.t_steps}, features), got {tuple(x.shape)}")
        out = torch.empty((x.shape[0], self.t_steps, self.hidden), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            check(_lib.lib().vmb_mla_embedded_mapping(self._h, int(level), ptr(x), x.shape[0], ptr(out), stream_ptr()),
                  "vmb_mla_embedded_mapping")
        return out

    def attention(self, level: int, h: torch.Tensor) -> torch.Tensor:
        """AttentionModule.forward of one level (eval mode, model.py:235-242): (B, T, hidden) -> (B, K)."""
        h = _need_cuda(h, "h")
        if h.dim() != 3 or h.shape[1] != self.t_steps or h.shape[2] != self.hidden:
            raise ValueError(f"expected (B, {self.t_steps}, {self.hidden}), got {tuple(h.shape)}")
        out = torch.empty((h.shape[0], self.n_classes), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            check(_lib.lib().vmb_mla_attention(self._h, int(level), ptr(h), h.shape[0], ptr(out), stream_ptr()),
                  "vmb_mla_attention")
        return out

    def forward(self, emb: torch.Tensor, fp32_crosscheck: bool = False) -> torch.Tensor:
        """(B, T, emb_in) fp32 CUDA -> (B, K) scores.  fp32_crosscheck=True runs the diagnostic fused CUDA-core kernel
        (vmb_mla_forward_fp32) instead of the tensor-core path."""
        emb = _need_cuda(emb, "embeddings")
        if emb.dim() != 3 or emb.shape[1] != self.t_steps or emb.shape[2] != self.emb_in:
            raise ValueError(f"expected (B, {self.t_steps}, {self.emb_in}), got {tuple(emb.shape)}")
        out = torch.empty((emb.shape[0], self.n_classes), device=self.device, dtype=torch.float32)
        fn, name = ((_lib.lib().vmb_mla_forward_fp32, "vmb_mla_forward_fp32") if fp32_crosscheck
                    else (_lib.lib().vmb_mla_forward, "vmb_mla_forward"))
        with torch.cuda.device(self.device):
            check(fn(self._h, ptr(emb), emb.shape[0], ptr(out), stream_ptr()), name)
        return out


class Pipeline:
    """waveform (n_clips, 160000) -> scores (n_clips, K): log-mel + VGGish + head, all inside the library."""

    def __init__(self, vggish: VggishHandle, mla: MlaHandle):
        if vggish.device != mla.device:
            raise ValueError("both handles must live on the same device")
        self.vggish, self.mla, self.device = vggish, mla, vggish.device
        self._ws: Optional[torch.Tensor] = None

    def forward(self, wave: torch.Tensor, want_embeddings: bool = False):
        self.vggish.check_saturation(synchronize=False)
        wave = _need_cuda(wave, "wave")
        if wave.dim() != 2:
            raise ValueError("wave must be (n_clips, n_samples)")
        n, ns = wave.shape
        if num_examples(ns) != self.mla.t_steps:
            raise ValueError(f"{ns} samples give {num_examples(ns)} examples per clip, the head needs {self.mla.t_steps}")
        scores = torch.empty((n, self.mla.n_classes), device=self.device, dtype=torch.float32)
        emb = torch.empty((n * self.mla.t_steps, 128), device=self.device, dtype=torch.float32) if want_embeddings else None
        if n == 0:
            return (scores, emb) if want_embeddings else scores
        with torch.cuda.device(self.device):
            need = int(_lib.lib().vmb_pipeline_workspace_bytes(n, ns))
            if self._ws is None or self._ws.numel() < need + 1024:
                self._ws = None
                self._ws = torch.empty(need + 1024, device=self.device, dtype=torch.uint8)
            base = (self._ws.data_ptr() + 1023) // 1024 * 1024
            check(_lib.lib().vmb_pipeline_forward(self.vggish.raw, self.mla.raw, ptr(wave), n, ns, ptr(scores), ptr(emb),
                                                  base, need, stream_ptr()), "vmb_pipeline_forward")
        return (scores, emb) if want_embeddings else scores

    def forward_host(self, wave_host: torch.Tensor, scores_host: Optional[torch.Tensor] = None,
                     clips_per_batch: int = 256) -> torch.Tensor:
        """End-to-end call with HOST buffers: H2D copy, compute and D2H copy all happen inside the library."""
        if wave_host.is_cuda or wave_host.dtype != torch.float32 or wave_host.dim() != 2:
            raise ValueError("wave_host must be a (n_clips, n_samples) fp32 CPU tensor (pinned for full speed)")
        wave_host = wave_host.contiguous()
        n, ns = wave_host.shape
        if scores_host is None:
            scores_host = torch.empty((n, self.mla.n_classes), dtype=torch.float32).pin_memory()
        with torch.cuda.device(self.device):
            check(_lib.lib().vmb_pipeline_forward_host(self.vggish.raw, self.mla.raw, wave_host.data_ptr(), n, ns,
                                                       scores_host.data_ptr(), clips_per_batch, stream_ptr()),
                  "vmb_pipeline_forward_host")
        return scores_host

    def submit_host(self, wave_host: torch.Tensor, scores_host: torch.Tensor, clips_per_batch: int = 64) -> int:
        """Asynchronous half of forward_host: enqueue copies + compute, return a ticket for wait_host().  Up to two
        calls may be in flight, so the H2D copy of call i+1 overlaps the compute of call i."""
        if wave_host.is_cuda or wave_host.dtype not in (torch.float32, torch.int16) or wave_host.dim() != 2 \
                or not wave_host.is_contiguous():
            raise ValueError("wave_host must be a contiguous (n_clips, n_samples) fp32 or int16 (PCM) CPU tensor")
        n, ns = wave_host.shape
        if tuple(scores_host.shape) != (n, self.mla.n_classes) or scores_host.dtype != torch.float32:
            raise ValueError("scores_host must be (n_clips, n_classes) fp32 on the host")
        with torch.cuda.device(self.device):
            fn = (_lib.lib().vmb_pipeline_submit_host_pcm16 if wave_host.dtype == torch.int16
                  else _lib.lib().vmb_pipeline_submit_host)
            ticket = fn(self.vggish.raw, self.mla.raw, wave_host.data_ptr(), n, ns, scores_host.data_ptr(),
                        clips_per_batch, stream_ptr())
        if ticket < 0:
            raise B200Error(f"vmb_pipeline_submit_host failed: {_lib.last_error()}")
        return ticket

    def wait_host(self, ticket: int) -> None:
        check(_lib.lib().vmb_pipeline_wait_host(self.vggish.raw, ticket), "vmb_pipeline_wait_host")
