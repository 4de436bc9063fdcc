"""Host-side mirror of the reference's attack interface on top of the C-ABI (include/avc_b200.h).

``Engine`` owns one ``avc_handle`` for one model on one GPU: it derives the hyper-parameters from the
model's ``state_dict()`` / module attributes (the reference keeps them in an external config.yaml,
data_utils.py:219-220), hands the weights to ``avc_load_weights`` and exposes ``emb_attack`` /
``e2e_attack`` / ``fb_attack`` / ``speaker_encoder`` / ``inference`` with the reference's argument
meaning (attack_utils.py:7-130, models.py:327-343, 472-485).  PyTorch is used for device memory,
the RNG draw of w0 and the CUDA stream only; all arithmetic runs in libavc_b200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import torch
from torch import Tensor, nn

from . import _lib
from ._lib import AttackArgs, AttackVarlenArgs, DecoderDesc, EncoderDesc, HeaderArgs, ModelDesc, WeightView


class AvcError(RuntimeError):
    pass


def _slope(mod) -> float:
    act = getattr(mod, "act", None)
    if isinstance(act, str):
        return 0.01 if act == "lrelu" else 0.0
    if isinstance(act, nn.LeakyReLU):
        return float(act.negative_slope)
    return 0.0


def _dropout_p(mod) -> float:
    d = getattr(mod, "dropout_layer", None)
    return float(getattr(d, "p", 0.0)) if d is not None else 0.0


def _encoder_desc(sd: Dict[str, Tensor], prefix: str, mod, dense: bool) -> EncoderDesc:
    d = EncoderDesc()
    ks = []
    i = 0
    while f"{prefix}conv_bank.{i}.weight" in sd:
        ks.append(int(sd[f"{prefix}conv_bank.{i}.weight"].shape[2]))
        i += 1
    if not ks or ks != list(range(1, len(ks) + 1)):
        raise ValueError(f"{prefix}: conv bank kernel sizes {ks} unsupported (need bank_scale == 1)")
    wb = sd[f"{prefix}conv_bank.0.weight"]
    d.c_bank, d.c_in, d.bank_size = int(wb.shape[0]), int(wb.shape[1]), len(ks)
    w1 = sd[f"{prefix}first_conv_layers.0.weight"]
    d.c_h, d.kernel_size = int(w1.shape[0]), int(w1.shape[2])
    n = 0
    while f"{prefix}first_conv_layers.{n}.weight" in sd:
        n += 1
    d.n_conv_blocks = n
    sub = list(getattr(mod, "subsample"))
    if len(sub) < n or n > _lib.AVC_MAX_BLOCKS:
        raise ValueError(f"{prefix}: subsample list {sub} does not cover {n} conv blocks")
    for l in range(n):
        d.subsample[l] = int(sub[l])
    if dense:
        nd = 0
        while f"{prefix}first_dense_layers.{nd}.weight" in sd:
            nd += 1
        d.n_dense_blocks = nd
        d.c_out = int(sd[f"{prefix}output_layer.weight"].shape[0])
    else:
        d.n_dense_blocks = 0
        d.c_out = int(sd[f"{prefix}mean_layer.weight"].shape[0])
    d.neg_slope = _slope(mod)
    if _dropout_p(mod) != 0.0:
        # the reference never calls .eval() (data_utils.py:220-221): p > 0 would be live noise
        raise ValueError(f"{prefix}: dropout_rate must be 0 (got {_dropout_p(mod)})")
    return d


def _decoder_desc(sd: Dict[str, Tensor], prefix: str, mod) -> DecoderDesc:
    if any(k.endswith("weight_orig") for k in sd if k.startswith(prefix)):
        raise ValueError("decoder: spectral_norm (sn=True) is not supported")
    d = DecoderDesc()
    wi = sd[f"{prefix}in_conv_layer.weight"]
    d.c_h, d.c_in = int(wi.shape[0]), int(wi.shape[1])
    d.c_cond = int(sd[f"{prefix}conv_affine_layers.0.weight"].shape[1])
    d.c_out = int(sd[f"{prefix}out_conv_layer.weight"].shape[0])
    d.kernel_size = int(sd[f"{prefix}first_conv_layers.0.weight"].shape[2])
    n = 0
    while f"{prefix}first_conv_layers.{n}.weight" in sd:
        n += 1
    d.n_conv_blocks = n
    up = list(getattr(mod, "upsample"))
    if len(up) < n or n > _lib.AVC_MAX_BLOCKS:
        raise ValueError(f"decoder: upsample list {up} does not cover {n} conv blocks")
    for l in range(n):
        d.upsample[l] = int(up[l])
    d.neg_slope = _slope(mod)
    if _dropout_p(mod) != 0.0:
        raise ValueError(f"decoder: dropout_rate must be 0 (got {_dropout_p(mod)})")
    return d


def _strides3(t: Tensor):
    return (C.c_int64 * 3)(*[int(s) for s in t.stride()])


class Engine:
    """One avc_handle bound to ``model``'s weights on one CUDA device."""

    def __init__(self, model: nn.Module, device: Optional[torch.device] = None):
        self._lib = _lib.load()
        if not torch.cuda.is_available():
            raise AvcError("attack_vc_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        sd = {k: v.detach() for k, v in model.state_dict().items()}
        if device is None:
            device = next(iter(sd.values())).device
        device = torch.device(device)
        if device.type != "cuda":
            raise AvcError("attack_vc_b200 needs the model on a CUDA device; there is no CPU fallback")
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        desc = ModelDesc()
        desc.speaker = _encoder_desc(sd, "speaker_encoder.", model.speaker_encoder, dense=True)
        desc.content = _encoder_desc(sd, "content_encoder.", model.content_encoder, dense=False)
        desc.decoder = _decoder_desc(sd, "decoder.", model.decoder)
        self.desc = desc
        self.c_in = int(desc.speaker.c_in)
        self.c_emb = int(desc.speaker.c_out)
        self._sessions = 0            # open AttackSession / HeaderSession objects: close() refuses while any is alive
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            rc = self._lib.avc_create(C.byref(h), C.byref(desc), self.device.index)
            if rc != 0:
                raise AvcError(f"avc_create failed ({rc}): {self._lib.avc_last_error(None).decode()}")
            self._h = h
            keep = []
            views = (WeightView * len(sd))()
            for i, (k, v) in enumerate(sd.items()):
                t = v.to(device=self.device, dtype=torch.float32).contiguous()
                keep.append(t)
                views[i].name = k.encode()
                views[i].data = t.data_ptr()
                views[i].ndim = t.dim()
                for j, s in enumerate(t.shape):
                    views[i].shape[j] = int(s)
            torch.cuda.synchronize(self.device)
            self._check(self._lib.avc_load_weights(self._h, views, len(sd)))
            del keep

    # ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_sessions", 0) > 0:
                raise AvcError(f"Engine.close(): {self._sessions} attack session(s) still open; end() them first")
            self._lib.avc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            msg = self._lib.avc_last_error(self._h).decode()
            if rc == -1:
                raise ValueError(f"libavc_b200: {msg}")
            raise AvcError(f"libavc_b200 error {rc}: {msg}")

    def _stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _utt(self, t: Tensor, name: str) -> Tensor:
        if not isinstance(t, Tensor):
            raise TypeError(f"{name} must be a torch.Tensor")
        if t.device.type != "cuda":
            raise AvcError(f"{name} is on {t.device}: attack_vc_b200 runs on CUDA only (no CPU fallback)")
        if t.device != self.device:
            raise AvcError(f"{name} is on {t.device} but the engine lives on {self.device}")
        if t.dtype != torch.float32:
            raise ValueError(f"{name} must be float32 (got {t.dtype})")
        if t.dim() != 3 or t.shape[1] != self.c_in:
            raise ValueError(f"{name} must have shape [B, {self.c_in}, T] (got {tuple(t.shape)})")
        return t

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.avc_kernel_launches(self._h))

    @property
    def launches_per_iter(self) -> int:
        return int(self._lib.avc_launches_per_iter(self._h))

    def decoder_frames(self, T_src: int) -> int:
        """Frames of the converted utterance for a source of ``T_src`` frames (avc_decoder_frames)."""
        return int(self._lib.avc_decoder_frames(self._h, int(T_src)))

    def min_frames(self, which: str = "speaker") -> int:
        """Shortest utterance the ``speaker`` / ``content`` encoder accepts: every reflect-padded conv input must be
        longer than its padding (models.py:23-28; the same rule avc_* enforces)."""
        d = self.desc.speaker if which == "speaker" else self.desc.content
        T = 1
        while True:
            Tl, ok = T, T > d.bank_size // 2
            for l in range(d.n_conv_blocks):
                ok = ok and Tl > d.kernel_size // 2
                Tl = -(-Tl // int(d.subsample[l]))
            if ok:
                return T
            T += 1

    # ------------------------------------------------------------------------------------------
    def _attack_args(self, kind, vc_tgt, adv_tgt, eps, n_iters, vc_src, w0, inv_norm, want_loss, want_grad, use_graph):
        if kind not in ("emb", "e2e", "fb"):
            raise NotImplementedError(kind)
        vc_tgt = self._utt(vc_tgt, "vc_tgt")
        adv_tgt = self._utt(adv_tgt, "adv_tgt")
        if kind != "emb":
            if vc_src is None:
                raise ValueError("vc_src is required for e2e and fb attacks")
            vc_src = self._utt(vc_src, "vc_src")
        else:
            vc_src = None
        B = vc_tgt.shape[0]
        if adv_tgt.shape[0] != B or (vc_src is not None and vc_src.shape[0] != B):
            raise ValueError("batch sizes of vc_src / vc_tgt / adv_tgt differ")
        n_iters = int(n_iters)
        if w0 is None:
            w0 = torch.zeros_like(vc_tgt).normal_(0, 1)
        w0 = self._utt(w0, "w0")
        if w0.shape != vc_tgt.shape:
            raise ValueError("w0 must have the shape of vc_tgt")
        out = torch.empty_like(vc_tgt)
        loss = torch.zeros(max(n_iters, 1), device=self.device, dtype=torch.float32) if want_loss else None
        grad = torch.zeros(vc_tgt.shape, device=self.device, dtype=torch.float32) if want_grad else None
        a = AttackArgs()
        a.vc_tgt, a.tgt_stride, a.B, a.T_tgt = vc_tgt.data_ptr(), _strides3(vc_tgt), B, vc_tgt.shape[2]
        a.adv_tgt, a.adv_stride, a.T_adv = adv_tgt.data_ptr(), _strides3(adv_tgt), adv_tgt.shape[2]
        if vc_src is not None:
            a.vc_src, a.src_stride, a.T_src = vc_src.data_ptr(), _strides3(vc_src), vc_src.shape[2]
        a.w0, a.w0_stride = w0.data_ptr(), _strides3(w0)
        a.adv_out, a.out_stride = out.data_ptr(), _strides3(out)
        a.loss_out = loss.data_ptr() if loss is not None else None
        a.grad_out = grad.data_ptr() if grad is not None else None
        a.eps, a.n_iters = float(eps), n_iters
        a.inv_norm = float(inv_norm) if inv_norm is not None else 0.0
        a.use_graph = 1 if use_graph else 0
        keep = (vc_tgt, adv_tgt, vc_src, w0, out, loss, grad)
        return a, keep

    def attack(self, kind: str, vc_tgt: Tensor, adv_tgt: Tensor, eps: float, n_iters: int,
               vc_src: Optional[Tensor] = None, w0: Optional[Tensor] = None, inv_norm: Optional[float] = None,
               want_loss: bool = False, want_grad: bool = False, use_graph: bool = True):
        """Run one attack.  Returns adv (same shape/strides as vc_tgt) or (adv, info) when
        want_loss / want_grad is set.  ``w0`` defaults to the reference's draw
        ``torch.zeros_like(vc_tgt).normal_(0, 1)`` (attack_utils.py:30,68,112)."""
        with torch.cuda.device(self.device):
            a, keep = self._attack_args(kind, vc_tgt, adv_tgt, eps, n_iters, vc_src, w0, inv_norm, want_loss, want_grad, use_graph)
            fn = {"emb": self._lib.avc_emb_attack, "e2e": self._lib.avc_e2e_attack, "fb": self._lib.avc_fb_attack}[kind]
            self._check(fn(self._h, C.byref(a), self._stream()))
        _, _, _, w0, out, loss, grad = keep
        if want_loss or want_grad:
            return out, {"losses": loss[:int(n_iters)] if loss is not None else None, "grad": grad, "w0": w0}
        return out

    def _packed(self, mels: Sequence[Tensor], name: str) -> Tensor:
        """[sum T_i, c_in] time-major block of utterances given as [T_i, c_in] mels: a view when they are consecutive
        contiguous views of one buffer (as AudioEngine.wav2mel_varlen returns them), else one torch.cat."""
        for i, m in enumerate(mels):
            if not isinstance(m, Tensor):
                raise TypeError(f"{name}[{i}] must be a torch.Tensor")
            if m.device.type != "cuda":
                raise AvcError(f"{name}[{i}] is on {m.device}: attack_vc_b200 runs on CUDA only (no CPU fallback)")
            if m.device != self.device:
                raise AvcError(f"{name}[{i}] is on {m.device} but the engine lives on {self.device}")
            if m.dtype != torch.float32 or m.dim() != 2 or m.shape[1] != self.c_in:
                raise ValueError(f"{name}[{i}] must be a float32 [T, {self.c_in}] mel (got {m.dtype} {tuple(m.shape)})")
        first, rows, consecutive = mels[0], 0, True
        for m in mels:
            consecutive = consecutive and m.is_contiguous() and m.untyped_storage().data_ptr() == first.untyped_storage().data_ptr() \
                and m.data_ptr() == first.data_ptr() + rows * self.c_in * 4
            rows += int(m.shape[0])
        if consecutive:
            return first.as_strided((rows, self.c_in), (self.c_in, 1))
        return torch.cat([m.contiguous() for m in mels])

    def attack_varlen(self, kind: str, vc_tgt: Sequence[Tensor], adv_tgt: Tensor, eps: float, n_iters: int,
                      vc_src: Optional[Tensor] = None, w0=None, inv_norm: Optional[float] = None,
                      want_loss: bool = False, want_grad: bool = False, use_graph: bool = True):
        """One attack over utterances of different lengths (avc_attack_varlen).  ``vc_tgt`` is a sequence of [T_i, 80]
        time-major mels; ``adv_tgt`` / ``vc_src`` are [B, 80, T] as in ``attack`` (batch stride 0 allowed).  ``w0`` is a
        sequence of [T_i, 80] (or one packed [sum T_i, 80] tensor); None draws it as ``Defender.draw_w0`` does, one
        utterance at a time in input order.  Returns the defended [T_i, 80] mels (views of one packed output), or
        ``(mels, info)`` when want_loss / want_grad is set: ``info["grad"]`` holds [T_i, 80] views too.  ``inv_norm``
        defaults as in ``attack``; the loss curve is summed over the batch."""
        if kind not in ("emb", "e2e", "fb"):
            raise NotImplementedError(kind)
        mels = list(vc_tgt)
        if not mels:
            raise ValueError("vc_tgt is empty")
        frames = [int(m.shape[0]) if isinstance(m, Tensor) and m.dim() == 2 else -1 for m in mels]
        B = len(mels)
        with torch.cuda.device(self.device):
            x = self._packed(mels, "vc_tgt")
            rows = x.shape[0]
            adv_tgt = self._utt(adv_tgt, "adv_tgt")
            if kind != "emb":
                if vc_src is None:
                    raise ValueError("vc_src is required for e2e and fb attacks")
                vc_src = self._utt(vc_src, "vc_src")
            else:
                vc_src = None
            if adv_tgt.shape[0] != B or (vc_src is not None and vc_src.shape[0] != B):
                raise ValueError("batch sizes of vc_src / vc_tgt / adv_tgt differ")
            if w0 is None:
                w0 = [torch.zeros_like(m.t().unsqueeze(0)).normal_(0, 1)[0].t() for m in mels]
            if isinstance(w0, Tensor):
                if w0.device != self.device or w0.dtype != torch.float32 or w0.dim() != 2 or w0.shape[1] != self.c_in:
                    raise ValueError(f"a packed w0 must be a float32 [sum T_i, {self.c_in}] tensor on {self.device}")
                w = w0.contiguous()
            else:
                w0 = list(w0)
                if len(w0) != B:
                    raise ValueError(f"w0 has {len(w0)} utterances, vc_tgt {B}")
                w = self._packed(w0, "w0")
                if [int(t.shape[0]) for t in w0] != frames:
                    raise ValueError("w0's utterance lengths differ from vc_tgt's")
            if w.shape[0] != rows:
                raise ValueError(f"w0 holds {w.shape[0]} frames, vc_tgt {rows} (sum of the utterance lengths)")
            n_iters = int(n_iters)
            out = torch.empty((rows, self.c_in), device=self.device, dtype=torch.float32)
            loss = torch.zeros(max(n_iters, 1), device=self.device, dtype=torch.float32) if want_loss else None
            grad = torch.zeros((rows, self.c_in), device=self.device, dtype=torch.float32) if want_grad else None
            fr = (C.c_int32 * B)(*frames)
            a = AttackVarlenArgs()
            a.vc_tgt, a.w0, a.adv_out = x.data_ptr(), w.data_ptr(), out.data_ptr()
            a.grad_out = grad.data_ptr() if grad is not None else None
            a.frames_host, a.B = fr, B
            a.adv_tgt, a.adv_stride, a.T_adv = adv_tgt.data_ptr(), _strides3(adv_tgt), adv_tgt.shape[2]
            if vc_src is not None:
                a.vc_src, a.src_stride, a.T_src = vc_src.data_ptr(), _strides3(vc_src), vc_src.shape[2]
            a.loss_out = loss.data_ptr() if loss is not None else None
            a.eps, a.n_iters = float(eps), n_iters
            a.inv_norm = float(inv_norm) if inv_norm is not None else 0.0
            a.use_graph = 1 if use_graph else 0
            self._check(self._lib.avc_attack_varlen(self._h, {"emb": 0, "e2e": 1, "fb": 2}[kind], C.byref(a), self._stream()))
        outs = list(out.split(frames))
        if want_loss or want_grad:
            return outs, {"losses": loss[:n_iters] if loss is not None else None,
                          "grad": list(grad.split(frames)) if grad is not None else None, "w0": w}
        return outs

    def begin(self, kind: str, vc_tgt: Tensor, adv_tgt: Tensor, eps: float, n_iters: int,
              vc_src: Optional[Tensor] = None, w0: Optional[Tensor] = None, inv_norm: Optional[float] = None,
              want_loss: bool = False, want_grad: bool = False, use_graph: bool = True) -> "AttackSession":
        """Open an attack session (avc_attack_begin): targets + loop invariants are computed and one
        iteration is captured; iterations are then enqueued with ``step(n)`` and ``end()`` returns adv."""
        with torch.cuda.device(self.device):
            a, keep = self._attack_args(kind, vc_tgt, adv_tgt, eps, n_iters, vc_src, w0, inv_norm, want_loss, want_grad, use_graph)
            sp = C.c_void_p()
            k = {"emb": 0, "e2e": 1, "fb": 2}[kind]
            self._check(self._lib.avc_attack_begin(self._h, k, C.byref(a), self._stream(), C.byref(sp)))
        return AttackSession(self, sp, keep, int(n_iters))

    # ---- universal perturbation header (models/header_model.py:25-68) ---------------------------------
    def _header_args(self, source, target, eps, lam, lr, n_iters, header0, inv_norm, want_loss, want_grad, use_graph):
        if source.dim() == 4:          # the reference's [B,1,80,T] -> the speaker encoder's [B,80,T] (a view)
            source = source.squeeze(1)
        if target.dim() == 4:
            target = target.squeeze(1)
        source, target = self._utt(source, "source_mel"), self._utt(target, "target_mel")
        B, _, T = source.shape
        if target.shape[0] != B:
            raise ValueError("batch sizes of source_mel / target_mel differ")
        if header0 is None:
            header0 = torch.zeros(self.c_in, T, device=self.device, dtype=torch.float32)   # header_model.py:22
        header0 = header0.reshape(self.c_in, -1)
        if header0.shape[1] != T or header0.device != self.device or header0.dtype != torch.float32:
            raise ValueError(f"header must be float32 [80, {T}] on {self.device}")
        n_iters = int(n_iters)
        out = torch.empty(self.c_in, T, device=self.device, dtype=torch.float32)
        loss = torch.zeros(max(n_iters, 1), device=self.device, dtype=torch.float32) if want_loss else None
        grad = torch.zeros(self.c_in, T, device=self.device, dtype=torch.float32) if want_grad else None
        a = HeaderArgs()
        a.source, a.src_stride, a.B, a.T = source.data_ptr(), _strides3(source), B, T
        a.target, a.tgt_stride, a.T_tgt = target.data_ptr(), _strides3(target), target.shape[2]
        a.header0, a.hdr_stride = header0.data_ptr(), (C.c_int64 * 2)(*[int(v) for v in header0.stride()])
        a.header_out, a.out_stride = out.data_ptr(), (C.c_int64 * 2)(*[int(v) for v in out.stride()])
        a.loss_out = loss.data_ptr() if loss is not None else None
        a.grad_out = grad.data_ptr() if grad is not None else None
        a.eps, a.lam, a.lr, a.n_iters = float(eps), float(lam), float(lr), n_iters
        a.inv_norm = float(inv_norm) if inv_norm is not None else 0.0
        a.use_graph = 1 if use_graph else 0
        return a, (source, target, header0, out, loss, grad)

    def header_optimize(self, source_mel: Tensor, target_mel: Tensor, num_iterations: int = 1000, epsilon: float = 0.1,
                        lambda_param: float = 0.5, lr: float = 1e-3, header0: Optional[Tensor] = None,
                        inv_norm: Optional[float] = None, want_loss: bool = False, want_grad: bool = False, use_graph: bool = True):
        """UniversalPerturbationHeader.optimize with this model's speaker encoder and Adam([header], lr)
        (header_model.py:25-68, train_header.py:46,77-81).  Returns the optimised header [1,1,80,T]
        (and an info dict when want_loss / want_grad)."""
        with torch.cuda.device(self.device):
            a, keep = self._header_args(source_mel, target_mel, epsilon, lambda_param, lr, num_iterations, header0, inv_norm,
                                        want_loss, want_grad, use_graph)
            self._check(self._lib.avc_header_optimize(self._h, C.byref(a), self._stream()))
        _, _, _, out, loss, grad = keep
        hdr = out.reshape(1, 1, self.c_in, -1)
        if want_loss or want_grad:
            return hdr, {"losses": loss[:int(num_iterations)] if loss is not None else None, "grad": grad}
        return hdr

    def header_begin(self, source_mel: Tensor, target_mel: Tensor, num_iterations: int, epsilon: float = 0.1,
                     lambda_param: float = 0.5, lr: float = 1e-3, header0: Optional[Tensor] = None,
                     inv_norm: Optional[float] = None, want_loss: bool = False, use_graph: bool = True) -> "HeaderSession":
        with torch.cuda.device(self.device):
            a, keep = self._header_args(source_mel, target_mel, epsilon, lambda_param, lr, num_iterations, header0, inv_norm,
                                        want_loss, False, use_graph)
            sp = C.c_void_p()
            self._check(self._lib.avc_header_begin(self._h, C.byref(a), self._stream(), C.byref(sp)))
        return HeaderSession(self, sp, keep, int(num_iterations))

    def speaker_encoder(self, x: Tensor) -> Tensor:
        x = self._utt(x, "x")
        with torch.cuda.device(self.device):
            emb = torch.empty(x.shape[0], self.c_emb, device=self.device, dtype=torch.float32)
            self._check(self._lib.avc_speaker_encoder(self._h, x.data_ptr(), _strides3(x), x.shape[0], x.shape[2],
                                                      emb.data_ptr(), self._stream()))
        return emb

    def inference(self, src: Tensor, tgt: Tensor) -> Tensor:
        src, tgt = self._utt(src, "src"), self._utt(tgt, "tgt")
        if src.shape[0] != tgt.shape[0]:
            raise ValueError("batch sizes differ")
        with torch.cuda.device(self.device):
            T_out = int(self._lib.avc_decoder_frames(self._h, src.shape[2]))
            out = torch.empty(src.shape[0], self.c_in, T_out, device=self.device, dtype=torch.float32)
            self._check(self._lib.avc_inference(self._h, src.data_ptr(), _strides3(src), src.shape[2], tgt.data_ptr(),
                                                _strides3(tgt), tgt.shape[2], src.shape[0], out.data_ptr(), self._stream()))
        return out

    # ---- per-kernel entry points (time-major tensors), used by tests -----------------------------
    def conv1d_fwd(self, x_tl: Tensor, w: Tensor, bias: Optional[Tensor], stride: int = 1, impl: int = 0) -> Tensor:
        B, T, c_in = x_tl.shape
        c_out, _, k = w.shape
        y = torch.empty(B, -(-T // stride), c_out, device=x_tl.device, dtype=torch.float32)
        self._check(self._lib.avc_conv1d_fwd(self._h, x_tl.contiguous().data_ptr(), w.contiguous().data_ptr(),
                                             bias.contiguous().data_ptr() if bias is not None else None, y.data_ptr(),
                                             B, T, c_in, c_out, k, stride, impl, self._stream()))
        return y

    def conv1d_dgrad(self, dy_tl: Tensor, w: Tensor, T: int, stride: int = 1, impl: int = 0) -> Tensor:
        B, _, c_out = dy_tl.shape
        _, c_in, k = w.shape
        dx = torch.empty(B, T, c_in, device=dy_tl.device, dtype=torch.float32)
        self._check(self._lib.avc_conv1d_dgrad(self._h, dy_tl.contiguous().data_ptr(), w.contiguous().data_ptr(),
                                               dx.data_ptr(), B, T, c_in, c_out, k, stride, impl, self._stream()))
        return dx

    def conv1d_wgrad(self, x_tl: Tensor, dy_tl: Tensor, k: int, stride: int = 1, bias: bool = True, impl: int = 1
                     ) -> Tuple[Tensor, Optional[Tensor]]:
        """d/dW and d/db of pad_layer + Conv1d (include/avc_b200.h avc_conv1d_wgrad_ex): x [B,T,c_in], dy [B,T_out,c_out]
        time-major -> dw [c_out,c_in,k], db [c_out].  impl 0 auto, 1 exact fp32 CUDA cores, 2 tcgen05 (TMA, 3xTF32)."""
        B, T, c_in = x_tl.shape
        c_out = dy_tl.shape[2]
        dw = torch.empty(c_out, c_in, k, device=x_tl.device, dtype=torch.float32)
        db = torch.empty(c_out, device=x_tl.device, dtype=torch.float32) if bias else None
        self._check(self._lib.avc_conv1d_wgrad_ex(self._h, x_tl.contiguous().data_ptr(), dy_tl.contiguous().data_ptr(),
                                                  dw.data_ptr(), db.data_ptr() if bias else None, B, T, c_in, c_out, k,
                                                  stride, int(impl), self._stream()))
        return dw, db

    def instnorm_adain_act_fwd(self, y: Tensor, cond: Optional[Tensor], res: Optional[Tensor], up: int, slope: float
                               ) -> Tuple[Tensor, Tensor]:
        B, T, Cc = y.shape
        out = torch.empty_like(y)
        stats = torch.empty(B, Cc, 2, device=y.device, dtype=torch.float32)
        self._check(self._lib.avc_instnorm_adain_act_fwd(
            self._h, y.contiguous().data_ptr(), cond.contiguous().data_ptr() if cond is not None else None,
            res.contiguous().data_ptr() if res is not None else None, up, out.data_ptr(), stats.data_ptr(), B, T, Cc,
            slope, self._stream()))
        return out, stats

    def instnorm_adain_act_bwd(self, g: Tensor, y: Tensor, stats: Tensor, cond: Optional[Tensor], slope: float
                               ) -> Tuple[Tensor, Tensor]:
        B, T, Cc = y.shape
        gy = torch.empty_like(y)
        gcond = torch.empty(B, 2 * Cc, device=y.device, dtype=torch.float32)
        self._check(self._lib.avc_instnorm_adain_act_bwd(
            self._h, g.contiguous().data_ptr(), y.contiguous().data_ptr(), stats.contiguous().data_ptr(),
            cond.contiguous().data_ptr() if cond is not None else None, gy.data_ptr(), gcond.data_ptr(), B, T, Cc,
            slope, self._stream()))
        return gy, gcond

    def unit_timing(self, reps: int) -> None:
        """avc_unit_timing: the three HBM-bound unit entry points repeat their kernel `reps` times and time it on the device."""
        self._check(self._lib.avc_unit_timing(self._h, int(reps)))

    def unit_last_ms(self) -> float:
        return float(self._lib.avc_unit_last_ms(self._h))

    def adam_tanh_step(self, g_adv: Tensor, x: Tensor, w: Tensor, m: Tensor, v: Tensor, eps: float, step: int) -> Tensor:
        adv = torch.empty_like(x)
        self._check(self._lib.avc_adam_tanh_step(self._h, g_adv.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(),
                                                 v.data_ptr(), adv.data_ptr(), x.numel(), eps, step, self._stream()))
        return adv


class AttackSession:
    """Handle of avc_attack_begin/step/end (include/avc_b200.h)."""

    def __init__(self, eng: Engine, sp, keep, n_iters: int):
        self.eng, self._s, self._keep, self.n_iters = eng, sp, keep, n_iters
        eng._sessions += 1

    @property
    def launches_per_iter(self) -> int:
        return int(self.eng._lib.avc_session_launches(self._s))

    def step(self, n: int = 1) -> None:
        self.eng._check(self.eng._lib.avc_attack_step(self._s, int(n), self.eng._stream()))

    def profile(self):
        """One eagerly launched iteration with CUDA events around every kernel ->
        list of (kind, ms, algorithmic flops, algorithmic bytes)."""
        n = self.launches_per_iter
        kind, ms = (C.c_int32 * n)(), (C.c_float * n)()
        fl, by = (C.c_double * n)(), (C.c_double * n)()
        self.eng._check(self.eng._lib.avc_session_profile(self._s, n, kind, ms, fl, by, self.eng._stream()))
        return [(int(kind[i]), float(ms[i]), float(fl[i]), float(by[i])) for i in range(n)]

    def end(self):
        if self._s is None:
            raise AvcError("session already ended")
        s, self._s = self._s, None
        self.eng._sessions -= 1
        self.eng._check(self.eng._lib.avc_attack_end(s, self.eng._stream()))
        _, _, _, w0, out, loss, grad = self._keep
        return out, {"losses": loss, "grad": grad, "w0": w0}

    def __del__(self):
        try:
            if self._s is not None:
                self.eng._sessions -= 1
                self.eng._lib.avc_attack_end(self._s, self.eng._stream())
                self._s = None
        except Exception:
            pass


class _DevMem:
    """CUDA array interface over a raw device pointer owned by the library (lives as long as the session)."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}


class HeaderSession:
    """avc_header_begin / avc_header_step / avc_attack_end.  ``step(n)`` runs whole iterations; a sharded
    caller alternates ``grad_half()``, an all-reduce of ``grad`` and ``apply_half()``."""

    def __init__(self, eng: Engine, sp, keep, n_iters: int):
        self.eng, self._s, self._keep, self.n_iters = eng, sp, keep, n_iters
        eng._sessions += 1
        n = C.c_int64()
        ptr = eng._lib.avc_header_grad_buffer(sp, C.byref(n))
        self.grad = torch.as_tensor(_DevMem(int(ptr), int(n.value)), device=eng.device)   # [T*80] time-major partial gradient

    def step(self, n: int = 1) -> None:
        self.eng._check(self.eng._lib.avc_header_step(self._s, int(n), 0, self.eng._stream()))

    def grad_half(self) -> None:
        self.eng._check(self.eng._lib.avc_header_step(self._s, 1, 1, self.eng._stream()))

    def apply_half(self) -> None:
        self.eng._check(self.eng._lib.avc_header_step(self._s, 1, 2, self.eng._stream()))

    def end(self):
        if self._s is None:
            raise AvcError("session already ended")
        s, self._s = self._s, None
        self.grad = None
        self.eng._sessions -= 1
        self.eng._check(self.eng._lib.avc_attack_end(s, self.eng._stream()))
        _, _, _, out, loss, _ = self._keep
        return out.reshape(1, 1, self.eng.c_in, -1), {"losses": loss}

    def __del__(self):
        try:
            if self._s is not None:
                self.eng._sessions -= 1
                self.eng._lib.avc_attack_end(self._s, self.eng._stream())
                self._s = None
        except Exception:
            pass


class SpeakerGradSession:
    """avc_spk_grad_begin / avc_spk_grad_step / avc_attack_end: the speaker-embedding loss of train_predictive.py:113-123
    and its gradient w.r.t. the perturbed batch.  The session owns four device tensors -- ``perturbed``, ``source``,
    ``target`` [B,80,T] to fill before each ``step()`` and ``grad`` [B,80,T] / ``loss`` [1] it writes."""

    def __init__(self, eng: "Engine", B: int, T: int, lambda_param: float = 0.5, inv_norm: float = 0.0, T_tgt: Optional[int] = None):
        self.eng = eng
        dev, c = eng.device, eng.c_in
        T_tgt = T if T_tgt is None else T_tgt
        self.perturbed = torch.zeros(B, c, T, device=dev)
        self.source = torch.zeros(B, c, T, device=dev)
        self.target = torch.zeros(B, c, T_tgt, device=dev)
        self.grad = torch.zeros(B, c, T, device=dev)
        self.loss = torch.zeros(1, device=dev)
        a = _lib.SpkGradArgs()
        a.perturbed, a.p_stride = self.perturbed.data_ptr(), _strides3(self.perturbed)
        a.source, a.s_stride = self.source.data_ptr(), _strides3(self.source)
        a.target, a.t_stride = self.target.data_ptr(), _strides3(self.target)
        a.grad_out, a.g_stride = self.grad.data_ptr(), _strides3(self.grad)
        a.loss_out = self.loss.data_ptr()
        a.B, a.T, a.T_tgt, a.lam, a.inv_norm, a.use_graph = B, T, T_tgt, lambda_param, float(inv_norm), 1
        sp = C.c_void_p()
        with torch.cuda.device(dev):
            torch.cuda.current_stream(dev).synchronize()
            eng._check(eng._lib.avc_spk_grad_begin(eng._h, C.byref(a), eng._stream(), C.byref(sp)))
        self._s = sp
        eng._sessions += 1

    def step(self) -> None:
        self.eng._check(self.eng._lib.avc_spk_grad_step(self._s, self.eng._stream()))

    def end(self) -> None:
        if self._s is not None:
            s, self._s = self._s, None
            self.eng._sessions -= 1
            self.eng._check(self.eng._lib.avc_attack_end(s, self.eng._stream()))

    def __del__(self):
        try:
            self.end()
        except Exception:
            pass


import weakref  # noqa: E402

_ENGINES: "weakref.WeakKeyDictionary[nn.Module, Tuple[Tuple, Engine]]" = weakref.WeakKeyDictionary()


def _fingerprint(model: nn.Module) -> Tuple:
    """(storage pointer, autograd version, 2-norm) per parameter.  The norms -- ONE multi-tensor kernel over all
    parameters and ONE device-to-host transfer, ~0.1 ms for the 4.9 M parameters of AdaIN-VC -- also catch in-place
    edits through ``p.data``, which do not bump ``_version``.  An edit that preserves every tensor's norm needs
    ``invalidate_engine(model)``."""
    ps = [p.detach() for p in model.parameters()]
    if not ps:
        return ()
    with torch.no_grad():
        norms = torch.stack(torch._foreach_norm(ps)).double().cpu().tolist()
    return tuple((p.data_ptr(), p._version, v) for p, v in zip(ps, norms))


def invalidate_engine(model: nn.Module) -> None:
    """Drop the cached engine of ``model`` (call after editing its weights in a way the fingerprint cannot see)."""
    hit = _ENGINES.pop(model, None)
    if hit is not None and hit[1]._sessions == 0:
        hit[1].close()


def engine_for(model: nn.Module) -> Engine:
    """Engine cache: one per LIVE model object (weak keys: a collected model releases its engine, and a new model that
    happens to reuse its id() or its allocator pointers can never be handed the old engine); rebuilt when a parameter
    was modified, replaced or moved."""
    sig = _fingerprint(model)
    hit = _ENGINES.get(model)
    if hit is not None and hit[0] == sig:
        return hit[1]
    if hit is not None and hit[1]._sessions == 0:
        hit[1].close()             # with sessions still open the old handle stays alive until they end (Engine.__del__)
    eng = Engine(model)
    _ENGINES[model] = (sig, eng)
    weakref.finalize(model, lambda e=eng: e._sessions == 0 and e.close())
    return eng
