"""Defend utterances from waveform to waveform on the GPU: the flow of the reference's ``attack.py:38-74`` as one library call.

Per utterance the reference runs ``file2mel`` -> ``normalize`` with the checkpoint's ``attr.pkl`` statistics
(data_utils.py:35-47) -> the ``[1, 80, T]`` view (attack.py:49-50) -> the attack -> ``denormalize`` -> ``mel2wav``.
``Defender.defend`` does the same for a whole list of utterances with three kinds of calls:

* ONE ragged front-end call (``avc_audio_wav2mel_varlen``, normalisation fused) over every target utterance plus the
  attack target and the conversion source;
* one ``Engine.attack`` per chunk of equal-length utterances (``group_by_length``; at most ``max_batch[kind]`` per chunk),
  each utterance with the normaliser a single ``attack.py`` run gives it, so that batching changes no result;
* ONE ragged back-end call (``avc_audio_mel2wav_varlen``, denormalisation fused) over every defended mel.

``librosa.load``, trimming and ``sf.write`` stay with the caller, as in ``audio.py``.  PyTorch allocates, copies and
draws the initial noise; every arithmetic step runs in libavc_b200.so.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor, nn

from .audio import AudioEngine, group_by_length
from .engine import AvcError, engine_for

KINDS = ("emb", "e2e", "fb")

# Utterances per attack call.  DESIGN "Data layout": an emb plan holds ~1.2 GB per 128 utterances of 512 frames, so 512 is
# ~5 GB (BASELINE configs[3] per GPU).  e2e / fb plans also hold the content encoder's and the decoder's activations: half.
DEFAULT_MAX_BATCH = {"emb": 512, "e2e": 256, "fb": 256}


def plan_chunks(frames: Sequence[int], max_batch: int) -> List[Tuple[int, List[int]]]:
    """Attack calls for utterances of ``frames[i]`` frames: equal lengths together (in order of first appearance), each
    group cut into chunks of at most ``max_batch`` -> [(T, [input indices]), ...]."""
    if max_batch < 1:
        raise ValueError(f"max_batch must be >= 1 (got {max_batch})")
    out = []
    for T, idx in group_by_length(frames):
        for i in range(0, len(idx), max_batch):
            out.append((T, idx[i:i + max_batch]))
    return out


def utterance_inv_norm(kind: str, c_emb: int, c_mel: int, T_out: int) -> float:
    """1 / D of ``nn.MSELoss`` for ONE utterance, as one attack.py run computes it (attack_utils.py:32,70,114): emb / fb
    compare embeddings [1, c_emb], e2e converted mels [1, c_mel, T_out]."""
    return 1.0 / float(c_emb if kind in ("emb", "fb") else c_mel * T_out)


class Defender:
    """A model, its speaker-normalisation statistics (``attr.pkl``'s ``mean`` / ``std``, [80] each) and the audio front-end
    and back-end, on one GPU.  ``model`` is an AdaIN-VC module (its engine comes from ``engine_for``) or an ``Engine``
    (or an object with its interface)."""

    def __init__(self, model, attr_mean, attr_std, audio: Optional[AudioEngine] = None, max_batch: Optional[Dict[str, int]] = None):
        # engine_for ties the engine's lifetime to the model's: keep the model alive as long as the defender
        self.model = model if isinstance(model, nn.Module) else None
        self.engine = engine_for(model) if isinstance(model, nn.Module) else model
        self.device = self.engine.device
        self.audio = audio if audio is not None else AudioEngine(device=self.device)
        if self.audio.device != self.device:
            raise AvcError(f"audio engine on {self.audio.device}, model on {self.device}")
        self.n_mels = self.audio.n_mels
        if self.n_mels != self.engine.c_in:
            raise ValueError(f"the audio front-end makes {self.n_mels}-bin mels, the model takes {self.engine.c_in}")
        self.mean = self._stat(attr_mean, "attr_mean")
        self.std = self._stat(attr_std, "attr_std")
        if not bool((self.std > 0).all()):
            raise ValueError("attr_std must be > 0 in every bin")
        self.max_batch = dict(DEFAULT_MAX_BATCH)
        self.max_batch.update(max_batch or {})
        for k in KINDS:
            if int(self.max_batch[k]) < 1:
                raise ValueError(f"max_batch[{k!r}] must be >= 1")
        self._events: Optional[_StageEvents] = None

    def _stat(self, x, name: str) -> Tensor:
        t = torch.as_tensor(x, dtype=torch.float32).to(self.device).reshape(-1).contiguous()
        if t.numel() != self.n_mels:
            raise ValueError(f"{name} must have {self.n_mels} entries (got {t.numel()})")
        if not bool(torch.isfinite(t).all()):
            raise ValueError(f"{name} must be finite")
        return t

    # ---- validation (everything raises before the first launch) -----------------------------------------------------
    def _wav(self, w, name: str) -> Tensor:
        if not isinstance(w, Tensor):
            raise TypeError(f"{name} must be a torch.Tensor")
        if w.device != self.device:
            raise AvcError(f"{name} is on {w.device}; the defender runs on {self.device} (no CPU fallback)")
        if w.dtype != torch.float32 or w.dim() != 1:
            raise ValueError(f"{name} must be a 1-D float32 waveform (got {w.dtype} {tuple(w.shape)})")
        return w

    def _frames(self, w: Tensor, name: str, min_frames: int) -> int:
        n, hop, n_fft = int(w.numel()), self.audio.hop_length, self.audio.n_fft
        if n <= n_fft // 2:
            raise ValueError(f"{name}: {n} samples are too short for the front-end's reflect padding (need > {n_fft // 2})")
        F = 1 + n // hop
        if F < min_frames:
            raise ValueError(f"{name}: {n} samples give {F} frames; the attack needs at least {min_frames}")
        return F

    # ---- the two audio ends --------------------------------------------------------------------------------------
    def wav2mel(self, wavs: Sequence[Tensor]) -> List[Tensor]:
        """file2mel + normalize (data_utils.py:35-40, 99-114): [n_frames, 80] per waveform, one ragged call."""
        return self.audio.wav2mel_varlen([self._wav(w, f"wavs[{i}]") for i, w in enumerate(wavs)], mean=self.mean, std=self.std)

    def mel2wav(self, mels: Sequence[Tensor], n_iter: int = 100) -> List[Tensor]:
        """denormalize + mel2wav (data_utils.py:43-47, 149-164): one waveform per normalised mel, one ragged call."""
        if int(n_iter) < 0:
            raise ValueError("n_iter must be >= 0")
        return self.audio.mel2wav_varlen(mels, n_iter=int(n_iter), mean=self.mean, std=self.std)

    # ---- the defence ---------------------------------------------------------------------------------------------
    def defend(self, vc_tgt: Sequence[Tensor], adv_tgt: Tensor, attack_type: str = "emb", eps: float = 0.1, n_iters: int = 1500,
               vc_src: Optional[Tensor] = None, griffin_lim_iters: int = 100, return_mels: bool = False):
        """attack.py on every waveform of ``vc_tgt`` (trimmed, on the device) against the one attack target ``adv_tgt``
        (and conversion source ``vc_src`` for e2e / fb).  Defaults as attack.py:95-113: emb attack, eps 0.1, 1500
        iterations; griffin_lim's 100 iterations (data_utils.py:173).  Returns the defended waveforms in input order, and
        with ``return_mels`` also the defended normalised mels ([n_frames, 80] each): ``(wavs, mels)``.

        Seeded like attack.py run on each file in turn: the initial noise of utterance i is drawn, in input order, exactly
        as attack_utils draws it for that utterance alone."""
        kind = attack_type
        if kind not in KINDS:
            raise ValueError(f"attack_type must be one of {KINDS} (got {kind!r})")
        if int(n_iters) < 0 or int(griffin_lim_iters) < 0:
            raise ValueError("n_iters and griffin_lim_iters must be >= 0")
        if kind != "emb" and vc_src is None:
            raise ValueError("vc_src is required for the e2e and fb attacks")
        tgts = [self._wav(w, f"vc_tgt[{i}]") for i, w in enumerate(vc_tgt)]
        if not tgts:
            return ([], []) if return_mels else []
        adv = self._wav(adv_tgt, "adv_tgt")
        src = self._wav(vc_src, "vc_src") if kind != "emb" else None
        spk_min = self.engine.min_frames("speaker")
        back_min = 2 + self.audio.n_fft // 2 // self.audio.hop_length        # hop (F - 1) > n_fft / 2 for the back-end
        frames = [self._frames(w, f"vc_tgt[{i}]", max(spk_min, back_min)) for i, w in enumerate(tgts)]
        self._frames(adv, "adv_tgt", spk_min)
        T_src = self._frames(src, "vc_src", self.engine.min_frames("content")) if src is not None else 0

        ev = _StageEvents(self.device)
        self._events = ev
        ev.record(0)
        # 1. front-end: the targets in chunk order, so that every chunk's mels are one contiguous [B_g, T, 80] block
        chunks = plan_chunks(frames, int(self.max_batch[kind]))
        order = [i for _, idx in chunks for i in idx]
        extra = [adv] + ([src] if src is not None else [])
        mels = self.wav2mel([tgts[i] for i in order] + extra)
        adv_mel = mels[len(order)]
        src_mel = mels[len(order) + 1] if src is not None else None
        ev.record(1)
        # 2. attacks
        where = {i: p for p, i in enumerate(order)}
        w0 = self.draw_w0([mels[where[i]] for i in range(len(tgts))])
        inv = utterance_inv_norm(kind, self.engine.c_emb, self.n_mels, self.engine.decoder_frames(T_src) if kind == "e2e" else 0)
        out: List[Optional[Tensor]] = [None] * len(tgts)
        pos = 0
        for T, idx in chunks:
            out_chunk = self._attack_chunk(kind, mels[pos:pos + len(idx)], [w0[i] for i in idx], adv_mel, src_mel, eps,
                                           int(n_iters), inv)
            for k, i in enumerate(idx):
                out[i] = out_chunk[k]
            pos += len(idx)
        ev.record(2)
        # 3. back-end, input order
        wavs = self.mel2wav(out, n_iter=int(griffin_lim_iters))  # type: ignore[arg-type]
        ev.record(3)
        return (wavs, out) if return_mels else wavs

    @staticmethod
    def draw_w0(mels: Sequence[Tensor]) -> List[Tensor]:
        """attack_utils' ``torch.zeros_like(vc_tgt).normal_(0, 1)`` on each utterance's [1, 80, T] view (attack.py:49-50),
        one utterance at a time, in the given order."""
        return [torch.zeros_like(m.t().unsqueeze(0)).normal_(0, 1) for m in mels]

    def _attack_chunk(self, kind: str, mels: Sequence[Tensor], w0: Sequence[Tensor], adv_mel: Tensor, src_mel: Optional[Tensor],
                      eps: float, n_iters: int, inv_norm: float) -> List[Tensor]:
        """One Engine.attack over equal-length utterances whose [T, 80] mels lie end to end in one buffer -> the defended
        [T, 80] mels (views of the attack's output, which keeps the input's time-major strides)."""
        B, T = len(mels), int(mels[0].shape[0])
        first = mels[0]
        blk = first.as_strided((B, self.n_mels, T), (T * self.n_mels, 1, self.n_mels))      # [B, 80, T] view, no copy
        for k, m in enumerate(mels):
            if m.data_ptr() != first.data_ptr() + k * T * self.n_mels * first.element_size():
                raise AvcError("internal: chunk mels are not contiguous")
        w = torch.empty_like(blk)
        for k, wk in enumerate(w0):
            w[k].copy_(wk[0])
        at = adv_mel.t().unsqueeze(0).expand(B, -1, -1)            # batch stride 0: the attack reads strides
        vs = src_mel.t().unsqueeze(0).expand(B, -1, -1) if src_mel is not None else None
        res = self.engine.attack(kind, blk, at, eps, n_iters, vc_src=vs, w0=w, inv_norm=inv_norm)
        return [res[k].t() for k in range(B)]

    @property
    def last_stage_ms(self) -> Dict[str, float]:
        """CUDA-event times of the last ``defend``: front-end, attacks, back-end (ms)."""
        return self._events.ms() if self._events is not None else {}

    @property
    def kernel_launches(self) -> int:
        return self.engine.kernel_launches + self.audio.kernel_launches


class _StageEvents:
    """CUDA events at the four stage boundaries of ``defend`` on the device's current stream (none off the GPU)."""

    NAMES = ("front_end", "attacks", "back_end")

    def __init__(self, device: torch.device):
        self.ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if device.type == "cuda" else None
        self.device = device

    def record(self, i: int) -> None:
        if self.ev is not None:
            self.ev[i].record(torch.cuda.current_stream(self.device))

    def ms(self) -> Dict[str, float]:
        if self.ev is None:
            return {}
        self.ev[3].synchronize()
        return {n: self.ev[i].elapsed_time(self.ev[i + 1]) for i, n in enumerate(self.NAMES)}
