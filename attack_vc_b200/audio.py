"""Host-side mirror of the reference's mel front-end / Griffin-Lim back-end (``data_utils.py:65-197``) on top of the C-ABI
(``avc_audio_*`` in include/avc_b200.h).  ``librosa.load`` / ``librosa.effects.trim`` (file I/O and silence trimming,
data_utils.py:93-96) stay with the caller; everything from the trimmed waveform to the normalised mel and back runs on the
GPU.  PyTorch supplies device memory and the stream only; there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from .engine import AvcError


def group_by_length(lengths: Sequence[int]) -> List[Tuple[int, List[int]]]:
    """Indices of equal-length items, in order of first appearance: [(length, [i, j, ...]), ...].  Utterances of one length
    form ONE batched call (the frames of the whole group are the rows of one GEMM per transform); ragged inputs therefore cost
    one call per distinct length, not one per utterance."""
    groups: Dict[int, List[int]] = {}
    for i, n in enumerate(lengths):
        groups.setdefault(int(n), []).append(i)
    return list(groups.items())


class AudioEngine:
    """One ``avc_audio_handle``: the preprocessing constants of ``config["preprocess"]`` (data_utils.py:214-220; the
    reference passes them as ``**config["preprocess"]`` to file2mel / mel2wav)."""

    def __init__(self, sample_rate: int = 24000, preemph: float = 0.97, n_fft: int = 2048, hop_length: int = 300,
                 win_length: int = 1200, n_mels: int = 80, ref_db: float = 20.0, max_db: float = 100.0,
                 top_db: Optional[float] = None, device: Optional[torch.device] = None):
        self._lib = _lib.load()
        if not torch.cuda.is_available():
            raise AvcError("attack_vc_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        device = torch.device("cuda" if device is None else device)
        if device.type != "cuda":
            raise AvcError("attack_vc_b200 runs on CUDA only; there is no CPU fallback")
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        self.n_mels, self.hop_length, self.n_fft = int(n_mels), int(hop_length), int(n_fft)
        self.top_db = top_db          # used by librosa.effects.trim on the host, kept for signature compatibility
        d = _lib.AudioDesc(int(sample_rate), int(n_fft), int(hop_length), int(win_length), int(n_mels), float(preemph), float(ref_db), float(max_db))
        h = C.c_void_p()
        rc = self._lib.avc_audio_create(C.byref(h), C.byref(d), self.device.index)
        if rc != 0:
            msg = self._lib.avc_audio_last_error(None).decode()
            raise (ValueError if rc == -1 else AvcError)(f"avc_audio_create failed ({rc}): {msg}")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.avc_audio_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            msg = self._lib.avc_audio_last_error(self._h).decode()
            raise (ValueError if rc == -1 else AvcError)(f"libavc_b200: {msg}")

    def _vec(self, x: Tensor, name: str, dim: int) -> Tensor:
        if not isinstance(x, Tensor) or x.device != self.device:
            raise AvcError(f"{name} must be a tensor on {self.device} (no CPU fallback)")
        if x.dtype != torch.float32 or x.dim() != dim:
            raise ValueError(f"{name} must be float32 with {dim} dimension(s) (got {x.dtype} {tuple(x.shape)})")
        return x.contiguous()

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.avc_audio_kernel_launches(self._h))

    def wav2mel(self, wav: Tensor) -> Tensor:
        """file2mel from the trimmed waveform on (data_utils.py:99-114): wav [n] -> mel [n_frames, n_mels];
        a batch of equal-length waveforms [B, n] -> [B, n_frames, n_mels] (one GEMM over all frames)."""
        batched = isinstance(wav, Tensor) and wav.dim() == 2
        wav = self._vec(wav, "wav", 2 if batched else 1)
        B, n = (int(wav.shape[0]), int(wav.shape[1])) if batched else (1, int(wav.numel()))
        F = int(self._lib.avc_audio_frames(self._h, n))
        with torch.cuda.device(self.device):
            mel = torch.empty(B, max(F, 0), self.n_mels, device=self.device, dtype=torch.float32)
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            self._check(self._lib.avc_audio_wav2mel_batch(self._h, wav.data_ptr(), B, n, mel.data_ptr(), st))
        return mel if batched else mel[0]

    def mel2wav(self, mel: Tensor, n_iter: int = 100) -> Tensor:
        """mel2wav (data_utils.py:120-165): mel [n_frames, n_mels] -> waveform [hop_length * (n_frames - 1)]."""
        batched = isinstance(mel, Tensor) and mel.dim() == 3          # [B, n_frames, n_mels]: equal-length utterances
        mel = self._vec(mel, "mel", 3 if batched else 2)
        if mel.shape[-1] != self.n_mels:
            raise ValueError(f"mel must have {self.n_mels} bins (got {mel.shape[-1]})")
        B, F = (int(mel.shape[0]), int(mel.shape[1])) if batched else (1, int(mel.shape[0]))
        n = int(self._lib.avc_audio_samples(self._h, F))
        with torch.cuda.device(self.device):
            wav = torch.empty(B, max(n, 0), device=self.device, dtype=torch.float32)
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            self._check(self._lib.avc_audio_mel2wav_batch(self._h, mel.data_ptr(), B, F, int(n_iter), wav.data_ptr(), st))
        return wav if batched else wav[0]

    def _norm_args(self, mean: Optional[Tensor], std: Optional[Tensor]) -> Tuple[Optional[int], Optional[int], tuple]:
        """Device pointers of the speaker-normalisation statistics (both or neither), plus the tensors to keep alive."""
        if (mean is None) != (std is None):
            raise ValueError("mean and std must be given together")
        if mean is None:
            return None, None, ()
        mean, std = self._vec(mean, "mean", 1), self._vec(std, "std", 1)
        if mean.numel() != self.n_mels or std.numel() != self.n_mels:
            raise ValueError(f"mean and std must have {self.n_mels} entries (got {mean.numel()}, {std.numel()})")
        return mean.data_ptr(), std.data_ptr(), (mean, std)

    def wav2mel_varlen(self, wavs: Sequence[Tensor], mean: Optional[Tensor] = None, std: Optional[Tensor] = None) -> List[Tensor]:
        """file2mel over utterances of ANY lengths in ONE call (avc_audio_wav2mel_varlen): the frames of all utterances are the
        rows of one GEMM.  With ``mean`` / ``std`` ([n_mels]) the mels come out speaker-normalised, ``(mel - mean) / std``
        (data_utils.py:35-40).  Returns [n_frames_u, n_mels] views of one buffer, in input order."""
        if len(wavs) == 0:
            return []
        flat = [self._vec(w, "wav", 1) for w in wavs]
        ns = [int(w.numel()) for w in flat]
        frames = [int(self._lib.avc_audio_frames(self._h, n)) for n in ns]
        m, s, keep = self._norm_args(mean, std)
        with torch.cuda.device(self.device):
            wav = torch.cat(flat) if len(flat) > 1 else flat[0]
            mel = torch.empty(max(sum(max(f, 0) for f in frames), 1), self.n_mels, device=self.device, dtype=torch.float32)
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            n_host = (C.c_int64 * len(ns))(*ns)
            self._check(self._lib.avc_audio_wav2mel_varlen(self._h, wav.data_ptr(), n_host, len(ns), m, s, mel.data_ptr(), st))
        del keep
        return list(mel.split(frames))

    def mel2wav_varlen(self, mels: Sequence[Tensor], n_iter: int = 100, mean: Optional[Tensor] = None,
                       std: Optional[Tensor] = None) -> List[Tensor]:
        """mel2wav over mels of ANY frame counts in ONE call (avc_audio_mel2wav_varlen; one Griffin-Lim loop for all of them).
        With ``mean`` / ``std`` the inputs are speaker-normalised mels, denormalised first (``x * std + mean``,
        data_utils.py:43-47).  Returns [hop_length * (n_frames_u - 1)] views of one buffer, in input order."""
        if len(mels) == 0:
            return []
        flat = [self._vec(x, "mel", 2) for x in mels]
        for x in flat:
            if x.shape[-1] != self.n_mels:
                raise ValueError(f"mel must have {self.n_mels} bins (got {x.shape[-1]})")
        frames = [int(x.shape[0]) for x in flat]
        ns = [int(self._lib.avc_audio_samples(self._h, f)) for f in frames]
        m, s, keep = self._norm_args(mean, std)
        with torch.cuda.device(self.device):
            mel = torch.cat(flat) if len(flat) > 1 else flat[0]
            wav = torch.empty(max(sum(max(n, 0) for n in ns), 1), device=self.device, dtype=torch.float32)
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            f_host = (C.c_int32 * len(frames))(*frames)
            self._check(self._lib.avc_audio_mel2wav_varlen(self._h, mel.data_ptr(), f_host, len(frames), int(n_iter), m, s,
                                                           wav.data_ptr(), st))
        del keep
        return list(wav.split(ns))

    def wav2mel_list(self, wavs: Sequence[Tensor]) -> List[Tensor]:
        """file2mel over utterances of ANY lengths (the reference loops over files, data_utils.py:65-117): equal-length
        waveforms are batched into one call each, results come back in input order."""
        out: List[Optional[Tensor]] = [None] * len(wavs)
        for _, idx in group_by_length([int(w.numel()) for w in wavs]):
            mel = self.wav2mel(torch.stack([self._vec(wavs[i], "wav", 1) for i in idx]))
            for k, i in enumerate(idx):
                out[i] = mel[k]
        return out  # type: ignore[return-value]

    def mel2wav_list(self, mels: Sequence[Tensor], n_iter: int = 100) -> List[Tensor]:
        """mel2wav over mels of ANY frame counts: one batched Griffin-Lim per distinct length, input order kept."""
        out: List[Optional[Tensor]] = [None] * len(mels)
        for _, idx in group_by_length([int(m.shape[0]) for m in mels]):
            wav = self.mel2wav(torch.stack([self._vec(mels[i], "mel", 2) for i in idx]), n_iter=n_iter)
            for k, i in enumerate(idx):
                out[i] = wav[k]
        return out  # type: ignore[return-value]
