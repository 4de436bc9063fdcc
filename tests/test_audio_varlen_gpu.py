"""Ragged batches of the mel front-end / Griffin-Lim back-end (avc_audio_wav2mel_varlen / avc_audio_mel2wav_varlen): one call
for utterances of any lengths equals the equal-length calls on each utterance alone, and the fused speaker normalisation
equals the unfused fp32 formula bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

LENS = [1025, 300 * 60 + 11, 7001, 24000, 300 * 33]          # 1025: one sample above the n_fft / 2 reflect-padding minimum


def tone(n, seed, sr=24000):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / sr
    w = 0.3 * np.sin(2 * np.pi * 220 * t) + 0.15 * np.sin(2 * np.pi * 1333 * t + 0.3) + 0.05 * np.sin(2 * np.pi * 5100 * t) + 0.02 * rng.standard_normal(n)
    return (w * np.hanning(n) ** 0.25).astype(np.float32)


def stats(seed=0):
    g = torch.Generator().manual_seed(seed)
    return (0.3 + 0.3 * torch.rand(80, generator=g)).cuda(), (0.1 + 0.2 * torch.rand(80, generator=g)).cuda()


@pytest.fixture(scope="module")
def audio():
    from attack_vc_b200.audio import AudioEngine
    return AudioEngine()


@pytest.fixture(scope="module")
def wavs():
    return [torch.from_numpy(tone(n, i)).cuda() for i, n in enumerate(LENS)]


def test_wav2mel_varlen_equals_single_calls(audio, wavs):
    """Rows are independent, so each utterance's mel equals the equal-length call on it alone.  The GEMM may split K
    differently for a different row count (chunked fp32 sums in another order): at most 1e-6 then."""
    l0 = audio.kernel_launches
    mels = audio.wav2mel_varlen(wavs)
    launches = audio.kernel_launches - l0
    identical = 0
    for w, m in zip(wavs, mels):
        one = audio.wav2mel(w)
        assert m.shape == one.shape == (1 + w.numel() // 300, 80)
        err = float((m - one).abs().max())
        assert err <= 1e-6, err
        identical += int(torch.equal(m, one))
    print(f"wav2mel_varlen: {identical} of {len(wavs)} utterances bit-identical to the single call; {launches} launches")
    l0 = audio.kernel_launches
    audio.wav2mel_varlen(wavs[:1])
    assert audio.kernel_launches - l0 == launches                  # one call whatever the number of lengths


def test_wav2mel_varlen_vs_oracle(audio, wavs):
    from oracle import audio_oracle as A
    for w, m in zip(wavs, audio.wav2mel_varlen(wavs)):
        ref = A.wav2mel(w.cpu().numpy().astype(np.float64))
        err = np.abs(m.cpu().numpy().astype(np.float64) - ref)
        assert err.max() < 1e-4 and err.mean() < 1e-5, (err.max(), err.mean())     # test_audio_gpu.py::test_wav2mel


@pytest.mark.parametrize("n_iter", [0, 3])
def test_mel2wav_varlen_equals_single_calls(audio, n_iter):
    from oracle import audio_oracle as A
    mels = [torch.from_numpy(A.wav2mel(tone(n, 20 + i).astype(np.float64))).cuda() for i, n in enumerate([300 * 120, 1500, 300 * 47 + 5])]
    out = audio.mel2wav_varlen(mels, n_iter=n_iter)
    tol_max, tol_l2 = (2e-3, 5e-4) if n_iter == 0 else (5e-2, 2e-2)   # test_audio_gpu.py::test_mel2wav_few_iterations
    for m, w in zip(mels, out):
        one = audio.mel2wav(m, n_iter=n_iter).double()
        assert w.shape == one.shape == (300 * (m.shape[0] - 1),)
        d = (w.double() - one).abs()
        assert float(d.max()) < tol_max * float(one.abs().max())
        assert float(d.norm()) < tol_l2 * float(one.norm())


def test_normalisation_bit_exact(audio, wavs):
    mean, std = stats()
    raw = audio.wav2mel_varlen(wavs)
    normed = audio.wav2mel_varlen(wavs, mean=mean, std=std)
    for r, x in zip(raw, normed):
        assert torch.equal(x, (r - mean) / std)                     # two correctly rounded fp32 ops, unfused
    mels = [x[: x.shape[0] // 2 + 5].contiguous() for x in normed[1:]]            # other frame counts, >= 5 each
    a = audio.mel2wav_varlen(mels, n_iter=2, mean=mean, std=std)
    b = audio.mel2wav_varlen([x * std + mean for x in mels], n_iter=2)
    for wa, wb in zip(a, b):
        assert torch.equal(wa, wb)


def test_varlen_errors(audio, wavs):
    from attack_vc_b200 import AvcError
    with pytest.raises(ValueError, match="too short"):
        audio.wav2mel_varlen([wavs[1], torch.zeros(1024, device="cuda"), wavs[2]])
    m = audio.wav2mel_varlen(wavs[1:3])
    with pytest.raises(ValueError):
        audio.mel2wav_varlen([m[0], torch.zeros(4, 80, device="cuda"), m[1]], n_iter=0)   # 900 samples: too short for GL
    with pytest.raises(ValueError):
        audio.mel2wav_varlen([m[0], torch.zeros(1, 80, device="cuda")], n_iter=0)
    with pytest.raises(ValueError):
        audio.wav2mel_varlen(wavs[:2], mean=torch.zeros(80, device="cuda"))                 # std missing
    with pytest.raises(AvcError):
        audio.wav2mel_varlen([wavs[0].cpu()])
    lib, h = audio._lib, audio._h
    n = (C.c_int64 * 2)(24000, 24000)
    f = (C.c_int32 * 2)(50, 50)
    buf = torch.zeros(2 * 24000, device="cuda")
    out = torch.zeros(200 * 80, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p, q = buf.data_ptr(), out.data_ptr()
    assert lib.avc_audio_wav2mel_varlen(h, None, n, 2, None, None, q, st) == -1
    assert lib.avc_audio_wav2mel_varlen(h, p, n, 2, None, None, None, st) == -1
    assert lib.avc_audio_wav2mel_varlen(h, p, None, 2, None, None, q, st) == -1
    assert lib.avc_audio_wav2mel_varlen(h, p, n, 0, None, None, q, st) == -1
    assert lib.avc_audio_wav2mel_varlen(h, p, n, 2, q, None, q, st) == -1                  # mean without std
    assert lib.avc_audio_mel2wav_varlen(h, None, f, 2, 0, None, None, p, st) == -1
    assert lib.avc_audio_mel2wav_varlen(h, q, f, 2, 0, None, None, None, st) == -1
    assert lib.avc_audio_mel2wav_varlen(h, q, None, 2, 0, None, None, p, st) == -1
    assert lib.avc_audio_mel2wav_varlen(h, q, f, 0, 0, None, None, p, st) == -1
    assert lib.avc_audio_mel2wav_varlen(h, q, f, 2, -1, None, None, p, st) == -1
    assert b"bad batch" in lib.avc_audio_last_error(h) or b"n_iter" in lib.avc_audio_last_error(h)
