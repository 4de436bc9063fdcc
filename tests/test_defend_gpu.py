"""Defender.defend (attack_vc_b200/defend.py) on the GPU: waveform -> normalised mel -> attack -> waveform for a list of
utterances equals attack.py's flow run on each utterance alone (hand-composed from the library's calls and attack_utils),
and the oracle end to end."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HOP = 300


def tone(n, seed, sr=24000):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / sr
    w = 0.3 * np.sin(2 * np.pi * 220 * t) + 0.15 * np.sin(2 * np.pi * 1333 * t + 0.3) + 0.05 * np.sin(2 * np.pi * 5100 * t) + 0.02 * rng.standard_normal(n)
    return (w * np.hanning(n) ** 0.25).astype(np.float32)


def wav(frames, seed, extra=0):
    return torch.from_numpy(tone(HOP * (frames - 1) + extra, seed)).cuda()


def stats():
    g = torch.Generator().manual_seed(0)
    return 0.3 + 0.3 * torch.rand(80, generator=g), 0.1 + 0.2 * torch.rand(80, generator=g)


@pytest.fixture(scope="module")
def defender(gpu_model):
    from attack_vc_b200 import Defender
    mean, std = stats()
    return Defender(gpu_model, mean, std)


def solo_chain(defender, gpu_model, kind, wavs, adv, src, n_iters, seed):
    """attack.py's flow composed by hand from library calls: front-end, attack_utils.<kind>_attack on each utterance's
    [1, 80, T] view in input order under one seed, back-end."""
    import attack_utils
    front = defender.wav2mel(list(wavs) + [adv] + ([src] if src is not None else []))
    at = front[len(wavs)].t().unsqueeze(0)
    vs = front[len(wavs) + 1].t().unsqueeze(0) if src is not None else None
    torch.manual_seed(seed)
    mels = []
    for m in front[:len(wavs)]:
        x = m.t().unsqueeze(0)                                          # strides (80 T, 1, 80), as attack.py:49-50
        if kind == "emb":
            r = attack_utils.emb_attack(gpu_model, x, at, 0.1, n_iters)
        elif kind == "e2e":
            r = attack_utils.e2e_attack(gpu_model, vs, x, at, 0.1, n_iters)
        else:
            r = attack_utils.fb_attack(gpu_model, vs, x, at, 0.1, n_iters)
        mels.append(r[0].t().contiguous())
    return front, mels


def wave_close(got, want, tol_max=2e-3, tol_l2=5e-4):
    """test_audio_gpu.py's tolerances for 0 Griffin-Lim iterations, relative to the peak / the norm."""
    d = (got.double() - want.double())
    assert got.shape == want.shape
    assert float(d.abs().max()) < tol_max * float(want.abs().max())
    assert float(d.norm()) < tol_l2 * float(want.double().norm())


@pytest.mark.parametrize("kind", ["emb", "e2e", "fb"])
def test_defend_equals_composed_chain(defender, gpu_model, kind):
    """3 utterances of 100 frames (one batched attack call, CUDA-core path) == batch-1 runs with the per-utterance
    normaliser; DESIGN "sharded batch equals unsharded": <= 5e-6.  The batch-mean normaliser does NOT reproduce them."""
    wavs = [wav(100, 10 + i, extra=17 * i) for i in range(3)]
    adv, src = wav(80, 30), wav(90, 31) if kind != "emb" else None
    torch.manual_seed(123)
    out, mels = defender.defend(wavs, adv, attack_type=kind, eps=0.1, n_iters=5, vc_src=src, griffin_lim_iters=0, return_mels=True)
    front, solo = solo_chain(defender, gpu_model, kind, wavs, adv, src, 5, 123)
    err = max(float((m - s).abs().max()) for m, s in zip(mels, solo))
    assert err <= 5e-6, err
    for w, s in zip(out, defender.mel2wav(solo, n_iter=0)):
        wave_close(w, s)
    # negative control: the same batch under nn.MSELoss's batch mean (inv_norm=None: 1 / (B D)) takes another trajectory
    torch.manual_seed(123)
    w0 = torch.stack([torch.zeros_like(m.t().unsqueeze(0)).normal_(0, 1)[0] for m in front[:3]])
    blk = torch.stack([m for m in front[:3]]).transpose(1, 2)
    at = front[3].t().unsqueeze(0).expand(3, -1, -1)
    vs = front[4].t().unsqueeze(0).expand(3, -1, -1) if src is not None else None
    wrong = defender.engine.attack(kind, blk, at, 0.1, 5, vc_src=vs, w0=w0)
    err_wrong = max(float((wrong[k].t() - solo[k]).abs().max()) for k in range(3))
    assert err_wrong > 20 * max(err, 1e-7), (err, err_wrong)


def test_defend_ragged_order_and_chunks(gpu_model):
    """3 distinct lengths out of order, max_batch 2: four attack calls, ONE back-end call, input order kept, each
    utterance equal to its batch-1 run."""
    from attack_vc_b200 import Defender
    mean, std = stats()
    d = Defender(gpu_model, mean, std, max_batch={"emb": 2})
    frames = [60, 45, 60, 80, 60]
    wavs = [wav(f, 40 + i) for i, f in enumerate(frames)]
    adv = wav(70, 50)
    back_calls = []
    inner = d.audio.mel2wav_varlen

    def counting(mels, **kw):
        back_calls.append([int(m.shape[0]) for m in mels])
        return inner(mels, **kw)
    d.audio.mel2wav_varlen = counting
    try:
        torch.manual_seed(7)
        out, mels = d.defend(wavs, adv, n_iters=4, griffin_lim_iters=2, return_mels=True)
    finally:
        del d.audio.mel2wav_varlen
    assert back_calls == [frames]
    _, solo = solo_chain(d, gpu_model, "emb", wavs, adv, None, 4, 7)
    for f, w, m, s in zip(frames, out, mels, solo):
        assert m.shape == (f, 80) and w.shape == (HOP * (f - 1),)
        assert float((m - s).abs().max()) <= 5e-6


def test_defend_tensor_core_batch(defender, gpu_model):
    """16 x 128 frames = 2048 GEMM rows: the attack runs on the tcgen05 plan, the solo runs on the batch-1 CUDA-core plan.
    Criteria of tests/test_attacks_gpu.py for batched tensor-core results: Adam at |g| ~ 1e-7 normalises the step, so an
    element whose gradient sits near zero may move by a whole lr-sized step the other way (eps * tanh' * 2 lr per
    iteration); everything else agrees to fp32 noise."""
    n = 3
    wavs = [wav(128, 60 + i) for i in range(16)]
    adv = wav(100, 80)
    torch.manual_seed(11)
    _, mels = defender.defend(wavs, adv, n_iters=n, griffin_lim_iters=0, return_mels=True)
    _, solo = solo_chain(defender, gpu_model, "emb", wavs, adv, None, n, 11)
    err = torch.stack([(m - s).abs() for m, s in zip(mels, solo)])
    assert float(err.median()) < 1e-6
    assert float((err > 1e-4).float().mean()) < 0.02
    assert float(err.max()) <= 2e-3 * n + 1e-6


def test_defend_vs_oracle(defender, cpu_model):
    """audio oracle -> normalize -> adainvc_oracle emb attack -> denormalize -> Griffin-Lim with 0 iterations.  Composed
    tolerances: the front-end is within 1e-4 (max) / 1e-5 (mean) of the fp64 oracle on the mel (test_audio_gpu.py), i.e.
    that over std after normalisation; the attack adds the batched-attack criteria above; the back-end with 0 iterations is
    linear in the magnitude 10^(5 mel): a mel error e (denormalised) moves it by ln(10) 5 e relative, on top of
    test_audio_gpu.py's 2e-3 (max) / 5e-4 (l2)."""
    from oracle import adainvc_oracle as O
    import norm_oracle as N
    from oracle import audio_oracle as A
    n = 3
    x, adv = wav(100, 90), wav(85, 91)
    torch.manual_seed(21)
    out, mels = defender.defend([x], adv, n_iters=n, griffin_lim_iters=0, return_mels=True)
    torch.manual_seed(21)
    w0 = torch.zeros_like(mels[0].t().unsqueeze(0)).normal_(0, 1).cpu()
    mean, std = (t.numpy() for t in stats())
    ref_x = N.normalize(A.wav2mel(x.cpu().numpy().astype(np.float64)), mean, std).astype(np.float32)
    ref_a = N.normalize(A.wav2mel(adv.cpu().numpy().astype(np.float64)), mean, std).astype(np.float32)
    o = O.run_attack("emb", cpu_model, torch.from_numpy(ref_x.T.copy())[None], torch.from_numpy(ref_a.T.copy())[None], 0.1, n, w0)
    ref_mel = o["adv"][0].t().numpy()
    err = np.abs(mels[0].cpu().numpy() - ref_mel)
    smin = float(std.min())
    assert np.median(err) < 1e-5 / smin + 1e-6, np.median(err)
    assert (err > 1e-4 / smin + 1e-5).mean() < 0.02
    assert err.max() <= 1e-4 / smin + 0.1 * 2e-3 * n + 1e-6, err.max()
    ref_wav = torch.from_numpy(A.mel2wav(N.denormalize(ref_mel, mean, std), n_iter=0))
    e = err * std                                                       # the same error in denormalised mel units
    k = np.log(10.0) * 5.0
    wave_close(out[0].cpu(), ref_wav, tol_max=2e-3 + k * float(e.max()), tol_l2=5e-4 + k * float(np.sqrt((e ** 2).mean())))


def test_defend_validation_before_launch(defender):
    from attack_vc_b200 import AvcError, Defender
    ok, adv = wav(60, 1), wav(60, 2)
    n0 = defender.kernel_launches
    with pytest.raises(AvcError):
        defender.defend([ok.cpu()], adv)                                # no CPU fallback
    with pytest.raises(AvcError):
        defender.defend([ok], adv.cpu())
    with pytest.raises(ValueError):
        defender.defend([ok.double()], adv)
    with pytest.raises(ValueError):
        defender.defend([ok], adv, attack_type="e2e")                   # vc_src required
    with pytest.raises(ValueError):
        defender.defend([ok], adv, attack_type="fb")
    with pytest.raises(ValueError):
        defender.defend([ok, torch.zeros(1024, device="cuda")], adv)    # too short for the front-end
    with pytest.raises(ValueError):
        defender.defend([ok, torch.zeros(HOP * 5, device="cuda")], adv)  # 6 frames: fewer than the speaker encoder takes
    with pytest.raises(ValueError):
        defender.defend([ok], adv, attack_type="e2e", vc_src=torch.zeros(HOP * 5, device="cuda"))
    with pytest.raises(ValueError):
        defender.defend([ok], adv, n_iters=-1)
    assert defender.kernel_launches == n0
    for mean, std in ((torch.zeros(79), torch.ones(80)), (torch.zeros(80), torch.zeros(80)),
                      (torch.full((80,), float("inf")), torch.ones(80))):
        with pytest.raises(ValueError):
            Defender(defender.engine, mean, std, audio=defender.audio)


def test_defender_keeps_its_model_alive():
    """engine_for closes a model's engine when the model is collected: a Defender built from a temporary model must keep
    it (and so its engine) alive."""
    import gc
    from attack_vc_b200 import Defender
    from attack_vc_b200.synthetic import SYNTH_CONFIG, ParamTree
    mean, std = stats()
    d = Defender(ParamTree(SYNTH_CONFIG, seed=0).to("cuda"), mean, std)
    gc.collect()
    out = d.defend([wav(40, 3)], wav(40, 4), n_iters=2, griffin_lim_iters=0)
    assert out[0].shape == (HOP * 39,) and bool(torch.isfinite(out[0]).all())
