"""Engine.attack_varlen (avc_attack_varlen) on the GPU: one ragged attack over utterances of different lengths equals
one Engine.attack per length group bit for bit when both run on the same tensor-core kernel, agrees with the CPU
oracle under the default routing, is served from the plan cache by exact length vector, validates before any launch,
and Defender.defend(..., mixed_lengths=True) equals the grouped defence."""
import pytest
import torch

pytestmark = pytest.mark.gpu

LENS = [160, 97, 160, 131, 97, 64]          # odd lengths at every sub-sampled level: partial pool windows, shifted edges
EPS, N_IT = 0.1, 4


def make_engine(gpu_model, monkeypatch, impl):
    from attack_vc_b200 import Engine
    monkeypatch.setenv("AVC_CONV_IMPL", str(impl))                      # read when the handle is created
    eng = Engine(gpu_model)
    monkeypatch.delenv("AVC_CONV_IMPL")
    return eng


def inputs(kind, lens, seed, T_adv=120, T_src=96):
    g = torch.Generator().manual_seed(seed)
    mels = [(torch.rand(T, 80, generator=g) * 2 - 1).cuda() for T in lens]
    w0 = [torch.randn(T, 80, generator=g).cuda() for T in lens]
    adv = (torch.rand(1, 80, T_adv, generator=g) * 2 - 1).cuda()
    src = (torch.rand(1, 80, T_src, generator=g) * 2 - 1).cuda() if kind != "emb" else None
    return mels, w0, adv, src


def inv_norm(eng, kind, T_src=96):
    return 1.0 / 128 if kind in ("emb", "fb") else 1.0 / (80 * eng.decoder_frames(T_src))


def grouped(eng, kind, mels, w0, adv, src, inv):
    """one Engine.attack per length group, outputs in input order; loss curves summed"""
    outs, grads, loss = [None] * len(mels), [None] * len(mels), 0.0
    for T in dict.fromkeys(int(m.shape[0]) for m in mels):
        idx = [i for i, m in enumerate(mels) if m.shape[0] == T]
        x = torch.stack([mels[i].t() for i in idx])
        w = torch.stack([w0[i].t() for i in idx])
        B = len(idx)
        vs = src.expand(B, -1, -1) if src is not None else None
        out, info = eng.attack(kind, x, adv.expand(B, -1, -1), EPS, N_IT, vc_src=vs, w0=w, inv_norm=inv, want_loss=True, want_grad=True)
        for k, i in enumerate(idx):
            outs[i], grads[i] = out[k].t(), info["grad"][k].t()
        loss = loss + info["losses"].double()
    return outs, grads, loss


def check_equal_to_grouped(eng, kind, lens, seed):
    mels, w0, adv, src = inputs(kind, lens, seed)
    inv = inv_norm(eng, kind)
    B = len(lens)
    vs = src.expand(B, -1, -1) if src is not None else None
    outs, info = eng.attack_varlen(kind, mels, adv.expand(B, -1, -1), EPS, N_IT, vc_src=vs, w0=w0, inv_norm=inv,
                                   want_loss=True, want_grad=True)
    ref, ref_g, ref_loss = grouped(eng, kind, mels, w0, adv, src, inv)
    for i in range(B):
        assert outs[i].shape == (lens[i], 80)
        assert torch.equal(outs[i], ref[i]), f"{kind} utterance {i} (T={lens[i]}): adv differs"
        assert torch.equal(info["grad"][i], ref_g[i]), f"{kind} utterance {i} (T={lens[i]}): grad differs"
    got = info["losses"].double()
    assert float(((got - ref_loss).abs() / ref_loss.abs()).max()) < 1e-6


@pytest.mark.parametrize("impl", [7, 6])
@pytest.mark.parametrize("kind", ["emb", "e2e", "fb"])
def test_varlen_bit_identical_to_grouped(gpu_model, monkeypatch, kind, impl):
    eng = make_engine(gpu_model, monkeypatch, impl)
    check_equal_to_grouped(eng, kind, LENS, seed=11)


def test_varlen_degenerate_cases(gpu_model, monkeypatch):
    eng = make_engine(gpu_model, monkeypatch, 7)
    Tmin = eng.min_frames("speaker")
    for lens in ([128, 128, 128], [113], [Tmin, 150, Tmin + 1]):
        check_equal_to_grouped(eng, "emb", lens, seed=len(lens))


def oracle_close(adv_gpu, o_adv):
    err = (adv_gpu.cpu() - o_adv).abs()
    assert float(err.median()) < 1e-6
    assert float((err > 1e-4).float().mean()) < 0.02
    assert float(err.max()) < 1e-3


@pytest.mark.parametrize("kind,B,lo,hi", [("emb", 512, 384, 640), ("e2e", 12, 80, 200), ("fb", 12, 80, 200)])
def test_varlen_default_routing_vs_oracle(engine, oracle, cpu_model, kind, B, lo, hi):
    g = torch.Generator().manual_seed(3)
    lens = [int(t) for t in torch.randint(lo, hi + 1, (B,), generator=g)]
    mels, w0, adv, src = inputs(kind, lens, seed=21)
    inv = inv_norm(engine, kind)
    vs = src.expand(B, -1, -1) if src is not None else None
    outs = engine.attack_varlen(kind, mels, adv.expand(B, -1, -1), EPS, 3, vc_src=vs, w0=w0, inv_norm=inv)
    for i in sorted(int(i) for i in torch.randperm(B, generator=g)[:4]):
        o = oracle.run_attack(kind, cpu_model, mels[i].t().unsqueeze(0).cpu(), adv.cpu(), EPS, 3, w0[i].t().unsqueeze(0).cpu(),
                              vc_src=src.cpu() if src is not None else None, inv_norm=inv)
        oracle_close(outs[i].t().unsqueeze(0), o["adv"])


def test_varlen_plan_cache_by_length_vector(engine):
    a, b = [150, 90, 120], [150, 120, 90]
    runs = []
    for lens in (a, b, a):
        mels, w0, adv, _ = inputs("emb", lens, seed=5)
        runs.append(engine.attack_varlen("emb", mels, adv.expand(3, -1, -1), EPS, N_IT, w0=w0))
    for x, y in zip(runs[0], runs[2]):
        assert torch.equal(x, y)


def test_varlen_validation_before_launch(gpu_model, engine, monkeypatch):
    from attack_vc_b200.engine import AvcError
    mels, w0, adv, _ = inputs("emb", [120, 100], seed=6)
    at = adv.expand(2, -1, -1)
    n0 = engine.kernel_launches
    short = torch.zeros(engine.min_frames("speaker") - 1, 80, device="cuda")
    with pytest.raises(ValueError, match="utterance 1 "):
        engine.attack_varlen("emb", [mels[0], short], at, EPS, 2, w0=[w0[0], short])
    with pytest.raises(ValueError):
        engine.attack_varlen("emb", mels, at, EPS, 2, w0=torch.cat(w0)[:-1])          # frames do not add up
    with pytest.raises(ValueError):
        engine.attack_varlen("emb", mels, at, EPS, 2, w0=[w0[1], w0[0]])              # lengths in the wrong order
    with pytest.raises(AvcError):
        engine.attack_varlen("emb", [mels[0].cpu(), mels[1]], at, EPS, 2, w0=w0)
    with pytest.raises(ValueError):
        engine.attack_varlen("emb", mels, adv.expand(3, -1, -1), EPS, 2, w0=w0)       # batch sizes differ
    assert engine.kernel_launches == n0
    simt = make_engine(gpu_model, monkeypatch, 1)
    n1 = simt.kernel_launches
    with pytest.raises(ValueError, match="ragged attacks run on the tensor-core kernels"):
        simt.attack_varlen("emb", mels, at, EPS, 2, w0=w0)
    assert simt.kernel_launches == n1


@pytest.mark.parametrize("kind", ["emb", "e2e", "fb"])
def test_defend_mixed_lengths_equals_grouped(gpu_model, monkeypatch, kind):
    from attack_vc_b200 import Defender
    from test_defend_gpu import stats, wav
    mean, std = stats()
    d_grouped = Defender(make_engine(gpu_model, monkeypatch, 7), mean, std, max_batch={kind: 2})
    d_mixed = Defender(make_engine(gpu_model, monkeypatch, 7), mean, std, max_batch={kind: 2})
    wavs = [wav(f, 40 + i) for i, f in enumerate([90, 130, 90, 111, 130])]
    adv, src = wav(100, 7), (wav(80, 8) if kind != "emb" else None)
    torch.manual_seed(9)
    _, m_grouped = d_grouped.defend(wavs, adv, attack_type=kind, n_iters=N_IT, vc_src=src, griffin_lim_iters=0, return_mels=True)
    torch.manual_seed(9)
    _, m_mixed = d_mixed.defend(wavs, adv, attack_type=kind, n_iters=N_IT, vc_src=src, griffin_lim_iters=0, return_mels=True,
                                mixed_lengths=True)
    for a, b in zip(m_grouped, m_mixed):
        assert torch.equal(a, b)
