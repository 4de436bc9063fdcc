"""Host side of the ragged attack without a GPU: the C layout of avc_attack_varlen_args, the length-sorted chunk plan, and
Defender.defend(..., mixed_lengths=True) with stand-ins for the engine and the audio ends (call plan, initial-noise
order, output order, validation before any call)."""
import ctypes as C

import pytest
import torch

from test_defend_cpu import HOP, _StubAudio, _StubEngine


def test_varlen_args_layout():
    from attack_vc_b200._lib import AttackVarlenArgs
    # include/avc_b200.h: 5 pointers, B, then the two strided [B, 80, T] operands, loss_out, eps, n_iters, inv_norm, use_graph
    assert AttackVarlenArgs.frames_host.offset == 32 and AttackVarlenArgs.B.offset == 40
    assert AttackVarlenArgs.adv_tgt.offset == 48 and AttackVarlenArgs.vc_src.offset == 88
    assert AttackVarlenArgs.inv_norm.offset % 8 == 0 and AttackVarlenArgs.inv_norm.offset == 144
    assert C.sizeof(AttackVarlenArgs) == 160


def test_plan_sorted_chunks():
    from attack_vc_b200.defend import plan_sorted_chunks
    assert plan_sorted_chunks([5, 3, 5, 7, 5], 2) == [[3, 0], [2, 4], [1]]      # longest first, ties in input order
    assert plan_sorted_chunks([4, 9, 6], 8) == [[1, 2, 0]]
    assert plan_sorted_chunks([], 3) == []
    with pytest.raises(ValueError):
        plan_sorted_chunks([1], 0)


class _StubRaggedEngine(_StubEngine):
    def attack_varlen(self, kind, vc_tgt, adv_tgt, eps, n_iters, vc_src=None, w0=None, inv_norm=None):
        mels = list(vc_tgt)
        self.calls.append(dict(kind=kind, frames=[int(m.shape[0]) for m in mels], inv_norm=inv_norm,
                               w0=[w.clone() for w in w0], adv_stride=adv_tgt.stride(), B_adv=adv_tgt.shape[0],
                               src_stride=None if vc_src is None else vc_src.stride(),
                               contiguous=all(m.data_ptr() == mels[0].data_ptr() + 4 * 80 * sum(x.shape[0] for x in mels[:k])
                                              for k, m in enumerate(mels))))
        return [m + w for m, w in zip(mels, w0)]


def _defender(max_batch):
    from attack_vc_b200.defend import Defender
    eng, aud = _StubRaggedEngine(), _StubAudio()
    return Defender(eng, torch.full((80,), 0.5), torch.full((80,), 0.2), audio=aud, max_batch=max_batch), eng, aud


@pytest.mark.parametrize("kind", ["emb", "e2e"])
def test_defend_mixed_lengths_plan_and_order(kind):
    frames = [20, 12, 20, 31, 20]
    wavs = [torch.full((HOP * (f - 1) + 7,), float(i + 1)) for i, f in enumerate(frames)]
    adv = torch.full((HOP * 15,), 100.0)
    src = torch.full((HOP * 17,), 200.0) if kind == "e2e" else None
    d, eng, aud = _defender({kind: 2})
    torch.manual_seed(5)
    wav_out, mels = d.defend(wavs, adv, attack_type=kind, eps=0.1, n_iters=3, vc_src=src, griffin_lim_iters=4,
                             return_mels=True, mixed_lengths=True)
    torch.manual_seed(5)
    want_w0 = [torch.zeros_like(torch.empty(f, 80).t().unsqueeze(0)).normal_(0, 1) for f in frames]   # input order
    plan = [[3, 0], [2, 4], [1]]                                        # sorted by length, chunks of at most 2
    assert [c["frames"] for c in eng.calls] == [[frames[i] for i in idx] for idx in plan]
    T_src = 1 + (HOP * 17) // HOP
    inv = 1.0 / 128 if kind == "emb" else 1.0 / (80 * (T_src + 3))
    for c, idx in zip(eng.calls, plan):
        assert c["kind"] == kind and c["inv_norm"] == inv
        assert c["contiguous"]                                          # one block of the front-end's buffer: no copy
        assert c["B_adv"] == len(idx) and (c["src_stride"] is None) == (kind == "emb")
        if len(idx) > 1:
            assert c["adv_stride"][0] == 0 and (c["src_stride"] is None or c["src_stride"][0] == 0)
        for k, i in enumerate(idx):
            assert torch.equal(c["w0"][k], want_w0[i][0].t())
    order = [3, 0, 2, 4, 1]
    extra = [adv.numel()] + ([src.numel()] if src is not None else [])
    assert aud.calls[0] == ("front", [wavs[i].numel() for i in order] + extra, True)
    assert aud.calls[1] == ("back", frames, 4, True) and len(aud.calls) == 2
    for i, (w, m) in enumerate(zip(wav_out, mels)):
        assert m.shape == (frames[i], 80)
        assert torch.equal(m, float(i + 1) + want_w0[i][0].t())
        assert w.shape == (HOP * (frames[i] - 1),)


def test_defend_mixed_lengths_validation():
    d, eng, aud = _defender({})
    ok = torch.zeros(HOP * 20)
    for kw in (dict(attack_type="fb"), dict(attack_type="nope"), dict(n_iters=-1)):
        with pytest.raises(ValueError):
            d.defend([ok], ok, mixed_lengths=True, **kw)
    with pytest.raises(ValueError):
        d.defend([ok, torch.zeros(HOP * 6)], ok, mixed_lengths=True)     # 7 frames: fewer than the encoder takes
    assert eng.calls == [] and aud.calls == []
