"""Host logic of the defence pipeline without a GPU: the normalize / denormalize oracle, the attack-call plan of
Defender.defend (grouping, chunking, per-utterance normaliser, initial-noise draw order, one front-end and one back-end
call) with stand-ins for the engine and the audio ends, and sharded_defend's variable-length gather under gloo."""
import ast
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import REFERENCE


def test_normalize_round_trip():
    import norm_oracle as N
    rng = np.random.default_rng(3)
    mel = rng.uniform(0, 1, (57, 80)).astype(np.float32)
    mean = rng.uniform(0.3, 0.6, 80).astype(np.float32)
    std = rng.uniform(0.1, 0.3, 80).astype(np.float32)
    x = N.normalize(mel, mean, std)
    assert x.shape == (57, 80) and x.dtype == np.float32
    np.testing.assert_array_equal(x[:, 5], (mel[:, 5] - mean[5]) / std[5])        # per mel bin, over the frames
    np.testing.assert_allclose(N.denormalize(x, mean, std), mel, rtol=0, atol=1e-6)
    np.testing.assert_array_equal(N.denormalize(x, mean, std), x * std + mean)


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(REFERENCE)),
                    reason="set ATTACK_VC_REFERENCE to a checkout of the original attack-vc project")
def test_normalize_matches_reference():
    """The reference's own normalize / denormalize (data_utils.py:35-47).  data_utils.py imports librosa, which is not
    installed, so the two functions are cut out of the file and compiled as they stand."""
    import inspect
    import norm_oracle as N
    tree = ast.parse(open(os.path.join(REFERENCE, "data_utils.py")).read())
    fns = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in ("normalize", "denormalize")]
    assert len(fns) == 2
    ns = {"np": np}
    exec(compile(ast.Module(body=fns, type_ignores=[]), "ref_data_utils_normalize", "exec"), ns)
    rng = np.random.default_rng(4)
    mel = rng.uniform(0, 1, (40, 80)).astype(np.float32)
    mean, std = rng.uniform(0.3, 0.6, 80).astype(np.float32), rng.uniform(0.1, 0.3, 80).astype(np.float32)

    def call(fn, x):
        if len(inspect.signature(fn).parameters) == 2:              # fn(mel, attr) with attr = {"mean": ..., "std": ...}
            return fn(x, {"mean": mean, "std": std})
        return fn(x, mean, std)
    np.testing.assert_array_equal(call(ns["normalize"], mel), N.normalize(mel, mean, std))
    np.testing.assert_array_equal(call(ns["denormalize"], mel), N.denormalize(mel, mean, std))


# ---- Defender.defend with stand-ins --------------------------------------------------------------------------------
HOP = 300


class _StubAudio:
    """Front-end: frame rows filled with the waveform's first sample; back-end: one sample per frame hop of row col 0."""
    n_mels, hop_length, n_fft, kernel_launches = 80, HOP, 2048, 0
    device = torch.device("cpu")

    def __init__(self):
        self.calls = []

    def wav2mel_varlen(self, wavs, mean=None, std=None):
        self.calls.append(("front", [int(w.numel()) for w in wavs], mean is not None))
        frames = [1 + int(w.numel()) // HOP for w in wavs]
        buf = torch.cat([torch.full((f, 80), float(w[0])) for f, w in zip(frames, wavs)])
        return list(buf.split(frames))

    def mel2wav_varlen(self, mels, n_iter=100, mean=None, std=None):
        self.calls.append(("back", [int(m.shape[0]) for m in mels], n_iter, mean is not None))
        return [m[:, 0].repeat_interleave(HOP)[: HOP * (m.shape[0] - 1)].clone() for m in mels]


class _StubEngine:
    device = torch.device("cpu")
    c_in, c_emb, kernel_launches = 80, 128, 0

    def __init__(self):
        self.calls = []

    def min_frames(self, which="speaker"):
        return 9

    def decoder_frames(self, T_src):
        return T_src + 3

    def attack(self, kind, vc_tgt, adv_tgt, eps, n_iters, vc_src=None, w0=None, inv_norm=None):
        self.calls.append(dict(kind=kind, B=vc_tgt.shape[0], T=vc_tgt.shape[2], inv_norm=inv_norm, w0=w0.clone(),
                               tgt_stride=vc_tgt.stride(), adv_stride=adv_tgt.stride(),
                               src_stride=None if vc_src is None else vc_src.stride()))
        out = torch.empty_like(vc_tgt)                 # keeps vc_tgt's strides, as Engine.attack does
        out.copy_(vc_tgt + w0)
        return out


def _defender(max_batch):
    from attack_vc_b200.defend import Defender
    eng, aud = _StubEngine(), _StubAudio()
    d = Defender(eng, torch.full((80,), 0.5), torch.full((80,), 0.2), audio=aud, max_batch=max_batch)
    return d, eng, aud


def test_plan_chunks():
    from attack_vc_b200.defend import plan_chunks
    assert plan_chunks([5, 3, 5, 7, 5], 2) == [(5, [0, 2]), (5, [4]), (3, [1]), (7, [3])]
    assert plan_chunks([4, 4, 4], 8) == [(4, [0, 1, 2])]
    assert plan_chunks([], 3) == []
    with pytest.raises(ValueError):
        plan_chunks([1], 0)


@pytest.mark.parametrize("kind", ["emb", "e2e"])
def test_defend_plan_and_w0_order(kind):
    frames = [20, 12, 20, 31, 20]
    wavs = [torch.full((HOP * (f - 1) + 7,), float(i + 1)) for i, f in enumerate(frames)]
    adv = torch.full((HOP * 15,), 100.0)
    src = torch.full((HOP * 17,), 200.0) if kind == "e2e" else None
    d, eng, aud = _defender({kind: 2})
    torch.manual_seed(5)
    wav_out, mels = d.defend(wavs, adv, attack_type=kind, eps=0.1, n_iters=3, vc_src=src, griffin_lim_iters=4, return_mels=True)
    # the initial noise: attack_utils' draw on each utterance's [1, 80, T] view, one utterance at a time, in INPUT order
    torch.manual_seed(5)
    want_w0 = [torch.zeros_like(torch.empty(f, 80).t().unsqueeze(0)).normal_(0, 1) for f in frames]
    # attack calls: equal lengths together, chunks of at most 2, the per-utterance normaliser, targets broadcast
    plan = [(20, [0, 2]), (20, [4]), (12, [1]), (31, [3])]
    assert [(c["T"], c["B"]) for c in eng.calls] == [(T, len(idx)) for T, idx in plan]
    T_src = 1 + (HOP * 17) // HOP
    inv = 1.0 / 128 if kind == "emb" else 1.0 / (80 * (T_src + 3))
    for c, (T, idx) in zip(eng.calls, plan):
        assert c["kind"] == kind and c["inv_norm"] == inv
        assert c["tgt_stride"] == (80 * T, 1, 80)                     # time-major [B, 80, T] view of the front-end's buffer
        assert (c["src_stride"] is None) == (kind == "emb")
        if c["B"] > 1:                                                 # one attack target / source, batch stride 0
            assert c["adv_stride"][0] == 0 and (c["src_stride"] is None or c["src_stride"][0] == 0)
        for k, i in enumerate(idx):
            assert torch.equal(c["w0"][k], want_w0[i][0])
    # one front-end call (targets in chunk order, then adv_tgt [, vc_src]), one back-end call in input order
    order = [0, 2, 4, 1, 3]
    extra = [adv.numel()] + ([src.numel()] if src is not None else [])
    assert aud.calls[0] == ("front", [wavs[i].numel() for i in order] + extra, True)
    assert aud.calls[1] == ("back", frames, 4, True) and len(aud.calls) == 2
    for i, (w, m) in enumerate(zip(wav_out, mels)):
        assert m.shape == (frames[i], 80) and m.is_contiguous()
        assert torch.equal(m, (float(i + 1) + want_w0[i][0]).t())
        assert w.shape == (HOP * (frames[i] - 1),)


def test_defend_validation():
    from attack_vc_b200.defend import Defender
    d, eng, aud = _defender({})
    ok = torch.zeros(HOP * 20)
    with pytest.raises(ValueError):
        d.defend([ok], ok, attack_type="fb")                            # vc_src required
    with pytest.raises(ValueError):
        d.defend([ok], ok, attack_type="nope")
    with pytest.raises(ValueError):
        d.defend([ok], ok, n_iters=-1)
    with pytest.raises(ValueError):
        d.defend([ok, torch.zeros(1000)], ok)                          # too short for the front-end
    with pytest.raises(ValueError):
        d.defend([torch.zeros(HOP * 6)], ok)                           # 7 frames: fewer than the encoder takes
    with pytest.raises(ValueError):
        d.defend([ok.double()], ok)
    with pytest.raises(ValueError):
        d.defend([ok.reshape(2, -1)], ok)
    assert eng.calls == [] and aud.calls == []                         # nothing ran
    for mean, std in ((torch.zeros(79), torch.ones(80)), (torch.zeros(80), torch.zeros(80)),
                      (torch.full((80,), float("nan")), torch.ones(80))):
        with pytest.raises(ValueError):
            Defender(_StubEngine(), mean, std, audio=_StubAudio())


# ---- sharded_defend under gloo -------------------------------------------------------------------------------------
class _StubDefender:
    device = torch.device("cpu")

    def defend(self, wavs, adv_tgt, **kw):
        return [torch.cat([w * 2 + adv_tgt[0], w[: int(w[0])]]) for w in wavs]      # lengths differ per utterance


def _inputs():
    return [torch.arange(n, dtype=torch.float32) + n for n in (9, 4, 12, 7, 5)], torch.full((3,), 0.5)


def _shard_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from attack_vc_b200.distributed import sharded_defend

        class Counting(_StubDefender):
            seen = []

            def defend(self, wavs, adv_tgt, **kw):
                self.seen.append(len(wavs))
                return super().defend(wavs, adv_tgt, **kw)
        d = Counting()
        wavs, adv = _inputs()
        out = sharded_defend(d, wavs, adv, attack_type="emb")
        q.put((rank, d.seen, [o.numpy().copy() for o in out]))
    finally:
        dist.destroy_process_group()


def test_sharded_defend_gloo():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    wavs, adv = _inputs()
    want = _StubDefender().defend(wavs, adv)
    assert [r[1] for r in res] == [[3], [2]]                           # contiguous slices of 3 and 2 utterances
    for _, _, out in res:                                              # every rank gets all, in input order, unpadded
        assert len(out) == 5
        for o, w in zip(out, want):
            np.testing.assert_array_equal(o, w.numpy())
