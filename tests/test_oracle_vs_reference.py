"""Oracle == unmodified reference, bit for bit, executed here.  Runs when ATTACK_VC_REFERENCE names a checkout of the
original project (it is not part of this repository).  Every case here is also pinned without it by tests/golden, in
test_oracle_golden.py: the AdaIN-VC forward and attack vectors were made from the reference; the vsmask_* vectors
(state-dict keys, header, PredictiveModel, trainer steps) were made from the oracle, which this module holds bit-identical
to the reference on the same cases.  Each file's "source" entry says which; tests/tools/make_golden.py remakes them from
the reference when ATTACK_VC_REFERENCE is set."""
import os
import sys

import pytest
import torch

from conftest import REFERENCE

pytestmark = pytest.mark.skipif(not (REFERENCE and os.path.isdir(REFERENCE)),
                                reason="set ATTACK_VC_REFERENCE to a checkout of the original attack-vc project")


@pytest.fixture(scope="module")
def ref_model(oracle):
    sys.path.insert(0, REFERENCE)
    try:
        import models as RM
    finally:
        sys.path.remove(REFERENCE)
    m = RM.AdaInVC(oracle.SYNTH_CONFIG)
    m.load_state_dict(oracle.make_state_dict(seed=0), strict=True)   # same keys + shapes as the reference
    return m


def test_state_dict_keys_match_reference(oracle, ref_model, cpu_model):
    assert list(ref_model.state_dict().keys()) == list(cpu_model.state_dict().keys())
    for (k, a), (_, b) in zip(ref_model.state_dict().items(), cpu_model.state_dict().items()):
        assert a.shape == b.shape, k
        assert torch.equal(a, b), k


@pytest.mark.parametrize("B,T,T_src", [(1, 128, 128), (3, 75, 43)])
def test_forward_bit_exact(oracle, ref_model, cpu_model, B, T, T_src):
    inp = oracle.make_inputs("e2e", B, T, seed=5, T_src=T_src)
    with torch.no_grad():
        assert torch.equal(ref_model.speaker_encoder(inp["vc_tgt"]), cpu_model.speaker_encoder(inp["vc_tgt"]))
        mu_r, ls_r = ref_model.content_encoder(inp["vc_src"])
        mu_o, ls_o = cpu_model.content_encoder(inp["vc_src"])
        assert torch.equal(mu_r, mu_o) and torch.equal(ls_r, ls_o)
        assert torch.equal(ref_model.inference(inp["vc_src"], inp["vc_tgt"]), cpu_model.inference(inp["vc_src"], inp["vc_tgt"]))


@pytest.mark.parametrize("kind", ["emb", "e2e", "fb"])
def test_attack_loop_bit_exact(oracle, ref_model, cpu_model, kind):
    sys.path.insert(0, REFERENCE)
    try:
        import attack_utils as RA
    finally:
        sys.path.remove(REFERENCE)
    inp = oracle.make_inputs(kind, 1, 48, seed=2)
    torch.manual_seed(77)
    w0 = torch.zeros_like(inp["vc_tgt"]).normal_(0, 1)
    torch.manual_seed(77)
    n = 4
    if kind == "emb":
        r = RA.emb_attack(ref_model, inp["vc_tgt"], inp["adv_tgt"], 0.1, n)
    elif kind == "e2e":
        r = RA.e2e_attack(ref_model, inp["vc_src"], inp["vc_tgt"], inp["adv_tgt"], 0.1, n)
    else:
        r = RA.fb_attack(ref_model, inp["vc_src"], inp["vc_tgt"], inp["adv_tgt"], 0.1, n)
    o = oracle.run_attack(kind, cpu_model, inp["vc_tgt"], inp["adv_tgt"], 0.1, n, w0, vc_src=inp.get("vc_src"))
    assert torch.equal(r.detach(), o["adv"])


def test_header_optimize_bit_exact(oracle, ref_model, cpu_model):
    """oracle.run_header == UniversalPerturbationHeader.optimize (models/header_model.py:25-68) with the AdaIN-VC
    speaker encoder and Adam([header], lr=1e-3) as train_header.py builds it."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_header_model", os.path.join(REFERENCE, "models", "header_model.py"))
    hm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(hm)
    inp = oracle.make_inputs("emb", 3, 100, seed=4)
    src, tgt = inp["vc_tgt"].unsqueeze(1) * 0.6, inp["adv_tgt"].unsqueeze(1) * 0.6      # some |x| > 1: the clamp is live
    assert float(src.abs().max()) > 1.0
    H = hm.UniversalPerturbationHeader(80, 100, device="cpu")
    opt = torch.optim.Adam([H.header], lr=1e-3)
    H.optimize(src, tgt, lambda m: ref_model.speaker_encoder(m.squeeze(1)), opt, num_iterations=5, epsilon=0.003,
               lambda_param=0.5)
    o = oracle.run_header(cpu_model, src, tgt, 5, epsilon=0.003)
    assert torch.equal(H.header.detach(), o["header"])
    assert float(o["header"].abs().max()) == pytest.approx(0.003, rel=1e-6)             # the eps clamp is live too


def _ref_predictive():
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_predictive_model", os.path.join(REFERENCE, "models", "predictive_model.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)          # by file path: models.py shadows the models/ directory (SURVEY 2 #8)
    return m.PredictiveModel()


def test_predictive_oracle_bit_exact():
    from oracle import predictive_oracle as P
    pm = _ref_predictive()
    sd = P.pm_make_state_dict(0)
    assert list(pm.state_dict().keys()) == list(sd.keys())
    pm.load_state_dict(sd, strict=True)
    x = torch.randn(3, 1, 80, 100, generator=torch.Generator().manual_seed(5))
    pm.eval()
    with torch.no_grad():
        assert torch.equal(pm(x), P.pm_forward(sd, x, training=False))
    pm.train()
    xin = x.clone().requires_grad_(True)
    out = pm(xin)
    loss = out.square().mean()
    loss.backward()
    t = P.pm_train_step(sd, x)
    assert torch.equal(out.detach(), t["out"]) and torch.equal(loss.detach(), t["loss"])
    for n, prm in pm.named_parameters():
        assert torch.equal(prm.grad, t["grads"][n]), n
    assert torch.equal(xin.grad, t["grad_x"])
    for k, v in t["new_stats"].items():
        assert torch.equal(pm.state_dict()[k], v), k


def _ref_weighted_constraint():
    """The reference's own apply_weighted_constraint (utils/audio.py:77-116).  utils/audio.py imports torchaudio, which is
    not installed, so the method's source is cut out of the file and compiled as it stands (nothing is restated)."""
    import ast
    src = open(os.path.join(REFERENCE, "utils", "audio.py")).read()
    tree = ast.parse(src)
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "MelSpectrogramConverter")
    fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "apply_weighted_constraint")
    mod = ast.Module(body=[fn], type_ignores=[])
    ns = {"torch": torch}
    exec(compile(mod, "ref_audio_apply_weighted_constraint", "exec"), ns)
    return lambda p, e1, e2, e3: ns["apply_weighted_constraint"](None, p, epsilon1=e1, epsilon2=e2, epsilon3=e3)


def _ref_train_steps(ref_model, sd, batches, eps):
    """The loop body of train_predictive.py:92-126 driven through the reference's PredictiveModel module, the reference's
    apply_weighted_constraint and the reference's AdaIN-VC speaker encoder, with the two documented repairs (crop to F
    mel rows, constraint on squeeze(1)).  Returns the losses, the final state dict and how many elements were clamped."""
    constraint = _ref_weighted_constraint()
    pm = _ref_predictive()
    pm.load_state_dict(sd, strict=True)
    enc = lambda m: ref_model.speaker_encoder(m.squeeze(1))
    opt = torch.optim.Adam(pm.parameters(), lr=1e-3)                       # train_predictive.py:57
    losses = []
    pm.train()                                                             # :64
    n_clamped = 0
    for source_mels, target_mels in batches:
        predicted = pm(source_mels)                                        # :92
        future_idx = 10
        perturbed = source_mels.clone()                                    # :100
        future_end = min(future_idx + predicted.shape[-1], perturbed.shape[-1])      # :101
        perturbed[:, :, :, future_idx:future_end] += predicted[:, :, :80, :future_end - future_idx]   # :102 + repair 1
        delta = (perturbed - source_mels).squeeze(1)                       # repair 2
        weighted = constraint(delta, *eps).unsqueeze(1)                    # :105-110
        n_clamped += int((weighted.squeeze(1) != delta).sum())
        perturbed = source_mels + weighted                                 # :111
        e_s, e_t, e_p = enc(source_mels), enc(target_mels), enc(perturbed)  # :114-116
        mse = torch.nn.MSELoss()
        loss = mse(e_p, e_t) - 0.5 * mse(e_p, e_s)                         # :119-122
        opt.zero_grad(); loss.backward(); opt.step()                       # :125-127
        losses.append(float(loss.detach()))
    return losses, pm.state_dict(), n_clamped


def test_vsmask_train_step_bit_exact(ref_model):
    """oracle.vsmask_train_oracle.train_steps == the reference's training loop (_ref_train_steps)."""
    from oracle import predictive_oracle as P
    from oracle import vsmask_train_oracle as V
    sd = P.pm_make_state_dict(0)
    g = torch.Generator().manual_seed(21)
    batches = [(0.5 * torch.randn(3, 1, 80, 100, generator=g), 0.5 * torch.randn(3, 1, 80, 100, generator=g)) for _ in range(3)]
    # eps an order of magnitude below the defaults: this synthetic model predicts |p| ~ 1e-2, and the clamp must be live
    eps = (0.01, 0.005, 0.008)
    losses, state, n_clamped = _ref_train_steps(ref_model, sd, batches, eps)
    assert n_clamped > 0                                                   # the clamp (and its mask in the backward) is exercised
    o = V.train_steps(sd, ref_model.speaker_encoder, batches, lr=1e-3, future_steps=10, eps=eps, lambda_param=0.5)
    assert o["losses"].tolist() == losses
    for k, v in state.items():
        if v.dtype.is_floating_point:
            assert torch.equal(v, o["state"][k]), k
