"""Oracle vs the committed golden vectors (generated from the reference by tests/tools/make_golden.py).
Runs everywhere (CPU), so the pin travels to the GPU box."""
import numpy as np
import pytest
import torch

CASES = ["emb_T128_it100", "e2e_T64_it20", "fb_T64_it20", "emb_B2_ragged_cli", "e2e_B2_ragged", "fb_B2_ragged"]


def test_model_forward_golden(oracle, cpu_model, golden):
    g = golden("model_fwd")
    with torch.no_grad():
        emb = cpu_model.speaker_encoder(torch.from_numpy(g["vc_tgt"]))
        mu, ls = cpu_model.content_encoder(torch.from_numpy(g["vc_src"]))
        out = cpu_model.inference(torch.from_numpy(g["vc_src"]), torch.from_numpy(g["vc_tgt"]))
    # same ATen ops, but thread count / ISA may differ from the generating run: allow fp32 noise
    np.testing.assert_allclose(emb.numpy(), g["emb"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(mu.numpy(), g["mu"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(ls.numpy(), g["log_sigma"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(out.numpy(), g["out"], rtol=0, atol=2e-5)


@pytest.mark.parametrize("name", CASES)
def test_attack_golden(oracle, cpu_model, golden, name):
    g = golden(name)
    kind = name.split("_")[0]
    n = int(g["n_iters"])
    n_run = min(n, 12)            # keep the CPU suite short; prefix of the trajectory is enough to pin it
    record = [int(k.split("_")[1]) for k in g if k.startswith("grad_") and int(k.split("_")[1]) < n_run]
    t = lambda k: torch.from_numpy(g[k])
    o = oracle.run_attack(kind, cpu_model, t("vc_tgt"), t("adv_tgt"), float(g["eps"]), n_run, t("w0"),
                          vc_src=t("vc_src") if "vc_src" in g else None, record_grads=record)
    np.testing.assert_allclose(o["losses"].numpy(), g["losses"][:n_run], rtol=2e-4)
    for i in record:
        ref = g[f"grad_{i}"]
        err = np.linalg.norm(o["grads"][i].numpy() - ref) / np.linalg.norm(ref)
        assert err < 1e-3, (i, err)
    if n_run == n:
        np.testing.assert_allclose(o["adv"].numpy(), g["adv"], rtol=0, atol=2e-5)
    # perturbation bound (attack_utils.py:40): |adv - x| <= eps up to one rounding of the sum
    assert np.abs(g["adv"] - g["vc_tgt"]).max() <= 0.1 * (1 + 1e-6)


# ---- VSMask side: the cases of test_oracle_vs_reference.py, pinned by tests/golden/vsmask_*.npz (tests/tools/make_golden.py) ----

def _check_sampled(g, prefix, tensors, rtol, atol):
    """Seeded element samples and whole-tensor norms stored by make_golden._sample_into."""
    assert {k.split("__")[2] for k in g if k.startswith(prefix + "__norm__")} == set(tensors)
    for name, t in tensors.items():
        a = t.detach().double().reshape(-1).numpy()
        np.testing.assert_allclose(a[g[f"{prefix}__idx__{name}"]], g[f"{prefix}__val__{name}"], rtol=rtol, atol=atol, err_msg=name)
        # atol too: the gradient of a conv bias that feeds BatchNorm is zero up to rounding
        np.testing.assert_allclose(np.linalg.norm(a), g[f"{prefix}__norm__{name}"], rtol=rtol, atol=atol, err_msg=name)


def test_state_dict_keys_golden(cpu_model, golden):
    from oracle.predictive_oracle import pm_make_state_dict
    g = golden("vsmask_keys")
    for tag, items in (("adainvc", cpu_model.state_dict().items()), ("predictive", pm_make_state_dict(0).items())):
        assert [k for k, _ in items] == g[f"{tag}_keys"].tolist()
        assert [",".join(map(str, v.shape)) for _, v in items] == g[f"{tag}_shapes"].tolist()


def test_header_optimize_golden(oracle, cpu_model, golden):
    g = golden("vsmask_header")
    inp = oracle.make_inputs("emb", 3, 100, seed=4)
    src, tgt = inp["vc_tgt"].unsqueeze(1) * 0.6, inp["adv_tgt"].unsqueeze(1) * 0.6
    o = oracle.run_header(cpu_model, src, tgt, 5, epsilon=0.003)
    # 1 vs 8 host threads move the 5-step header by up to 6e-7 (of its 3e-3 bound)
    np.testing.assert_allclose(o["header"].numpy(), g["header"], rtol=0, atol=5e-6)


def test_predictive_golden(golden):
    from oracle import predictive_oracle as P
    g = golden("vsmask_predictive")
    sd = P.pm_make_state_dict(0)
    x = torch.randn(3, 1, 80, 100, generator=torch.Generator().manual_seed(5))
    t = P.pm_train_step(sd, x)
    np.testing.assert_allclose(t["loss"].numpy(), g["loss"], rtol=1e-5)
    _check_sampled(g, "out", {"eval": P.pm_forward(sd, x, training=False), "train": t["out"], "grad_x": t["grad_x"]}, 1e-4, 1e-7)
    _check_sampled(g, "grad", t["grads"], 1e-4, 1e-8)
    _check_sampled(g, "stats", t["new_stats"], 1e-5, 1e-7)


def test_vsmask_train_golden(cpu_model, golden):
    from oracle import predictive_oracle as P
    from oracle import vsmask_train_oracle as V
    g = golden("vsmask_train")
    sd = P.pm_make_state_dict(0)
    gen = torch.Generator().manual_seed(21)
    batches = [(0.5 * torch.randn(3, 1, 80, 100, generator=gen), 0.5 * torch.randn(3, 1, 80, 100, generator=gen)) for _ in range(3)]
    o = V.train_steps(sd, cpu_model.speaker_encoder, batches, lr=1e-3, future_steps=10, eps=(0.01, 0.005, 0.008), lambda_param=0.5)
    np.testing.assert_allclose(o["losses"].numpy(), g["losses"], rtol=1e-5)
    _check_sampled(g, "update", {k: v - sd[k] for k, v in o["state"].items() if v.dtype.is_floating_point}, 1e-3, 1e-6)
