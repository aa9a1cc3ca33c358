"""Pins the CPU oracle (oracle/convtasnet_oracle.py) against golden vectors minted from the unmodified
reference by tests/golden/make_golden.py.  CPU only."""
import os

import pytest
import torch

import convtasnet_oracle as O

# fp32 CPU restatement vs fp32 CPU reference: same ATen ops in (almost) the same order.
RTOL, ATOL = 1e-5, 2e-6
# torch.set_num_threads() of tests/golden/make_golden.py, which minted the fixtures
MINT_THREADS = 8


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)


@pytest.mark.parametrize("name", ["tiny_gln", "tiny_cln", "tiny_softmax", "small_relu_3spk", "paper_2spk", "paper_3spk_short"])
def test_model_cases(golden_dir, name):
    rec = _load(golden_dir, name)
    cfg = O.OracleConfig(**rec["cfg"])
    sd = O.synth_state_dict(cfg, seed=rec["wseed"])
    assert abs(float(sum(v.double().abs().sum() for v in sd.values())) - rec["weight_abs_sum"]) < 1e-6 * rec["weight_abs_sum"]
    assert sum(v.numel() for v in sd.values()) == rec["n_params"]
    mixture, sources = O.synth_batch(rec["batch"], cfg.n_sources, rec["T"], seed=rec["xseed"])
    with torch.no_grad():
        out, latent = O.conv_tasnet_fwd(mixture, sd, cfg)
        loss, perm = O.pit_neg_sisdr(out, sources)
        loss_b, perm_b = O.pit_neg_sisdr(out, sources, batch_mean=False)
    if "out_stride" in rec:
        s = rec["out_stride"]
        a, b = rec["latent_stride"]
        torch.testing.assert_close(out[..., ::s], rec["out"], rtol=RTOL, atol=ATOL)
        torch.testing.assert_close(latent[:, :, ::a, ::b], rec["latent"], rtol=RTOL, atol=ATOL)
    else:
        torch.testing.assert_close(out, rec["out"], rtol=RTOL, atol=ATOL)
        torch.testing.assert_close(latent, rec["latent"], rtol=RTOL, atol=ATOL)
    assert abs(float(out.double().sum()) - rec["out_sum"]) < 1e-3
    assert torch.equal(perm, rec["perm"]) and torch.equal(perm_b, rec["perm_b"])
    torch.testing.assert_close(loss, rec["loss"], rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(loss_b, rec["loss_b"], rtol=1e-5, atol=1e-4)


def test_paper_param_count(golden_dir):
    # SURVEY.md section 6: 4,984,881 parameters for the 2-speaker paper config
    assert _load(golden_dir, "paper_2spk")["n_params"] == 4984881


def test_norms(golden_dir):
    m = _load(golden_dir, "modules")
    one, zero = torch.ones(3), torch.zeros(3)
    torch.testing.assert_close(O.gln(m["gln_arange_in"], one, zero), m["gln_arange_out"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(O.cln(m["gln_arange_in"], one, zero), m["cln_arange_out"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(O.gln(m["gln_in"], m["gln_gamma"], m["gln_beta"]), m["gln_out"], rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(O.cln(m["gln_in"], m["gln_gamma"], m["gln_beta"]), m["cln_out"], rtol=1e-5, atol=2e-6)


def test_encoder_decoder(golden_dir):
    m = _load(golden_dir, "modules")
    keys = [k for k in m if k.startswith("encdec_")]
    assert len(keys) == 3
    for k in keys:
        r = m[k]
        _, N, L, S, T, relu = k.split("_")
        w = O.encoder_fwd(r["x"], r["We"], int(S[1:]), relu=bool(int(relu)))
        torch.testing.assert_close(w, r["w"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(O.decoder_fwd(w, r["Wd"], int(S[1:])), r["y"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("causal", [0, 1])
def test_tdcn(golden_dir, causal):
    r = _load(golden_dir, "modules")[f"tdcn_causal{causal}"]
    cfg = O.OracleConfig(**r["cfg"])
    sd = O.synth_state_dict(cfg, seed=r["wseed"])
    y = O.tdcn_fwd(r["x"], sd, "separator.tdcn.", kernel_size=3, num_blocks=2, num_layers=4, dilated=True,
                   causal=bool(causal), nonlinear=True, norm=True, eps=O.EPS)
    torch.testing.assert_close(y, r["y"], rtol=1e-5, atol=2e-6)


def test_pit_sisdr(golden_dir):
    m = _load(golden_dir, "modules")
    r = m["pit_selftest"]
    loss, pat = O.pit_neg_sisdr(r["input"], r["target"])
    assert torch.equal(pat, r["pattern"])
    torch.testing.assert_close(loss, r["loss"], rtol=1e-6, atol=1e-5)
    for S in (2, 3, 4):
        r = m[f"pit_S{S}"]
        loss_b, pat = O.pit_neg_sisdr(r["input"], r["target"], batch_mean=False)
        assert torch.equal(pat, r["pattern"]) and pat.dtype == torch.int64
        torch.testing.assert_close(loss_b, r["loss_b"], rtol=1e-6, atol=1e-5)
        torch.testing.assert_close(O.sisdr(r["input"], r["target"]), r["sisdr"], rtol=1e-6, atol=1e-5)
    t = m["sisdr_limits_in"]
    torch.testing.assert_close(O.sisdr(t, torch.zeros_like(t)), m["sisdr_zero_target"], rtol=1e-6, atol=1e-4)
    torch.testing.assert_close(O.sisdr(t, t.clone()), m["sisdr_perfect"], rtol=1e-6, atol=1e-4)
    r = m["pit_tie"]
    l, p = O.pit_neg_sisdr(r["input"], r["target"], batch_mean=False)
    assert torch.equal(p, r["pattern"])
    torch.testing.assert_close(l, r["loss_b"], rtol=1e-6, atol=1e-5)


def test_autograd_over_the_oracle_matches_reference_backward(golden_dir):
    """The training checker (torch autograd over the oracle) is pinned to the reference's own ``loss.backward()``
    (tests/golden/make_golden.py: grad_case, paper hyper-parameters, 3 speakers, batch 2, T = 8000): loss, permutation and
    all 343 gradient tensors (fp64 sums + every 97th element).

    The fp32 gradients of the PReLU slopes are sums over ~2e6 terms with heavy cancellation: they move by up to 25 % of the
    tensor's largest entry with the order of the CPU reduction, which follows torch's thread count.  The fixture was minted
    with MINT_THREADS threads (make_golden.py), so the test runs with the same count on any machine."""
    threads = torch.get_num_threads()
    torch.set_num_threads(MINT_THREADS)
    try:
        _check_autograd_over_the_oracle(golden_dir)
    finally:
        torch.set_num_threads(threads)


def _check_autograd_over_the_oracle(golden_dir):
    rec = _load(golden_dir, "paper_3spk_grad")
    cfg = O.OracleConfig(**rec["cfg"])
    sd = {k: v.clone().requires_grad_(True) for k, v in O.synth_state_dict(cfg, seed=rec["wseed"]).items()}
    mixture, sources = O.synth_batch(rec["batch"], cfg.n_sources, rec["T"], seed=rec["xseed"])
    out, _ = O.conv_tasnet_fwd(mixture, sd, cfg)
    loss, perm = O.pit_neg_sisdr(out, sources)
    loss.backward()
    assert torch.equal(perm, rec["perm"])
    torch.testing.assert_close(loss.detach(), rec["loss"], rtol=0, atol=1e-4)
    assert len(rec["grads"]) == 343
    for k, g in rec["grads"].items():
        mine = sd[k].grad
        assert tuple(mine.shape) == g["shape"], k
        tol = 2e-4 * g["absmax"] + 1e-12
        assert float((mine.flatten()[::rec["stride"]] - g["sample"]).abs().max()) <= tol, k
        assert abs(float(mine.double().sum()) - g["sum"]) <= 2e-4 * (g["sumsq"] * mine.numel()) ** 0.5 + 1e-9, k
    # and in fp64 (the noise-free answer the GPU tests are anchored on): oracle autograd in double == reference backward in double
    sd64 = {k: v.double().clone().requires_grad_(True) for k, v in O.synth_state_dict(cfg, seed=rec["wseed"]).items()}
    out64, _ = O.conv_tasnet_fwd(mixture.double(), sd64, cfg)
    loss64, _ = O.pit_neg_sisdr(out64, sources.double())
    loss64.backward()
    assert abs(float(loss64) - rec["loss64"]) < 1e-9
    for k, g in rec["grads"].items():
        assert float((sd64[k].grad.flatten()[::rec["stride"]] - g["sample64"]).abs().max()) <= 1e-9 * max(1.0, g["absmax64"]), k


def test_sdr_oracle_vs_reference_golden(golden_dir):
    """oracle sdr() (src/criterion/sdr.py:6-20) against the values the reference produced (criteria.pt)"""
    rec = torch.load(os.path.join(golden_dir, "criteria.pt"), weights_only=False)
    for name, r in rec.items():
        torch.testing.assert_close(O.sdr(r["input"], r["target"]), r["sdr"], rtol=1e-6, atol=1e-5, msg=lambda m: f"{name}: {m}")
        torch.testing.assert_close(torch.clamp(O.sisdr(r["input"], r["target"]), max=20.0).mean(dim=tuple(range(1, r["input"].dim() - 1)))
                                   if r["input"].dim() > 2 else torch.clamp(O.sisdr(r["input"], r["target"]), max=20.0),
                                   r["ClippedSISDR_20"], rtol=1e-5, atol=1e-4)


def test_multichannel_oracle_vs_reference_golden(golden_dir):
    """in_channels = 2 (4-D input, conv_tasnet.py:138-141,167-168): oracle == reference on the stereo fixture"""
    r = torch.load(os.path.join(golden_dir, "tiny_stereo.pt"), weights_only=False)
    cfg = O.OracleConfig(**r["cfg"])
    out, latent = O.conv_tasnet_fwd(r["mixture"], O.synth_state_dict(cfg, seed=r["wseed"]), cfg)
    assert out.shape == r["out"].shape == (2, 3, 2, 1501)
    torch.testing.assert_close(out, r["out"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(latent, r["latent"], rtol=1e-5, atol=1e-6)
