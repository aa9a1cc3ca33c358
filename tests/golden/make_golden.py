#!/usr/bin/env python
"""Mint golden vectors from the UNMODIFIED reference (run in the build container only).

    python tests/golden/make_golden.py          # writes tests/golden/*.pt

The reference (/root/reference/src) is imported as-is; nothing is copied from it.
Weights and inputs come from the deterministic generators in oracle/convtasnet_oracle.py
(``synth_state_dict`` / ``synth_batch``) and are loaded into the reference modules with
``load_state_dict(strict=True)`` -- which also proves the key names / shapes / order of
``state_dict_spec`` match the reference.  Outputs are stored as small fixtures; the paper-size
case stores a strided subsample plus fp64 checksums.

/root/reference does not exist on the GPU box: tests only read the committed .pt files.
"""
import os
import sys
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF_SRC = "/root/reference/src"

sys.path.insert(0, REF_SRC)
warnings.simplefilter("ignore")
from models.conv_tasnet import ConvTasNet  # noqa: E402  (reference)
from models.tdcn import TimeDilatedConvNet  # noqa: E402
from models.filterbank import Encoder, Decoder  # noqa: E402
from modules.norm import GlobalLayerNorm, CumulativeLayerNorm1d  # noqa: E402
from criterion.sdr import NegSISDR, sisdr  # noqa: E402
from criterion.pit import PIT1d  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import convtasnet_oracle as O  # noqa: E402

torch.set_num_threads(8)


def build_reference(cfg: O.OracleConfig):
    m = ConvTasNet(
        cfg.n_basis, cfg.kernel_size, stride=cfg.stride, enc_basis="trainable", dec_basis="trainable",
        enc_nonlinear=cfg.enc_nonlinear,
        sep_hidden_channels=cfg.sep_hidden_channels, sep_bottleneck_channels=cfg.sep_bottleneck_channels,
        sep_skip_channels=cfg.sep_skip_channels, sep_kernel_size=cfg.sep_kernel_size,
        sep_num_blocks=cfg.sep_num_blocks, sep_num_layers=cfg.sep_num_layers,
        dilated=cfg.dilated, separable=cfg.separable, sep_nonlinear=cfg.sep_nonlinear, sep_norm=cfg.sep_norm,
        mask_nonlinear=cfg.mask_nonlinear, causal=cfg.causal, n_sources=cfg.n_sources, eps=cfg.eps, in_channels=cfg.in_channels)
    return m


def model_case(name, cfg: O.OracleConfig, batch, T, wseed, xseed, subsample=None):
    ref = build_reference(cfg)
    ref_keys = [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    spec = [(k, tuple(s)) for k, s in O.state_dict_spec(cfg)]
    assert ref_keys == spec, "state_dict_spec does not match the reference for " + name
    sd = O.synth_state_dict(cfg, seed=wseed)
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    mixture, sources = O.synth_batch(batch, cfg.n_sources, T, seed=xseed)
    with torch.no_grad():
        out, latent = ref.extract_latent(mixture)
        crit = PIT1d(NegSISDR(), n_sources=cfg.n_sources)
        loss, perm = crit(out, sources)
        loss_b, perm_b = crit(out, sources, batch_mean=False)
        # fp64 run of the same reference = noise-floor estimate
        ref64 = build_reference(cfg).double()
        ref64.load_state_dict({k: v.double() for k, v in sd.items()})
        out64, _ = ref64.extract_latent(mixture.double())
    rec = {
        "name": name, "cfg": cfg.to_dict(), "batch": batch, "T": T, "wseed": wseed, "xseed": xseed,
        "weight_abs_sum": float(sum(v.double().abs().sum() for v in sd.values())),
        "loss": loss.clone(), "perm": perm.clone(), "loss_b": loss_b.clone(), "perm_b": perm_b.clone(),
        "out_sum": float(out.double().sum()), "out_sumsq": float((out.double() ** 2).sum()),
        "out_absmax": float(out.abs().max()),
        "fp32_vs_fp64_maxabs": float((out.double() - out64).abs().max()),
        "n_params": sum(v.numel() for v in sd.values()),
    }
    if subsample is None:
        rec["out"] = out.clone()
        rec["latent"] = latent.clone()
    else:
        rec["out_stride"] = subsample
        rec["out"] = out[..., ::subsample].clone()
        rec["latent_stride"] = (37, 53)
        rec["latent"] = latent[:, :, ::37, ::53].clone()
    path = os.path.join(HERE, name + ".pt")
    torch.save(rec, path)
    print(f"{name}: out {tuple(out.shape)} absmax {rec['out_absmax']:.4f} loss {float(loss):.6f} "
          f"perm {perm.tolist()} fp32-vs-fp64 {rec['fp32_vs_fp64_maxabs']:.2e} -> {os.path.getsize(path)} B")


def grad_case(name, cfg: O.OracleConfig, batch, T, wseed, xseed, stride=97):
    """Reference-side TRAINING golden: ``loss.backward()`` of the unmodified reference through PIT1d(NegSISDR)
    (egs/wsj0-mix/common/src/driver.py:146-150).  Stores, per parameter tensor, fp64 (sum, sumsq, absmax) of the gradient
    and every ``stride``-th element of its flattened values (the full set is 20 MB at the paper size) -- once in the reference's
    own fp32 and once from the SAME reference modules in fp64.  At this size the fp32 backward is itself 3e-4 (median) to 3e-2
    (PReLU slopes, some 1x1 weights) away from the fp64 answer, relative to each tensor's largest entry, so a second fp32
    implementation can only be asked to be as close to the fp64 answer as the reference's fp32 is (``fp32_vs_fp64_maxabs``)."""
    sd = O.synth_state_dict(cfg, seed=wseed)
    mixture, sources = O.synth_batch(batch, cfg.n_sources, T, seed=xseed)
    crit = PIT1d(NegSISDR(), n_sources=cfg.n_sources)

    def run(dtype):
        ref = build_reference(cfg).to(dtype)
        ref.load_state_dict({k: v.to(dtype) for k, v in sd.items()}, strict=True)
        ref.train()
        out = ref(mixture.to(dtype))
        loss, perm = crit(out, sources.to(dtype))
        loss.backward()
        return ref, out, loss, perm

    ref, out, loss, perm = run(torch.float32)
    ref64, _, loss64, perm64 = run(torch.float64)      # the same reference modules in double = the noise-free answer
    assert torch.equal(perm, perm64)
    g64 = {k: p.grad.detach() for k, p in ref64.named_parameters()}
    grads = {}
    for k, p in ref.named_parameters():
        g = p.grad.detach()
        d = g64[k]
        grads[k] = {"sum": float(g.double().sum()), "sumsq": float((g.double() ** 2).sum()), "absmax": float(g.abs().max()),
                    "sample": g.flatten()[::stride].clone(), "shape": tuple(g.shape),
                    "sample64": d.flatten()[::stride].clone(), "sum64": float(d.sum()), "absmax64": float(d.abs().max()),
                    "fp32_vs_fp64_maxabs": float((g.double() - d).abs().max())}
    rec = {"name": name, "cfg": cfg.to_dict(), "batch": batch, "T": T, "wseed": wseed, "xseed": xseed, "stride": stride,
           "loss": loss.detach().clone(), "loss64": float(loss64), "perm": perm.clone(), "grads": grads,
           "out_absmax": float(out.detach().abs().max())}
    path = os.path.join(HERE, name + ".pt")
    torch.save(rec, path)
    print(f"{name}: loss {float(loss):.6f} perm {perm.tolist()} {len(grads)} gradient tensors -> {os.path.getsize(path)} B")


def checkpoint_case():
    """A trainer checkpoint written the way the reference's TrainerBase.save_model does (egs/wsj0-mix/common/src/driver.py:208-226):
    get_config() + state_dict + optimizer / bookkeeping entries, from the unmodified reference model (tiny_gln weights)."""
    cfg = O.OracleConfig(n_basis=16, kernel_size=4, sep_hidden_channels=16, sep_bottleneck_channels=8, sep_skip_channels=8,
                         sep_num_blocks=2, sep_num_layers=3, causal=False)
    ref = build_reference(cfg)
    ref.load_state_dict(O.synth_state_dict(cfg, seed=11), strict=True)
    opt = torch.optim.Adam(ref.parameters(), lr=1e-3)
    config = ref.get_config()
    config['state_dict'] = ref.state_dict()
    config['optim_dict'] = opt.state_dict()
    config['best_loss'], config['no_improvement'] = float('infinity'), 0
    config['train_loss'], config['valid_loss'] = torch.zeros(3), torch.zeros(3)
    config['epoch'] = 1
    path = os.path.join(HERE, "ref_ckpt_tiny_gln.pth")
    torch.save(config, path)
    print("ref_ckpt_tiny_gln.pth ->", os.path.getsize(path), "B; config keys", sorted(k for k in config if k != 'state_dict'))


def dprnn_cases():
    """DPRNN-TasNet (BASELINE cfg4) goldens from the unmodified reference: transform.py modules, one tiny model, and the cfg4
    hyper-parameters (N=64 L=2 F=64 H=128 K=250 P=125 B=6) on a short batch (strided subsample + fp64 checksums)."""
    from models.dprnn_tasnet import DPRNNTasNet  # reference
    from models.transform import Segment1d, OverlapAdd1d
    import dprnn_oracle as DO
    rec = {}
    g = torch.Generator().manual_seed(17)
    for (B, Fc, T, K, P) in [(2, 3, 5, 3, 2), (2, 6, 103, 10, 5), (1, 4, 40, 7, 3)]:
        x = torch.randn(B, Fc, T, generator=g)
        seg = Segment1d(K, P)(x)
        rec[f"segment_{B}_{Fc}_{T}_{K}_{P}"] = {"x": x, "seg": seg, "ola": OverlapAdd1d(K, P)(seg)}
    torch.save(rec, os.path.join(HERE, "dprnn_modules.pt"))
    for name, cfg, batch, T, sub in [
        ("dprnn_tiny", DO.DPRNNConfig(n_basis=16, kernel_size=4, sep_hidden_channels=12, sep_bottleneck_channels=8, sep_chunk_size=10,
                                      sep_hop_size=5, sep_num_blocks=2, n_sources=2), 2, 203, None),
        ("dprnn_cfg4_short", DO.DPRNNConfig(n_basis=64, kernel_size=2, sep_hidden_channels=128, sep_bottleneck_channels=64,
                                            sep_chunk_size=250, sep_hop_size=125, sep_num_blocks=6, n_sources=2), 2, 4000, 13),
    ]:
        ref = DPRNNTasNet(cfg.n_basis, cfg.kernel_size, stride=cfg.stride, enc_basis="trainable", dec_basis="trainable", enc_nonlinear=None,
                          sep_hidden_channels=cfg.sep_hidden_channels, sep_bottleneck_channels=cfg.sep_bottleneck_channels,
                          sep_chunk_size=cfg.sep_chunk_size, sep_hop_size=cfg.sep_hop_size, sep_num_blocks=cfg.sep_num_blocks,
                          sep_norm=True, mask_nonlinear="sigmoid", causal=False, rnn_type="lstm", n_sources=cfg.n_sources, eps=cfg.eps)
        ref_keys = [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
        assert ref_keys == [(k, tuple(sh)) for k, sh in DO.state_dict_spec(cfg)], "dprnn state_dict_spec does not match the reference"
        sd = DO.synth_state_dict(cfg, seed=31)
        ref.load_state_dict(sd, strict=True)
        ref.eval()
        mixture, sources = O.synth_batch(batch, cfg.n_sources, T, seed=32)
        with torch.no_grad():
            out, latent = ref.extract_latent(mixture)
            loss, perm = PIT1d(NegSISDR(), n_sources=cfg.n_sources)(out, sources)
        r = {"name": name, "cfg": cfg.to_dict(), "batch": batch, "T": T, "wseed": 31, "xseed": 32, "loss": loss.clone(), "perm": perm.clone(),
             "out_sum": float(out.double().sum()), "out_sumsq": float((out.double() ** 2).sum()), "out_absmax": float(out.abs().max())}
        if sub is None:
            r["out"], r["latent"] = out.clone(), latent.clone()
        else:
            r["out_stride"] = sub
            r["out"] = out[..., ::sub].clone()
            r["latent_stride"] = (7, 29)
            r["latent"] = latent[:, :, ::7, ::29].clone()
        path = os.path.join(HERE, name + ".pt")
        torch.save(r, path)
        print(f"{name}: out {tuple(out.shape)} absmax {r['out_absmax']:.4f} loss {float(loss):.6f} perm {perm.tolist()} -> {os.path.getsize(path)} B")


def module_cases():
    rec = {}
    # gLN / cLN: the reference's own self-test input (src/modules/norm.py:107-116) + a random one
    g = torch.Generator().manual_seed(7)
    x_ar = torch.arange(30, dtype=torch.float).view(2, 3, 5)
    x_rn = torch.randn(3, 24, 301, generator=g) * 2.0 + 0.7
    gam = 1.0 + 0.3 * torch.randn(24, generator=g)
    bet = 0.2 * torch.randn(24, generator=g)
    gl = GlobalLayerNorm(3)
    rec["gln_arange_in"], rec["gln_arange_out"] = x_ar, gl(x_ar).detach()
    gl = GlobalLayerNorm(24)
    gl.load_state_dict({"norm.weight": gam, "norm.bias": bet})
    rec["gln_in"], rec["gln_gamma"], rec["gln_beta"], rec["gln_out"] = x_rn, gam, bet, gl(x_rn).detach()
    cl = CumulativeLayerNorm1d(24)
    cl.load_state_dict({"gamma": gam.view(1, 24, 1), "beta": bet.view(1, 24, 1)})
    rec["cln_out"] = cl(x_rn).detach()
    cl3 = CumulativeLayerNorm1d(3)
    rec["cln_arange_out"] = cl3(x_ar).detach()

    # Encoder / Decoder
    for (N, L, S, T, relu) in [(32, 16, 8, 400, False), (20, 4, 2, 131, True), (64, 2, 1, 96, False)]:
        key = f"N{N}_L{L}_S{S}_T{T}_{int(relu)}"
        enc = Encoder(1, N, kernel_size=L, stride=S, nonlinear="relu" if relu else None)
        dec = Decoder(N, 1, kernel_size=L, stride=S)
        We = (torch.rand(N, 1, L, generator=g) * 2 - 1) / L ** 0.5
        Wd = (torch.rand(N, 1, L, generator=g) * 2 - 1) / L ** 0.5
        enc.load_state_dict({"conv1d.weight": We})
        dec.load_state_dict({"conv_transpose1d.weight": Wd})
        x = torch.randn(3, 1, T, generator=g)
        w = enc(x).detach()
        y = dec(w).detach()
        rec["encdec_" + key] = {"We": We, "Wd": Wd, "x": x, "w": w, "y": y}

    # TimeDilatedConvNet standalone (separable, prelu, norm) causal and non-causal
    for causal in (False, True):
        cfg = O.OracleConfig(n_basis=8, kernel_size=4, sep_hidden_channels=24, sep_bottleneck_channels=12,
                             sep_skip_channels=10, sep_num_blocks=2, sep_num_layers=4, causal=causal)
        tdcn = TimeDilatedConvNet(12, hidden_channels=24, skip_channels=10, kernel_size=3, num_blocks=2, num_layers=4,
                                  dilated=True, separable=True, causal=causal, nonlinear="prelu", norm=True)
        full = O.synth_state_dict(cfg, seed=5)
        sub = {k[len("separator.tdcn."):]: v for k, v in full.items() if k.startswith("separator.tdcn.")}
        tdcn.load_state_dict(sub, strict=True)
        x = torch.randn(2, 12, 157, generator=g)
        rec[f"tdcn_causal{int(causal)}"] = {"cfg": cfg.to_dict(), "wseed": 5, "x": x, "y": tdcn(x).detach()}

    # SI-SDR / PIT: the reference self-test (src/criterion/pit.py:226-265: seed 111, randint(2,(4,2,1024))) + S=3,4
    torch.manual_seed(111)
    inp = torch.randint(2, (4, 2, 1024), dtype=torch.float)
    tgt = torch.randint(2, (4, 2, 1024), dtype=torch.float)
    crit = PIT1d(NegSISDR(), n_sources=2)
    loss, pattern = crit(inp, tgt)
    rec["pit_selftest"] = {"input": inp, "target": tgt, "loss": loss, "pattern": pattern}
    for S in (2, 3, 4):   # batch 2 keeps modules.pt under 1 MB; T = 3000 keeps the long per-pair reductions
        e = torch.randn(2, S, 3000, generator=g)
        t = torch.randn(2, S, 3000, generator=g)
        # make some estimates close to permuted targets so the permutation is non-trivial
        perm = torch.randperm(S, generator=g)
        if torch.equal(perm, torch.arange(S)):
            perm = perm.roll(1)
        e = 0.3 * e + t[:, perm]
        crit = PIT1d(NegSISDR(), n_sources=S)
        loss_b, pattern = crit(e, t, batch_mean=False)
        loss, _ = crit(e, t)
        rec[f"pit_S{S}"] = {"input": e, "target": t, "loss_b": loss_b, "loss": loss, "pattern": pattern,
                            "sisdr": sisdr(e, t)}
    # SI-SDR limits quoted in SURVEY.md 8a-12: zero target, perfect estimate, tie (identical estimates)
    t = torch.randn(2, 2, 500, generator=g)
    rec["sisdr_zero_target"] = sisdr(t, torch.zeros_like(t))
    rec["sisdr_perfect"] = sisdr(t, t.clone())
    rec["sisdr_limits_in"] = t
    e_tie = t[:, :1].repeat(1, 2, 1)
    crit = PIT1d(NegSISDR(), n_sources=2)
    l_tie, p_tie = crit(e_tie, t, batch_mean=False)
    rec["pit_tie"] = {"input": e_tie, "target": t, "loss_b": l_tie, "pattern": p_tie}
    path = os.path.join(HERE, "modules.pt")
    torch.save(rec, path)
    print("modules ->", os.path.getsize(path), "B")


def multichannel_case():
    """in_channels = n_mics = 2 (the 4-D input form, conv_tasnet.py:138-141,167-168; the MUSDB18 recipes): reference forward on a seeded
    stereo mixture, 3 sources"""
    cfg = O.OracleConfig(n_basis=32, kernel_size=8, sep_hidden_channels=48, sep_bottleneck_channels=16, sep_skip_channels=24,
                         sep_num_blocks=2, sep_num_layers=3, causal=False, n_sources=3, in_channels=2)
    ref = build_reference(cfg)
    assert [(k, tuple(v.shape)) for k, v in ref.state_dict().items()] == [(k, tuple(s)) for k, s in O.state_dict_spec(cfg)]
    sd = O.synth_state_dict(cfg, seed=31)
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    g = torch.Generator().manual_seed(32)
    mixture = 0.3 * torch.randn(2, 1, 2, 1501, generator=g)
    with torch.no_grad():
        out, latent = ref.extract_latent(mixture)
    rec = {"cfg": cfg.to_dict(), "wseed": 31, "mixture": mixture, "out": out.clone(), "latent": latent.clone()}
    path = os.path.join(HERE, "tiny_stereo.pt")
    torch.save(rec, path)
    print("tiny_stereo: out", tuple(out.shape), "->", os.path.getsize(path), "B")


def criteria_case():
    """SDR / NegSDR (src/criterion/sdr.py:6-110) and the clipped SI-SDR classes (:233-327) of the reference on seeded inputs; the
    estimates are noisy copies of the targets so that SDR spans roughly -5 .. 35 dB"""
    from criterion.sdr import SDR, NegSDR, ClippedSISDR, ClippedNegSISDR, sdr
    g = torch.Generator().manual_seed(77)
    rec = {}
    for name, shape in (("2d", (5, 1003)), ("3d", (3, 2, 1600)), ("4d", (2, 3, 2, 801))):
        tgt = torch.randn(shape, generator=g)
        noise = torch.randn(shape, generator=g) * torch.logspace(-2, 0.3, shape[0]).view(-1, *([1] * (len(shape) - 1)))
        est = tgt + noise
        r = {"input": est, "target": tgt, "sdr": sdr(est, tgt)}
        for red in ("mean", "sum", None):
            r[f"SDR_{red}"] = SDR(reduction=red)(est, tgt, batch_mean=False)
            r[f"NegSDR_{red}_bm"] = NegSDR(reduction=red)(est, tgt, batch_mean=True)
        r["ClippedSISDR_20"] = ClippedSISDR(max=20.0)(est, tgt, batch_mean=False)
        r["ClippedNegSISDR_-15"] = ClippedNegSISDR(min=-15.0)(est, tgt, batch_mean=False)
        r["ClippedNegSISDR_none_bm"] = ClippedNegSISDR(min=-15.0, reduction=None)(est, tgt, batch_mean=True)
        rec[name] = r
    path = os.path.join(HERE, "criteria.pt")
    torch.save(rec, path)
    print("criteria ->", os.path.getsize(path), "B")


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "criteria":
        criteria_case()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "stereo":
        multichannel_case()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "modules":
        module_cases()
        return
    paper = dict(n_basis=512, kernel_size=16, sep_hidden_channels=512, sep_bottleneck_channels=128,
                 sep_skip_channels=128, sep_num_blocks=3, sep_num_layers=8)
    if len(sys.argv) > 1 and sys.argv[1] == "softmax":
        tiny = dict(n_basis=16, kernel_size=4, sep_hidden_channels=16, sep_bottleneck_channels=8, sep_skip_channels=8,
                    sep_num_blocks=2, sep_num_layers=3)
        model_case("tiny_softmax", O.OracleConfig(**tiny, causal=False, mask_nonlinear="softmax"), batch=2, T=203, wseed=14, xseed=24)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "ckpt":
        checkpoint_case()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "dprnn":
        dprnn_cases()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "grad":   # mint only the training golden (the forward fixtures are unchanged)
        grad_case("paper_3spk_grad", O.OracleConfig(**paper, causal=False, n_sources=3), batch=2, T=8000, wseed=113, xseed=113)
        return
    tiny = dict(n_basis=16, kernel_size=4, sep_hidden_channels=16, sep_bottleneck_channels=8, sep_skip_channels=8,
                sep_num_blocks=2, sep_num_layers=3)
    model_case("tiny_gln", O.OracleConfig(**tiny, causal=False), batch=2, T=203, wseed=11, xseed=21)
    model_case("tiny_cln", O.OracleConfig(**tiny, causal=True), batch=2, T=203, wseed=12, xseed=22)
    model_case("tiny_softmax", O.OracleConfig(**tiny, causal=False, mask_nonlinear="softmax"), batch=2, T=203, wseed=14, xseed=24)
    small = dict(n_basis=64, kernel_size=16, sep_hidden_channels=96, sep_bottleneck_channels=32, sep_skip_channels=48,
                 sep_num_blocks=2, sep_num_layers=5)
    model_case("small_relu_3spk", O.OracleConfig(**small, causal=False, n_sources=3, enc_nonlinear="relu"),
               batch=3, T=2500, wseed=13, xseed=23)
    paper = dict(n_basis=512, kernel_size=16, sep_hidden_channels=512, sep_bottleneck_channels=128,
                 sep_skip_channels=128, sep_num_blocks=3, sep_num_layers=8)
    model_case("paper_2spk", O.OracleConfig(**paper, causal=False, n_sources=2), batch=2, T=32000, wseed=111, xseed=111,
               subsample=61)
    model_case("paper_3spk_short", O.OracleConfig(**paper, causal=False, n_sources=3), batch=1, T=8000, wseed=112,
               xseed=112, subsample=17)
    module_cases()
    grad_case("paper_3spk_grad", O.OracleConfig(**paper, causal=False, n_sources=3), batch=2, T=8000, wseed=113, xseed=113)
    dprnn_cases()
    checkpoint_case()


if __name__ == "__main__":
    main()
