"""Codebook training step (GPU) against the REAL reference: tests/golden/vqgan_train_small.npz holds two optimisation steps of the
unmodified reference VQGAN (train mode, perceptual_weight = 0, Adam betas (0.5, 0.9)) produced by oracle/make_golden.py —
loss terms, codes, per-parameter gradient norms and projections for ALL 120+ tensors, full gradients / weights for a dozen of them,
and the EMA-updated codebook.  Tolerances: the reference's own harness uses atol = rtol = 1e-5 on single layers
(viewformer/utils/testing.py:98); a 40-layer backward pass in fp32 with a different summation order lands at ~1e-4 relative."""
import os

import numpy as np
import pytest
import torch

from oracle import synth
from oracle.make_golden import SMALL_VQ, vq_images
from viewformer_b200.config import VQGANConfig

pytestmark = pytest.mark.gpu

# VF_TRAIN_TC: "1" (default) runs dense layers and 3x3 stride-1 convs on the exact split-fp16 tensor-core GEMM, "0" keeps the whole
# backward pass on the fp32 CUDA-core kernels (conv_wgrad with Linear layouts, the SIMT tied head and data gradients)
# Each golden training test below runs on the default path; a *_cuda_core twin runs the same checks, at the same tolerances, with
# VF_TRAIN_TC=0.


def test_vqgan_training_step_matches_reference(golden_dir, monkeypatch):
    _vqgan_training_step_vs_golden(golden_dir, "1", monkeypatch)


def test_vqgan_training_step_cuda_core_matches_reference(golden_dir, monkeypatch):
    _vqgan_training_step_vs_golden(golden_dir, "0", monkeypatch)


def _vqgan_training_step_vs_golden(golden_dir, train_tc, monkeypatch):
    from viewformer_b200 import VQGAN
    from viewformer_b200.train import VQGANTrainer
    monkeypatch.setenv("VF_TRAIN_TC", train_tc)
    g = np.load(os.path.join(golden_dir, "vqgan_train_small.npz"))
    cfg = VQGANConfig(**dict(SMALL_VQ, perceptual_weight=0.0))
    model = VQGAN(cfg, precision="fp32").load_state_dict(synth.make_vqgan_state_dict(cfg, 5))
    tr = VQGANTrainer(model, bucket_bytes=1 << 16)                 # small buckets: exercises the bucket bookkeeping
    assert tr.use_tc == (train_tc == "1")
    assert len(tr.buckets) > 3
    names = [str(n) for n in g["names"]]
    gen = torch.Generator().manual_seed(99)
    probe = None
    for step in range(2):
        x = vq_images(3, cfg.image_size, 2000 + step)
        loss = tr.forward_backward(x)
        torch.cuda.synchronize()
        assert sorted(tr.launched) == list(range(len(tr.buckets)))              # every gradient bucket was closed exactly once
        print(f"[train step {step}] loss {float(loss):.6f} (ref {float(g[f'loss{step}']):.6f}) rec {float(tr.last['rec_loss']):.6f} quant {float(tr.last['quant_loss']):.6f}")
        assert np.array_equal(tr.last["codes"].cpu().numpy(), g[f"codes{step}"])
        assert abs(float(loss) - float(g[f"loss{step}"])) < 2e-5 * max(1.0, abs(float(g[f"loss{step}"])))
        assert abs(float(tr.last["rec_loss"]) - float(g[f"rec{step}"])) < 2e-5 and abs(float(tr.last["quant_loss"]) - float(g[f"quant{step}"])) < 2e-5
        grads = tr.export_gradients()
        assert set(grads) == set(names)
        if probe is None:
            probe = {n: torch.randn(grads[n].shape, generator=gen) for n in names}
        worst = 0.0
        for i, n in enumerate(names):
            gn, gd = float(grads[n].norm()), float((grads[n] * probe[n]).sum())
            rn, rd = float(g[f"gnorm{step}"][i]), float(g[f"gdot{step}"][i])
            # conv biases that feed a GroupNorm with one channel per group have an exactly-zero true gradient: both sides hold rounding
            # noise (~1e-8) there, hence the absolute floor
            e = max(abs(gn - rn), abs(gd - rd)) / max(rn, 1e-4)
            worst = max(worst, e)
            assert e < 3e-3, f"step {step} {n}: |g| {gn:.6e} vs {rn:.6e}, <g,probe> {gd:.6e} vs {rd:.6e}"
        full = [k[len(f"g{step}."):] for k in g.files if k.startswith(f"g{step}.")]
        wfull = 0.0
        for n in full:
            ref = torch.from_numpy(g[f"g{step}.{n}"])
            err = float((grads[n] - ref).abs().max() / ref.abs().max().clamp_min(1e-4))
            wfull = max(wfull, err)
            assert err < 2e-3, f"step {step} grad {n}: max rel err {err:.3e}"
        print(f"[train step {step} VF_TRAIN_TC={train_tc}] gradients: worst norm/projection rel err {worst:.2e} over {len(names)} tensors; "
              f"worst element-wise {wfull:.2e} over {len(full)} tensors")
        tr.optimizer_step()
        sd = tr.export_state_dict()
        wp = 0.0
        for i, n in enumerate(names):
            pd, rd = float((sd[n] * probe[n]).sum()), float(g[f"pdot{step}"][i])
            wp = max(wp, abs(pd - rd) / max(abs(rd), float(probe[n].norm()) * cfg.learning_rate))
        for n in full:
            ref = torch.from_numpy(g[f"p{step}.{n}"])
            d = (sd[n] - ref).abs()
            # Adam's first steps move every weight by ~lr * sign(g): elements whose gradient is at rounding level may flip sign
            frac_bad = float((d > 0.05 * cfg.learning_rate).float().mean())
            assert frac_bad < 0.02, f"step {step} weight {n}: {frac_bad:.3%} elements differ by more than 5% of lr"
        emb = model._w["q"]["emb"].cpu().numpy()
        # step 1 starts from weights that already differ by Adam's sign flips of rounding-level gradients: looser there
        np.testing.assert_allclose(emb, g[f"emb{step}"], rtol=2e-4 if step == 0 else 5e-3, atol=2e-5 if step == 0 else 2e-4)
        print(f"[train step {step}] post-Adam weight projections: worst rel err {wp:.2e}")
    # the model serves inference with the trained weights (state_dict round trip through the reference key names)
    m2 = VQGAN(cfg, precision="fp32").load_state_dict(tr.export_state_dict())
    xq = vq_images(2, cfg.image_size, 7)
    assert torch.equal(m2.encode(xq)[2], model.encode(xq)[2])


def test_vqgan_training_step_full_size_matches_reference(golden_dir):
    """BASELINE configs[3] model (VQGANConfig defaults, 67.9 M parameters, 128x128 images): one optimisation step on a batch of 2 against
    the REAL reference (tests/golden/vqgan_train_full.npz): loss terms, the 128 codes, gradient norm and projection of all 342 tensors,
    post-Adam weight projections and the EMA-updated codebook."""
    from viewformer_b200 import VQGAN
    from viewformer_b200.train import VQGANTrainer
    g = np.load(os.path.join(golden_dir, "vqgan_train_full.npz"))
    cfg = VQGANConfig(perceptual_weight=0.0)
    model = VQGAN(cfg, precision="fp32").load_state_dict(synth.make_vqgan_state_dict(cfg, 5))
    tr = VQGANTrainer(model)
    names = [str(n) for n in g["names"]]
    x = vq_images(2, cfg.image_size, 3000)
    loss = tr.forward_backward(x)
    torch.cuda.synchronize()
    print(f"[full-size train step] loss {float(loss):.6f} (ref {float(g['loss']):.6f}) rec {float(tr.last['rec_loss']):.6f} quant {float(tr.last['quant_loss']):.6f}; "
          f"{len(tr.buckets)} gradient buckets")
    assert np.array_equal(tr.last["codes"].cpu().numpy(), g["codes"])
    assert abs(float(loss) - float(g["loss"])) < 2e-5 * max(1.0, abs(float(g["loss"])))
    assert abs(float(tr.last["rec_loss"]) - float(g["rec"])) < 2e-5 and abs(float(tr.last["quant_loss"]) - float(g["quant"])) < 2e-5
    grads = tr.export_gradients()
    assert set(grads) == set(names)
    gen = torch.Generator().manual_seed(99)
    probe = {n: torch.randn(grads[n].shape, generator=gen) for n in names}
    worst = 0.0
    for i, n in enumerate(names):
        gn, gd = float(grads[n].norm()), float((grads[n] * probe[n]).sum())
        rn, rd = float(g["gnorm"][i]), float(g["gdot"][i])
        e = max(abs(gn - rn), abs(gd - rd)) / max(rn, 1e-4)
        worst = max(worst, e)
        assert e < 5e-3, f"{n}: |g| {gn:.6e} vs {rn:.6e}, <g,probe> {gd:.6e} vs {rd:.6e}"
    print(f"[full-size train step] gradients: worst norm/projection rel err {worst:.2e} over {len(names)} tensors")
    tr.optimizer_step()
    emb = model._w["q"]["emb"].double().cpu()
    ge = torch.Generator().manual_seed(7)
    assert abs(float(emb.norm()) - float(g["emb_norm"])) < 1e-5 * float(g["emb_norm"])
    assert abs(float((emb * torch.randn(emb.shape, generator=ge).double()).sum()) - float(g["emb_dot"])) < 2e-4 * float(g["emb_norm"])


def test_vqgan_commit_quantizer_training_step_matches_reference(golden_dir, monkeypatch):
    """``VQGAN(quantizer="commit")`` = the reference's gradient-trained ``Quantize`` (utils_th.py:75-124, beta = 0.25) in place of QuantizeEMA:
    two optimisation steps against tests/golden/vqgan_train_commit_small.npz (the real reference VQGAN with its own Quantize class dropped
    in, oracle/make_golden.py) — loss (1 + beta) * mean((q - z)^2), codes, gradients of every tensor incl. the codebook, post-Adam codebook."""
    _vqgan_commit_training_step_vs_golden(golden_dir, "1", monkeypatch)


def test_vqgan_commit_quantizer_training_step_cuda_core_matches_reference(golden_dir, monkeypatch):
    _vqgan_commit_training_step_vs_golden(golden_dir, "0", monkeypatch)


def _vqgan_commit_training_step_vs_golden(golden_dir, train_tc, monkeypatch):
    from viewformer_b200 import VQGAN
    from viewformer_b200.train import VQGANTrainer
    monkeypatch.setenv("VF_TRAIN_TC", train_tc)
    g = np.load(os.path.join(golden_dir, "vqgan_train_commit_small.npz"))
    cfg = VQGANConfig(**dict(SMALL_VQ, perceptual_weight=0.0))
    sd = synth.make_vqgan_state_dict(cfg, 5)
    sd = {k: v for k, v in sd.items() if not k.startswith("quantize.") or k == "quantize.embeddings"}
    sd["quantize.embeddings"] = torch.from_numpy(g["emb_init"])
    model = VQGAN(cfg, precision="fp32", quantizer="commit", beta=0.25).load_state_dict(sd)
    assert "quantize.counter" not in model.expected_keys()
    tr = VQGANTrainer(model, bucket_bytes=1 << 16)
    assert tr.use_tc == (train_tc == "1")
    names = [str(n) for n in g["names"]]
    assert "quantize.embeddings" in names
    gen = torch.Generator().manual_seed(99)
    probe = None
    for step in range(2):
        x = vq_images(3, cfg.image_size, 2000 + step)
        loss = tr.forward_backward(x)
        torch.cuda.synchronize()
        assert sorted(tr.launched) == list(range(len(tr.buckets)))
        print(f"[commit-quantizer train step {step}] loss {float(loss):.6f} (ref {float(g[f'loss{step}']):.6f}) quant {float(tr.last['quant_loss']):.6f}")
        assert np.array_equal(tr.last["codes"].cpu().numpy(), g[f"codes{step}"])
        assert abs(float(loss) - float(g[f"loss{step}"])) < 2e-5 * max(1.0, abs(float(g[f"loss{step}"])))
        assert abs(float(tr.last["quant_loss"]) - float(g[f"quant{step}"])) < 2e-5
        grads = tr.export_gradients()
        assert set(grads) == set(names)
        if probe is None:
            probe = {n: torch.randn(grads[n].shape, generator=gen) for n in names}
        worst = 0.0
        for i, n in enumerate(names):
            gn, gd = float(grads[n].norm()), float((grads[n] * probe[n]).sum())
            rn, rd = float(g[f"gnorm{step}"][i]), float(g[f"gdot{step}"][i])
            e = max(abs(gn - rn), abs(gd - rd)) / max(rn, 1e-4)
            worst = max(worst, e)
            # step 0 is the parity check proper (identical weights on both sides).  Step 1 starts from weights AND a codebook that differ by
            # Adam's +-lr sign flips wherever a first-step gradient sits at rounding level, which moves the early-layer gradients by a few
            # per cent; there the loss, the codes and the order of magnitude of every gradient are checked.
            assert e < (3e-3 if step == 0 else 0.15), f"step {step} {n}: |g| {gn:.6e} vs {rn:.6e}, <g,probe> {gd:.6e} vs {rd:.6e}"
        for n in [k[len(f"g{step}."):] for k in g.files if k.startswith(f"g{step}.")]:
            ref = torch.from_numpy(g[f"g{step}.{n}"])
            err = float((grads[n] - ref).abs().max() / ref.abs().max().clamp_min(1e-4))
            assert err < (2e-3 if step == 0 else 0.15), f"step {step} grad {n}: max rel err {err:.3e}"
        print(f"[commit-quantizer train step {step} VF_TRAIN_TC={train_tc}] gradients: worst norm/projection rel err {worst:.2e} over {len(names)} tensors")
        tr.optimizer_step()
        emb = model._w["q"]["emb"].cpu()
        ref = torch.from_numpy(g[f"p{step}.quantize.embeddings"])
        frac_bad = float(((emb - ref).abs() > 0.05 * cfg.learning_rate).float().mean())
        assert frac_bad < 0.02, f"step {step}: {frac_bad:.3%} codebook elements differ by more than 5% of lr after Adam"
        # the lookup tables follow the gradient step (transposed copy, |e|^2, decode table)
        assert torch.allclose(model._w["q"]["et"].cpu(), emb.t(), atol=0) and torch.allclose(model._w["q"]["esq"].cpu(), (emb * emb).sum(0), rtol=1e-5)
    m2 = VQGAN(cfg, precision="fp32", quantizer="commit").load_state_dict(tr.export_state_dict())
    xq = vq_images(2, cfg.image_size, 7)
    assert torch.equal(m2.encode(xq)[2], model.encode(xq)[2])


def test_migt_training_step_matches_oracle_autograd(golden_dir, monkeypatch):
    """MIGT.train_step (migt.py:464-505): three optimisation steps against tests/golden/migt_train_small.npz — gradients from torch
    autograd through the oracle's forward, optimizer / schedule restated from models/utils.py (oracle/make_golden.py).  The fixture is
    reproduced by the reference's own MIGT.train_step executed over oracle/tf_shim.py (tests/test_reference_on_shim.py, CPU, container)."""
    _migt_training_step_vs_golden(golden_dir, "1", monkeypatch)


def test_migt_training_step_cuda_core_matches_oracle_autograd(golden_dir, monkeypatch):
    _migt_training_step_vs_golden(golden_dir, "0", monkeypatch)


def _migt_training_step_vs_golden(golden_dir, train_tc, monkeypatch):
    from viewformer_b200 import MIGT
    from viewformer_b200.train_migt import MIGTTrainer
    from viewformer_b200.config import MIGTConfig
    from oracle.make_golden import MIGT_TRAIN, MIGT_TRAIN_WARMUP
    from oracle import migt_oracle as mo
    monkeypatch.setenv("VF_TRAIN_TC", train_tc)
    g = np.load(os.path.join(golden_dir, "migt_train_small.npz"))
    cfg = MIGTConfig(**MIGT_TRAIN)
    model = MIGT(cfg, precision="fp32").load_state_dict(synth.make_migt_state_dict(cfg, 9))
    tr = MIGTTrainer(model, warmup_steps=MIGT_TRAIN_WARMUP, bucket_bytes=1 << 18)
    assert tr.use_tc == (train_tc == "1")
    assert len(tr.buckets) > 2
    names = [str(n) for n in g["names"]]
    gen = torch.Generator().manual_seed(77)
    probe = {k: torch.randn(tuple(tr.p[k].shape), generator=gen) for k in names}
    full = [k[3:] for k in g.files if k.startswith("g0.")]
    B, T = 2, 4
    for step in range(3):
        codes = synth.make_codes(B, T, n_embed=cfg.n_embeddings, seed=50 + step)
        cams = mo.normalize_cameras(mo.to_relative_cameras(synth.make_cameras(B, T, seed=60 + step))[0])
        assert abs(tr.learning_rate() - float(g[f"lr{step}"])) < 1e-9
        loss = tr.forward_backward(cams, codes)
        torch.cuda.synchronize()
        assert sorted(tr.launched) == list(range(len(tr.buckets)))
        print(f"[migt train step {step}] loss {float(loss):.6f} (ref {float(g[f'loss{step}']):.6f}) lr {tr.learning_rate():.2e}")
        assert abs(float(loss) - float(g[f"loss{step}"])) < 3e-5 * abs(float(g[f"loss{step}"]))
        np.testing.assert_allclose(tr.last["ce_loss"].cpu().numpy(), g[f"ce{step}"], rtol=3e-5)
        np.testing.assert_allclose(tr.last["pose_loss"].cpu().numpy(), g[f"pose{step}"], rtol=1e-4)
        grads = tr.gradients()
        worst = 0.0
        for i, n in enumerate(names):
            gn, gd = float(grads[n].norm()), float((grads[n] * probe[n]).sum())
            rn, rd = float(g[f"gnorm{step}"][i]), float(g[f"gdot{step}"][i])
            e = max(abs(gn - rn), abs(gd - rd)) / max(rn, 1e-4)
            worst = max(worst, e)
            assert e < 3e-3, f"step {step} {n}: |g| {gn:.6e} vs {rn:.6e}, <g,probe> {gd:.6e} vs {rd:.6e}"
        wfull = 0.0
        for n in full:
            ref = torch.from_numpy(g[f"g{step}.{n}"])
            err = float((grads[n] - ref).abs().max() / ref.abs().max().clamp_min(1e-4))
            wfull = max(wfull, err)
            assert err < 2e-3, f"step {step} grad {n}: max rel err {err:.3e}"
        print(f"[migt train step {step} VF_TRAIN_TC={train_tc}] gradients: worst norm/projection rel err {worst:.2e} over {len(names)} tensors; worst element-wise {wfull:.2e}")
        tr.optimizer_step()
        sd = tr.state_dict()
        lr = max(float(g[f"lr{step}"]), 1e-12)
        for n in full:
            ref = torch.from_numpy(g[f"p{step}.{n}"])
            d = (sd[n] - ref).abs()
            frac_bad = float((d > 0.05 * lr + 1e-7).float().mean())
            assert frac_bad < 0.02, f"step {step} weight {n}: {frac_bad:.3%} elements differ by more than 5% of lr"
    # trained weights serve inference through the ordinary model class
    m2 = MIGT(cfg, precision="fp32").load_state_dict(tr.state_dict())
    out = m2(dict(input_ids=codes, poses=cams))
    assert torch.isfinite(out["logits"]).all()


def test_migt_dynamic_pose_loss_and_weight_schedule():
    """use_dynamic_pose_loss (DynamicLossWeightingCriterion, migt.py:107-120) + a non-constant localization_weight schedule
    (utils/schedules.py; evaluated at the train counter, migt.py:446): loss and gradients of the trainer against torch autograd through the
    oracle's forward at the same step; the inference-mode ``compute_losses=True`` call reports the same loss."""
    from viewformer_b200 import MIGT
    from viewformer_b200.train_migt import MIGTTrainer
    from viewformer_b200.config import MIGTConfig
    from viewformer_b200.schedules import parse
    from oracle.make_golden import MIGT_TRAIN
    from oracle import migt_oracle as mo
    sched = "warmup(cosine(1,0.25,40),4)"
    cfg = MIGTConfig(**dict(MIGT_TRAIN, use_dynamic_pose_loss=True, localization_weight=sched, total_steps=50))
    sd = synth.make_migt_state_dict(cfg, 11)
    sd["pose_loss_weighting_criterion.pos_ori_weights"] = torch.tensor([0.3, -1.2])
    model = MIGT(cfg, precision="fp32").load_state_dict(sd)
    tr = MIGTTrainer(model, warmup_steps=2, bucket_bytes=1 << 18)
    B, T = 3, 4
    codes = synth.make_codes(B, T, n_embed=cfg.n_embeddings, seed=91)
    cams = mo.normalize_cameras(mo.to_relative_cameras(synth.make_cameras(B, T, seed=92))[0])
    for step in (0, 3, 17):
        tr.iterations = step
        lw = parse(sched).with_total_steps(50)(step)
        assert abs(tr.loc_weight - lw) < 1e-12
        loss = tr.forward_backward(cams, codes)
        torch.cuda.synchronize()
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        o = mo.forward(leaves, cfg, dict(input_ids=codes, poses=cams), compute_losses=True, localization_weight=lw)
        ref = o["loss"].mean()
        ref.backward()
        print(f"[migt dynamic pose loss] step {step}: localization_weight {lw:.4f} loss {float(loss):.6f} (oracle {float(ref):.6f})")
        assert abs(float(loss) - float(ref)) < 3e-5 * abs(float(ref))
        grads = tr.gradients()
        for k in ("pose_loss_weighting_criterion.pos_ori_weights", "pose_classifier.c_proj.weight", "pose_classifier.c_fc.bias", "h.1.mlp.c_fc.weight", "ln_f.gamma"):
            want = leaves[k].grad if leaves[k].grad is not None else torch.zeros_like(leaves[k])
            err = float((grads[k] - want).abs().max() / want.abs().max().clamp_min(1e-5))
            assert err < 3e-3, f"step {step} grad {k}: rel err {err:.3e}"
    model._train_counter = 17
    out = model(dict(input_ids=codes, poses=cams), compute_losses=True)
    assert abs(float(out["loss"].mean()) - float(ref)) < 3e-5 * abs(float(ref))
    assert abs(out["localization_weight"] - lw) < 1e-9 and abs(out["dynamic_loss_weight_ori"] + 1.2) < 1e-6


def test_migt_training_step_full_size_matches_oracle_autograd(golden_dir):
    """Full-size transformer (MIGTConfig defaults: 12 layers, d = 768): loss terms and the gradient of all 156 tensors of one training step
    (B = 1, T = 5, dropout 0) against torch autograd through the oracle (tests/golden/migt_train_full.npz, reproduced by the reference's own
    train_step over oracle/tf_shim.py in tests/test_reference_on_shim.py)."""
    from viewformer_b200 import MIGT
    from viewformer_b200.train_migt import MIGTTrainer
    from viewformer_b200.config import MIGTConfig
    from oracle import migt_oracle as mo
    g = np.load(os.path.join(golden_dir, "migt_train_full.npz"))
    cfg = MIGTConfig(dropout=0.0, label_smoothing=0.1, localization_weight="0.7", total_steps=100, learning_rate=1e-4)
    model = MIGT(cfg, precision="fp32").load_state_dict(synth.make_migt_state_dict(cfg, 13))
    tr = MIGTTrainer(model)
    B, T = 1, 5
    codes = synth.make_codes(B, T, n_embed=cfg.n_embeddings, seed=70)
    cams = mo.normalize_cameras(mo.to_relative_cameras(synth.make_cameras(B, T, seed=71))[0])
    loss = tr.forward_backward(cams, codes)
    torch.cuda.synchronize()
    print(f"[migt full-size train step] loss {float(loss):.6f} (ref {float(g['loss']):.6f})")
    assert abs(float(loss) - float(g["loss"])) < 3e-5 * abs(float(g["loss"]))
    np.testing.assert_allclose(tr.last["ce_loss"].cpu().numpy(), g["ce"], rtol=3e-5)
    np.testing.assert_allclose(tr.last["pose_loss"].cpu().numpy(), g["pose"], rtol=2e-4)
    names = [str(n) for n in g["names"]]
    grads = tr.gradients()
    gen = torch.Generator().manual_seed(78)
    worst = 0.0
    for i, n in enumerate(names):
        pr = torch.randn(tuple(grads[n].shape), generator=gen)
        gn, gd = float(grads[n].norm()), float((grads[n] * pr).sum())
        rn, rd = float(g["gnorm"][i]), float(g["gdot"][i])
        e = max(abs(gn - rn), abs(gd - rd)) / max(rn, 1e-4)
        worst = max(worst, e)
        assert e < 3e-3, f"{n}: |g| {gn:.6e} vs {rn:.6e}, <g,probe> {gd:.6e} vs {rd:.6e}"
    print(f"[migt full-size train step] gradients: worst norm/projection rel err {worst:.2e} over {len(names)} tensors")


def _vqgan_grads(train_tc, monkeypatch):
    from viewformer_b200 import VQGAN
    from viewformer_b200.train import VQGANTrainer
    monkeypatch.setenv("VF_TRAIN_TC", train_tc)
    cfg = VQGANConfig(**dict(SMALL_VQ, perceptual_weight=0.0))
    tr = VQGANTrainer(VQGAN(cfg, precision="fp32").load_state_dict(synth.make_vqgan_state_dict(cfg, 5)))
    assert tr.use_tc == (train_tc == "1")
    loss = float(tr.forward_backward(vq_images(3, cfg.image_size, 2000)))
    return loss, tr.export_gradients()


def _migt_grads(train_tc, monkeypatch):
    from viewformer_b200 import MIGT
    from viewformer_b200.train_migt import MIGTTrainer
    from viewformer_b200.config import MIGTConfig
    from oracle.make_golden import MIGT_TRAIN, MIGT_TRAIN_WARMUP
    from oracle import migt_oracle as mo
    monkeypatch.setenv("VF_TRAIN_TC", train_tc)
    cfg = MIGTConfig(**MIGT_TRAIN)
    tr = MIGTTrainer(MIGT(cfg, precision="fp32").load_state_dict(synth.make_migt_state_dict(cfg, 9)), warmup_steps=MIGT_TRAIN_WARMUP)
    assert tr.use_tc == (train_tc == "1")
    codes = synth.make_codes(2, 4, n_embed=cfg.n_embeddings, seed=50)
    cams = mo.normalize_cameras(mo.to_relative_cameras(synth.make_cameras(2, 4, seed=60))[0])
    loss = float(tr.forward_backward(cams, codes))
    return loss, tr.gradients()


PATHS_TOL = 4e-5        # measured on a B200 (1000 W): VQGAN 7.7e-6 (a GroupNorm gamma), MIGT 1.1e-6


@pytest.mark.parametrize("model", ["vqgan", "migt"])
def test_cuda_core_and_tensor_core_backward_agree(model, monkeypatch):
    """Both backward paths are fp32-faithful, so on the same weights and batch their gradients agree tensor by tensor far more closely
    than either agrees with the reference's golden norms.  A bias gradient sum(dy) is formed from the same terms as its weight gradient
    sum(x dy), so its rounding is measured against the larger of the two: a conv bias in front of a GroupNorm with one channel per
    group has an exactly-zero true gradient, and both paths hold rounding noise there."""
    run = _vqgan_grads if model == "vqgan" else _migt_grads
    loss_tc, g_tc = run("1", monkeypatch)
    loss_cc, g_cc = run("0", monkeypatch)
    assert set(g_tc) == set(g_cc)
    print(f"[{model} backward paths] loss tensor-core {loss_tc:.8f} CUDA-core {loss_cc:.8f}")
    assert abs(loss_tc - loss_cc) < 1e-5 * abs(loss_tc)
    errs = {}
    for n in g_tc:
        scale = float(g_tc[n].abs().max())
        if n.endswith(".bias") and n[:-5] + ".weight" in g_tc:
            scale = max(scale, float(g_tc[n[:-5] + ".weight"].abs().max()))
        errs[n] = float((g_tc[n] - g_cc[n]).abs().max()) / max(scale, 1e-30)
    top = sorted(errs.items(), key=lambda kv: -kv[1])[:4]
    print(f"[{model} backward paths] worst per-tensor max error / max|g| over {len(errs)} tensors: " + ", ".join(f"{n} {e:.2e}" for n, e in top))
    bad = {n: e for n, e in errs.items() if e >= PATHS_TOL}
    assert not bad, f"gradients of the two backward paths differ: {bad}"


# one tensor per dropout site: embeddings, attention probabilities, attention output, MLP output; plus the pose embedding
FD_TENSORS = ["wpe.embeddings", "h.0.attn.c_attn.weight", "h.1.attn.c_proj.weight", "h.1.mlp.c_proj.weight", "pose_embedding.c_fc.weight"]
# measured on a B200 (1000 W): control (dropout 0) 4.0e-3, dropout 0.1 3.7e-3, both at pose_embedding.c_fc.weight; with the attention-
# output mask of the backward pass taken from the MLP-output site the dropout run reaches 2.0e-2 .. 3.5e-2
FD_TOL = 1e-2


def _migt_fd_errors(dropout):
    """Central differences of the trainer's own loss along a unit direction per tensor, against <g, v>.  The dropout masks depend only
    on (seed, iterations, site) and forward_backward does not advance iterations, so every evaluation sees the same masks.
    The direction is half the normalised analytic gradient, half random: along a purely random direction <g, v> ~ |g| / sqrt(numel),
    and the step h that moves the loss by 1e-3 of itself (well above its fp32 rounding) leaves the linear regime.  An analytic gradient
    that is wrong anywhere in the tensor still shows, through both halves."""
    from viewformer_b200 import MIGT
    from viewformer_b200.train_migt import MIGTTrainer
    from viewformer_b200.config import MIGTConfig
    from oracle.make_golden import MIGT_TRAIN, MIGT_TRAIN_WARMUP
    from oracle import migt_oracle as mo
    cfg = MIGTConfig(**dict(MIGT_TRAIN, dropout=dropout))
    tr = MIGTTrainer(MIGT(cfg, precision="fp32").load_state_dict(synth.make_migt_state_dict(cfg, 9)), warmup_steps=MIGT_TRAIN_WARMUP, seed=3)
    assert tr.use_tc
    tr.iterations = 5
    codes = synth.make_codes(2, 4, n_embed=cfg.n_embeddings, seed=50)
    cams = mo.normalize_cameras(mo.to_relative_cameras(synth.make_cameras(2, 4, seed=60))[0])

    def loss_at():
        tr._wsplit = {}                         # as optimizer_step does: the split-fp16 weight copies follow tr.p
        return float(tr.forward_backward(cams, codes))

    loss0 = loss_at()
    grads = tr.gradients()
    gen = torch.Generator().manual_seed(5)
    errs = {}
    for name in FD_TENSORS:
        p = tr.p[name]
        gd = grads[name].double()
        r = torch.randn(tuple(p.shape), generator=gen, dtype=torch.float64)
        v = gd / gd.norm() + r / r.norm()
        v /= v.norm()
        gv = float((gd * v).sum())
        h = 1e-3 * abs(loss0) / abs(gv)
        orig = p.clone()
        p.copy_((orig.double() + h * v.to(p.device)).float())
        lp = loss_at()
        p.copy_((orig.double() - h * v.to(p.device)).float())
        lm = loss_at()
        p.copy_(orig)
        fd = (lp - lm) / (2 * h)
        errs[name] = abs(fd - gv) / abs(gv)
        print(f"[migt FD dropout={dropout}] {name}: <g,v> {gv:.6e} central difference {fd:.6e} (h {h:.2e}) rel err {errs[name]:.2e}")
    assert loss_at() == loss0                   # the weights are restored
    return tr, loss0, errs, loss_at


def test_migt_dropout_gradients_match_finite_differences():
    """MIGT with dropout 0.1 (the config default) at all four dropout sites: the analytic gradient of the trainer against central
    differences of its own loss.  The same harness at dropout 0, where the gradient is validated against the oracle golden, measures
    the accuracy of the finite differences; the dropout run is held to the same bound.  A missing 1/(1-rate) at one site would move
    that site's gradients by ~11%, a mask from the wrong site by far more."""
    _, loss_ctl, errs_ctl, _ = _migt_fd_errors(0.0)
    tr, loss_do, errs_do, loss_at = _migt_fd_errors(0.1)
    print(f"[migt FD] worst rel err: control {max(errs_ctl.values()):.2e}, dropout 0.1 {max(errs_do.values()):.2e} (bound {FD_TOL:.0e})")
    assert max(errs_ctl.values()) < FD_TOL
    assert max(errs_do.values()) < FD_TOL
    # the loss is a deterministic function of (weights, batch, seed, iterations): no forward kernel accumulates with atomics
    assert loss_at() == loss_do
    assert loss_do != loss_ctl
    tr.iterations += 1
    assert loss_at() != loss_do                 # new masks at the next step
