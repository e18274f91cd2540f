"""TEST INFRASTRUCTURE — regenerate tests/golden/*.npz from the REAL reference (container only).

    python -m oracle.make_golden

VQGAN fixtures are produced by the unmodified reference modules loaded from /root/reference
(oracle/ref_loader.py); weights and inputs come from oracle/synth.py so that the GPU box (which has no
/root/reference) can rebuild the same state_dict and compare its outputs with these files.
MIGT fixtures (migt_small / migt_full / migt_train_*) are written from the restatement (oracle/migt_oracle.py) and REPRODUCED by the
reference's own TensorFlow sources executed over oracle/tf_shim.py (tests/test_reference_on_shim.py); migt_reference_shim.npz is written
directly from that reference-on-shim run.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import synth, ref_loader, migt_oracle  # noqa: E402
from viewformer_b200.config import VQGANConfig, MIGTConfig  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

SMALL_VQ = dict(ch=32, ch_mult=[1, 2, 2], attn_resolutions=[8], image_size=32, embed_dim=16,
                z_channels=16, n_embed=64)
SMALL_MIGT = dict(n_layer=2, n_head=4, d_model=128, sequence_size=4, n_loss_skip=1)


def vq_images(n, size, seed):
    u8 = synth.make_images_uint8(1, n, size=size, seed=seed)[0]            # [n,H,W,3]
    return migt_oracle.images_to_float(u8).permute(0, 3, 1, 2).contiguous()


def golden_vqgan(tag, overrides, n_images, seed):
    cfg = VQGANConfig(**overrides)
    sd = synth.make_vqgan_state_dict(cfg, seed)
    ref = ref_loader.build_reference_vqgan(sd, **overrides)
    x = vq_images(n_images, cfg.image_size, 1000 + seed)
    with torch.no_grad():
        z = ref.quant_conv(ref.encoder(x))
        quant, diff, codes = ref.encode(x)
        dec = ref.decode_code(codes)
        rec, diff2, _, _ = ref(x)
    full = tag == "small"
    np.savez_compressed(
        os.path.join(OUT, f"vqgan_{tag}.npz"),
        seed=seed, n_images=n_images,
        z=z.numpy(), codes=codes.numpy(), diff=diff.numpy(),
        quant_sample=quant[:1].numpy(),
        dec=(dec if full else dec[:, :, ::4, ::4]).numpy(), dec0=dec[0].numpy(),
        dec_mean=dec.mean().numpy(), dec_std=dec.std().numpy(),
        rec_absmean=(rec - x).abs().mean().numpy())
    print(tag, "codes", codes.shape, "diff", float(diff), "dec std", float(dec.std()))


def golden_quantizer():
    """QuantizeEMA training branch + Quantize(beta=.25) on a seeded z (utils_th.py:46-64, 93-120)."""
    _, uth, _ = ref_loader.load_reference_modules()
    g = torch.Generator().manual_seed(7)
    D, K = 16, 64
    q = uth.QuantizeEMA(D, K)
    E = synth._uniform((D, K), 3 ** 0.5, g)
    q.embeddings.copy_(E)
    z = torch.randn((3, D, 4, 4), generator=g)
    q.train()
    outs = {}
    for step in range(2):
        quant, diff, ids = q(z)
        outs[f"ids{step}"] = ids.numpy()
        outs[f"diff{step}"] = diff.detach().numpy()
        outs[f"emb{step}"] = q.embeddings.clone().numpy()
        outs[f"cs{step}"] = q.ema_cluster_size_hidden.clone().numpy()
        outs[f"dw{step}"] = q.ema_dw_hidden.clone().numpy()
    q2 = uth.Quantize(D, K)
    with torch.no_grad():
        q2.embeddings.copy_(E)
    quant, loss, ids = q2(z)
    np.savez_compressed(os.path.join(OUT, "quantizer.npz"), E=E.numpy(), z=z.numpy(),
                        commit_loss=loss.detach().numpy(), commit_ids=ids.numpy(), **outs)
    print("quantizer ok")


def golden_lookup():
    """Nearest-neighbour indices of the reference's own expression (utils_th.py:36-41) on seeded rows,
    including adversarial near-ties (midpoints of two codes)."""
    g = torch.Generator().manual_seed(11)
    D, K = 256, 1024
    E = synth._uniform((D, K), 3 ** 0.5, g)
    z = torch.randn((4096, D), generator=g)
    a = torch.randint(0, K, (512,), generator=g)
    b = torch.randint(0, K, (512,), generator=g)
    mid = 0.5 * (E[:, a] + E[:, b]).t() + 1e-3 * torch.randn((512, D), generator=g)
    z = torch.cat([z, mid, E[:, :64].t().contiguous()], 0)
    dist = z.pow(2).sum(1, keepdim=True) - 2 * z @ E + E.pow(2).sum(0, keepdim=True)
    idx = (-dist).max(1)[1]
    d64 = (z.double()[:, :, None] - E.double()[None]).pow(2).sum(1)
    top2 = d64.topk(2, dim=1, largest=False)
    np.savez_compressed(os.path.join(OUT, "vq_lookup.npz"), seed=11, idx=idx.numpy(),
                        idx_f64=top2.indices[:, 0].numpy(), gap_f64=(top2.values[:, 1] - top2.values[:, 0]).numpy())
    print("lookup: fp32 vs fp64 mismatches", int((idx != top2.indices[:, 0]).sum()))


def golden_migt():
    for tag, overrides, B, T in (("small", SMALL_MIGT, 2, 4), ("full", {}, 1, 10)):
        cfg = MIGTConfig(**overrides)
        sd = synth.make_migt_state_dict(cfg, 3)
        codes = synth.make_codes(B, T, seed=5)
        cams = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(B, T, seed=6))[0])
        ids = torch.cat([codes[:, :-1], torch.full_like(codes[:, :1], cfg.n_embeddings)], 1)
        with torch.no_grad():
            o = migt_oracle.forward(sd, cfg, dict(input_ids=ids, poses=cams))
            o2 = migt_oracle.forward(sd, cfg, dict(input_ids=codes, poses=cams[:, :-1]))
        last = o["logits"][:, -1]
        np.savez_compressed(os.path.join(OUT, f"migt_{tag}.npz"), B=B, T=T,
                            logits_last=last[:1].numpy().astype(np.float32),
                            argmax_last=last.argmax(-1).numpy(),
                            pose_last=migt_oracle.reduce_cameras(o2["pose_prediction"][:, -1:], -2).numpy())
        print("migt", tag, "logit std", float(last.std()))


def golden_vqgan_train():
    """Two optimisation steps of the REAL reference codebook (vqgan_th.py:395-423, 443-445; train mode: QuantizeEMA updates the
    codebook; perceptual_weight = 0 because LPIPS weights are not available): loss, gradients and post-step weights."""
    overrides = dict(SMALL_VQ, perceptual_weight=0.0)
    cfg = VQGANConfig(**overrides)
    sd = synth.make_vqgan_state_dict(cfg, 5)
    ref = ref_loader.build_reference_vqgan(sd, **overrides)
    ref.train()
    opt = torch.optim.Adam(ref.parameters(), lr=cfg.learning_rate, betas=(0.5, 0.9))          # configure_optimizers
    g = torch.Generator().manual_seed(99)
    names = [n for n, _ in ref.named_parameters()]
    probe = {n: torch.randn(p.shape, generator=g) for n, p in ref.named_parameters()}
    keep = ["encoder.conv_in.weight", "encoder.down.0.block.0.norm1.weight", "encoder.down.1.downsample.conv.weight", "encoder.mid.attn_1.q.weight",
            "encoder.mid.attn_1.proj_out.bias", "quant_conv.weight", "post_quant_conv.bias", "decoder.up.1.upsample.conv.weight",
            "decoder.up.0.block.2.conv2.weight", "decoder.up.0.block.0.nin_shortcut.weight", "decoder.conv_out.bias", "decoder.norm_out.bias"]
    out = dict(names=np.array(names))
    for step in range(2):
        x = vq_images(3, cfg.image_size, 2000 + step)
        opt.zero_grad()
        xrec, qloss, _, codes = ref(x)
        loss, log = ref._compute_loss(qloss, x, xrec, split="train")
        loss.backward()
        out[f"loss{step}"] = loss.detach().numpy()
        out[f"rec{step}"] = log["train/rec_loss"].numpy()
        out[f"quant{step}"] = log["train/quant_loss"].numpy()
        out[f"codes{step}"] = codes.numpy()
        out[f"gnorm{step}"] = np.array([float(p.grad.norm()) for _, p in ref.named_parameters()])
        out[f"gdot{step}"] = np.array([float((p.grad * probe[n]).sum()) for n, p in ref.named_parameters()])
        for k in keep:
            out[f"g{step}.{k}"] = dict(ref.named_parameters())[k].grad.numpy().copy()
        opt.step()
        out[f"pdot{step}"] = np.array([float((p.detach() * probe[n]).sum()) for n, p in ref.named_parameters()])
        for k in keep:
            out[f"p{step}.{k}"] = dict(ref.named_parameters())[k].detach().numpy().copy()
        out[f"emb{step}"] = ref.quantize.embeddings.numpy().copy()
    np.savez_compressed(os.path.join(OUT, "vqgan_train_small.npz"), **out)
    print("train golden: losses", float(out["loss0"]), float(out["loss1"]))


def golden_vqgan_train_full():
    """ONE optimisation step of the real reference codebook at the FULL BASELINE size (VQGANConfig defaults: 128x128 images, ch 128,
    ch_mult [1,1,2,2,4], 1024 x 256 codebook; 67.9 M parameters), batch of 2: loss terms, codes, gradient norm and a random projection of
    every parameter tensor, the EMA-updated codebook's projections.  Small file: no full tensors."""
    overrides = dict(perceptual_weight=0.0)
    cfg = VQGANConfig(**overrides)
    sd = synth.make_vqgan_state_dict(cfg, 5)
    ref = ref_loader.build_reference_vqgan(sd, **overrides)
    ref.train()
    opt = torch.optim.Adam(ref.parameters(), lr=cfg.learning_rate, betas=(0.5, 0.9))
    g = torch.Generator().manual_seed(99)
    names = [n for n, _ in ref.named_parameters()]
    probe = {n: torch.randn(p.shape, generator=g) for n, p in ref.named_parameters()}
    x = vq_images(2, cfg.image_size, 3000)
    opt.zero_grad()
    xrec, qloss, _, codes = ref(x)
    loss, log = ref._compute_loss(qloss, x, xrec, split="train")
    loss.backward()
    out = dict(names=np.array(names), loss=loss.detach().numpy(), rec=log["train/rec_loss"].numpy(), quant=log["train/quant_loss"].numpy(),
               codes=codes.numpy(),
               gnorm=np.array([float(p.grad.norm()) for _, p in ref.named_parameters()]),
               gdot=np.array([float((p.grad * probe[n]).sum()) for n, p in ref.named_parameters()]))
    opt.step()
    out["pdot"] = np.array([float((p.detach() * probe[n]).sum()) for n, p in ref.named_parameters()])
    e = ref.quantize.embeddings
    ge = torch.Generator().manual_seed(7)
    out["emb_norm"] = np.float64(e.double().norm())
    out["emb_dot"] = np.float64((e.double() * torch.randn(e.shape, generator=ge).double()).sum())
    np.savez_compressed(os.path.join(OUT, "vqgan_train_full.npz"), **out)
    print("train golden (full size): loss", float(out["loss"]), "tensors", len(names))


def golden_vqgan_train_commit():
    """The same two optimisation steps with the reference's OTHER quantizer, ``Quantize`` (utils_th.py:75-124: gradient-trained codebook,
    beta = 0.25 commitment term), dropped into the real reference VQGAN in place of QuantizeEMA — both classes return
    (quantize, loss, indices), so VQGAN.forward / _compute_loss run unchanged."""
    overrides = dict(SMALL_VQ, perceptual_weight=0.0)
    cfg = VQGANConfig(**overrides)
    sd = synth.make_vqgan_state_dict(cfg, 5)
    ref = ref_loader.build_reference_vqgan(sd, **overrides)
    import sys
    Quantize = sys.modules["viewformer.models.utils_th"].Quantize
    ref.quantize = Quantize(cfg.embed_dim, cfg.n_embed, beta=0.25)
    with torch.no_grad():
        ref.quantize.embeddings.copy_(sd["quantize.embeddings"] * 0.5)        # a codebook at the scale of the encoder output
    ref.train()
    opt = torch.optim.Adam(ref.parameters(), lr=cfg.learning_rate, betas=(0.5, 0.9))
    g = torch.Generator().manual_seed(99)
    names = [n for n, _ in ref.named_parameters()]
    probe = {n: torch.randn(p.shape, generator=g) for n, p in ref.named_parameters()}
    keep = ["quantize.embeddings", "quant_conv.weight", "post_quant_conv.bias", "encoder.conv_in.weight", "decoder.conv_out.bias"]
    out = dict(names=np.array(names), emb_init=ref.quantize.embeddings.detach().numpy().copy())
    for step in range(2):
        x = vq_images(3, cfg.image_size, 2000 + step)
        opt.zero_grad()
        xrec, qloss, _, codes = ref(x)
        loss, log = ref._compute_loss(qloss, x, xrec, split="train")
        loss.backward()
        out[f"loss{step}"] = loss.detach().numpy()
        out[f"quant{step}"] = log["train/quant_loss"].numpy()
        out[f"codes{step}"] = codes.numpy()
        out[f"gnorm{step}"] = np.array([float(p.grad.norm()) for _, p in ref.named_parameters()])
        out[f"gdot{step}"] = np.array([float((p.grad * probe[n]).sum()) for n, p in ref.named_parameters()])
        for k in keep:
            out[f"g{step}.{k}"] = dict(ref.named_parameters())[k].grad.numpy().copy()
        opt.step()
        for k in keep:
            out[f"p{step}.{k}"] = dict(ref.named_parameters())[k].detach().numpy().copy()
    np.savez_compressed(os.path.join(OUT, "vqgan_train_commit_small.npz"), **out)
    print("train (commit quantizer) golden: losses", float(out["loss0"]), float(out["loss1"]), "names", len(names))


def keras_adamw_reference(params, grads, m, v, step, lr, wd, betas=(0.9, 0.999), eps=1e-8):
    """Restatement of AdamWeightDecay._resource_apply_dense (models/utils.py:507-523) on top of Keras Adam (TF 2.4
    optimizer_v2/adam.py, non-amsgrad): decoupled decay for names without "bias" (the exclusion patterns "LayerNorm" / "layer_norm"
    never match this model's variable names), then var -= lr_t * m / (sqrt(v) + eps), lr_t = lr sqrt(1-b2^t)/(1-b1^t).  step is 1-based."""
    b1, b2 = betas
    lr_t = lr * (1 - b2 ** step) ** 0.5 / (1 - b1 ** step)
    for k in params:
        if wd > 0 and "bias" not in k:
            params[k] -= lr * wd * params[k]
        m[k] += (grads[k] - m[k]) * (1 - b1)
        v[k] += (grads[k] * grads[k] - v[k]) * (1 - b2)
        params[k] -= lr_t * m[k] / (v[k].sqrt() + eps)


def warmup_cosine(step, init_lr, warmup, total):
    """WarmUp(CosineDecay) of models/utils.py:310-416 as create_optimizer builds it."""
    import math
    if warmup and step < warmup:
        return init_lr * step / warmup
    decay_steps = max(1, total - warmup)
    t = min(max(step - warmup, 0), decay_steps) / decay_steps
    return init_lr * 0.5 * (1 + math.cos(math.pi * t))


MIGT_TRAIN = dict(SMALL_MIGT, dropout=0.0, weight_decay=0.01, total_steps=10, learning_rate=1e-3, label_smoothing=0.05, localization_weight="0.5",
                  image_generation_weight=0.8, pose_multiplier=1.0)
MIGT_TRAIN_WARMUP = 2


def golden_migt_train():
    """Three optimisation steps of the transformer: gradients by torch autograd through the oracle's forward (compute_losses=True,
    dropout 0), optimizer / schedule restated above.  Reproduced by three calls of the reference's own MIGT.train_step executed over
    oracle/tf_shim.py (tests/test_reference_on_shim.py)."""
    cfg = MIGTConfig(**MIGT_TRAIN)
    sd = {k: v.clone() for k, v in synth.make_migt_state_dict(cfg, 9).items()}
    B, T = 2, 4
    m = {k: torch.zeros_like(v) for k, v in sd.items()}
    vv = {k: torch.zeros_like(v) for k, v in sd.items()}
    out = {}
    KEEP = ("h.0.attn.c_attn.weight", "h.1.mlp.c_proj.bias", "h.1.ln_2.gamma", "ln_f.beta", "pose_classifier.c_proj.weight",
            "pose_embedding.c_fc.weight", "wpe.embeddings", "h.1.attn.c_proj.weight")
    for step in range(3):
        codes = synth.make_codes(B, T, n_embed=cfg.n_embeddings, seed=50 + step)
        cams = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(B, T, seed=60 + step))[0])
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        o = migt_oracle.forward(leaves, cfg, dict(input_ids=codes, poses=cams), compute_losses=True, localization_weight=0.5)
        loss = o["loss"].mean()
        loss.backward()
        grads = {k: (leaves[k].grad if leaves[k].grad is not None else torch.zeros_like(leaves[k])) for k in sd}
        out[f"loss{step}"] = loss.detach().numpy()
        out[f"ce{step}"] = o["ce_loss"].detach().numpy()
        out[f"pose{step}"] = o["pose_loss"].detach().numpy()
        names = list(sd.keys())
        if step == 0:
            gen = torch.Generator().manual_seed(77)
            probe = {k: torch.randn(sd[k].shape, generator=gen) for k in names}
            out["names"] = np.array(names)
        out[f"gnorm{step}"] = np.array([float(grads[k].norm()) for k in names])
        out[f"gdot{step}"] = np.array([float((grads[k] * probe[k]).sum()) for k in names])
        for k in KEEP:
            out[f"g{step}.{k}"] = grads[k].numpy().astype(np.float32)
        lr = warmup_cosine(step, cfg.learning_rate, MIGT_TRAIN_WARMUP, cfg.total_steps)
        with torch.no_grad():
            keras_adamw_reference(sd, grads, m, vv, step + 1, lr, cfg.weight_decay)
        out[f"lr{step}"] = np.float32(lr)
        out[f"pdot{step}"] = np.array([float((sd[k] * probe[k]).sum()) for k in names])
        for k in KEEP:
            out[f"p{step}.{k}"] = sd[k].numpy().copy()
    np.savez_compressed(os.path.join(OUT, "migt_train_small.npz"), **out)
    print("migt train golden: losses", [float(out[f"loss{i}"]) for i in range(3)])


def golden_migt_train_full():
    """One optimisation step of the FULL-size transformer (MIGTConfig defaults: 12 layers, d = 768, 12 heads, 1024 + 2 tokens), B = 1,
    T = 5 views, dropout 0: loss terms, gradient norm + projection of every tensor (autograd through the oracle; reproduced by the
    reference's own train_step over oracle/tf_shim.py, tests/test_reference_on_shim.py)."""
    cfg = MIGTConfig(dropout=0.0, label_smoothing=0.1, localization_weight="0.7", total_steps=100, learning_rate=1e-4)
    sd = {k: v.clone() for k, v in synth.make_migt_state_dict(cfg, 13).items()}
    B, T = 1, 5
    codes = synth.make_codes(B, T, n_embed=cfg.n_embeddings, seed=70)
    cams = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(B, T, seed=71))[0])
    leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    o = migt_oracle.forward(leaves, cfg, dict(input_ids=codes, poses=cams), compute_losses=True, localization_weight=0.7)
    loss = o["loss"].mean()
    loss.backward()
    names = list(sd.keys())
    gen = torch.Generator().manual_seed(78)
    probe = {k: torch.randn(sd[k].shape, generator=gen) for k in names}
    grads = {k: (leaves[k].grad if leaves[k].grad is not None else torch.zeros_like(leaves[k])) for k in names}
    out = dict(names=np.array(names), loss=loss.detach().numpy(), ce=o["ce_loss"].detach().numpy(), pose=o["pose_loss"].detach().numpy(),
               gnorm=np.array([float(grads[k].norm()) for k in names]), gdot=np.array([float((grads[k] * probe[k]).sum()) for k in names]))
    np.savez_compressed(os.path.join(OUT, "migt_train_full.npz"), **out)
    print("migt train golden (full size): loss", float(out["loss"]), "tensors", len(names))


REF_SHIM_CASES = [
    ("generate", {}), ("localize", {}), ("losses", {}), ("explicit", {}),
    ("generate", dict(localization_weight="0")),
    ("losses", dict(label_smoothing=0.1, pose_multiplier=0.3, image_generation_weight=0.7, localization_weight="cosine(2.0,0.5,100)")),
    ("losses", dict(use_dynamic_pose_loss=True)),
]
REF_SHIM_BASE = dict(n_layer=2, n_head=4, d_model=64, sequence_size=4, n_embeddings=40, token_image_size=2, n_loss_skip=1)


def ref_shim_inputs(cfg, variant, B=2, T=4):
    codes = synth.make_codes(B, T, n_embed=cfg.n_embeddings, side=cfg.token_image_size, seed=5)
    cams = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(B, T, seed=6))[0])
    if variant == "generate":
        return dict(input_ids=torch.cat([codes[:, :-1], torch.full_like(codes[:, :1], cfg.n_embeddings)], 1), poses=cams), False
    if variant == "localize":
        return dict(input_ids=codes, poses=cams[:, :-1]), False
    if variant == "losses":
        return dict(input_ids=codes, poses=cams), True
    return dict(input_ids=codes, poses=cams, output_poses=cams.flip(1).contiguous(), localization_tokens=codes.flip(0).contiguous()), False


def golden_migt_reference_shim():
    """Outputs of the REFERENCE's own migt.py / branching_attention.py executed over oracle/tf_shim.py (TensorFlow cannot be installed;
    see that file) for seven call patterns of MIGT.call, plus generate_batch_predictions of evaluate_transformer.py with the real torch
    codebook.  tests/test_oracle_pinned.py compares the oracle with this file wherever /root/reference is absent."""
    out = {}
    for i, (variant, extra) in enumerate(REF_SHIM_CASES):
        kw = dict(REF_SHIM_BASE, **extra)
        cfg = MIGTConfig(**kw)
        sd = synth.make_migt_state_dict(cfg, 3)
        dyn = [0.3, -2.0] if kw.get("use_dynamic_pose_loss") else None
        model = ref_loader.build_reference_migt(sd, dynamic_pose_weights=dyn, **kw)
        inputs, losses = ref_shim_inputs(cfg, variant)
        model._train_counter.assign(7)
        with torch.no_grad():
            r = model({k: v.clone() for k, v in inputs.items()}, compute_losses=losses, training=False)
        for k in ("logits", "loss", "pose_prediction", "ce_loss", "pose_loss", "pose_pos_loss", "pose_ori_loss", "localization_weight"):
            if k in r:
                out[f"c{i}.{k}"] = torch.as_tensor(r[k]).detach().float().numpy()
        out[f"c{i}.n_streams"] = np.int64(len(r["hidden_states"]))
    ev, _ = ref_loader.load_reference_evaluate()
    vcfg = VQGANConfig(**SMALL_VQ)
    vq = ref_loader.build_reference_vqgan(synth.make_vqgan_state_dict(vcfg, 0), **SMALL_VQ)
    kw = dict(REF_SHIM_BASE, n_embeddings=vcfg.n_embed, token_image_size=8)
    cfg = MIGTConfig(**kw)
    model = ref_loader.build_reference_migt(synth.make_migt_state_dict(cfg, 3), **kw)
    images = synth.make_images_uint8(2, 4, size=vcfg.image_size, seed=11)
    cams = synth.make_cameras(2, 4, seed=12)
    with torch.no_grad():
        r = ev.generate_batch_predictions(model, ref_loader.ReferenceCodebookNHWC(vq), images.clone(), cams.clone())
    out["gen.images"] = torch.as_tensor(r["generated_images"]).numpy()
    out["gen.cameras"] = torch.as_tensor(r["generated_cameras"]).float().numpy()
    np.savez_compressed(os.path.join(OUT, "migt_reference_shim.npz"), **out)
    print("reference-on-shim golden:", len(out), "arrays")


EVALUATOR_CASES = [  # (tag, n, gt size, generated size, Evaluator(image_size), seed)
    ("same", 5, 64, 64, None, 21),          # no resize: integer-exact inputs on both sides
    ("up", 3, 96, 48, None, 22),            # generated image upsampled bilinearly to the ground truth's size (evaluate_transformer.py:42-45)
    ("down", 3, 96, 48, 32, 22),            # both brought down to Evaluator(image_size=32)
]


def evaluator_cameras(seed=23, n=7):
    gt = synth.make_cameras(1, n, seed=seed)[0]
    g = torch.Generator().manual_seed(seed + 1)
    gen = gt.clone()
    gen[:, :3] += 0.3 * torch.randn((n, 3), generator=g)
    gen[:, 3:] += 0.2 * torch.randn((n, 4), generator=g)              # un-normalised on purpose: the metric normalises
    return gt, gen


def golden_evaluator_reference_shim():
    """The reference's own Evaluator (evaluate/evaluate_transformer.py:22-67) and metric classes (utils/metrics.py) executed over
    oracle/tf_shim.py on integer-built synthetic images (oracle/synth.py::make_metric_pair): the numbers viewformer_b200.metrics.Evaluator
    has to reproduce on the GPU.  LPIPS is replaced by zeros (VGG weights are not available offline) and not stored."""
    ev, _ = ref_loader.load_reference_evaluate()                      # installs oracle/tf_shim.py as `tensorflow`
    import tensorflow as tf
    metrics = sys.modules["viewformer.utils.metrics"]
    metrics.LPIPSMetric._lpips_pool["vgg"] = lambda a, b: torch.zeros(a.shape[0])
    out = {}
    for tag, n, gs, ns, image_size, seed in EVALUATOR_CASES:
        gt, gen = synth.make_metric_pair(n, gs, ns, seed)
        E = ev.Evaluator(image_size)
        E.update_with_image(tf.convert_to_tensor(gt.numpy()), tf.convert_to_tensor(gen.numpy()))
        r = E.result()
        for k in ("mse", "rmse", "mae", "psnr", "ssim"):
            out[f"{tag}.{k}"] = np.float64(r[k])
        out[f"{tag}.input_sums"] = np.asarray([int(gt.sum()), int(gen.sum())], np.int64)      # guards the regeneration of the inputs
    gt_c, gen_c = evaluator_cameras()
    E = ev.Evaluator()
    E.update_with_camera(tf.convert_to_tensor(gt_c.numpy()), tf.convert_to_tensor(gen_c.numpy()))
    r = E.result()
    for k in ("loc-angle", "loc-dist", "loc-angle-med", "loc-dist-med"):
        out[f"cam.{k}"] = np.float64(r[k])
    # the function-level ssim() with its default K1 (what image_metrics()['ssim'] returns) next to SSIMMetric's K1 = 1
    gt, gen = synth.make_metric_pair(5, 64, 64, 21)
    out["same.ssim_default_k1"] = np.float64(torch.as_tensor(metrics.ssim(gt.float().numpy() / 255, gen.float().numpy() / 255)).double().mean())
    np.savez_compressed(os.path.join(OUT, "evaluator_reference_shim.npz"), **out)
    print("evaluator golden:", {k: float(v) for k, v in out.items() if not k.endswith("sums")})


# ----------------------------------------------------------------------------------------------- reference_outputs.npz
# What the tests that compare with the reference's own code read from it, so that they run on every machine.  Each function below
# runs the reference exactly as the test named in its docstring used to, and stores the reference's side of the comparison.
# Float arrays are stored as a fixed seeded sample of their elements (sample_index) and their shape (`<key>.shape`).

def _json(obj):
    import json
    return np.array(json.dumps(obj))


def sample_index(key, numel, k):
    """The flat indices of the stored sample of array ``key``: all of them up to ``k`` elements, else ``k`` drawn with a seed taken from the
    key's name (the tests recompute them from the name and the number of stored values)."""
    import zlib
    if numel <= k:
        return torch.arange(numel)
    return torch.randperm(numel, generator=torch.Generator().manual_seed(zlib.crc32(key.encode()))).narrow(0, 0, k).sort().values


def _sampled(out, key, t, k=512):
    a = torch.as_tensor(t).detach().float()
    out[key] = a.reshape(-1)[sample_index(key, a.numel(), k)].numpy()
    out[key + ".shape"] = np.asarray(tuple(a.shape), np.int64)


def reference_outputs():
    return np.load(os.path.join(OUT, "reference_outputs.npz"))


def at_reference_sample(G, key, t):
    """(``t`` at the elements stored for reference array ``key``, the stored reference values); ``t`` must have the reference's shape."""
    a = torch.as_tensor(t).detach().float()
    assert tuple(a.shape) == tuple(G[key + ".shape"]), (key, tuple(a.shape), tuple(G[key + ".shape"]))
    want = torch.from_numpy(G[key])
    return a.reshape(-1)[sample_index(key, a.numel(), want.numel())], want


def _crc(t):
    """CRC-32 of a uint8 image array (an input the caller hands back: only its identity is stored)."""
    import zlib
    return zlib.crc32(np.ascontiguousarray(torch.as_tensor(t).as_subclass(torch.Tensor).numpy()).tobytes())


def ref_vqgan_restatement(out):
    """test_oracle_pinned.py::test_vqgan_restatement_equals_real_reference."""
    cfg = VQGANConfig(**SMALL_VQ)
    ref = ref_loader.build_reference_vqgan(synth.make_vqgan_state_dict(cfg, 5), **SMALL_VQ)
    x = torch.rand(3, 3, cfg.image_size, cfg.image_size, generator=torch.Generator().manual_seed(1)) * 2 - 1
    with torch.no_grad():
        q, d, c = ref.encode(x)
        dec, d2, q2, c2 = ref(x)
    assert torch.equal(c, c2) and torch.equal(q, q2) and float(d) == float(d2)
    out.update({"vqgan.codes": c.numpy(), "vqgan.diff": d.numpy()})
    _sampled(out, "vqgan.quant", q)
    _sampled(out, "vqgan.dec", dec)


SCHEDULE_CASES = ["0", "1", "0.5", "2.5e-1", " 3 ", "linear(1,3,10)", "linear(0,0,5)", "linear(1,2)", "cosine(2,0)", "cosine(0,0)",
                  "cosine(2.0,0.5,100)", "warmup(1,2000)", "warmup(0,7)", "warmup(cosine(1,0.5,100),4)", "warmup(linear(0,2,50),10)",
                  "warmup(warmup(1,3),5)"]
SCHEDULE_STEPS = (0, 1, 2, 4, 5, 10, 54, 100, 150, 199, 200, 1000, 2000, 5000)


def ref_schedules_and_configs(out):
    """test_oracle_pinned.py::test_schedules_equal_the_reference_module and ::test_config_fields_and_defaults_equal_the_reference_dataclasses:
    utils/schedules.py and models/config.py as shipped."""
    import dataclasses
    ref_loader.load_reference_modules()
    R = sys.modules["viewformer.utils.schedules"]
    sch = []
    for c in SCHEDULE_CASES:
        r = R.Schedule.from_str(c)
        rt = r.with_total_steps(200)
        sch.append(dict(case=c, str=str(r), is_zero=bool(r.is_zero()), str_total=str(rt), values=[float(rt(t, "float64")) for t in SCHEDULE_STEPS]))
    nested = "warmup(cosine(1,0.5),4)"
    try:
        R.Schedule.from_str(nested).with_total_steps(200)(3)
        nested_error = None
    except Exception as e:
        nested_error = type(e).__name__
    out["schedules"] = _json(dict(steps=list(SCHEDULE_STEPS), cases=sch, step_form_is_none=R.Schedule.from_str("step(1,2)") is None,
                                  nested=nested, nested_error=nested_error))
    RC = sys.modules["viewformer.models.config"]
    cfgs = {}
    for name in ("VQGANConfig", "MIGTConfig"):
        inst = getattr(RC, name)()
        cfgs[name] = dict(fields={f.name: str(getattr(inst, f.name)) for f in dataclasses.fields(getattr(RC, name))},
                          model=inst.model, model_type=inst.model_type)
    cfgs["MIGTConfig"]["localization_weight"] = str(RC.MIGTConfig().localization_weight)
    cfgs["VQGANConfig"]["stride"] = RC.VQGANConfig().stride
    out["configs"] = _json(cfgs)


def latent_code_scenes():
    scenes = []
    for i in range(4):
        fr = np.zeros((6, 8, 8, 3), np.uint8)
        fr[:, :2, :2, 0] = (10 * i + np.arange(6))[:, None, None]
        scenes.append(dict(frames=fr, cameras=np.full((6, 7), i, np.float32)))
    return scenes


def ref_latent_code_transformer(out):
    """test_data_formats.py::test_latent_code_transformer_equals_the_reference_class: commands/generate_codes.py's LatentCodeTransformer
    with a stand-in codebook that returns the top-left 2x2 pixels of channel 0 as codes."""
    ref_mod, restore = ref_loader.load_reference_generate_codes()

    class Cfg:
        image_size, stride, batch_size = 8, 4, 5

    class RefCodebook(torch.nn.Module):
        config, calls = Cfg, []

        def encode(self, x):                                 # NCHW float in [-1, 1], as _convert_image_type hands it over
            self.calls.append(len(x))
            return None, None, ((x[:, 0, :2, :2] + 1) / 2 * 255).round().to(torch.int64)
    try:
        rcb = RefCodebook()
        tr = ref_mod.LatentCodeTransformer(rcb, batch_size=5, device="cpu")
        info = tr.update_dataset_info({})
        feats = {str(f): tr.output_features(f) for f in (None, ["frames", "cameras"], ["frames", "cameras-gqn"])}
        want = list(tr("train", iter([dict(s) for s in latent_code_scenes()])))
    finally:
        restore()
    out["lct.meta"] = _json(dict(dataset_info=info, output_features=feats, encoder_calls=rcb.calls, n_scenes=len(want)))
    for i, w in enumerate(want):
        out[f"lct.codes{i}"] = np.asarray(w["codes"])
        out[f"lct.cameras{i}"] = np.asarray(w["cameras"])


REF_CALL_CASES = [("generate", {}), ("localize", {}), ("losses", {}), ("explicit", {}),
                  ("generate", dict(localization_weight="0")), ("losses", dict(localization_weight="0")),
                  ("losses", dict(label_smoothing=0.1, pose_multiplier=0.3, image_generation_weight=0.7, localization_weight="cosine(2.0,0.5,100)")),
                  ("losses", dict(use_dynamic_pose_loss=True, localization_weight="warmup(linear(1.0,0.2,50),10)")),
                  ("generate", dict(token_image_size=4, n_head=2, sequence_size=6))]
REF_CALL_STEP = 7


def _var(model, key):
    suffix = "/" + key.replace(".", "/")
    hits = [v for v in model.variables if ("/" + v.name[:-2].replace(".", "/")).endswith(suffix)]
    assert len(hits) == 1, (key, [v.name for v in hits])
    return hits[0]


def ref_migt_calls(out):
    """test_reference_on_shim.py::test_reference_call_equals_oracle_forward: MIGT.call of the reference over the shim."""
    for i, (variant, extra) in enumerate(REF_CALL_CASES):
        kw = dict(REF_SHIM_BASE, **extra)
        cfg = MIGTConfig(**kw)
        sd = synth.make_migt_state_dict(cfg, 3)
        dyn = [0.3, -2.0] if kw.get("use_dynamic_pose_loss") else None
        model = ref_loader.build_reference_migt(sd, dynamic_pose_weights=dyn, **kw)
        inputs, losses = ref_shim_inputs(cfg, variant, T=cfg.sequence_size)
        model._train_counter.assign(REF_CALL_STEP)
        with torch.no_grad():
            r = model({k: v.clone() for k, v in inputs.items()}, compute_losses=losses, training=False)
            lw = float(model.localization_weight(REF_CALL_STEP)) if model.use_localization else 0.0
        p = f"call{i}."
        out[p + "use_localization"] = np.bool_(model.use_localization)
        out[p + "lw"] = np.float64(lw)
        for k in ("logits", "loss", "pose_prediction", "ce_loss", "pose_loss", "pose_pos_loss", "pose_ori_loss", "localization_weight"):
            if k in r:
                _sampled(out, p + k, r[k], k=512)
        out[p + "n_hidden"] = np.int64(len(r["hidden_states"]))
        for j, h in enumerate(r["hidden_states"]):
            _sampled(out, p + f"hidden{j}", h, k=256)


def ref_migt_fixtures(out):
    """test_reference_on_shim.py::test_reference_reproduces_committed_forward_fixture, ::test_reference_train_step_reproduces_committed_train_fixture,
    ::test_reference_train_step_gradients_full_size, ::test_reference_dynamic_pose_weights_gradient."""
    for tag, overrides, B, T in (("small", dict(n_layer=2, n_head=4, d_model=128, sequence_size=4, n_loss_skip=1), 2, 4), ("full", {}, 1, 10)):
        cfg = MIGTConfig(**overrides)
        model = ref_loader.build_reference_migt(synth.make_migt_state_dict(cfg, 3), **overrides)
        codes = synth.make_codes(B, T, seed=5)
        cams = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(B, T, seed=6))[0])
        ids = torch.cat([codes[:, :-1], torch.full_like(codes[:, :1], cfg.n_embeddings)], 1)
        with torch.no_grad():
            last = model(dict(input_ids=ids, poses=cams), training=False)["logits"][:, -1]
            o2 = model(dict(input_ids=codes, poses=cams[:, :-1]), training=False)
            pose = model.reduce_cameras(o2["pose_prediction"][:, -1:], -2)
        _sampled(out, f"fwd_{tag}.logits_last", last[:1], k=1024)
        out[f"fwd_{tag}.argmax_last"] = last.argmax(-1).numpy()
        out[f"fwd_{tag}.pose_last"] = torch.as_tensor(pose).float().numpy()

    kw = dict(MIGT_TRAIN)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 9)
    model = ref_loader.build_reference_migt(sd, **kw)
    utils = sys.modules["viewformer.models.utils"]
    opt, _ = utils.create_optimizer(cfg.learning_rate, num_train_steps=cfg.total_steps, num_warmup_steps=MIGT_TRAIN_WARMUP,
                                    weight_decay_rate=cfg.weight_decay)
    model.compile(optimizer=opt)
    G = np.load(os.path.join(OUT, "migt_train_small.npz"))
    names = [str(n) for n in G["names"]]
    gen = torch.Generator().manual_seed(77)
    probe = {k: torch.randn(sd[k].shape, generator=gen) for k in names}
    keep = [k[3:] for k in G.files if k.startswith("p0.")]
    losses = []
    for step in range(3):
        codes = synth.make_codes(2, 4, n_embed=cfg.n_embeddings, seed=50 + step)
        cams = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(2, 4, seed=60 + step))[0])
        model._train_counter.assign(step)
        metrics = model.train_step((cams, codes))
        losses.append(float(metrics["loss"]))
        out[f"train_small.pdot{step}"] = np.array([float((_var(model, k).detach() * probe[k]).sum()) for k in names])
        for j, k in enumerate(keep):
            _sampled(out, f"train_small.p{step}.{k}", _var(model, k).detach(), k=256)
    out["train_small.meta"] = _json(dict(optimizer=type(opt).__name__, iterations=int(opt.iterations), keep=keep))
    out["train_small.losses"] = np.array(losses)

    class Recorder:
        def apply_gradients(self, grads_and_vars):
            self.pairs = [(g, v) for g, v in grads_and_vars]

    kw = dict(dropout=0.0, label_smoothing=0.1, localization_weight="0.7", total_steps=100, learning_rate=1e-4)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 13)
    model = ref_loader.build_reference_migt(sd, **kw)
    rec = Recorder()
    model.compile(optimizer=rec)
    codes = synth.make_codes(1, 5, n_embed=cfg.n_embeddings, seed=70)
    cams = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(1, 5, seed=71))[0])
    metrics = model.train_step((cams, codes))
    names = [str(n) for n in np.load(os.path.join(OUT, "migt_train_full.npz"))["names"]]
    grads = {id(v): g for g, v in rec.pairs}
    gen = torch.Generator().manual_seed(78)
    probe = {k: torch.randn(sd[k].shape, generator=gen) for k in names}
    gn, gd = [], []
    for k in names:
        g = grads[id(_var(model, k))]
        g = torch.zeros_like(sd[k]) if g is None else g
        gn.append(float(g.norm()))
        gd.append(float((g * probe[k]).sum()))
    out["train_full.names"] = np.array(names)
    out["train_full.gnorm"], out["train_full.gdot"] = np.array(gn), np.array(gd)
    for k in ("loss", "ce_loss", "pose_loss"):
        out[f"train_full.{k}"] = np.float64(float(metrics[k]))

    kw = dict(REF_SHIM_BASE, dropout=0.0, use_dynamic_pose_loss=True, localization_weight="0.5")
    cfg = MIGTConfig(**kw)
    model = ref_loader.build_reference_migt(synth.make_migt_state_dict(cfg, 4), dynamic_pose_weights=[0.2, -1.5], **kw)
    rec = Recorder()
    model.compile(optimizer=rec)
    inputs, _ = ref_shim_inputs(cfg, "losses")
    model.train_step((inputs["poses"], inputs["input_ids"]))
    g_ref = [g for g, v in rec.pairs if v.name.startswith("pos_ori_weights")]
    assert len(g_ref) == 1
    out["dyn.grad_pos_ori_weights"] = torch.as_tensor(g_ref[0]).float().numpy()
    _sampled(out, "dyn.grad_h0_c_attn_weight", [g for g, v in rec.pairs if v.name.endswith("h.0/attn/c_attn/weight:0")][0], k=1024)


def ref_evaluation_callers(out):
    """test_reference_on_shim.py::test_reference_generate_batch_predictions_equal_oracle, ::test_reference_allimg_script_equals_oracle,
    ::test_codebook_evaluation_script_equals_oracle_and_fixture, ::test_reference_test_step_and_predict_step_equal_the_oracle_expectations:
    the evaluation scripts as shipped, with the real torch codebook and the real MIGT on the shim."""
    ev, mc = ref_loader.load_reference_evaluate()
    vcfg = VQGANConfig(**SMALL_VQ)
    vq = ref_loader.build_reference_vqgan(synth.make_vqgan_state_dict(vcfg, 0), **SMALL_VQ)
    codebook = ref_loader.ReferenceCodebookNHWC(vq)
    small = dict(n_layer=2, n_head=4, d_model=64, sequence_size=4, n_embeddings=vcfg.n_embed, token_image_size=8, n_loss_skip=1)
    for augment, loc in (("relative", "1"), ("relative", "0"), ("no", "1")):
        kw = dict(small, augment_poses=augment, localization_weight=loc)
        model = ref_loader.build_reference_migt(synth.make_migt_state_dict(MIGTConfig(**kw), 3), **kw)
        images = synth.make_images_uint8(2, 4, size=vcfg.image_size, seed=11)
        cams = synth.make_cameras(2, 4, seed=12)
        p = f"gbp.{augment}.{loc}."
        with torch.no_grad():
            r = ev.generate_batch_predictions(model, codebook, images.clone(), cams.clone())
            for k in ("generated_images", "ground_truth_cameras", "generated_cameras"):
                out[p + k] = torch.as_tensor(r[k]).as_subclass(torch.Tensor).numpy()
            out[p + "ground_truth_images.crc32"] = np.int64(_crc(r["ground_truth_images"]))
            if model.use_localization:
                r = mc.generate_batch_predictions(model, codebook, images.clone(), cams.clone())
                out[p + "multictx.generated_images"] = torch.as_tensor(r["generated_images"]).as_subclass(torch.Tensor).numpy()
                out[p + "multictx.generated_cameras"] = torch.as_tensor(r["generated_cameras"]).as_subclass(torch.Tensor).numpy()

    R = os.path.join(ref_loader.REFERENCE_ROOT, "viewformer", "evaluate", "evaluate_transformer_multictx_allimg.py")
    al = ref_loader._load("viewformer.evaluate.evaluate_transformer_multictx_allimg", R)
    model = ref_loader.build_reference_migt(synth.make_migt_state_dict(MIGTConfig(**small), 3), **small)
    images = synth.make_images_uint8(3, 4, size=vcfg.image_size, seed=41)
    cams = synth.make_cameras(3, 4, seed=42)
    with torch.no_grad():
        codes = al.encode_images(images.clone(), codebook_model=codebook)
        gen_cams, gen_codes = al.run_with_batchsize(al.transformer_predict, 2, cams.clone(), codes, transformer_model=model)
        gen_images = al.decode_code(gen_codes, codebook_model=codebook)
    for k, v in (("codes", codes), ("generated_cameras", gen_cams), ("generated_codes", gen_codes), ("generated_images", gen_images)):
        out["allimg." + k] = torch.as_tensor(v).as_subclass(torch.Tensor).numpy()

    ec = ref_loader._load("viewformer.evaluate.evaluate_codebook",
                          os.path.join(ref_loader.REFERENCE_ROOT, "viewformer", "evaluate", "evaluate_codebook.py"))
    metrics = sys.modules["viewformer.utils.metrics"]
    metrics.LPIPSMetric._lpips_pool["vgg"] = lambda a, b: torch.zeros(a.shape[0])       # LPIPS needs VGG weights: not available offline
    import tensorflow as tf
    for size in (vcfg.image_size, 48):
        images = synth.make_images_uint8(1, 3, size=size, seed=51)[0]
        with torch.no_grad():
            r = ec.generate_batch_predictions(codebook, tf.convert_to_tensor(images.numpy()))
        out[f"codebook{size}.generated_images"] = torch.as_tensor(r["generated_images"]).as_subclass(torch.Tensor).numpy()
        out[f"codebook{size}.ground_truth_images.crc32"] = np.int64(_crc(r["ground_truth_images"]))
        if size != vcfg.image_size:                                   # the dataset resize rule in front of the encoder
            out[f"codebook{size}.resized"] = sys.modules["viewformer.data._common"].resize(images.numpy(), vcfg.image_size)
    gt, gen = synth.make_metric_pair(5, 64, 64, 21)
    E = ec.Evaluator()
    E.update_state(tf.convert_to_tensor(gt.numpy()), tf.convert_to_tensor(gen.numpy()))
    r = E.result()
    out["codebook.evaluator"] = _json(dict(keys=list(r), values={k: float(r[k]) for k in ("mse", "rmse", "mae", "psnr", "ssim")},
                                           img_rgbl1=float(E.get_progress_bar_info()["img_rgbl1"])))

    model = ref_loader.build_reference_migt(synth.make_migt_state_dict(MIGTConfig(**small), 3), **small)
    model.codebook_model = codebook
    codes = synth.make_codes(3, 4, n_embed=vcfg.n_embed, side=8, seed=5)
    rel = migt_oracle.normalize_cameras(migt_oracle.to_relative_cameras(synth.make_cameras(3, 4, seed=6))[0])
    with torch.no_grad():
        for m in model.metrics:
            m.reset_states()
        res = model.test_step((tf.constant(rel.numpy()), codes.clone()))
        ps = model.predict_step((tf.constant(rel.numpy()), codes.clone()))
    out["steps.test_step"] = _json({k: float(v) for k, v in res.items()})
    out["steps.latent_code"] = torch.as_tensor(ps["latent_code"]).long().numpy()
    out["steps.image_shapes"] = np.asarray([tuple(ps["decoded_image"].shape), tuple(ps["ground_truth_image"].shape)], np.int64)


def ref_process_batch(out):
    """test_reference_on_shim.py::test_process_batch_equals_the_reference_function: train/train_transformer.py:31-64, the function's own
    source cut out of the file with ast and executed over the shim."""
    import ast
    import math
    import tensorflow as tf
    ref_loader.load_reference_migt()
    path = os.path.join(ref_loader.REFERENCE_ROOT, "viewformer", "train", "train_transformer.py")
    fn = [n for n in ast.parse(open(path).read()).body if isinstance(n, ast.FunctionDef) and n.name == "process_batch"]
    assert len(fn) == 1
    ns = dict(tf=tf, geometry=sys.modules["viewformer.utils.geometry_tf"], math=math)
    exec(compile(ast.Module(body=fn, type_ignores=[]), path, "exec"), ns)
    cams = synth.make_cameras(3, 5, seed=8)
    toks = synth.make_codes(3, 5, n_embed=16, side=2, seed=9)
    for name, x in (("window", cams[0]), ("batch", cams)):
        for augment in ("relative", "no", "simple", "advanced"):
            for split in ("train", "test"):
                torch.manual_seed(123)
                want, wt = ns["process_batch"](tf.constant(x.numpy()), toks, augment, split)
                assert wt is toks
                out[f"process_batch.{name}.{augment}.{split}"] = torch.as_tensor(want).as_subclass(torch.Tensor).numpy()


def _attribute_paths(root, max_depth=5):
    """{id(variable): ['a/b/0/c', ...]}: every path of public attribute names / list indices from ``root`` to a shim Variable."""
    tf_shim = sys.modules["oracle.tf_shim"]
    found = {}

    def walk(obj, path, depth, seen):
        if isinstance(obj, tf_shim.Variable):
            found.setdefault(id(obj), []).append("/".join(path))
            return
        if depth == max_depth or id(obj) in seen:
            return
        if isinstance(obj, (list, tuple)):
            items = [(str(i), v) for i, v in enumerate(obj)]
        elif isinstance(obj, tf_shim.Layer):
            items = [(k, v) for k, v in vars(obj).items() if not k.startswith("_")]
        else:
            return
        for name, v in items:
            walk(v, path + [name], depth + 1, seen | {id(obj)})
    walk(root, [], 0, frozenset())
    return found


def ref_object_paths(out):
    """test_reference_on_shim.py::test_checkpoint_object_paths_are_the_reference_models_attribute_names: the attribute paths from the real
    reference MIGT object to each of its variables (the names a TF2 object-based checkpoint is keyed by)."""
    kw = dict(REF_SHIM_BASE, use_dynamic_pose_loss=True)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 3)
    model = ref_loader.build_reference_migt(sd, dynamic_pose_weights=[0.3, -2.0], **kw)
    paths = _attribute_paths(model)
    keys = list(sd) + ["pose_loss_weighting_criterion.pos_ori_weights"]
    dyn = [v for v in model.variables if v.name.startswith("pos_ori_weights")]
    assert len(dyn) == 1
    table = {}
    for k in keys:
        v = dyn[0] if k == "pose_loss_weighting_criterion.pos_ori_weights" else _var(model, k)
        table[k] = dict(paths=sorted(paths.get(id(v), [])), shape=list(v.shape))
    root = sorted(k for k in vars(model) if not k.startswith("_"))
    out["object_paths"] = _json(dict(variables=table, root_attributes=root, wpe_has_embeddings=hasattr(model.wpe, "embeddings"),
                                     pos_ori_weights=torch.as_tensor(dyn[0]).detach().tolist()))


def ref_metrics(out):
    """test_reference_on_shim.py::test_ssim_of_the_gpu_tests_and_the_k1_quirk_follow_the_reference, ::test_allow_nan_mean_counts_nan_as_zero_
    with_full_weight_like_the_reference, ::test_multi_context_evaluator_equals_the_reference_class, ::test_evaluator_fixture_is_what_the_
    reference_evaluator_computes: utils/metrics.py and the Evaluator classes of the evaluation scripts."""
    import tensorflow as tf
    ev, mc = ref_loader.load_reference_evaluate()
    metrics = sys.modules["viewformer.utils.metrics"]
    metrics.LPIPSMetric._lpips_pool["vgg"] = lambda a, b: torch.zeros(a.shape[0])
    gt, gen = synth.make_metric_pair(4, 64, 64, 5)
    A, B = gt.float() / 255, gen.float() / 255
    out["ssim.default_k1"] = torch.as_tensor(metrics.ssim(A.numpy(), B.numpy())).double().numpy()
    out["ssim.k1_is_1"] = np.float64(torch.as_tensor(metrics.ssim(A.numpy(), B.numpy(), 1)).double().mean())
    m = metrics.SSIMMetric()
    m.update_state(gt.numpy(), gen.numpy())
    out["ssim.metric_class"] = np.float64(float(m.result()))

    a = torch.tensor([[0., 0, 0, 1, 0, 0, 0], [1, 1, 1, 1, 0, 0, 0], [2, 0, 0, 1, 0, 0, 0]])
    b = torch.tensor([[3., 4, 0, 1, 0, 0, 0], [float("nan"), 1, 1, 1, 0, 0, 0], [2, 0, 1, 1, 0, 0, 0]])
    m = metrics.CameraPositionError()
    m.update_state(tf.convert_to_tensor(a.numpy()), tf.convert_to_tensor(b.numpy()))
    out["nan_mean.camera_position_error"] = np.float64(float(m.result()))

    B_, T = 4, 4
    gt_cams = synth.make_cameras(1, B_, seed=31)[0]
    g = torch.Generator().manual_seed(32)
    gen_cams = gt_cams[:, None].repeat(1, T, 1) + 0.2 * torch.randn((B_, T, 7), generator=g)
    gt_img, _ = synth.make_metric_pair(B_, 16, 16, 33)
    gen_img = torch.stack([synth.make_metric_pair(B_, 16, 16, 40 + i)[1] for i in range(T)], 1)
    ref = mc.MultiContextEvaluator(T)
    ref.update_state(tf.convert_to_tensor(gt_cams.numpy()), tf.convert_to_tensor(gen_cams.numpy()), tf.convert_to_tensor(gt_img.numpy()),
                     tf.convert_to_tensor(gen_img.numpy()))
    r = ref.result()
    out["multictx"] = _json(dict(keys=list(r), values={k: {m: float(r[k][m]) for m in ("loc-angle", "loc-dist", "loc-angle-med", "loc-dist-med")}
                                                       for k in r},
                                 cam_loc=float(ref.get_progress_bar_info()["cam_loc"])))

    res = {}
    for tag, n, gs, ns, image_size, seed in EVALUATOR_CASES:
        gt, gen = synth.make_metric_pair(n, gs, ns, seed)
        E = ev.Evaluator(image_size)
        E.update_with_image(tf.convert_to_tensor(gt.numpy()), tf.convert_to_tensor(gen.numpy()))
        rr = E.result()
        res[tag] = dict(input_sums=[int(gt.sum()), int(gen.sum())], **{k: float(rr[k]) for k in ("mse", "rmse", "mae", "psnr", "ssim")})
    out["evaluator"] = _json(res)


REGISTRY_SMALL_VQ = dict(ch=32, ch_mult=[1, 2], attn_resolutions=[8], image_size=16, embed_dim=8, z_channels=8, n_embed=16, num_res_blocks=1)


def ref_state_dict_keys(out):
    """test_registry_boundary.py::test_b200_codebook_state_dict_keys_are_the_reference_models: the reference VQGAN's state_dict keys
    (vqgan_th.py), without its loss modules."""
    ref = ref_loader.build_reference_vqgan(**REGISTRY_SMALL_VQ)
    out["vqgan.state_dict_keys"] = np.array(sorted(k for k in ref.state_dict() if not k.startswith(("perceptual_loss.", "loss."))))


def golden_reference_outputs():
    out = {}
    ref_state_dict_keys(out)
    ref_vqgan_restatement(out)
    ref_schedules_and_configs(out)
    ref_latent_code_transformer(out)
    ref_migt_calls(out)
    ref_migt_fixtures(out)
    ref_evaluation_callers(out)
    ref_process_batch(out)
    ref_object_paths(out)
    ref_metrics(out)
    np.savez_compressed(os.path.join(OUT, "reference_outputs.npz"), **out)
    print("reference outputs:", len(out), "arrays,", os.path.getsize(os.path.join(OUT, "reference_outputs.npz")), "bytes")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    golden_lookup()
    golden_quantizer()
    golden_vqgan("small", SMALL_VQ, 2, 0)
    golden_vqgan("full", {}, 4, 0)
    golden_migt()
    golden_vqgan_train()
    golden_vqgan_train_commit()
    golden_vqgan_train_full()
    golden_migt_train()
    golden_migt_train_full()
    golden_migt_reference_shim()
    golden_evaluator_reference_shim()
    golden_reference_outputs()
