"""Pins the CPU oracle: restatement == golden vectors produced by the REAL reference (tests/golden/*.npz,
oracle/make_golden.py), restatement == what the real reference modules returned (tests/golden/reference_outputs.npz), and the
structural invariants that stand in for the (un-runnable) TensorFlow transformer."""
import json
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import synth, vqgan_oracle as vo, migt_oracle as mo
from oracle.make_golden import SMALL_VQ, SMALL_MIGT, vq_images, reference_outputs, at_reference_sample
from viewformer_b200.config import VQGANConfig, MIGTConfig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _g(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_vqgan_small_matches_reference_golden(golden_dir):
    g = _g(golden_dir, "vqgan_small.npz")
    cfg = VQGANConfig(**SMALL_VQ)
    sd = synth.make_vqgan_state_dict(cfg, int(g["seed"]))
    x = vq_images(int(g["n_images"]), cfg.image_size, 1000 + int(g["seed"]))
    with torch.no_grad():
        quant, diff, codes, z = vo.encode(sd, cfg, x, return_pre_quant=True)
        dec = vo.decode_code(sd, cfg, codes)
    assert np.array_equal(codes.numpy(), g["codes"])                       # bit-exact indices
    np.testing.assert_allclose(z.numpy(), g["z"], atol=1e-6, rtol=1e-6)
    np.testing.assert_allclose(float(diff), float(g["diff"]), rtol=1e-6)
    np.testing.assert_allclose(dec.numpy(), g["dec"], atol=1e-6, rtol=1e-6)


def test_vqgan_full_matches_reference_golden(golden_dir):
    g = _g(golden_dir, "vqgan_full.npz")
    cfg = VQGANConfig()
    sd = synth.make_vqgan_state_dict(cfg, int(g["seed"]))
    x = vq_images(int(g["n_images"]), cfg.image_size, 1000 + int(g["seed"]))
    torch.set_num_threads(os.cpu_count())
    with torch.no_grad():
        quant, diff, codes, z = vo.encode(sd, cfg, x, return_pre_quant=True)
        dec = vo.decode_code(sd, cfg, codes)
    assert np.array_equal(codes.numpy(), g["codes"])
    np.testing.assert_allclose(z.numpy(), g["z"], atol=2e-5, rtol=1e-5)
    np.testing.assert_allclose(dec[0].numpy(), g["dec0"], atol=2e-5, rtol=1e-5)
    np.testing.assert_allclose(dec[:, :, ::4, ::4].numpy(), g["dec"], atol=2e-5, rtol=1e-5)


def test_vqgan_restatement_equals_real_reference():
    """The reference VQGAN's encode() and forward() (what oracle/make_golden.py::ref_vqgan_restatement stored) == the restatement:
    identical codes; quantised latents, reconstruction and commitment loss to float32 rounding (they were computed on another machine)."""
    R = reference_outputs()
    cfg = VQGANConfig(**SMALL_VQ)
    sd = synth.make_vqgan_state_dict(cfg, 5)
    x = torch.rand(3, 3, cfg.image_size, cfg.image_size, generator=torch.Generator().manual_seed(1)) * 2 - 1
    with torch.no_grad():
        qo, do, co = vo.encode(sd, cfg, x)
        deco, *_ = vo.forward(sd, cfg, x)
    assert np.array_equal(co.numpy(), R["vqgan.codes"])
    for key, got in (("vqgan.quant", qo), ("vqgan.dec", deco)):
        g, w = at_reference_sample(R, key, got)
        np.testing.assert_allclose(g.numpy(), w.numpy(), atol=1e-6, rtol=1e-6, err_msg=key)
    np.testing.assert_allclose(float(do), float(R["vqgan.diff"]), rtol=1e-6)


def test_quantizer_training_branch_matches_reference_golden(golden_dir):
    g = _g(golden_dir, "quantizer.npz")
    E, z = torch.from_numpy(g["E"]), torch.from_numpy(g["z"])
    sd = {"quantize.embeddings": E.clone(), "quantize.ema_cluster_size_hidden": torch.zeros(E.shape[1]),
          "quantize.ema_dw_hidden": torch.zeros_like(E), "quantize.counter": torch.tensor(0)}
    for step in range(2):
        q, diff, ids, new = vo.quantize_ema(sd, z, training=True)
        sd.update(new)
        assert np.array_equal(ids.numpy(), g[f"ids{step}"])
        np.testing.assert_allclose(float(diff), float(g[f"diff{step}"]), rtol=1e-6)
        np.testing.assert_allclose(sd["quantize.embeddings"].numpy(), g[f"emb{step}"], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(sd["quantize.ema_dw_hidden"].numpy(), g[f"dw{step}"], rtol=1e-6, atol=1e-7)
    q, loss, ids = vo.quantize_commit(E, z)
    assert np.array_equal(ids.numpy(), g["commit_ids"])
    np.testing.assert_allclose(float(loss), float(g["commit_loss"]), rtol=1e-6)


def test_c_lookup_oracle_matches_reference_expression(golden_dir):
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libvq_oracle.so"))
    g = _g(golden_dir, "vq_lookup.npz")
    E, z = synth.make_lookup_inputs(int(g["seed"]))
    z = z[:1024].contiguous()                     # bounded: the scalar C loop is slow
    idx = np.empty(z.shape[0], dtype=np.int64)
    lib.vq_oracle_lookup(ctypes.c_void_p(z.data_ptr()), ctypes.c_void_p(E.data_ptr()), ctypes.c_int64(z.shape[0]),
                         ctypes.c_int(256), ctypes.c_int(1024), idx.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(0))
    assert np.array_equal(idx, g["idx"][:1024])
    assert np.array_equal(vo.vq_lookup(E, z).numpy(), g["idx"][:1024])


def test_migt_restatement_regression_and_invariants(golden_dir):
    g = _g(golden_dir, "migt_small.npz")
    cfg = MIGTConfig(**SMALL_MIGT)
    sd = synth.make_migt_state_dict(cfg, 3)
    B, T = int(g["B"]), int(g["T"])
    codes = synth.make_codes(B, T, seed=5)
    cams = mo.normalize_cameras(mo.to_relative_cameras(synth.make_cameras(B, T, seed=6))[0])
    ids = torch.cat([codes[:, :-1], torch.full_like(codes[:, :1], cfg.n_embeddings)], 1)
    with torch.no_grad():
        o1 = mo.forward(sd, cfg, dict(input_ids=ids, poses=cams))
        np.testing.assert_allclose(o1["logits"][:1, -1].numpy(), g["logits_last"], atol=1e-5, rtol=1e-5)
        assert np.array_equal(o1["logits"][:, -1].argmax(-1).numpy(), g["argmax_last"])
        # invariant (i): single-stream logits at the last view == 3-stream stream-1 logits at the last slot
        ctx_c = torch.cat([cams[:, :-1], torch.zeros_like(cams[:, :1])], 1)
        o3 = mo.forward(sd, cfg, dict(input_ids=ids, poses=ctx_c, output_poses=cams[:, -1:].repeat(1, T, 1),
                                      localization_tokens=codes[:, -1:].repeat(1, T, 1, 1)))
        assert (o1["logits"][:, -1] - o3["logits"][:, -1]).abs().max() < 1e-4
        # invariant (ii): context hidden states do not depend on the query view => KV cache is exact
        cams2 = cams.clone()
        cams2[:, -1, :3] += 1.0
        o2 = mo.forward(sd, cfg, dict(input_ids=ids, poses=cams2))
        assert torch.equal(o1["hidden_states"][0][:, :-1], o2["hidden_states"][0][:, :-1])


def test_camera_helpers_round_trip():
    cams = synth.make_cameras(3, 5)
    rel, tr = mo.to_relative_cameras(cams)
    assert rel[:, 0, :3].abs().max() < 1e-6 and (rel[:, 0, 3] - 1).abs().max() < 1e-6
    back = mo.from_relative_cameras(rel, tr)
    assert (back - cams).abs().max() < 1e-5


def test_oracle_matches_reference_on_shim_fixture(golden_dir):
    """tests/golden/migt_reference_shim.npz holds outputs of the reference's OWN migt.py / branching_attention.py /
    evaluate_transformer.py executed over oracle/tf_shim.py (written by oracle/make_golden.py::golden_migt_reference_shim in the
    container, where tests/test_reference_on_shim.py runs the same comparison live).  The restatement must reproduce every array."""
    from oracle.make_golden import REF_SHIM_CASES, REF_SHIM_BASE, ref_shim_inputs
    from oracle import vqgan_oracle
    g = _g(golden_dir, "migt_reference_shim.npz")
    for i, (variant, extra) in enumerate(REF_SHIM_CASES):
        kw = dict(REF_SHIM_BASE, **extra)
        cfg = MIGTConfig(**kw)
        sd = synth.make_migt_state_dict(cfg, 3)
        if kw.get("use_dynamic_pose_loss"):
            sd["pose_loss_weighting_criterion.pos_ori_weights"] = torch.tensor([0.3, -2.0])
        inputs, losses = ref_shim_inputs(cfg, variant)
        use_loc = str(kw.get("localization_weight", "1")) != "0"
        lw = float(g[f"c{i}.localization_weight"]) if f"c{i}.localization_weight" in g.files else 1.0
        with torch.no_grad():
            o = mo.forward(sd, cfg, inputs, compute_losses=losses, use_localization=use_loc, localization_weight=lw)
        assert len(o["hidden_states"]) == int(g[f"c{i}.n_streams"])
        keys = [k[len(f"c{i}."):] for k in g.files if k.startswith(f"c{i}.") and not k.endswith(("n_streams", "localization_weight"))]
        assert "logits" in keys and ("pose_prediction" in keys) == use_loc and ("pose_prediction" in o) == use_loc
        for k in keys:
            want = torch.from_numpy(g[f"c{i}.{k}"])
            got = torch.as_tensor(o[k]).float()
            assert got.shape == want.shape, (i, k)
            assert float((got - want).abs().max()) <= 2e-6 * max(1.0, float(want.abs().max())), (i, variant, k)
    # generate_batch_predictions of evaluate_transformer.py (real torch codebook + MIGT on the shim) vs the two oracles chained
    vcfg = VQGANConfig(**SMALL_VQ)
    vsd = synth.make_vqgan_state_dict(vcfg, 0)
    kw = dict(REF_SHIM_BASE, n_embeddings=vcfg.n_embed, token_image_size=8)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 3)
    images = synth.make_images_uint8(2, 4, size=vcfg.image_size, seed=11)
    cams = synth.make_cameras(2, 4, seed=12)
    with torch.no_grad():
        o = mo.generate_batch_predictions(lambda inp: mo.forward(sd, cfg, inp), lambda x: vo.encode(vsd, vcfg, x)[-1],
                                          lambda c: vo.decode_code(vsd, vcfg, c), cfg, images, cams)
    diff = (o["generated_images"].int() - torch.from_numpy(g["gen.images"]).int()).abs()
    assert int(diff.max()) <= 1 and float((diff > 0).float().mean()) < 1e-3        # uint8 views: the codebook restatement may round one LSB apart
    assert float((o["generated_cameras"] - torch.from_numpy(g["gen.cameras"])).abs().max()) < 1e-5


def test_schedules_equal_the_reference_module():
    """viewformer_b200/schedules.py against the reference's utils/schedules.py (pure Python, imported as shipped): same parse, same string
    form, same is_zero, same values on a grid of steps — localization_weight schedules of MIGT (migt.py:280-283, :446).  One deliberate
    difference: warmup(cosine(a,b),n).with_total_steps(T) raises TypeError in the reference (WarmupSchedule does not forward the horizon to
    its inner schedule); here the horizon is forwarded and the schedule evaluates.  The reference's side is stored in
    tests/golden/reference_outputs.npz (oracle/make_golden.py::ref_schedules_and_configs)."""
    from oracle.make_golden import SCHEDULE_CASES
    from viewformer_b200.schedules import parse
    R = json.loads(str(reference_outputs()["schedules"]))
    assert [r["case"] for r in R["cases"]] == SCHEDULE_CASES
    for r in R["cases"]:
        c, o = r["case"], parse(r["case"])
        assert r["str"] == str(o) and r["is_zero"] == o.is_zero(), c
        o = o.with_total_steps(200)
        assert r["str_total"] == str(o), c
        for t, rv in zip(R["steps"], r["values"]):
            ov = float(o(t))
            assert abs(rv - ov) <= 1e-6 * max(1.0, abs(rv)), (c, t, rv, ov)         # the reference computes in float32 inside
    assert R["step_form_is_none"]
    with pytest.raises(ValueError):
        parse("step(1,2)")
    assert R["nested"] == "warmup(cosine(1,0.5),4)" and R["nested_error"] == "TypeError"
    assert abs(float(parse(R["nested"]).with_total_steps(200)(3)) - 0.75) < 1e-9


def test_config_fields_and_defaults_equal_the_reference_dataclasses():
    """viewformer_b200/config.py against models/config.py:62-119 imported as shipped: the same field names (= the config.json schema of
    the published checkpoints) and the same defaults; `localization_weight` is kept as the string and parsed where it is used.  The
    reference's fields and defaults are stored in tests/golden/reference_outputs.npz (oracle/make_golden.py::ref_schedules_and_configs)."""
    import dataclasses
    from viewformer_b200 import config as C
    RC = json.loads(str(reference_outputs()["configs"]))
    for name in ("VQGANConfig", "MIGTConfig"):
        r, o = RC[name], getattr(C, name)
        rf, of = set(r["fields"]), {f.name for f in dataclasses.fields(o)}
        assert rf - of <= {"model"} and not (of - rf), (name, rf ^ of)
        oi = o()
        assert r["model"] == oi.model and r["model_type"] == oi.model_type
        for k in sorted(rf & of):
            assert r["fields"][k] == str(getattr(oi, k)) or k == "localization_weight", (name, k)
    assert RC["MIGTConfig"]["localization_weight"] == "1.0" and C.MIGTConfig().localization_weight == "1"
    assert RC["VQGANConfig"]["stride"] == C.VQGANConfig().stride == 16
