"""The reference's OWN transformer sources, run once (oracle/make_golden.py::golden_reference_outputs) with oracle/tf_shim.py answering
``import tensorflow``: viewformer/models/migt.py, models/branching_attention.py, models/utils.py (create_optimizer, WarmUp,
AdamWeightDecay), utils/{tensorflow,geometry_tf,metrics,schedules}.py and evaluate/evaluate_transformer{,_multictx,_multictx_allimg}.py,
evaluate_codebook.py.  What those runs returned is stored in tests/golden/reference_outputs.npz (float arrays as a fixed seeded sample of
their elements), and each test below holds this repository's code to it.  The shim restates only leaf tensor ops; its own semantics are
checked below against TensorFlow's documented behaviour.

What this pins:
  * oracle/migt_oracle.py::forward == MIGT.call (migt.py:338-455) for the generate() call, the localisation call, compute_losses with
    label smoothing / pose multiplier / schedules / dynamic pose weights, explicit output_poses + localization_tokens, use_localization off;
  * the COMMITTED fixtures the GPU parity tests consume (tests/golden/migt_small.npz, migt_full.npz, migt_train_small.npz,
    migt_train_full.npz) are what the reference's code computes: forward, MIGT.train_step (GradientTape, clip, AdamWeightDecay under
    WarmUp(CosineDecay)) — so CUDA == fixture (tests -m gpu) and fixture == reference (here) close the chain;
  * generate_batch_predictions of the evaluation scripts == the oracle's restatements (oracle/vqgan_oracle.py stands in for the reference
    codebook, which tests/test_oracle_pinned.py pins to the reference's).
Stored and recomputed values come from different machines: float comparisons keep the tolerances of a live comparison, uint8 views
produced through the codebook may differ by one LSB in a few pixels (as in test_oracle_pinned.py::test_oracle_matches_reference_on_shim_fixture)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import synth, migt_oracle as mo, vqgan_oracle as vo
from oracle.make_golden import reference_outputs, at_reference_sample
from viewformer_b200.config import MIGTConfig, VQGANConfig

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SMALL = dict(n_layer=2, n_head=4, d_model=64, sequence_size=4, n_embeddings=40, token_image_size=2, n_loss_skip=1)


@pytest.fixture(scope="module")
def tf():
    from oracle import tf_shim
    yield tf_shim.install()
    tf_shim.uninstall()                       # later test modules must not see a `tensorflow` in sys.modules


@pytest.fixture(scope="module")
def R():
    return reference_outputs()


def _close(got, key, R, rel):
    """got (full array) against the stored sample of reference array `key`: max |diff| <= rel * max(1, max |reference|)."""
    g, w = at_reference_sample(R, key, got)
    assert torch.isfinite(g).all(), key
    scale = max(1.0, float(torch.as_tensor(got).detach().float().abs().max()))
    assert float((g - w).abs().max()) <= rel * scale, (key, float((g - w).abs().max()))


def _same_u8(got, want, frac=1e-3):
    d = (torch.as_tensor(got).int() - torch.as_tensor(want).int()).abs()
    assert tuple(d.shape) == tuple(torch.as_tensor(want).shape)
    assert int(d.max()) <= 1 and float((d > 0).float().mean()) < frac, (int(d.max()), float((d > 0).float().mean()))


def _crc(t):
    import zlib
    return zlib.crc32(np.ascontiguousarray(torch.as_tensor(t).numpy()).tobytes())


def _small_codebook():
    from oracle import make_golden as mg
    vcfg = VQGANConfig(**mg.SMALL_VQ)
    vsd = synth.make_vqgan_state_dict(vcfg, 0)
    return vcfg, (lambda x: vo.encode(vsd, vcfg, x)[-1]), (lambda c: vo.decode_code(vsd, vcfg, c))


# ------------------------------------------------------------------------------------------------ the shim's own semantics
def test_shim_ops_follow_documented_tensorflow_semantics(tf):
    x = tf.reshape(tf.range(24), [2, 3, 4])
    assert x.shape.as_list() == [2, 3, 4] and tf.shape(x).tolist() == [2, 3, 4] and tf.rank(x) == 3
    a, b = tf.split(x, 2, axis=-1)                                   # an int = NUMBER of equal parts (torch.split: size of a part)
    assert a.shape == (2, 3, 2) and b[0, 0].tolist() == [2, 3]
    p, q = tf.split(x, (1, 3), axis=-1)
    assert p.shape == (2, 3, 1) and q.shape == (2, 3, 3)
    assert tf.repeat(tf.range(3), 2).tolist() == [0, 0, 1, 1, 2, 2]  # element-wise, not tiling
    assert tf.tile(tf.range(3), [2]).tolist() == [0, 1, 2, 0, 1, 2]
    assert tf.one_hot([0, 2], 3).tolist() == [[1, 0, 0], [0, 0, 1]]
    assert tf.gather(tf.constant([[1., 2.], [3., 4.], [5., 6.]]), tf.constant([[2, 0]])).tolist() == [[[5, 6], [1, 2]]]
    assert tf.constant(3).dtype == tf.int32 and tf.constant(3.0).dtype == tf.float32 and tf.constant(3, "float32").dtype == tf.float32
    assert tf.constant(np.zeros(2, np.uint8)).dtype == tf.uint8       # numpy arrays keep their dtype
    g = tf.constant([3.0, 4.0])
    assert torch.allclose(tf.clip_by_norm(g, 1.0), torch.tensor([0.6, 0.8])) and torch.equal(tf.clip_by_norm(g, 10.0), torch.tensor([3.0, 4.0]))
    assert torch.allclose(tf.linalg.l2_normalize(g, axis=-1), torch.tensor([0.6, 0.8]))
    assert torch.equal(tf.linalg.l2_normalize(tf.zeros([2]), axis=-1, epsilon=1e-12), torch.zeros(2))      # x * rsqrt(max(sum x^2, eps))
    u8 = tf.constant(np.array([0, 1, 128, 255], np.uint8))
    f = tf.image.convert_image_dtype(u8, tf.float32)
    assert torch.equal(f, u8.float() * torch.tensor(1 / 255, dtype=torch.float32))
    assert tf.image.convert_image_dtype(tf.constant([0.0, 0.5, 0.999, 1.0]), tf.uint8).tolist() == [0, 127, 255, 255]    # x * 255.5, truncated
    logits = tf.constant([[1.0, 2.0, 3.0]])
    lp = torch.log_softmax(logits, -1)
    assert torch.allclose(tf.nn.sparse_softmax_cross_entropy_with_logits(tf.constant([2]), logits), -lp[:, 2])
    assert torch.allclose(tf.nn.softmax_cross_entropy_with_logits(tf.constant([[0.5, 0.5, 0.0]]), logits), -(0.5 * lp[:, 0] + 0.5 * lp[:, 1]))
    assert torch.allclose(tf.losses.mse(tf.constant([[1.0, 3.0]]), tf.constant([[0.0, 0.0]])), torch.tensor([5.0]))
    assert torch.allclose(tf.nn.gelu(tf.constant([1.0])), torch.tensor([0.8413447]))                       # exact erf form
    assert torch.equal(tf.matmul(tf.ones([2, 3]), tf.ones([4, 3]), transpose_b=True), torch.full((2, 4), 3.0))
    assert tf.ones(tf.shape(tf.zeros([5, 2]))[0], "float32").shape == (5,)                                  # scalar shape -> 1-D
    init = tf.keras.initializers.TruncatedNormal(0.02)                # positional argument = MEAN (stddev stays 0.05), as in Keras
    w = init([4000])
    assert abs(float(w.mean()) - 0.02) < 5e-3 and float((w - 0.02).abs().max()) <= 0.1 + 1e-6
    ln = tf.keras.layers.LayerNormalization(epsilon=1e-5, name="ln")
    y = ln(tf.constant([[1.0, 2.0, 3.0, 6.0]]))
    assert abs(float(y.mean())) < 1e-6 and [v.name for v in ln.variables] == ["ln/gamma:0", "ln/beta:0"]
    sched = tf.keras.experimental.CosineDecay(2.0, 10)
    assert abs(float(sched(0)) - 2.0) < 1e-6 and abs(float(sched(5)) - 1.0) < 1e-6 and abs(float(sched(20))) < 1e-6


def test_shim_adam_matches_torch_adam(tf):
    """The Adam base under the reference's AdamWeightDecay: Keras' epsilon-outside-the-bias-correction form.  Against torch.optim.Adam,
    whose epsilon sits inside (eps_hat = eps * sqrt(1 - b2^t)), the two agree when eps is negligible."""
    w = tf.Variable(torch.linspace(-1, 1, 7))
    opt = tf.keras.optimizers.Adam(learning_rate=0.01, beta_1=0.9, beta_2=0.999, epsilon=1e-12)
    p = torch.nn.Parameter(torch.linspace(-1, 1, 7))
    ref = torch.optim.Adam([p], lr=0.01, betas=(0.9, 0.999), eps=1e-12)
    for step in range(4):
        g = torch.sin(torch.arange(7.0) + step)
        opt.apply_gradients([(g, w)])
        p.grad = g.clone()
        ref.step()
    assert float((w.detach() - p.detach()).abs().max()) < 1e-6 and int(opt.iterations) == 4


# ------------------------------------------------------------------------------------------------ MIGT.call == oracle.forward
CASES = [("generate", {}), ("localize", {}), ("losses", {}), ("explicit", {}),
         ("generate", dict(localization_weight="0")), ("losses", dict(localization_weight="0")),
         ("losses", dict(label_smoothing=0.1, pose_multiplier=0.3, image_generation_weight=0.7, localization_weight="cosine(2.0,0.5,100)")),
         ("losses", dict(use_dynamic_pose_loss=True, localization_weight="warmup(linear(1.0,0.2,50),10)")),
         ("generate", dict(token_image_size=4, n_head=2, sequence_size=6))]


@pytest.mark.parametrize("variant,extra", CASES)
def test_reference_call_equals_oracle_forward(R, variant, extra):
    """MIGT.call of the reference (training=False, train counter at step 7) == oracle.forward: every output and every stream's hidden state."""
    from oracle.make_golden import REF_CALL_CASES, ref_shim_inputs
    i = REF_CALL_CASES.index((variant, extra))
    p = f"call{i}."
    kw = dict(SMALL, **extra)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 3)
    if kw.get("use_dynamic_pose_loss"):
        sd = dict(sd, **{"pose_loss_weighting_criterion.pos_ori_weights": torch.tensor([0.3, -2.0])})
    inputs, losses = ref_shim_inputs(cfg, variant, T=cfg.sequence_size)
    use_loc = bool(R[p + "use_localization"])
    lw = float(R[p + "lw"])
    with torch.no_grad():
        o = mo.forward(sd, cfg, inputs, compute_losses=losses, use_localization=use_loc, localization_weight=lw)
    assert len(o["hidden_states"]) == int(R[p + "n_hidden"])
    keys = ["logits", "loss"] + [k for k in ("pose_prediction", "ce_loss", "pose_loss", "pose_pos_loss", "pose_ori_loss") if p + k in R.files]
    assert all(k in o for k in keys) and ("pose_prediction" in o) == (p + "pose_prediction" in R.files)
    for k in keys:
        _close(o[k], p + k, R, 1e-6)
    for j, h in enumerate(o["hidden_states"]):
        _close(h, p + f"hidden{j}", R, 1e-6)
    if losses and use_loc:
        _, reported = at_reference_sample(R, p + "localization_weight", torch.tensor(lw))
        assert abs(float(reported) - lw) < 1e-7


# ------------------------------------------------------------------------------------------------ committed fixtures == reference
@pytest.mark.parametrize("tag,overrides,B,T", [("small", dict(n_layer=2, n_head=4, d_model=128, sequence_size=4, n_loss_skip=1), 2, 4), ("full", {}, 1, 10)])
def test_reference_reproduces_committed_forward_fixture(R, tag, overrides, B, T):
    """tests/golden/migt_{small,full}.npz (what tests/test_models_gpu.py compares the CUDA transformer with; `full` = the 12-layer,
    d = 768 BASELINE model) against what the reference's MIGT.call + reduce_cameras computed on the same weights and inputs."""
    G = np.load(os.path.join(GOLDEN, f"migt_{tag}.npz"))
    assert (int(G["B"]), int(G["T"])) == (B, T)
    fixture, ref = at_reference_sample(R, f"fwd_{tag}.logits_last", torch.from_numpy(G["logits_last"]))
    assert float((ref - fixture).abs().max()) < 2e-5
    assert np.array_equal(R[f"fwd_{tag}.argmax_last"], G["argmax_last"])
    assert float(np.abs(R[f"fwd_{tag}.pose_last"] - G["pose_last"]).max()) < 1e-6


def test_reference_train_step_reproduces_committed_train_fixture(R):
    """Three calls of the reference's MIGT.train_step — GradientTape over its forward, per-tensor clip, its own create_optimizer →
    AdamWeightDecay under WarmUp(CosineDecay) — land on the post-step weights of tests/golden/migt_train_small.npz, the file the CUDA
    trainer is compared with in tests/test_train_gpu.py."""
    meta = json.loads(str(R["train_small.meta"]))
    assert meta["optimizer"] == "AdamWeightDecay" and meta["iterations"] == 3
    G = np.load(os.path.join(GOLDEN, "migt_train_small.npz"))
    keep = [k[3:] for k in G.files if k.startswith("p0.")]
    assert len(keep) >= 6 and keep == meta["keep"]
    for step in range(3):
        pdot = R[f"train_small.pdot{step}"]
        assert np.max(np.abs(pdot - G[f"pdot{step}"]) / (np.abs(G[f"pdot{step}"]) + 1e-3)) < 2e-5, step
        for k in keep:
            fixture, ref = at_reference_sample(R, f"train_small.p{step}.{k}", torch.from_numpy(G[f"p{step}.{k}"]))
            assert float((ref - fixture).abs().max()) < 1e-6, (step, k)
    want = np.cumsum([float(G[f"loss{i}"]) for i in range(3)]) / np.arange(1, 4)
    assert np.allclose(R["train_small.losses"], want, rtol=1e-5)     # running mean of the per-step losses (tf.metrics.Mean)


def test_reference_train_step_gradients_full_size(R):
    """The 12-layer, d = 768 model (MIGTConfig defaults), label smoothing 0.1, localization weight 0.7: loss terms and the gradient of
    every tensor as the reference's train_step computes them == tests/golden/migt_train_full.npz (norm and a random projection)."""
    G = np.load(os.path.join(GOLDEN, "migt_train_full.npz"))
    assert [str(n) for n in R["train_full.names"]] == [str(n) for n in G["names"]]
    assert abs(float(R["train_full.loss"]) - float(G["loss"])) < 1e-5 * abs(float(G["loss"]))
    assert abs(float(R["train_full.ce_loss"]) - float(G["ce"].mean())) < 1e-5 and abs(float(R["train_full.pose_loss"]) - float(G["pose"].mean())) < 1e-5
    cfg = MIGTConfig(dropout=0.0, label_smoothing=0.1, localization_weight="0.7", total_steps=100, learning_rate=1e-4)
    sd = synth.make_migt_state_dict(cfg, 13)
    gen = torch.Generator().manual_seed(78)
    for i, k in enumerate(str(n) for n in G["names"]):
        pn = float(torch.randn(sd[k].shape, generator=gen).norm())
        assert abs(float(R["train_full.gnorm"][i]) - G["gnorm"][i]) <= 2e-4 * G["gnorm"][i] + 1e-7, k
        assert abs(float(R["train_full.gdot"][i]) - G["gdot"][i]) <= 2e-4 * G["gnorm"][i] * pn + 1e-7, k


def test_reference_dynamic_pose_weights_gradient(R):
    """use_dynamic_pose_loss: the learned (pos, ori) log-weights are trainable variables of the reference model; their gradient through
    DynamicLossWeightingCriterion (migt.py:107-120), as its train_step hands it to the optimizer, == autograd through the oracle."""
    from oracle.make_golden import ref_shim_inputs
    kw = dict(SMALL, dropout=0.0, use_dynamic_pose_loss=True, localization_weight="0.5")
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 4)
    inputs, _ = ref_shim_inputs(cfg, "losses")
    leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    leaves["pose_loss_weighting_criterion.pos_ori_weights"] = torch.tensor([0.2, -1.5], requires_grad=True)
    o = mo.forward(leaves, cfg, inputs, compute_losses=True, localization_weight=0.5)
    o["loss"].mean().backward()
    g_ref = torch.from_numpy(R["dyn.grad_pos_ori_weights"])
    assert float((g_ref - leaves["pose_loss_weighting_criterion.pos_ori_weights"].grad).abs().max()) < 1e-6
    got, want = at_reference_sample(R, "dyn.grad_h0_c_attn_weight", leaves["h.0.attn.c_attn.weight"].grad)
    assert float((got - want).abs().max()) < 1e-6


# ------------------------------------------------------------------------------------------------ the evaluation callers
@pytest.mark.parametrize("augment,loc", [("relative", "1"), ("relative", "0"), ("no", "1")])
def test_reference_generate_batch_predictions_equal_oracle(R, augment, loc):
    """evaluate_transformer.py:97-146 and evaluate_transformer_multictx.py:37-95 as shipped — with the REAL reference torch codebook
    behind an NHWC adapter and the real MIGT on the shim — against oracle.generate_batch_predictions{,_multictx}: uint8 views, codes and
    cameras."""
    vcfg, enc, dec = _small_codebook()
    kw = dict(n_layer=2, n_head=4, d_model=64, sequence_size=4, n_embeddings=vcfg.n_embed, token_image_size=8, n_loss_skip=1,
              augment_poses=augment, localization_weight=loc)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 3)
    images = synth.make_images_uint8(2, 4, size=vcfg.image_size, seed=11)
    cams = synth.make_cameras(2, 4, seed=12)
    use_loc = loc != "0"
    p = f"gbp.{augment}.{loc}."

    def fwd(inp):
        return mo.forward(sd, cfg, inp, use_localization=use_loc)
    with torch.no_grad():
        o = mo.generate_batch_predictions(fwd, enc, dec, cfg, images, cams, use_localization=use_loc)
    want = R[p + "generated_images"]
    assert want.dtype == np.uint8 and want.shape == (2, 32, 32, 3) and float(want.std()) > 5
    _same_u8(o["generated_images"], want)
    assert _crc(o["ground_truth_images"]) == int(R[p + "ground_truth_images.crc32"])
    for k in ("ground_truth_cameras", "generated_cameras"):
        assert float((torch.from_numpy(R[p + k]) - o[k]).abs().max()) < 1e-6, k
    assert (p + "multictx.generated_images" in R.files) == use_loc         # the 3-stream script needs the pose head
    if use_loc:
        with torch.no_grad():
            o = mo.generate_batch_predictions_multictx(fwd, enc, dec, cfg, images, cams)
        assert R[p + "multictx.generated_images"].shape == (2, 4, 32, 32, 3)
        _same_u8(o["generated_images"], R[p + "multictx.generated_images"])
        assert float((torch.from_numpy(R[p + "multictx.generated_cameras"]) - o["generated_cameras"]).abs().max()) < 1e-6


def test_reference_allimg_script_equals_oracle(R):
    """evaluate_transformer_multictx_allimg.py:15-88 as shipped (encode_images, transformer_predict, run_with_batchsize, decode_code):
    what viewformer_b200.evaluate mirrors and tests/test_eval_gpu.py::test_transformer_predict_and_steps_match_oracle compares with
    oracle.generate_batch_predictions_multictx.  The script blanks the LAST context camera with zeros where the multictx script keeps
    it (allimg:28 vs multictx:64) — the outputs must not depend on it (the query streams only see strictly earlier views)."""
    vcfg, enc, dec = _small_codebook()
    kw = dict(n_layer=2, n_head=4, d_model=64, sequence_size=4, n_embeddings=vcfg.n_embed, token_image_size=8, n_loss_skip=1)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 3)
    images = synth.make_images_uint8(3, 4, size=vcfg.image_size, seed=41)
    cams = synth.make_cameras(3, 4, seed=42)
    with torch.no_grad():
        o = mo.generate_batch_predictions_multictx(lambda d: mo.forward(sd, cfg, d), enc, dec, cfg, images, cams)
        want_codes = enc(mo.images_to_float(images.reshape(-1, *images.shape[2:])).permute(0, 3, 1, 2).contiguous()).reshape(3, 4, 8, 8)
    assert R["allimg.codes"].shape == (3, 4, 8, 8) and np.array_equal(R["allimg.codes"].astype(np.int64), want_codes.numpy())
    assert np.array_equal(R["allimg.generated_codes"].astype(np.int64), o["generated_codes"].long().numpy())
    assert float((torch.from_numpy(R["allimg.generated_cameras"]) - o["generated_cameras"]).abs().max()) < 1e-6
    _same_u8(o["generated_images"], R["allimg.generated_images"])


def test_process_batch_equals_the_reference_function(R):
    """train/train_transformer.py:31-64 (the pose augmentation mapped over every training sample): the function's own source text,
    cut out of the reference file with ast and executed over the shim with the reference's geometry_tf, against
    viewformer_b200.data.process_batch — every augment mode, both splits, random modes under the same seed (the shim draws from torch's
    global generator, in the order the reference's expressions are evaluated)."""
    from viewformer_b200.data import process_batch
    cams = synth.make_cameras(3, 5, seed=8)                             # [B, T, 7]: the loader maps over [T, 7] windows, batches also work
    toks = synth.make_codes(3, 5, n_embed=16, side=2, seed=9)
    for name, x in (("window", cams[0]), ("batch", cams)):
        for augment in ("relative", "no", "simple", "advanced"):
            for split in ("train", "test"):
                want = torch.from_numpy(R[f"process_batch.{name}.{augment}.{split}"])
                torch.manual_seed(123)
                got, gt = process_batch(x.clone(), toks, augment, split)
                assert gt is toks
                assert float((want - got).abs().max()) < 2e-6, (augment, split)
                assert bool((got[..., 3] >= 0).all()) and float((got[..., 3:].norm(dim=-1) - 1).abs().max()) < 1e-5
                if augment in ("simple", "advanced"):                    # random modes act on the train split only
                    same = float((got - process_batch(x.clone(), toks, "no", split)[0]).abs().max()) < 1e-6
                    assert same == (split != "train")
    with pytest.raises(ValueError):
        process_batch(cams[0], toks, "bogus", "train")


# ---------------------------------------------------------------------------------------- evaluation metrics (utils/metrics.py, Evaluator)
def test_shim_image_ops_follow_documented_tensorflow_semantics(tf):
    """The leaf ops utils/metrics.py adds to the shim's surface: tf.nn.depthwise_conv2d (NHWC, filter [fh,fw,in,mult], output channel
    k*mult + q), tf.image.psnr, tf.image.convert_image_dtype(uint8 -> float = /255), Keras MeanSquaredError (CAST, no rescale)."""
    rng = np.random.default_rng(0)
    x = rng.standard_normal((2, 5, 6, 3)).astype(np.float32)
    w = rng.standard_normal((2, 3, 3, 2)).astype(np.float32)
    y = tf.nn.depthwise_conv2d(tf.constant(x), tf.constant(w), strides=[1, 1, 1, 1], padding="VALID").numpy()
    want = np.zeros((2, 4, 4, 6), np.float32)
    for k in range(3):
        for q in range(2):
            for i in range(4):
                for j in range(4):
                    want[:, i, j, k * 2 + q] = (x[:, i:i + 2, j:j + 3, k] * w[:, :, k, q]).sum((1, 2))
    assert y.shape == want.shape and np.allclose(y, want, atol=1e-5)
    a = rng.integers(0, 256, (2, 8, 8, 3), dtype=np.uint8)
    b = rng.integers(0, 256, (2, 8, 8, 3), dtype=np.uint8)
    fa, fb = tf.image.convert_image_dtype(a, "float32"), tf.image.convert_image_dtype(b, "float32")
    assert fa.dtype == tf.float32 and np.allclose(fa.numpy(), a / 255.0, atol=1e-7)
    mse = ((a / 255.0 - b / 255.0) ** 2).mean((1, 2, 3))
    assert np.allclose(tf.image.psnr(fa, fb, 1).numpy(), 10 * np.log10(1 / mse), atol=1e-4)
    m = tf.keras.metrics.MeanSquaredError("mse")
    m.update_state(a, b)
    assert abs(float(m.result()) - ((a.astype(np.float64) - b) ** 2).mean()) < 1e-2               # 0..255 scale: uint8 is cast, not rescaled
    m = tf.keras.metrics.MeanAbsoluteError("mae")
    m.update_state(a, b)
    assert abs(float(m.result()) - np.abs(a.astype(np.float64) - b).mean()) < 1e-3


def test_evaluator_fixture_is_what_the_reference_evaluator_computes(R, golden_dir):
    """tests/golden/evaluator_reference_shim.npz (what viewformer_b200.metrics.Evaluator is held to on the GPU,
    tests/test_vs_reference_evaluator_gpu.py) against what the reference's own Evaluator (evaluate_transformer.py:22-67) computed."""
    from oracle import make_golden as G
    ref = json.loads(str(R["evaluator"]))
    g = np.load(os.path.join(golden_dir, "evaluator_reference_shim.npz"))
    for tag, n, gs, ns, image_size, seed in G.EVALUATOR_CASES:
        gt, gen = synth.make_metric_pair(n, gs, ns, seed)
        assert [int(gt.sum()), int(gen.sum())] == g[f"{tag}.input_sums"].tolist() == ref[tag]["input_sums"]
        for k in ("mse", "rmse", "mae", "psnr", "ssim"):
            assert abs(ref[tag][k] - float(g[f"{tag}.{k}"])) <= 1e-6 * abs(ref[tag][k]), (tag, k)
    # what follows from HOW the reference calls its metrics: mse / mae on the 0..255 scale, rmse^2 == mse
    assert abs(float(g["same.mse"]) - float(g["same.rmse"]) ** 2) < 1e-3 * float(g["same.mse"]) and float(g["same.mae"]) > 1.0


def test_ssim_of_the_gpu_tests_and_the_k1_quirk_follow_the_reference(R):
    """(a) the fp64 restatement tests/test_eval_gpu.py::ssim_ref that the CUDA kernel is compared with equals the reference's ssim()
    (utils/metrics.py:17-73) with its default K1 = 0.01; (b) SSIMMetric — the class the evaluators use — passes 1 as the THIRD positional
    argument, which is K1, not the data range (metrics.py:183): its value is ssim(K1 = 1), measurably different."""
    import importlib
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    T = importlib.import_module("test_eval_gpu")
    gt, gen = synth.make_metric_pair(4, 64, 64, 5)
    A, B = gt.float() / 255, gen.float() / 255
    ref_default = torch.from_numpy(R["ssim.default_k1"])
    assert torch.allclose(T.ssim_ref(A, B), ref_default, atol=2e-6)
    ref_k1 = float(R["ssim.k1_is_1"])
    assert abs(float(R["ssim.metric_class"]) - ref_k1) < 1e-6
    assert abs(ref_k1 - float(ref_default.mean())) > 1e-4


def test_allow_nan_mean_counts_nan_as_zero_with_full_weight_like_the_reference(R):
    """metrics.py:76-88 replaces NaN by 0 and then computes the weight from is_nan of the CLEANED values: a NaN camera error counts as 0
    with weight 1.  viewformer_b200.metrics.Mean(nan="zero") reproduces that for loc-angle / loc-dist."""
    from viewformer_b200.metrics import Evaluator
    a = torch.tensor([[0., 0, 0, 1, 0, 0, 0], [1, 1, 1, 1, 0, 0, 0], [2, 0, 0, 1, 0, 0, 0]])
    b = torch.tensor([[3., 4, 0, 1, 0, 0, 0], [float("nan"), 1, 1, 1, 0, 0, 0], [2, 0, 1, 1, 0, 0, 0]])
    assert abs(float(R["nan_mean.camera_position_error"]) - 2.0) < 1e-6                 # (5 + 0 + 1) / 3, not (5 + 1) / 2
    ours = Evaluator()
    ours.update_with_camera(a, b)
    assert abs(ours.result()["loc-dist"] - 2.0) < 1e-6


def test_multi_context_evaluator_equals_the_reference_class(R):
    """evaluate_transformer_multictx.py:13-34 as shipped against viewformer_b200.metrics.MultiContextEvaluator: same ctxNN keys, same
    camera statistics per context size (the image half of each Evaluator needs the GPU: tests/test_vs_reference_evaluator_gpu.py)."""
    from viewformer_b200.metrics import MultiContextEvaluator
    ref = json.loads(str(R["multictx"]))
    B, T = 4, 4
    gt_cams = synth.make_cameras(1, B, seed=31)[0]                                     # [B, 7] the target view's camera
    g = torch.Generator().manual_seed(32)
    gen_cams = gt_cams[:, None].repeat(1, T, 1) + 0.2 * torch.randn((B, T, 7), generator=g)
    ours = MultiContextEvaluator(T)
    ours.update_state(gt_cams, gen_cams)                                               # cameras only: nothing touches the device
    o = ours.result()
    assert ref["keys"] == list(o) == ["ctx01", "ctx02", "ctx03"]
    for k in ref["keys"]:
        for m in ("loc-angle", "loc-dist", "loc-angle-med", "loc-dist-med"):
            assert abs(ref["values"][k][m] - o[k][m]) < 2e-6 * max(1.0, abs(o[k][m])), (k, m)
    assert set(ours.get_progress_bar_info()) == {"img_psnr", "cam_loc", "cam_ang"}
    assert abs(ref["cam_loc"] - ours.get_progress_bar_info()["cam_loc"]) < 2e-6


def test_checkpoint_object_paths_are_the_reference_models_attribute_names(R):
    """A TF2 object-based checkpoint (what model.save_weights writes and utils/tensorflow.py:57-61 loads) is keyed by the Python
    attribute names along the path from the model to each variable.  The stored table lists, for every state_dict key, each path of
    public attribute names / list indices that leads from the REAL reference MIGT object to that key's variable (found independently by
    its Keras variable name); tf_checkpoint.object_paths(key)[0] must be one of them — this is what caught 'wpe' (a variable hanging off
    the model itself, not wpe/embeddings) and pose_criterion/pose_classifier (not pose_classifier at the root)."""
    from viewformer_b200 import tf_checkpoint as tfc
    ref = json.loads(str(R["object_paths"]))
    kw = dict(SMALL, use_dynamic_pose_loss=True)
    sd = synth.make_migt_state_dict(MIGTConfig(**kw), 3)
    table = ref["variables"]
    assert set(table) == set(sd) | {"pose_loss_weighting_criterion.pos_ori_weights"}
    assert table["pose_loss_weighting_criterion.pos_ori_weights"]["shape"] == [2] and ref["pos_ori_weights"] == pytest.approx([0.3, -2.0])
    for k in table:
        assert tfc.object_paths(k)[0] in table[k]["paths"], (k, table[k]["paths"])
        if k in sd:
            assert table[k]["shape"] == list(sd[k].shape), k
    # the literal dotted form is NOT an attribute path of the real model for these two groups
    assert "pose_classifier" not in ref["root_attributes"] and not ref["wpe_has_embeddings"]


def test_codebook_evaluation_script_equals_oracle_and_fixture(R, golden_dir):
    """evaluate/evaluate_codebook.py as shipped: its generate_batch_predictions (encode -> decode round trip, BASELINE configs[0]) with the
    REAL torch codebook equals the oracle's encode / decode_code / float_to_images chain — what viewformer_b200.evaluate
    .generate_codebook_predictions is compared with on the GPU — and its Evaluator reports the image numbers of the committed fixture."""
    vcfg, enc, dec = _small_codebook()
    for size in (vcfg.image_size, 48):                                  # 48 -> 32: the dataset resize rule in front of the encoder
        images = synth.make_images_uint8(1, 3, size=size, seed=51)[0]
        x = images if size == vcfg.image_size else torch.from_numpy(R[f"codebook{size}.resized"])
        with torch.no_grad():
            want = mo.float_to_images(dec(enc(mo.images_to_float(x).permute(0, 3, 1, 2).contiguous())).permute(0, 2, 3, 1))
        _same_u8(want, R[f"codebook{size}.generated_images"])
        assert _crc(images) == int(R[f"codebook{size}.ground_truth_images.crc32"])
    ref = json.loads(str(R["codebook.evaluator"]))
    g = np.load(os.path.join(golden_dir, "evaluator_reference_shim.npz"))
    assert ref["keys"] == ["mse", "rmse", "mae", "psnr", "lpips", "ssim"]
    for k in ("mse", "rmse", "mae", "psnr", "ssim"):
        assert abs(ref["values"][k] - float(g["same." + k])) <= 1e-6 * abs(ref["values"][k])
    assert abs(ref["img_rgbl1"] - ref["values"]["mae"]) < 1e-9


def test_reference_test_step_and_predict_step_equal_the_oracle_expectations(R):
    """migt.py:507-541 as shipped, with the real torch codebook attached: the quantities tests/test_eval_gpu.py holds MIGT.test_step /
    predict_step to (mean loss of call(compute_losses=True), token accuracy beyond the first n_loss_skip views, teacher-forced argmax
    tokens and their decoded images) are what the reference's own steps returned."""
    from oracle import make_golden as mg
    vcfg = VQGANConfig(**mg.SMALL_VQ)
    kw = dict(n_layer=2, n_head=4, d_model=64, sequence_size=4, n_embeddings=vcfg.n_embed, token_image_size=8, n_loss_skip=1)
    cfg = MIGTConfig(**kw)
    sd = synth.make_migt_state_dict(cfg, 3)
    codes = synth.make_codes(3, 4, n_embed=cfg.n_embeddings, side=8, seed=5)
    rel = mo.normalize_cameras(mo.to_relative_cameras(synth.make_cameras(3, 4, seed=6))[0])
    with torch.no_grad():
        o = mo.forward(sd, cfg, dict(input_ids=codes, poses=rel), compute_losses=True)
    res = json.loads(str(R["steps.test_step"]))
    assert {"loss", "ce_loss", "acc", "localization_weight", "psnr", "pose_loss", "pose_pos_loss", "pose_ori_loss", "pose_pos_err", "pose_ori_err"} <= set(res)
    assert abs(res["loss"] - float(o["loss"].mean())) < 1e-5 * abs(float(o["loss"].mean()))
    acc = float((o["logits"].argmax(-1)[:, 1:] == codes[:, 1:]).float().mean())
    assert abs(res["acc"] - acc) < 1e-6 and res["psnr"] > 0
    assert np.array_equal(R["steps.latent_code"], o["logits"].argmax(-1).numpy())
    assert R["steps.image_shapes"].tolist() == [[12, 32, 32, 3], [12, 32, 32, 3]]
