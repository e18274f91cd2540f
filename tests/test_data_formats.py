"""TFRecord / tf.train.Example codec, token-dataset loader and the generate-codes scene re-batching logic (CPU)."""
import os

import numpy as np
import pytest
import torch

from viewformer_b200 import data as D


def test_example_codec_roundtrip_and_known_bytes(tmp_path):
    feats = dict(codes=np.arange(-3, 200, dtype=np.int64), cameras=np.linspace(-1, 1, 14, dtype=np.float32), frames=[b"\x89PNG...", b"jpeg"])
    buf = D.encode_example(feats)
    got = D.decode_example(buf)
    assert np.array_equal(got["codes"], feats["codes"]) and np.array_equal(got["cameras"], feats["cameras"]) and got["frames"] == feats["frames"]
    # known answer: Example{features{feature{key:"a" value{int64_list{value:[1]}}}}} as protoc encodes it (packed int64)
    assert D.encode_example(dict(a=np.asarray([1], np.int64))) == bytes.fromhex("0a0c0a0a0a0161120 51a030a0101".replace(" ", ""))
    path = str(tmp_path / "x.tfrecord")
    with D.TFRecordWriter(path) as w:
        w.write(buf)
        w.write(b"")
    recs = list(D.read_tfrecords(path, verify=True))
    assert recs == [buf, b""]
    raw = bytearray(open(path, "rb").read())
    raw[20] ^= 0xFF
    open(path, "wb").write(bytes(raw))
    with pytest.raises(ValueError):
        list(D.read_tfrecords(path, verify=True))


def test_token_dataset_windows_and_sharding(tmp_path):
    rng = np.random.default_rng(0)
    scenes = [dict(cameras=rng.standard_normal((t, 7)).astype(np.float32) + 100 * i, codes=np.full((t, 2, 2), i, np.int64))
              for i, t in enumerate([9, 4, 13, 3, 8, 8, 8, 21])]
    D.write_token_dataset(str(tmp_path), "train", scenes, token_image_size=2, scenes_per_shard=3)
    seq = 4
    batches = list(D.load_token_dataset(str(tmp_path), batch_size=2, sequence_size=seq, token_image_size=2, split="train", repeat=1, seed=3))
    assert all(p.shape == (2, seq, 7) and t.shape == (2, seq, 2, 2) for p, t in batches)
    n_windows = sum(t // seq for t in [9, 4, 13, 3, 8, 8, 8, 21])
    assert len(batches) == n_windows // 2
    for p, t in batches:
        for b in range(2):
            sid = int(t[b, 0, 0, 0])
            assert (t[b] == sid).all() and torch.allclose(p[b].mean(), torch.tensor(100.0 * sid), atol=3.0)     # a window never mixes scenes
            assert len({tuple(v.tolist()) for v in p[b]}) == seq                                             # distinct views
    capped = list(D.load_token_dataset(str(tmp_path), 1, seq, 2, split="train", repeat=1, max_windows_per_environment=1))
    assert len(capped) == sum(1 for t in [9, 4, 13, 3, 8, 8, 8, 21] if t >= seq)
    # the reference's own knob: take(k) on a one-sample dataset (tfrecord_dataset.py:177-181) -> k >= 1 keeps everything, 0 nothing
    assert len(list(D.load_token_dataset(str(tmp_path), 1, seq, 2, split="train", repeat=1, max_samples_per_environment=1))) == n_windows
    assert len(list(D.load_token_dataset(str(tmp_path), 1, seq, 2, split="train", repeat=1, max_samples_per_environment=0))) == 0
    # the training transform (train_transformer.py:113: partial(process_batch, augment=config.augment_poses)) is applied per window
    import functools
    rel = list(D.load_token_dataset(str(tmp_path), 2, seq, 2, split="train", repeat=1, seed=3, transform=functools.partial(D.process_batch, augment="relative")))
    assert len(rel) == len(batches)
    for p, t in rel:
        assert p.dtype == torch.float32 and p.shape == (2, seq, 7) and t.dtype == torch.int64
        assert float(p[:, 0, :3].abs().max()) < 1e-5 and torch.allclose(p[:, 0, 3:], torch.tensor([1.0, 0, 0, 0]).expand(2, 4), atol=1e-5)   # first view = identity
        assert float((p[..., 3:].norm(dim=-1) - 1).abs().max()) < 1e-5 and bool((p[..., 3] >= 0).all())
    r0 = list(D.load_token_dataset(str(tmp_path), 2, seq, 2, split="train", repeat=1, rank=0, world=2))
    r1 = list(D.load_token_dataset(str(tmp_path), 2, seq, 2, split="train", repeat=1, rank=1, world=2))
    s0 = {int(t[b, 0, 0, 0]) for _, t in r0 for b in range(t.shape[0])}
    s1 = {int(t[b, 0, 0, 0]) for _, t in r1 for b in range(t.shape[0])}
    assert not (s0 & s1) and all(p.shape[0] == 1 for p, _ in r0 + r1)        # disjoint file shards, local batch = global / world


def test_latent_code_transformer_rebatches_across_scenes():
    class FakeCodebook:
        class config:
            image_size, stride, batch_size = 8, 4, 5
        device = "cpu"
        calls = []

        def encode_u8(self, x):
            self.calls.append(len(x))
            return x[:, :2, :2, 0].to(torch.int64)          # "codes" = top-left pixels: traceable back to the frame

    import viewformer_b200._lib as L
    orig = L.resize_u8
    L.resize_u8 = lambda x, size, method=None: x            # no device in this test
    try:
        cb = FakeCodebook()
        tr = D.LatentCodeTransformer(cb, batch_size=5)
        assert tr.update_dataset_info({})["token_image_size"] == 2
        scenes = []
        for i, t in enumerate([3, 7, 1, 4]):
            fr = np.zeros((t, 8, 8, 3), np.uint8)
            fr[:, :2, :2, 0] = (10 * i + np.arange(t))[:, None, None]
            scenes.append(dict(frames=fr, cameras=np.full((t, 7), i, np.float32)))
        out = list(tr("train", iter(scenes)))
        assert [len(o["codes"]) for o in out] == [3, 7, 1, 4]
        for i, o in enumerate(out):
            assert (o["cameras"] == i).all() and np.array_equal(o["codes"][:, 0, 0], 10 * i + np.arange(len(o["codes"])))
        assert cb.calls == [5, 5, 5]                          # 15 frames encoded in full batches of 5 across scene boundaries
    finally:
        L.resize_u8 = orig


def test_frames_feature_png_roundtrip(tmp_path):
    """The raw-dataset side of generate-codes (commands/generate_codes.py:58-66): scenes carry `frames` as a bytes_list of encoded
    images; decode_frames turns them into the uint8 [T,H,W,3] array LatentCodeTransformer takes (PNG is lossless, so exact)."""
    import io
    PIL = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(4)
    frames = rng.integers(0, 256, (3, 20, 24, 3), dtype=np.uint8)
    blobs = []
    for f in frames:
        buf = io.BytesIO()
        PIL.fromarray(f).save(buf, format="PNG")
        blobs.append(buf.getvalue())
    cams = rng.standard_normal((3, 7)).astype(np.float32)
    path = str(tmp_path / "raw.tfrecord")
    with D.TFRecordWriter(path) as w:
        w.write(D.encode_example(dict(frames=blobs, cameras=cams)))
    (rec,) = list(D.read_tfrecords(path, verify=True))
    ex = D.decode_example(rec)
    assert list(ex["frames"]) == blobs
    got = D.decode_frames(ex["frames"])
    assert got.dtype == np.uint8 and got.shape == frames.shape and np.array_equal(got, frames)
    assert np.array_equal(np.asarray(ex["cameras"], np.float32).reshape(3, 7), cams)


def test_latent_code_transformer_equals_the_reference_class():
    """commands/generate_codes.py:20-78 (the reference's LatentCodeTransformer, run as shipped with a stand-in for webdataset's three
    filters and a stand-in codebook returning the top-left 2x2 pixels of channel 0; stored by oracle/make_golden.py::ref_latent_code_transformer)
    against data.LatentCodeTransformer on the same scenes with the same stand-in codebook: same scenes out, same codes, same cameras, same
    encoder batch sizes.  Equal-length scenes: with ragged scenes the reference mis-assigns the carried-over frames (it assumes they belong
    to a scene as long as the next batch's first one, generate_codes.py:63) — this implementation keeps a queue."""
    import json
    from oracle.make_golden import reference_outputs, latent_code_scenes
    R = reference_outputs()
    ref = json.loads(str(R["lct.meta"]))

    class Cfg:
        image_size, stride, batch_size = 8, 4, 5

    class OurCodebook:
        config, device, calls = Cfg, "cpu", []

        def encode_u8(self, x):                              # NHWC uint8
            self.calls.append(len(x))
            return x[:, :2, :2, 0].to(torch.int64)

    import viewformer_b200._lib as L
    orig = L.resize_u8
    L.resize_u8 = lambda x, size, method=None: x            # frames already have the codebook's size; no device in this test
    try:
        ocb = OurCodebook()
        our_tr = D.LatentCodeTransformer(ocb, batch_size=5)
        assert our_tr.update_dataset_info({}) == ref["dataset_info"] == {"token_image_size": 2}
        for feats in (None, ["frames", "cameras"], ["frames", "cameras-gqn"]):
            assert our_tr.output_features(feats) == ref["output_features"][str(feats)]
        got = list(our_tr("train", iter([dict(s) for s in latent_code_scenes()])))
    finally:
        L.resize_u8 = orig
    assert len(got) == ref["n_scenes"] == 4 and ocb.calls == ref["encoder_calls"] == [5, 5, 5, 5, 4]
    for i, g in enumerate(got):
        assert np.array_equal(R[f"lct.codes{i}"], np.asarray(g["codes"])) and np.array_equal(R[f"lct.cameras{i}"], np.asarray(g["cameras"]))
