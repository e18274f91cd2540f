"""``generate()`` — the reference's novel-view synthesis entry point, B200-native.

Mirrors ``generate_batch_predictions(transformer_model, codebook_model, images, cameras)`` of
viewformer/evaluate/evaluate_transformer.py:97-146 (same argument meaning, same result dict), so that
evaluate_co3d.py:33,74 / evaluate_sevenscenes.py:14,262 / generate_images.py:7,29 keep working when the
models are the viewformer_b200 ones.  Camera pre/post-processing (a few floats per scene) is host-side
torch on whatever device the cameras live on; all image / token work runs in libvf_b200 kernels.
"""
import torch

from . import _lib as L


# --------------------------------------------------------------------------- quaternion helpers (utils/geometry_tf.py:6-13,44-91)
def quaternion_multiply(q1, q2):
    w1, x1, y1, z1 = q1.unbind(-1)
    w2, x2, y2, z2 = q2.unbind(-1)
    return torch.stack((-x1 * x2 - y1 * y2 - z1 * z2 + w1 * w2,
                        x1 * w2 + y1 * z2 - z1 * y2 + w1 * x2,
                        -x1 * z2 + y1 * w2 + z1 * x2 + w1 * y2,
                        x1 * y2 - y1 * x2 + z1 * w2 + w1 * z2), -1)


def quaternion_conjugate(q):
    return torch.cat((q[..., :1], -q[..., 1:]), -1)


def quaternion_rotate(point, q):
    p = torch.cat([torch.zeros_like(point[..., :1]), point], -1)
    return quaternion_multiply(quaternion_multiply(q, p), quaternion_conjugate(q))[..., 1:]


def quaternion_normalize(x, epsilon=1e-12):
    return x * torch.rsqrt(torch.clamp((x * x).sum(-1, keepdim=True), min=epsilon))


def quaternion_remove_sign(x):
    return x * (2 * (x[..., :1] >= 0).to(x.dtype) - 1)


def reduce_cameras(x, axis=-2):
    """migt.py:150-154 + 123-129."""
    x = torch.as_tensor(x)
    q = quaternion_remove_sign(quaternion_normalize(x[..., 3:])).mean(axis)
    q = quaternion_remove_sign(quaternion_normalize(q))
    return torch.cat((x[..., :3].mean(axis), q), -1)


def to_relative_cameras(cameras):
    """evaluate_transformer.py:70-78."""
    xyz, quat = cameras[..., :3], cameras[..., 3:]
    t_xyz, t_q = xyz[..., :1, :], quat[..., :1, :]
    inv = quaternion_conjugate(t_q).expand_as(quat)
    return torch.cat((quaternion_rotate(xyz - t_xyz, inv), quaternion_multiply(inv, quat)), -1), torch.cat((t_xyz, t_q), -1)


def from_relative_cameras(cameras, transform):
    """evaluate_transformer.py:81-87."""
    t_xyz, t_q = transform[..., :3], transform[..., 3:]
    xyz, quat = cameras[..., :3], cameras[..., 3:]
    t_qe = t_q.expand_as(quat)
    return torch.cat((quaternion_rotate(xyz, t_qe) + t_xyz, quaternion_multiply(t_qe, quat)), -1)


def normalize_cameras(cameras):
    """evaluate_transformer.py:90-94."""
    return torch.cat((cameras[..., :3], quaternion_remove_sign(quaternion_normalize(cameras[..., 3:]))), -1)


# --------------------------------------------------------------------------- generate
def generate_batch_predictions(transformer_model, codebook_model, images, cameras, *, encode_target=None):
    """images uint8 [B,T,H,W,3] (host or device), cameras f32 [B,T,7] ->
    dict(ground_truth_images [B,H,W,3] u8, generated_images [B,H,W,3] u8, ground_truth_cameras [B,7],
         generated_cameras [B,7]) — evaluate_transformer.py:97-146.

    ``encode_target``: the reference encodes all T views and, when the model localises, runs a second
    forward on the true codes of the target view (:134-136).  Default: encode the target only when that
    second forward is needed (skipping it does not change any returned value, SURVEY.md Appendix A.18).
    """
    _dev = getattr(codebook_model, "device", None)
    if _dev is not None and _dev.type == "cuda" and _dev.index is not None and _dev.index != torch.cuda.current_device():
        with torch.cuda.device(_dev):            # kernels launch on the current device's stream: make the models' device current
            return generate_batch_predictions(transformer_model, codebook_model, images, cameras, encode_target=encode_target)
    dev = transformer_model.device
    images = torch.as_tensor(images)
    cameras = torch.as_tensor(cameras)
    if cameras.dtype != torch.float32:
        cameras = cameras.to(torch.float32)
    gt_cam = cameras[:, -1]
    relative = transformer_model.config.augment_poses == "relative"
    cams_dev, transform = L.cameras_prepare(cameras.to(dev, non_blocking=True).contiguous(), relative)   # :99-102, one launch

    B, T = images.shape[:2]
    size = codebook_model.config.image_size
    use_loc = transformer_model.use_localization
    if encode_target is None:
        encode_target = use_loc
    img_dev = images.to(device=dev, non_blocking=True) if images.device != dev else images
    side = transformer_model.token_image_size
    n_enc = T if encode_target else T - 1
    if not img_dev.is_contiguous():
        img_dev = img_dev.contiguous()
    if images.shape[2] != size or images.shape[3] != size:        # resize_tf (evaluate_transformer.py:104, data/_common.py:19-62)
        img_dev = L.resize_u8(img_dev[:, :n_enc].reshape((-1,) + tuple(img_dev.shape[2:])).contiguous(), size)
        img_dev = img_dev.reshape((B, n_enc) + tuple(img_dev.shape[1:]))
        if img_dev.shape[2] != size or img_dev.shape[3] != size:      # the rule leaves images with one side == size unchanged
            raise ValueError(f"{images.shape[2]}x{images.shape[3]} images do not resize to the codebook's {size}x{size} under the dataset "
                             "resize rule (it returns them unchanged when one side already matches)")
    codes = codebook_model.encode_u8(img_dev, first_views=n_enc).reshape(B, n_enc, side, side)

    gen_codes = transformer_model.generate_codes(codes[:, : T - 1], cams_dev)
    gen_images = codebook_model.decode_code_u8(gen_codes)

    if use_loc:
        out = transformer_model(dict(input_ids=codes, poses=cams_dev[:, :-1].contiguous()))
        gen_cam = reduce_cameras(out["pose_prediction"][:, -1:], -2)
    else:
        gen_cam = cams_dev[:, :1]
    if relative:
        gen_cam = L.cameras_from_relative(gen_cam.to(dev).contiguous(), transform)
    return dict(ground_truth_images=images[:, -1], generated_images=gen_images, ground_truth_cameras=gt_cam,
                generated_cameras=gen_cam[:, -1], generated_codes=gen_codes)


class GraphedPredictions:
    """``generate_batch_predictions`` for a fixed (scenes, views) shape, captured once into a CUDA graph and replayed: one
    cudaGraphLaunch per batch instead of ~380 kernel launches (each tcgen05 / streaming kernel is 10-1000 us long, so the
    launch gaps of the eager path are ~5 % of a step).  Inputs are copied into static device buffers (from pinned host memory
    or from device tensors), outputs live in static device tensors that the next call overwrites.

    Only the non-localising configuration is graph-safe: camera localisation ends in a host-side quaternion mean
    (``reduce_cameras``), which a capture cannot contain."""

    def __init__(self, transformer_model, codebook_model, scenes, views, warmup=2):
        if transformer_model.use_localization:
            raise NotImplementedError("GraphedPredictions: the localisation branch reduces cameras on the host; use generate_batch_predictions")
        dev = transformer_model.device
        size = codebook_model.config.image_size
        self.device = dev
        self.images = torch.zeros((scenes, views, size, size, 3), dtype=torch.uint8, device=dev)
        self.cameras = torch.zeros((scenes, views, 7), dtype=torch.float32, device=dev)
        self.cameras[..., 3] = 1.0                                   # identity quaternions for the warm-up passes
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                                # warm-up outside the capture: lazy one-time setup, allocator pools
            for _ in range(max(1, warmup)):
                generate_batch_predictions(transformer_model, codebook_model, self.images, self.cameras)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        n0 = L.launch_count()
        with torch.cuda.graph(self.graph):
            self.outputs = generate_batch_predictions(transformer_model, codebook_model, self.images, self.cameras)
        self.launches_per_replay = L.launch_count() - n0             # libvf_b200 kernel-launching calls recorded in the graph

    def __call__(self, images, cameras):
        self.images.copy_(torch.as_tensor(images), non_blocking=True)
        self.cameras.copy_(torch.as_tensor(cameras), non_blocking=True)
        self.graph.replay()
        return self.outputs


def generate_batch_predictions_multictx(transformer_model, codebook_model, images, cameras):
    """Multi-context variant — viewformer/evaluate/evaluate_transformer_multictx.py:37-95: one 3-stream forward yields,
    for every context size i, the query view rendered from context views 0..i-1 (stream 1) and the query localised
    against them (stream 2).  Returns generated_images [B,T,H,W,3] u8 and generated_cameras [B,T,7]."""
    _dev = getattr(codebook_model, "device", None)
    if _dev is not None and _dev.type == "cuda" and _dev.index is not None and _dev.index != torch.cuda.current_device():
        with torch.cuda.device(_dev):            # kernels launch on the current device's stream: make the models' device current
            return generate_batch_predictions_multictx(transformer_model, codebook_model, images, cameras)
    dev = transformer_model.device
    images = torch.as_tensor(images)
    cameras = torch.as_tensor(cameras)
    if cameras.dtype != torch.float32:
        cameras = cameras.to(torch.float32)
    gt_cam = cameras[:, -1]
    relative = transformer_model.config.augment_poses == "relative"
    cams, transform = L.cameras_prepare(cameras.to(dev, non_blocking=True).contiguous(), relative)
    B, T = images.shape[:2]
    side = transformer_model.token_image_size
    img_dev = images.to(device=dev, non_blocking=True) if images.device != dev else images
    codes = codebook_model.encode_u8(img_dev.contiguous(), first_views=T).reshape(B, T, side, side)
    mask = torch.full_like(codes[:, :1], transformer_model.mask_token)
    input_ids = torch.cat([codes[:, :-1], mask], 1)                                    # :61-62
    context_cameras = torch.cat([cams[:, :-1], torch.zeros_like(cams[:, :1])], 1)      # :63
    out = transformer_model(dict(input_ids=input_ids, poses=context_cameras,
                                 localization_tokens=codes[:, -1:].repeat(1, T, 1, 1).contiguous(),
                                 output_poses=cams[:, -1:].repeat(1, T, 1).contiguous()))       # :66-73
    logits = out["logits"]
    gen_codes = L.argmax_rows(logits.reshape(-1, logits.shape[-1])).reshape(B * T, side, side)   # :76
    gen_images = codebook_model.decode_code_u8(gen_codes)
    gen_images = gen_images.reshape((B, T) + tuple(gen_images.shape[1:]))
    gen_cam = reduce_cameras(out["pose_prediction"], -2)                               # :77  [B,T,7]
    if relative:
        gen_cam = L.cameras_from_relative(gen_cam.to(dev).contiguous(), transform)
    return dict(ground_truth_images=images[:, -1], generated_images=gen_images, ground_truth_cameras=gt_cam,
                generated_cameras=gen_cam)
