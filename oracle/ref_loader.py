"""TEST INFRASTRUCTURE — import the *real* reference torch VQGAN from /root/reference.

Container only (the GPU box has no /root/reference).  Three absent third-party modules are stubbed
(aparse.Literal, pytorch_lightning.LightningModule, lpips.LPIPS -> zeros); the reference sources are
loaded in place by file path — nothing is copied.  Recipe from SURVEY.md §8(c).
"""
import importlib.util
import os
import sys
import types
import typing

import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("VIEWFORMER_REFERENCE", "/root/reference")


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "viewformer", "models", "vqgan_th.py"))


class _ZeroLPIPS(nn.Module):
    def __init__(self, **kw):
        super().__init__()

    def forward(self, a, b):
        return torch.zeros(a.shape[0], 1, 1, 1)


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


_cache = {}


def load_reference_modules():
    """Returns (config_module, utils_th_module, vqgan_th_module) of the real reference."""
    if "mods" in _cache:
        return _cache["mods"]
    if not available():
        raise RuntimeError("reference sources not present at %s" % REFERENCE_ROOT)
    if "aparse" not in sys.modules:
        ap = types.ModuleType("aparse")
        ap.Literal = typing.Literal
        sys.modules["aparse"] = ap
    if "pytorch_lightning" not in sys.modules:
        pl = types.ModuleType("pytorch_lightning")
        pl.LightningModule = nn.Module
        sys.modules["pytorch_lightning"] = pl
    if "lpips" not in sys.modules:
        lp = types.ModuleType("lpips")
        lp.LPIPS = _ZeroLPIPS
        sys.modules["lpips"] = lp
    for pkg in ("viewformer", "viewformer.utils", "viewformer.models"):
        if pkg not in sys.modules:
            p = types.ModuleType(pkg)
            p.__path__ = []
            sys.modules[pkg] = p
    R = os.path.join(REFERENCE_ROOT, "viewformer")
    _load("viewformer.utils.schedules", R + "/utils/schedules.py")
    cfg = _load("viewformer.models.config", R + "/models/config.py")
    uth = _load("viewformer.models.utils_th", R + "/models/utils_th.py")
    vq = _load("viewformer.models.vqgan_th", R + "/models/vqgan_th.py")
    _cache["mods"] = (cfg, uth, vq)
    return _cache["mods"]


def build_reference_vqgan(state_dict=None, **cfg_overrides):
    """Instantiate the real reference VQGAN (eval mode — see SURVEY.md §8 a6 quirk)."""
    cfg_mod, _, vq = load_reference_modules()
    cfg = cfg_mod.VQGANConfig(**cfg_overrides)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        model = vq.VQGAN(cfg)
    if state_dict is not None:
        model.load_state_dict(state_dict, strict=True)
    return model.eval()


def load_reference_registry(extra_paths=()):
    """Executes the REAL ``viewformer/models/__init__.py`` (AutoModel / AutoModelTH / load_config and the two override tables)
    as the package ``viewformer.models``.  ``extra_paths`` are appended to the package ``__path__`` (how a maintainer's copied
    shim modules become importable as ``viewformer.models.<shim>``)."""
    load_reference_modules()
    R = os.path.join(REFERENCE_ROOT, "viewformer", "models")
    spec = importlib.util.spec_from_file_location("viewformer.models", os.path.join(R, "__init__.py"),
                                                  submodule_search_locations=[R] + list(extra_paths))
    m = importlib.util.module_from_spec(spec)
    sys.modules["viewformer.models"] = m
    spec.loader.exec_module(m)
    return m


# ----------------------------------------------------------------------------------------------- the TensorFlow half, on oracle/tf_shim.py
def migt_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "viewformer", "models", "migt.py"))


def load_reference_migt():
    """Executes the reference's transformer sources UNMODIFIED from /root/reference — models/migt.py, models/branching_attention.py,
    models/utils.py (WarmUp, AdamWeightDecay, create_optimizer), utils/tensorflow.py (shape_list), utils/geometry_tf.py,
    utils/metrics.py, utils/schedules.py — with oracle/tf_shim.py answering ``import tensorflow``.  Returns the ``migt`` module."""
    if "migt" in _cache:
        return _cache["migt"]
    if not migt_available():
        raise RuntimeError("reference sources not present at %s" % REFERENCE_ROOT)
    from oracle import tf_shim
    tf_shim.install()
    load_reference_registry()                                       # the real viewformer.models package (config, registry)
    R = os.path.join(REFERENCE_ROOT, "viewformer")
    # (utils/__init__.py itself is not executed: it pulls tqdm / requests download helpers that are not on this path)
    sys.modules["viewformer.utils"].__path__ = [os.path.join(R, "utils")]
    for name in ("geometry_tf", "tensorflow", "metrics"):
        _load("viewformer.utils." + name, os.path.join(R, "utils", name + ".py"))
        setattr(sys.modules["viewformer.utils"], name, sys.modules["viewformer.utils." + name])
    m = importlib.import_module("viewformer.models.migt")           # resolves .branching_attention / .config / .utils from the real directory
    _cache["migt"] = m
    return m


_TF_NAME = {"wpe.embeddings": "wpe/embeddings"}


def build_reference_migt(state_dict, dynamic_pose_weights=None, **cfg_overrides):
    """The real reference MIGT (constructed by its own __init__, which runs one forward to create the variables) with every variable
    overwritten from ``state_dict`` (keys of viewformer_b200.MIGT / oracle.synth: 'h.0.attn.c_attn.weight', 'wpe.embeddings', ...).
    Variable names come from the shim's call-time scopes ('migt/h.0/attn/c_attn/weight:0'); each state_dict key must match exactly one."""
    migt = load_reference_migt()
    cfg_mod = sys.modules["viewformer.models.config"]
    sched = sys.modules["viewformer.utils.schedules"]
    kw = dict(cfg_overrides)
    if isinstance(kw.get("localization_weight"), (str, int, float)):
        kw["localization_weight"] = sched.Schedule.from_str(str(kw["localization_weight"]))
    model = migt.MIGT(cfg_mod.MIGTConfig(**kw))
    variables = {v.name[:-2]: v for v in model.variables}           # strip ':0'
    used = set()
    for key, val in state_dict.items():
        suffix = "/" + key.replace(".", "/")
        # layer names contain dots ('h.0'): compare with dots turned into slashes on both sides
        hits = [n for n in variables if ("/" + n.replace(".", "/")).endswith(suffix)]
        if not hits and key.startswith("pose_classifier.") and not model.use_localization:
            continue                                                # the pose head is never called, Keras never builds its variables
        if len(hits) != 1:
            raise KeyError(f"state_dict key {key} matches {hits} among the reference's variables")
        v = variables[hits[0]]
        if tuple(v.shape) != tuple(val.shape):
            raise ValueError(f"{key}: reference variable {hits[0]} has shape {tuple(v.shape)}, state_dict {tuple(val.shape)}")
        v.assign(val)
        used.add(hits[0])
    left = sorted(set(variables) - used)
    if dynamic_pose_weights is not None:
        variables["pos_ori_weights"].assign(torch.as_tensor(dynamic_pose_weights, dtype=torch.float32))
        left = [n for n in left if n != "pos_ori_weights"]
    left = [n for n in left if n != "pos_ori_weights"]              # keeps its initial [0, -3] unless given
    if left:
        raise KeyError(f"reference variables without a state_dict entry: {left}")
    return model


def load_reference_evaluate():
    """The reference's evaluation callers, executed unmodified on the shim: evaluate/evaluate_transformer.py (generate_batch_predictions,
    to_relative_cameras, from_relative_cameras, normalize_cameras) and evaluate/evaluate_transformer_multictx.py.  Argument-parsing
    decorators (aparse.click / ConditionalType) and the dataset loader table are stubbed — they are not on the path."""
    if "evaluate" in _cache:
        return _cache["evaluate"]
    load_reference_migt()
    R = os.path.join(REFERENCE_ROOT, "viewformer")
    ap = sys.modules["aparse"]
    if not hasattr(ap, "click"):
        click = types.SimpleNamespace(command=lambda *a, **k: (lambda f: f))
        ap.click = click
        ap.ConditionalType = lambda name, table, default=None: typing.Any
    common = _load("viewformer.utils._common", os.path.join(R, "utils", "_common.py"))
    for n in ("SplitIndices", "unique", "batch_slice", "batch_len", "single", "dict_replace", "is_torch_model"):
        if hasattr(common, n):
            setattr(sys.modules["viewformer.utils"], n, getattr(common, n))
    for pkg, sub in (("viewformer.data", "data"), ("viewformer.evaluate", "evaluate")):
        if pkg not in sys.modules:
            p = types.ModuleType(pkg)
            p.__path__ = []
            sys.modules[pkg] = p
    loaders = types.ModuleType("viewformer.data.loaders")
    loaders.get_loaders = lambda: {}
    sys.modules["viewformer.data.loaders"] = loaders
    _load("viewformer.data._common", os.path.join(R, "data", "_common.py"))
    ev = _load("viewformer.evaluate.evaluate_transformer", os.path.join(R, "evaluate", "evaluate_transformer.py"))
    mc = _load("viewformer.evaluate.evaluate_transformer_multictx", os.path.join(R, "evaluate", "evaluate_transformer_multictx.py"))
    _cache["evaluate"] = (ev, mc)
    return _cache["evaluate"]


class ReferenceCodebookNHWC:
    """The real reference torch codebook (vqgan_th.VQGAN, NCHW) behind the TF-flavour calls the evaluation scripts make
    (models/vqgan.py:284-301: NHWC images in, NHWC images out) — a pure layout adapter."""

    def __init__(self, vqgan):
        self.model, self.config = vqgan, vqgan.config

    def encode(self, x):
        with torch.no_grad():
            q, diff, codes = self.model.encode(torch.as_tensor(x).as_subclass(torch.Tensor).permute(0, 3, 1, 2).contiguous())
        return q.permute(0, 2, 3, 1), diff, codes

    def decode_code(self, codes, training=False):
        with torch.no_grad():
            return self.model.decode_code(torch.as_tensor(codes).as_subclass(torch.Tensor).long()).permute(0, 2, 3, 1).contiguous()


def load_reference_generate_codes():
    """commands/generate_codes.py loaded as shipped, with stand-ins for what is not on this path: `webdataset.filters` (three generators
    restating the documented behaviour of map_ / unbatched_ / batched_ with the default collation), aparse.click, viewformer.data
    .transform_dataset; TensorFlow is made un-importable for the duration so that the script's own `except ImportError` branch runs."""
    import numpy as np
    load_reference_modules()
    ap = sys.modules["aparse"]
    if not hasattr(ap, "click"):                          # the same stand-ins load_reference_evaluate installs
        ap.click = types.SimpleNamespace(command=lambda *a, **k: (lambda f: f))
    if not hasattr(ap, "ConditionalType"):
        ap.ConditionalType = lambda name, table, default=None: typing.Any
    utils = sys.modules["viewformer.utils"]
    if not hasattr(utils, "SplitIndices"):
        utils.SplitIndices = object
    data = sys.modules.get("viewformer.data")
    if data is None:
        data = types.ModuleType("viewformer.data")
        data.__path__ = []
        sys.modules["viewformer.data"] = data
    data.transform_dataset = lambda *a, **k: None

    def collate(samples):
        cols = list(zip(*samples))
        out = []
        for c in cols:
            if isinstance(c[0], (int, float)):
                out.append(np.array(list(c)))
            elif isinstance(c[0], torch.Tensor):
                out.append(torch.stack(list(c)))
            elif isinstance(c[0], np.ndarray):
                out.append(np.array(list(c)))
            else:
                out.append(list(c))
        return out

    def map_(data, f):
        for s in data:
            yield f(s)

    def unbatched_(data):
        for s in data:
            for i in range(len(s[0])):
                yield tuple(x[i] for x in s)

    def batched_(data, batchsize=20, partial=True):
        batch = []
        for s in data:
            if len(batch) >= batchsize:
                yield collate(batch)
                batch = []
            batch.append(s)
        if batch and (len(batch) == batchsize or partial):
            yield collate(batch)

    wds = types.ModuleType("webdataset")
    wds.filters = types.SimpleNamespace(map_=map_, unbatched_=unbatched_, batched_=batched_)
    saved_wds, saved_tf = sys.modules.get("webdataset"), sys.modules.pop("tensorflow", None)
    sys.modules["webdataset"] = wds
    sys.modules["tensorflow"] = None                      # `import tensorflow` -> ImportError, as on a torch-only machine
    try:
        path = os.path.join(REFERENCE_ROOT, "viewformer", "commands", "generate_codes.py")
        spec = importlib.util.spec_from_file_location("viewformer_commands_generate_codes_ref", path)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
    finally:
        if saved_tf is not None:
            sys.modules["tensorflow"] = saved_tf
        else:
            sys.modules.pop("tensorflow", None)
    return m, (lambda: sys.modules.__setitem__("webdataset", saved_wds) if saved_wds is not None else sys.modules.pop("webdataset", None))
