"""The drop-in boundary, exercised through the REAL reference registry (viewformer/models/__init__.py:15-59):
AutoModelTH.from_config / AutoModel.from_config must hand out viewformer_b200 objects, both with the run-time patch
(viewformer_b200.compat.install) and with the three shim files of integration/ placed on the package path.
CPU-only: constructing the model objects touches no device (weights are laid out at load_state_dict).
The registry tests execute the reference package itself and skip where its sources are absent; the state_dict keys they compare are
also held to the reference's, stored in tests/golden/reference_outputs.npz, everywhere."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from oracle import ref_loader  # noqa: E402

needs_reference = pytest.mark.skipif(not ref_loader.available(), reason="the reference package's sources are not present")


def _fresh_registry(extra_paths=()):
    for k in [k for k in sys.modules if k.startswith("viewformer.models.") and "b200" in k]:
        del sys.modules[k]
    return ref_loader.load_reference_registry(extra_paths)


@needs_reference
def test_unpatched_registry_returns_reference_class():
    reg = _fresh_registry()
    cfg = reg.load_config({"model": "vqgan", "ch": 32, "ch_mult": [1, 2], "attn_resolutions": [], "image_size": 16, "embed_dim": 8,
                           "z_channels": 8, "n_embed": 16, "num_res_blocks": 1})
    m = reg.AutoModelTH.from_config(cfg)
    assert type(m).__module__ == "viewformer.models.vqgan_th"


@needs_reference
@pytest.mark.parametrize("how", ["install", "shim_files"])
def test_registry_hands_out_b200_models(how):
    from viewformer_b200 import compat, VQGAN, MIGT
    if how == "install":
        reg = compat.install(_fresh_registry())
    else:
        reg = _fresh_registry([os.path.join(ROOT, "integration", "viewformer", "models")])
        reg._TH_REPOSITORY.update({"vqgan": ("vqgan_b200_th", "VQGAN")})                                   # the lines INTEGRATION.md documents
        reg._TF_REPOSITORY.update({"vqgan": ("vqgan_b200", "VQGAN"), "migt": ("migt_b200", "MIGT")})
    vcfg = reg.load_config({"model": "vqgan"})              # the reference's own config object goes in
    th = reg.AutoModelTH.from_config(vcfg)
    assert isinstance(th, VQGAN) and type(th) is compat.VQGAN_TH
    assert th.config.image_size == 128 and th.config.stride == 16 and th.config.n_embed == 1024
    tf_ = reg.AutoModel.from_config(vcfg)
    assert type(tf_) is compat.VQGAN_TF and isinstance(tf_, VQGAN)
    tcfg = reg.load_config({"model": "migt", "localization_weight": "cosine(1,0,100)" if False else "1"})
    tr = reg.AutoModel.from_config(tcfg)
    assert isinstance(tr, MIGT) and tr.mask_token == 1024 and tr.localization_token == 1025 and tr.use_localization
    # state_dict keys of the b200 codebook are the reference's (strict load both ways)
    ref_model = ref_loader.build_reference_vqgan(ch=32, ch_mult=[1, 2], attn_resolutions=[8], image_size=16, embed_dim=8,
                                                 z_channels=8, n_embed=16, num_res_blocks=1)
    small = reg.AutoModelTH.from_config(reg.load_config({"model": "vqgan", "ch": 32, "ch_mult": [1, 2], "attn_resolutions": [8],
                                                         "image_size": 16, "embed_dim": 8, "z_channels": 8, "n_embed": 16,
                                                         "num_res_blocks": 1}))
    want = {k for k in ref_model.state_dict() if not k.startswith(("perceptual_loss.", "loss."))}
    assert set(small.expected_keys()) == want


def test_b200_codebook_state_dict_keys_are_the_reference_models():
    """Strict loading both ways needs the b200 codebook to expect exactly the reference VQGAN's state_dict keys (its loss modules aside)."""
    from oracle.make_golden import REGISTRY_SMALL_VQ, reference_outputs
    from viewformer_b200 import compat
    from viewformer_b200.config import VQGANConfig
    small = compat.VQGAN_TH(VQGANConfig(**REGISTRY_SMALL_VQ))
    assert sorted(small.expected_keys()) == [str(k) for k in reference_outputs()["vqgan.state_dict_keys"]]


def test_tf_flavour_rejects_nchw_input():
    """ADVICE r1: a layout mistake must fail before any kernel runs."""
    import torch
    from viewformer_b200 import compat
    m = compat.VQGAN_TF()
    m._w = {}                                  # pretend weights are present: the layout check comes first
    with pytest.raises(ValueError, match="NHWC"):
        m.encode(torch.zeros(2, 3, 128, 128))
    with pytest.raises(ValueError, match="NCHW"):
        compat.VQGAN_TH.encode(m, torch.zeros(2, 128, 128, 3))
