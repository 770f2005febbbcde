"""TEST INFRASTRUCTURE ONLY -- imports the UNMODIFIED reference from the checkout named by $OMT_REFERENCE_ROOT.

Used by oracle/make_golden.py to record the reference's outputs as tests/golden/*.pt;
the tests compare against those files and never import this module.

Recipe follows SURVEY.md Appendix D: the packages the reference imports but the
image lacks (pytorch_lightning, timm, fairscale, imageio) are stubbed; none of
the stubs touch hot-path arithmetic.  LPIPS is replaced by a dummy because its
constructor downloads VGG16 (modules/lpips.py:59,123).
"""
import os
import sys
import types
import argparse
import warnings

import torch
import torch.nn as nn

REF_ROOT = os.environ.get("OMT_REFERENCE_ROOT", "")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isdir(os.path.join(REF_ROOT, "OmniTokenizer"))


_loaded = None


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def load():
    """Returns (omnitokenizer module, base module) of the reference."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError(f"reference tree not found at OMT_REFERENCE_ROOT={REF_ROOT!r} (a checkout of the reference)")
    warnings.filterwarnings("ignore")

    class _LM(nn.Module):  # stands in for pl.LightningModule
        def save_hyperparameters(self, *a, **k):
            pass

        def log(self, *a, **k):
            pass

        @property
        def global_step(self):
            return 0

    _mod("pytorch_lightning", LightningModule=_LM, LightningDataModule=object, Trainer=object)
    _mod("pytorch_lightning.callbacks", Callback=object, ModelCheckpoint=object, LearningRateMonitor=object)
    _mod("pytorch_lightning.utilities")
    _mod("pytorch_lightning.utilities.distributed", rank_zero_only=lambda f: f)
    _mod("pytorch_lightning.loggers", WandbLogger=object)
    _mod("timm")
    _mod("timm.scheduler")
    _mod("timm.scheduler.cosine_lr", CosineLRScheduler=object)
    _mod("timm.models")
    _mod("timm.models.layers", trunc_normal_=nn.init.trunc_normal_, DropPath=nn.Identity,
         to_2tuple=lambda x: (x, x))
    _mod("fairscale")
    _mod("fairscale.nn", checkpoint_wrapper=lambda m, *a, **k: m)
    _mod("imageio")
    pkg = types.ModuleType("OmniTokenizer")
    pkg.__path__ = [os.path.join(REF_ROOT, "OmniTokenizer")]  # skip __init__.py (data.py deps)
    sys.modules["OmniTokenizer"] = pkg
    import OmniTokenizer.omnitokenizer as ot
    import OmniTokenizer.base as base

    class _NoLPIPS(nn.Module):
        def forward(self, a, b):
            return torch.zeros(a.shape[0], 1, 1, 1)

    ot.LPIPS = _NoLPIPS
    _loaded = (ot, base)
    return _loaded


CANON = ("--patch_embed linear --patch_size 8 --temporal_patch_size 4 --spatial_depth 4 --temporal_depth 4 "
         "--embedding_dim 512 --disc_layers 3 --enc_block ttww --dec_block tttt --twod_window_size 8 "
         "--causal_in_temporal_transformer --causal_in_peg --dim_head 64 --heads 8 --apply_noise --apply_blur "
         "--spatial_pos rope --n_codes 8192 --codebook_dim 8 --l2_code --commitment_weight 1.0 "
         "--no_random_restart --resolution 256 --sequence_length 17 --norm_type batch").split()


def make_args(argv=None):
    ot, base = load()
    p = argparse.ArgumentParser()
    p = base.VQGAN.add_model_specific_args(p)
    p = ot.VQGAN.add_model_specific_args(p)
    for f, d in (("--resolution", 256), ("--sequence_length", 17), ("--image_channels", 3),
                 ("--sample_every_n_frames", 1)):
        p.add_argument(f, type=int, default=d)  # normally from VideoData.add_data_specific_args
    return p.parse_args(CANON if argv is None else argv)


def make_model(argv=None, seed=0, perturb=True):
    """Canonical reference model with seeded random weights (SURVEY.md 8d)."""
    ot, _ = load()
    args = make_args(argv)
    torch.manual_seed(seed)
    m = ot.VQGAN(args)
    m.codebook._need_init = False
    if perturb:
        perturb_state(m, seed + 1)
    return m.eval(), args


def perturb_state(m, seed=1):
    """Move scales / LN affine / biases off their ones/zeros init so a kernel that ignores them fails."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in list(m.named_parameters()) + list(m.named_buffers()):
            if name.startswith(("image_discriminator", "video_discriminator", "perceptual_model")):
                continue
            if name.endswith(("q_scale", "k_scale", "norm.gamma", "norm_out.gamma")) or \
               (name.endswith(".weight") and p.ndim == 1):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
            elif name.endswith(".bias") and p.ndim == 1:
                p.copy_((torch.rand(p.shape, generator=g) - 0.5) * 0.2)
            elif name.endswith("relative_position_bias_table"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.5)
