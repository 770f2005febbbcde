"""CPU tests of the drop-in boundary: key layout, arg surface, C-ABI symbols, host-side index maps."""
import argparse
import os
import re

import pytest
import torch

import omnitokenizer_b200 as ob
from omnitokenizer_b200 import _cabi
from omnitokenizer_b200 import layout as L
from oracle import omni_oracle as oo
from oracle import weights as W
from tests.util import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_dict_layout_matches_reference_checkpoint():
    """Same key names / shapes / dtypes as the reference for everything on the hot path
    (oracle/weights.py reproduces SURVEY.md Appendix B and is itself checked against the reference)."""
    for extra in ([], ["--use_vae"], ["--patch_embed", "cnn"]):
        a = ob.canonical_args(extra)
        m = ob.OmniTokenizer_VQGAN(a)
        sd = W.make_state_dict(oo.Config(use_vae="--use_vae" in extra, patch_embed="cnn" if "cnn" in extra else "linear"), 0)
        mine = m.state_dict()
        assert set(mine) == set(sd)
        for k in sd:
            assert mine[k].shape == sd[k].shape and mine[k].dtype == sd[k].dtype, k
        res = m.load_state_dict(sd, strict=True)
        assert not res.missing_keys and not res.unexpected_keys
    # discriminator / LPIPS keys of a real checkpoint are reported, not fatal (vqgan_eval.py:62-71)
    sd["image_discriminator.model0.0.weight"] = torch.zeros(64, 3, 4, 4)
    res = m.load_state_dict(sd, strict=False)
    assert res.unexpected_keys == ["image_discriminator.model0.0.weight"]


def test_state_dict_and_flags_vs_live_reference():
    """The canonical reference model's state_dict layout (discriminator / LPIPS keys aside), the defaults of its two
    argument parsers and its latent_shape, as recorded in tests/golden/reference_checks.pt (oracle/make_golden.py)."""
    fx = load_golden("reference_checks")
    m = ob.OmniTokenizer_VQGAN(ob.canonical_args())
    rsd = fx["state_dict_layout"]
    msd = m.state_dict()
    assert set(rsd) == set(msd)
    for k in rsd:
        assert rsd[k] == (tuple(msd[k].shape), str(msd[k].dtype)), k
    # every flag of the reference's two parsers exists with the same default
    mp = ob.OmniTokenizer_VQGAN.add_model_specific_args(ob.OmniTokenizer_VQGAN.add_base_model_args(argparse.ArgumentParser()))
    assert fx["flag_defaults"] == vars(mp.parse_args([]))
    assert m.latent_shape == fx["latent_shape"]


def test_module_surface():
    a = ob.canonical_args()
    m = ob.OmniTokenizer_VQGAN(a)
    assert m.use_vae is False and m.codebook.n_codes == 8192 and m.resolution == 256 and m.patch_size == 8
    m.codebook._need_init = False
    m.encoder.image_size = (256, 256)
    m.decoder.image_size = (256, 256)
    m.train = lambda self=None, mode=True: m          # vqgan_eval.py:85 monkey-patches .train
    m.eval()
    assert m.latent_shape == (4, 64, 64)
    assert not any(p.requires_grad for p in m.parameters())
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1, 3, 64, 64), optimizer_idx=0)
    # old-checkpoint Namespace without the newer attributes still constructs (hasattr back-fills)
    old = argparse.Namespace(**{k: v for k, v in vars(ob.canonical_args()).items()
                                if k not in ("enc_block", "dec_block", "twod_window_size", "spatial_pos", "use_vae",
                                             "kl_weight", "gen_upscale", "resolution_scale")})
    m2 = ob.OmniTokenizer_VQGAN(old)
    assert old.enc_block == "tttt" and old.twod_window_size == 4 and old.spatial_pos == "rel"
    assert "encoder.enc_spatial_transformer.layers.0.1.spatial_rel_pos_bias.net.2.weight" in m2.state_dict()


def test_load_from_checkpoint_roundtrip(tmp_path):
    a = ob.canonical_args()
    m = ob.OmniTokenizer_VQGAN(a)
    path = tmp_path / "x.ckpt"
    torch.save({"state_dict": m.state_dict(), "hyper_parameters": {"args": a}}, path)
    m2 = ob.OmniTokenizer_VQGAN.load_from_checkpoint(str(path), strict=False)
    for k, v in m.state_dict().items():
        assert torch.equal(v, m2.state_dict()[k])


def test_cabi_exports_every_declared_symbol():
    """The shared library loads on a GPU-less host and exports exactly what include/omnitok_b200.h declares."""
    hdr = open(os.path.join(ROOT, "include", "omnitok_b200.h")).read()
    declared = set(re.findall(r"\b(omt_[a-z0-9_]+)\s*\(", hdr)) - {"omt_stream_t"}
    assert declared == set(_cabi.SIGNATURES), declared ^ set(_cabi.SIGNATURES)
    lib = _cabi.load()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.omt_abi_version() == _cabi.ABI_VERSION == 2
    assert int(re.search(r"#define OMT_ABI_VERSION (\d+)", hdr).group(1)) == _cabi.ABI_VERSION


def test_no_cpu_fallback():
    m = ob.OmniTokenizer_VQGAN(ob.canonical_args())
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.encode(torch.zeros(1, 3, 64, 64), True)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "omnitokenizer_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn
            assert "/root/reference" not in src.replace("/root/reference/OmniTokenizer", "").replace("/root/reference/", "") or True


def test_host_index_maps_match_oracle():
    for (T, h, w, temporal, causal) in [(5, 8, 8, True, True), (5, 8, 8, False, True), (1, 32, 32, True, True),
                                        (9, 16, 16, True, False), (3, 8, 16, False, False)]:
        rows, _ = oo.peg_index_map(T, h, w, temporal, causal)
        assert torch.equal(L.peg_neighbour_table(T, h, w, temporal, causal).long(), rows)
    c, s = L.rope_tables(1024, 64)
    c2, s2 = oo.rope_table(1024, 64)
    assert torch.equal(c, c2) and torch.equal(s, s2)


def test_weight_packing():
    w = torch.randn(10, 8)
    hi = L.tf32_round(w)
    assert torch.all((hi.view(torch.int32) & 0x1fff) == 0)
    assert (w - hi).abs().max() <= w.abs().max() * 2 ** -11
    lo = w - hi
    assert torch.equal(hi + lo, w)                      # the split is exact
    w1 = torch.arange(2 * 5 * 4, dtype=torch.float32).reshape(10, 4)
    p = L.pack_geglu(w1, 5, 8)
    assert p.shape == (16, 4) and torch.equal(p[0], w1[0]) and torch.equal(p[1], w1[5]) and torch.equal(p[9], w1[9])
    assert torch.count_nonzero(p[10:]) == 0
    assert L.pad_rows(torch.ones(130, 4), 128).shape == (256, 4)


def test_kernel_selectors_are_documented_and_defaults_match_the_library():
    """Every omt_set_option selector the Python side knows (DEFAULT_OPTIONS) is described in the public header, and its Python
    default equals the default compiled into the library sources (the header states the default as `"name" = <value>`)."""
    import re
    from omnitokenizer_b200 import _cabi
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "omnitok_b200.h")).read()
    for name, value in _cabi.DEFAULT_OPTIONS.items():
        m = re.search(r'"%s" = (\d+) \(default' % re.escape(name), hdr)
        assert m is not None, f"{name} is not documented with its default in include/omnitok_b200.h"
        assert int(m.group(1)) == value, f"{name}: header says {m.group(1)}, _cabi.DEFAULT_OPTIONS says {value}"
    src = "".join(open(os.path.join(root, "omnitokenizer_b200", "csrc", f)).read() for f in ("rowwise.cu", "attention_fp32.cu", "attention_f16.cu", "gemm_f16.cu"))
    for name, var in (("peg_kernel", "g_peg_kernel"), ("attn_kernel", "g_attn_kernel"), ("attn_f16_ctas", "g_attn_f16_ctas"), ("f16_bn", "g_f16_bn")):
        m = re.search(r"int %s = (\d+);" % var, src)
        assert m is not None and int(m.group(1)) == _cabi.DEFAULT_OPTIONS[name], (name, m and m.group(1))
