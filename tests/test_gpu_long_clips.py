"""GPU tests for clips past 17 latent frames: the chunked temporal attention kernel at op level, the model against the
reference's long-clip fixtures and the oracle at full size, the properties batch sharding relies on, and the shape limit."""
import os

import pytest
import torch

from oracle import omni_oracle as oo
from oracle import weights as W
from tests.util import build_model, check_sub, golden_setup, load_golden, namespace_from_cfg

pytestmark = pytest.mark.gpu
PIX_TOL = 1e-3
MATHS = ["fp32", "3xtf32", "f16x3"]
# the conservative kernel set of test_gpu_model.py and the shipped defaults
VARIANTS = {"base": dict(OMT_ATTN_F16="0", OMT_STATIC_U="0", OMT_PEG_KERNEL="3", OMT_ATTN_CTAS="1"), "default": dict()}


def _cabi():
    from omnitokenizer_b200 import _cabi
    _cabi.load()
    return _cabi


def _rand(shape, seed, device):
    return (torch.rand(shape, generator=torch.Generator().manual_seed(seed)) - 0.5).mul_(2).to(device)


def _temporal(cabi, qkv, o, planes, B, T, N, causal, row0=0):
    p = qkv.data_ptr() + row0 * 1536 * 4
    hi, lo = (None, None) if planes is None else (planes[0][row0:], planes[1][row0:])
    cabi.call("omt_attn_temporal", p, 1536, p + 2048, 1536, p + 4096, 1536, None if o is None else o[row0:], hi, lo, 512,
              B, T, N, 8, 8.0, causal)


@pytest.mark.parametrize("B,N", [(2, 64), (3, 7)])       # 3 * 7 = 21 sequences: not a multiple of the 4 per CTA
@pytest.mark.parametrize("causal", [0, 1])
@pytest.mark.parametrize("T", [18, 32, 33, 66, 129, 257])
def test_temporal_attention_long(cuda, T, causal, B, N):
    cabi = _cabi()
    M = B * T * N
    qkv = _rand((M, 1536), 70 + T, cuda)
    q, k, v = qkv[:, :512], qkv[:, 512:1024], qkv[:, 1024:]

    def seq(t):
        return t.double().view(B, T, N, 8, 64).permute(0, 2, 3, 1, 4)                # (B,N,H,T,D)
    s = (seq(q) @ seq(k).transpose(-1, -2)) * 8.0
    if causal:
        s = s.masked_fill(torch.ones(T, T, dtype=torch.bool, device=cuda).triu(1), float("-inf"))
    want = (torch.softmax(s, dim=-1) @ seq(v)).permute(0, 3, 1, 2, 4).reshape(M, 512)

    o = torch.full((M, 512), float("nan"), device=cuda)
    _temporal(cabi, qkv, o, None, B, T, N, causal)
    # un-normalised random q,k give |scale*q.k| ~ 50: exp() carries |s|*2^-24 ~ 3e-6 relative error per term
    err = (o.double() - want).abs().max().item()
    assert err < 2e-5, err
    planes = torch.full((2, M, 512), -1, dtype=torch.int16, device=cuda)          # fp16 NaN bit pattern
    _temporal(cabi, qkv, None, planes, B, T, N, causal)
    rec = planes[0].view(torch.float16).double() + planes[1].view(torch.float16).double() * 2.0 ** -11
    err = (rec - want).abs().max().item()
    assert err < 2e-5, err
    # a slice of the batch reproduces its rows bit for bit (the property batch sharding relies on)
    o2 = torch.full_like(o, float("nan"))
    _temporal(cabi, qkv, o2, None, 1, T, N, causal, row0=(B - 1) * T * N)
    assert torch.equal(o2[(B - 1) * T * N:], o[(B - 1) * T * N:])


@pytest.fixture(params=list(VARIANTS))
def variant(request, monkeypatch):
    for k in ("OMT_ATTN_F16", "OMT_STATIC_U", "OMT_PEG_KERNEL", "OMT_ATTN_CTAS"):
        monkeypatch.delenv(k, raising=False)
    for k, v in VARIANTS[request.param].items():
        monkeypatch.setenv(k, v)
    return request.param


@pytest.mark.parametrize("math", MATHS)
@pytest.mark.parametrize("name", ["vid73x64", "vid261x64"])
def test_long_clip_matches_golden(cuda, variant, name, math):
    fx = load_golden(name)
    cfg, sd, x = golden_setup(fx)
    m = build_model(cfg, sd, cuda, math)
    emb, idx = m.encode(x.to(cuda), False, include_embeddings=True)
    assert tuple(idx.shape) == tuple(fx["idx"].shape)
    mism = int((idx.cpu() != fx["idx"].long()).sum())
    assert mism == 0, f"{mism}/{idx.numel()} code indices differ from the reference ({math}, {variant})"
    check_sub(fx["emb"], emb, 1e-5, "embeddings")
    rec = m.decode(idx, False)
    err = check_sub(fx["rec"], rec, PIX_TOL, "reconstruction")
    print(f"{name} [{math}, {variant}]: idx mismatches 0/{idx.numel()}, max |dpixel| {err:.2e}")


@pytest.mark.parametrize("math", MATHS)
def test_long_clip_vae_matches_golden(cuda, variant, math):
    fx = load_golden("vae_vid73x64")
    cfg, sd, x = golden_setup(fx)
    m = build_model(cfg, sd, cuda, math)
    _orig = torch.randn
    try:       # the reference draws the noise from the global CPU RNG (vae.py:16); inject the recorded draw
        torch.randn = lambda *a, **k: fx["noise"].clone()
        z = m.encode(x.to(cuda), False)
    finally:
        torch.randn = _orig
    check_sub(fx["z"], z, 1e-4, "vae latent")
    rec = m.decode(z.permute(0, 2, 3, 4, 1), False)
    check_sub(fx["rec"], rec, PIX_TOL, "vae reconstruction")


_ORACLE_CACHE = {}


def _oracle(shape, cfg, sd, x):
    if shape not in _ORACLE_CACHE:
        oo.USE_LIBRARY_OPS = True          # torch's fused CPU ops (tests/test_oracle.py pins both forms)
        try:
            torch.set_num_threads(min(16, os.cpu_count() or 1))
            with torch.no_grad():
                idx = oo.encode(sd, cfg, x)
                _ORACLE_CACHE[shape] = idx, oo.decode(sd, cfg, idx, False)
        finally:
            oo.USE_LIBRARY_OPS = False
    return _ORACLE_CACHE[shape]


@pytest.mark.parametrize("math", ["3xtf32", "f16x3"])
@pytest.mark.parametrize("shape", [(1, 3, 129, 256, 256), (1, 3, 257, 256, 256)])     # T' = 33, T' = 65
def test_long_clip_full_size_parity(cuda, shape, math):
    cfg = oo.Config()
    sd = W.make_state_dict(cfg, 11)
    x = W.synthetic_input(shape, 323)
    m = build_model(cfg, sd, cuda, math)
    idx = m.encode(x.to(cuda), False)
    rec = m.decode(idx, False)
    idx_o, rec_o = _oracle(shape, cfg, sd, x)
    mism = int((idx.cpu() != idx_o).sum())
    err = float((rec.cpu() - rec_o).abs().max())
    print(f"{shape} [{math}]: idx mismatches {mism}/{idx.numel()}, max |dpixel| {err:.2e}")
    assert mism == 0
    assert err <= PIX_TOL


@pytest.mark.parametrize("math", ["3xtf32", "f16x3"])
def test_long_clip_batch_properties(cuda, math):
    """3 clips of 129 frames at 128^2 (T' = 33) through the public API: shards equal the full batch bit for bit, decode_u8
    equals the torch uint8 expression on decode, and flat indices decode like the 5-D form."""
    import omnitokenizer_b200 as ob
    cfg = oo.Config(resolution=128)
    os.environ["OMT_MATH"] = math
    m = ob.OmniTokenizer_VQGAN(namespace_from_cfg(cfg, sequence_length=129))
    m.load_state_dict(W.make_state_dict(cfg, 12), strict=False)
    m.codebook._need_init = False
    m = m.to(cuda).eval()
    x = W.synthetic_input((3, 3, 129, 128, 128), 655).to(cuda)
    full = m.encode(x, False)
    assert tuple(full.shape) == (3, 33, 16, 16)
    assert torch.equal(m.encode(x[1:2], False), full[1:2])
    rec = m.decode(full, False)
    assert torch.equal(m.decode(full[1:3], False), rec[1:3])
    assert torch.equal(m.decode_u8(full, False), oo.to_u8(rec))
    assert torch.equal(m.decode(full.reshape(3, -1), False), rec)


def test_shape_limit(cuda):
    cfg = oo.Config()
    eng = build_model(cfg, W.make_state_dict(cfg, 0), cuda, "fp32").engine()
    # 1025 frames at 256^2: T' = 257 latent frames of 1024 tokens, 1536 fp32 QKV columns per token
    bmax = (2 ** 31 - 1) // (257 * 1024 * 1536)
    assert bmax == 5
    with pytest.raises(ValueError, match=f"at most {bmax} clips"):
        eng._shape((8, 3, 1025, 256, 256))
    with pytest.raises(ValueError, match=f"at most {bmax} clips"):
        eng._shape((bmax + 1, 3, 1025, 256, 256))
    assert eng._shape((bmax, 3, 1025, 256, 256))[4] == 257
    assert eng._ws == {}
