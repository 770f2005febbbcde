"""CPU tests: the oracle restatement vs the committed golden vectors (made by the UNMODIFIED reference,
oracle/make_golden.py)."""
import pytest
import torch

from oracle import omni_oracle as oo
from oracle import weights as W
from tests.util import check_sub, golden_setup, load_golden

FAST = ["img64", "vid5x64", "vae_vid5x64", "vae_img64", "cnn_vid5x64"]


@pytest.mark.parametrize("name", FAST + ["vid9x128_b2", "img256_cfg1"])
def test_oracle_matches_golden(name):
    fx = load_golden(name)
    cfg, sd, x = golden_setup(fx)
    is_image = x.ndim == 4
    with torch.no_grad():
        if not cfg.use_vae:
            emb, idx = oo.encode(sd, cfg, x, include_embeddings=True)
            assert torch.equal(idx, fx["idx"].long()), "code indices differ from the reference"
            check_sub(fx["emb"], emb, 1e-6, "embeddings")
            rec = oo.decode(sd, cfg, idx, is_image)
            check_sub(fx["rec"], rec, 2e-5, "reconstruction")
            if is_image:
                rec_flat = oo.decode(sd, cfg, idx.reshape(idx.shape[0], -1), True)
                assert (rec_flat - rec).abs().max().item() <= fx["rec_flat_maxdiff"] + 1e-6
        else:
            z = oo.encode(sd, cfg, x, noise=fx["noise"])
            check_sub(fx["z"], z, 2e-5, "vae latent")
            rec = oo.decode(sd, cfg, z if is_image else z.permute(0, 2, 3, 4, 1), is_image)
            check_sub(fx["rec"], rec, 5e-5, "vae reconstruction")


@pytest.mark.parametrize("name", ["img64", "vid5x64"])
def test_oracle_transformer_taps(name):
    fx = load_golden(name)
    cfg, sd, x = golden_setup(fx)
    taps = {}
    with torch.no_grad():
        h, hw = oo.encoder(sd, cfg, x, taps)
        B, T, N, C = taps["encoder_out"].shape
        # reference temporal-transformer output is laid out (b h w) t d
        ref_layout = taps["encoder_out"].permute(0, 2, 1, 3).reshape(B * N, T, C)
        check_sub(fx["tap:encoder.enc_temporal_transformer"], ref_layout, 2e-5, "enc temporal out")


def test_oracle_forward_log_image_stats():
    fx = load_golden("img64")
    cfg, sd, x = golden_setup(fx)
    with torch.no_grad():
        fr, frr, xx, xr, vq = oo.forward_log_image(sd, cfg, x)
    check_sub(fx["fwd_rec"], xr, 2e-5, "forward recon")
    assert torch.equal(vq["encodings"], fx["idx"].long())
    for k in ("commitment_loss", "perplexity", "avg_usage"):
        assert abs(float(vq[k]) - float(fx["fwd"][k])) <= 1e-5 * max(1.0, abs(float(fx["fwd"][k]))), k
    assert int((vq["batch_usage"] > 0).sum()) == fx["fwd"]["batch_usage_nnz"]


def test_peg_scrambled_map_is_a_permutation_free_gather():
    rows, f = oo.peg_index_map(5, 8, 8, temporal=True, causal=True)
    assert rows.shape == (5 * 64, 27)
    assert int(rows.max()) < 5 * 64 and int(rows.min()) == -1
    # centre tap (kt=2 causal, kh=1, kw=1) is the identity
    assert torch.equal(rows[:, 2 * 9 + 4], torch.arange(5 * 64))


def test_frame_count_assert():
    cfg = oo.Config()
    sd = W.make_state_dict(cfg, 0)
    with pytest.raises(AssertionError):
        oo.encode(sd, cfg, torch.zeros(1, 3, 6, 64, 64))


@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (1, 3, 5, 64, 64)])
def test_oracle_matches_live_reference(shape):
    """encode / decode of the reference itself on weight seed 3 (tests/golden/reference_checks.pt, oracle/make_golden.py)."""
    fx = load_golden("reference_checks")["parity"][shape]
    cfg, sd, x = golden_setup(fx)
    is_image = x.ndim == 4
    with torch.no_grad():
        emb_o, idx_o = oo.encode(sd, cfg, x, include_embeddings=True)
        rec_o = oo.decode(sd, cfg, idx_o, is_image)
    assert torch.equal(fx["idx"].long(), idx_o)
    check_sub(fx["emb"], emb_o, 1e-6, "embeddings")
    check_sub(fx["rec"], rec_o, 2e-5, "reconstruction")


def test_library_op_form_agrees_with_restatement():
    """bench.py times the oracle with torch's fused library ops (the reference's own calls); both forms
    must produce the same codes and pixels."""
    fx = load_golden("vid5x64")
    cfg, sd, x = golden_setup(fx)
    try:
        oo.USE_LIBRARY_OPS = True
        with torch.no_grad():
            idx = oo.encode(sd, cfg, x)
            rec = oo.decode(sd, cfg, idx, False)
    finally:
        oo.USE_LIBRARY_OPS = False
    assert torch.equal(idx, fx["idx"].long())
    check_sub(fx["rec"], rec, 2e-5, "reconstruction (library-op form)")


# ---- numerics model of the tensor-core path (DESIGN.md section 4) -------------------------------------------------
def _tf32_rna(x):
    """round-to-nearest (ties away) to 10 explicit mantissa bits: the kernels' tf32_rn / layout.tf32_round."""
    return ((x.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def _tf32_trunc(x):
    """what the tensor core does to an fp32 operand of a kind::tf32 MMA: the low 13 mantissa bits are ignored."""
    return (x.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def _mm_3xtf32(a, b):
    ah, bh = _tf32_rna(a), _tf32_rna(b)
    al, bl = _tf32_trunc(a - ah), _tf32_trunc(b - bh)
    return (al @ bh + ah @ bl) + ah @ bh          # the kernels' order: A_lo.W_hi, A_hi.W_lo, A_hi.W_hi, fp32 accumulate


def _mm_tf32(a, b):
    return _tf32_trunc(a) @ _tf32_trunc(b)


def test_layout_tf32_round_is_rna():
    from omnitokenizer_b200 import layout as L
    x = torch.randn(4096, generator=torch.Generator().manual_seed(3)) * 3.0
    assert torch.equal(L.tf32_round(x), _tf32_rna(x))
    lo = x - L.tf32_round(x)
    assert (lo.abs() <= x.abs() * 2.0 ** -11 * (1 + 1e-6)).all()        # |lo| <= half a tf32 ulp
    assert torch.equal(L.tf32_round(x) + lo, x)                          # the split is lossless in fp32


@pytest.mark.parametrize("name", ["vid9x128_b2", "img256_cfg1"])
def test_3xtf32_numerics_model_keeps_code_indices(name, monkeypatch):
    """Every tensor-core product of the CUDA path (nn.Linear layers + spatial attention core) replaced by an
    emulation of 3xTF32 (hi/lo split, three fp32-accumulated products): indices stay bit-exact vs the reference's
    golden vectors and pixels stay within 1e-3 (north_star).  Single-pass TF32 is ~1000x less accurate: it is a
    throughput mode only (on the GPU it flips ~6/5120 indices of cfg-3)."""
    fx = load_golden(name)
    cfg, sd, x = golden_setup(fx)
    is_image = x.ndim == 4
    err = {}
    with torch.no_grad():
        for label, model in (("3xtf32", _mm_3xtf32), ("tf32", _mm_tf32)):
            monkeypatch.setattr(oo, "MATMUL_MODEL", model)
            emb, idx = oo.encode(sd, cfg, x, include_embeddings=True)
            rec = oo.decode(sd, cfg, fx["idx"].long(), is_image)      # decode the reference's codes: isolates decoder error
            err[label] = (int((idx != fx["idx"].long()).sum()), check_sub(fx["rec"], rec, 1.0, "reconstruction"))
    assert err["3xtf32"][0] == 0, f"3xTF32 model flipped {err['3xtf32'][0]} indices"
    assert err["3xtf32"][1] <= 1e-4, err
    assert err["tf32"][1] > 20 * err["3xtf32"][1], err                 # the single-pass mode is far off fp32 grade


def test_consumer_restatements_match_live_reference():
    """SURVEY.md 8f: Net2NetTransformer.encode_to_z (lm_transformer.py:258-268) run UNBOUND on a stub carrying the reference
    VQGAN, against the oracle's restatement; plus shift_dim / the eval script's uint8 expression.  The reference's answers
    are recorded in tests/golden/reference_checks.pt (oracle/make_golden.py)."""
    golden = load_golden("reference_checks")
    fx = golden["encode_to_z"]
    cfg, sd, x = golden_setup(fx)
    for n in (0, 2):
        with torch.no_grad():
            emb_o, tgt_o = oo.encode_to_z(sd, cfg, x, False, n)
        assert torch.equal(fx[n]["targets"].long(), tgt_o) and (fx[n]["emb"] - emb_o).abs().max().item() < 1e-5
    assert torch.equal(golden["eval_u8"]["u8"], oo.to_u8(golden["eval_u8"]["video"]))


@pytest.mark.parametrize("strategy", ["average", "first"])
def test_inflate_gen_matches_live_reference(strategy):
    """Checkpoint tooling (SURVEY.md 8f-4): omnitokenizer_b200.ckpt.inflate_gen vs OmniTokenizer/utils.py:11 on a synthetic
    checkpoint, key for key and bit for bit (the reference's output is recorded as, per key, "input" where it kept the input
    tensor and a sha256 of dtype, shape and bytes elsewhere); the inflated checkpoint then loads into the module without
    missing keys."""
    import omnitokenizer_b200 as ob
    from omnitokenizer_b200.ckpt import inflate_gen
    from oracle.make_golden import tensor_digest
    fx = load_golden("reference_checks")["inflate_gen"]
    sd = W.make_state_dict(oo.Config(), 4)
    assert W.fingerprint(sd) == fx["fingerprint"]
    a, b = inflate_gen(sd, 4, 8, strategy), fx[strategy]
    assert a.keys() == b.keys()
    assert all(torch.equal(a[k], sd[k]) if b[k] == "input" else tensor_digest(a[k]) == b[k] for k in a)
    m = ob.OmniTokenizer_VQGAN(ob.canonical_args())
    res = m.load_state_dict(a, strict=False)
    assert not res.missing_keys
