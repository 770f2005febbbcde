"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.pt by running the UNMODIFIED reference
(a checkout of FoundationVision/OmniTokenizer, loaded by oracle/ref_loader.py) on seeded synthetic weights and inputs.

    OMT_REFERENCE_ROOT=<checkout> python -m oracle.make_golden [fixture names]

With no names every fixture is rewritten.  The tests only read the fixtures, so they run without the reference.
Each fixture stores the weight/input recipe (cfg overrides, seeds, fingerprint) and the reference outputs.
"""
import argparse
import hashlib
import os
import sys

import torch

from . import ref_loader as rl
from . import omni_oracle as oo
from . import weights as W

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = [
    # name, argv extras, input shape, weight seed, input seed
    ("img64", [], (1, 3, 64, 64), 0, 1234),
    ("vid5x64", [], (1, 3, 5, 64, 64), 0, 1235),
    ("vid9x128_b2", [], (2, 3, 9, 128, 128), 1, 1236),
    ("img256_cfg1", [], (1, 3, 256, 256), 0, 1237),
    ("vae_vid5x64", ["--use_vae"], (1, 3, 5, 64, 64), 2, 1238),
    ("vae_img64", ["--use_vae"], (2, 3, 64, 64), 2, 1239),
    # patch_embed='cnn' (Conv3d + eval BatchNorm); its decoder only handles the configured resolution
    ("cnn_vid5x64", ["--patch_embed", "cnn", "--resolution", "64"], (1, 3, 5, 64, 64), 4, 1240),
]


# Reconstructions of at most this many values (every 64x64 case) are stored whole; larger ones (cfg-1 at 256^2, the B=2
# 9x128^2 video) as a strided sample + checksum, which keeps every fixture under 1 MB.
REC_CAP = 65_536


def _sub(t, cap=200_000):
    """Keep fixtures small: full tensor if small, else a deterministic strided sample + checksum."""
    t = t.detach().contiguous()
    if t.numel() <= cap:
        return {"full": t.clone()}
    flat = t.reshape(-1)
    step = flat.numel() // cap + 1
    return {"stride": step, "sample": flat[::step].clone(), "sum64": float(flat.double().sum()),
            "abs64": float(flat.double().abs().sum()), "shape": tuple(t.shape)}


def _recipe(cfg, sd, x, wseed, xseed):
    """the keys tests/util.golden_setup rebuilds (cfg, state_dict, input) from"""
    return {"use_vae": cfg.use_vae, "patch_embed": cfg.patch_embed, "resolution": cfg.resolution, "shape": tuple(x.shape),
            "wseed": wseed, "xseed": xseed, "fingerprint": W.fingerprint(sd), "x_sum64": float(x.double().sum())}


def tensor_digest(t):
    """sha256 of a tensor's dtype, shape and bytes: a bit-exact comparison without storing the tensor"""
    t = t.detach().contiguous().cpu()
    return hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode() + t.view(torch.uint8).numpy().tobytes()).hexdigest()


DISCRIMINATOR_KEYS = ("image_discriminator", "video_discriminator", "perceptual_model")


def reference_checks():
    """What the reference answers for the checks of the drop-in surface (tests/test_boundary.py) and of the oracle's
    restatements (tests/test_oracle.py): state_dict layout and flag defaults, encode / decode on weight seed 3,
    Net2NetTransformer.encode_to_z run unbound on a stub, the eval script's uint8 expression, and utils.inflate_gen."""
    ot, base = rl.load()
    fx = {"torch": torch.__version__}
    ref, args = rl.make_model(perturb=False)
    fx["state_dict_layout"] = {k: (tuple(v.shape), str(v.dtype)) for k, v in ref.state_dict().items()
                               if not k.startswith(DISCRIMINATOR_KEYS)}
    parser = ot.VQGAN.add_model_specific_args(base.VQGAN.add_model_specific_args(argparse.ArgumentParser()))
    fx["flag_defaults"] = vars(parser.parse_args([]))
    fx["latent_shape"] = tuple(ref.latent_shape)

    cfg = oo.Config.from_args(args)
    sd = W.make_state_dict(cfg, 3)
    ref.load_state_dict(sd, strict=False)
    fx["parity"] = {}
    for shape in ((1, 3, 64, 64), (1, 3, 5, 64, 64)):
        x = W.synthetic_input(shape, 99)
        is_image = x.ndim == 4
        with torch.no_grad():
            emb, idx = ref.encode(x, is_image, include_embeddings=True)
            rec = ref.decode(idx, is_image)
        fx["parity"][shape] = dict(_recipe(cfg, sd, x, 3, 99), idx=idx.to(torch.int16), emb=_sub(emb), rec=_sub(rec, cap=REC_CAP))

    import types
    import OmniTokenizer.lm_transformer as lt
    from OmniTokenizer.utils import inflate_gen, shift_dim
    x = W.synthetic_input((1, 3, 9, 64, 64), 55)
    fx["encode_to_z"] = _recipe(cfg, sd, x, 3, 55)
    for n in (0, 2):
        stub = types.SimpleNamespace(vtokens=False, first_stage_model=ref, sample_every_n_latent_frames=n)
        emb, tgt = lt.Net2NetTransformer.encode_to_z(stub, x, False)
        fx["encode_to_z"][n] = {"emb": emb.clone(), "targets": tgt.to(torch.int16)}
    v = torch.rand((2, 3, 5, 8, 8), generator=torch.Generator().manual_seed(56)) - 0.5
    fx["eval_u8"] = {"video": v, "u8": shift_dim(torch.clamp(v + 0.5, 0, 1) * 255, 1, -1).byte()}

    sd4 = W.make_state_dict(oo.Config(), 4)
    fx["inflate_gen"] = {"fingerprint": W.fingerprint(sd4)}
    for strategy in ("average", "first"):
        out = inflate_gen(sd4, 4, 8, strategy=strategy)
        fx["inflate_gen"][strategy] = {k: ("input" if torch.equal(v, sd4[k]) else tensor_digest(v)) for k, v in out.items()}
    return fx


def main(names=()):
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    names = set(names) or {c[0] for c in CASES} | {"reference_checks"}
    if "reference_checks" in names:
        torch.save(reference_checks(), os.path.join(OUT, "reference_checks.pt"))
        print("reference_checks", os.path.getsize(os.path.join(OUT, "reference_checks.pt")) // 1024, "KiB")
    for name, extra, shape, wseed, xseed in CASES:
        if name not in names:
            continue
        m, args = rl.make_model(rl.CANON + extra, perturb=False)
        cfg = oo.Config.from_args(args)
        sd = W.make_state_dict(cfg, wseed)
        res = m.load_state_dict(sd, strict=False)
        assert not res.unexpected_keys
        m.codebook._need_init = False
        x = W.synthetic_input(shape, xseed)
        is_image = x.ndim == 4
        fx = {"name": name, "use_vae": cfg.use_vae, "patch_embed": cfg.patch_embed, "resolution": cfg.resolution,
              "shape": shape, "wseed": wseed, "xseed": xseed,
              "fingerprint": W.fingerprint(sd), "x_sum64": float(x.double().sum()),
              "torch": torch.__version__}
        taps = {}
        hooks = []
        for tn in ("encoder.enc_spatial_transformer", "encoder.enc_temporal_transformer",
                   "decoder.dec_temporal_transformer", "decoder.dec_spatial_transformer"):
            mod = dict(m.named_modules())[tn]
            hooks.append(mod.register_forward_hook(lambda _m, _i, o, tn=tn: taps.__setitem__(tn, o.detach().clone())))
        with torch.no_grad():
            if not cfg.use_vae:
                emb, idx = m.encode(x, is_image, include_embeddings=True)
                rec = m.decode(idx, is_image)
                fx["idx"] = idx.to(torch.int16 if cfg.n_codes <= 32767 else torch.int32)
                fx["emb"] = _sub(emb)
                fx["rec"] = _sub(rec, cap=REC_CAP)
                # flat-index decode convention (omnitokenizer.py:271-288) only valid at cfg.resolution
                if is_image:
                    rec_flat = m.decode(idx.reshape(idx.shape[0], -1), True)
                    fx["rec_flat_maxdiff"] = float((rec_flat - rec).abs().max())
                    # forward(log_image=True) works on CPU for images only (omnitokenizer.py:401 .cuda())
                    m.codebook.call_cnt = 0
                    fr, frr, xx, xr, vq = m(x, log_image=True)
                    fx["fwd_rec"] = _sub(xr, cap=REC_CAP)
                    fx["fwd"] = {k: (v.clone() if v.ndim == 0 else None) for k, v in vq.items()
                                 if isinstance(v, torch.Tensor)}
                    fx["fwd"]["batch_usage_nnz"] = int((vq["batch_usage"] > 0).sum())
                    fx["fwd"]["batch_usage_max"] = float(vq["batch_usage"].max())
            else:
                h = m.pre_vq_conv(m.encoder(x, is_image))          # (B,16,T',h,w)
                noise = torch.rand(h.shape[0], h.shape[1] // 2, *h.shape[2:],
                                   generator=torch.Generator().manual_seed(xseed + 1)) * 2 - 1
                # reproduce vae.py:15-17 with a recorded noise tensor instead of the global RNG
                mean, logvar = torch.chunk(h, 2, dim=1)
                z = mean + torch.exp(0.5 * torch.clamp(logvar, -30.0, 20.0)) * noise
                # cross-check against the reference's own sampler by forcing its RNG draw
                _orig = torch.randn
                try:
                    torch.randn = lambda *a, **k: noise.clone()
                    z_ref = m.encode(x, is_image)
                finally:
                    torch.randn = _orig
                zz = z.squeeze(2) if is_image else z
                assert torch.equal(z_ref, zz)
                rec = m.decode(z_ref if is_image else z_ref.permute(0, 2, 3, 4, 1), is_image)
                fx["noise"] = noise
                fx["z"] = _sub(z_ref)
                fx["rec"] = _sub(rec, cap=REC_CAP)
        for h_ in hooks:
            h_.remove()
        for tn, v in taps.items():
            fx["tap:" + tn] = _sub(v, cap=20_000)
        path = os.path.join(OUT, name + ".pt")
        torch.save(fx, path)
        print(name, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
