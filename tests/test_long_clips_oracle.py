"""CPU tests: the oracle against the reference's long-clip fixtures (scripts/make_long_goldens.py): T' = 19 and T' = 66
latent frames, past the 17 frames of the register-resident temporal attention kernel and the 64 of PEG v4."""
import pytest
import torch

from oracle import omni_oracle as oo
from tests.util import check_sub, golden_setup, load_golden

LONG_CASES = ["vid73x64", "vid261x64", "vae_vid73x64"]


@pytest.mark.parametrize("name", LONG_CASES)
def test_oracle_matches_long_clip_golden(name):
    fx = load_golden(name)
    cfg, sd, x = golden_setup(fx)
    with torch.no_grad():
        if not cfg.use_vae:
            emb, idx = oo.encode(sd, cfg, x, include_embeddings=True)
            assert torch.equal(idx, fx["idx"].long()), "code indices differ from the reference"
            check_sub(fx["emb"], emb, 1e-6, "embeddings")
            rec = oo.decode(sd, cfg, idx, False)
            check_sub(fx["rec"], rec, 2e-5, "reconstruction")
        else:
            z = oo.encode(sd, cfg, x, noise=fx["noise"])
            check_sub(fx["z"], z, 2e-5, "vae latent")
            rec = oo.decode(sd, cfg, z.permute(0, 2, 3, 4, 1), False)
            check_sub(fx["rec"], rec, 5e-5, "vae reconstruction")
