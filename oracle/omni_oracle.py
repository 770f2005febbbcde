"""TEST INFRASTRUCTURE ONLY -- CPU fp32 restatement of the OmniTokenizer VQGAN encode/decode path.

This is the parity oracle for the CUDA path.  Only tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs may import it; the product
package (omnitokenizer_b200/) never does.

It is a *functional* restatement over a reference-layout ``state_dict`` (same key
names as the reference checkpoint, SURVEY.md Appendix B): plain torch fp32 ops on
CPU, written from the arithmetic spec (SURVEY.md Appendix A), not copied from the
reference.  Activations are kept in ONE canonical layout ``X[B, T', N, C]`` (the
reference's ``(b t) (h w) d`` tensor); the temporal blocks index it through the
``(b n) t`` view exactly the way the CUDA kernels do, so the index maps here
(scrambled PEG, window partition, patch order) are the ones the kernels use.

Pinning: tests/test_oracle.py checks every function here against the committed
golden vectors in tests/golden/, which oracle/make_golden.py recorded from the
UNMODIFIED reference itself.

Reference citations are relative to the reference's OmniTokenizer/ directory.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
SD = Dict[str, Tensor]

# When True the oracle calls the same torch LIBRARY ops the reference calls (F.conv3d for PEG,
# F.scaled_dot_product_attention, F.layer_norm, F.gelu) instead of the explicit restatements.
# Same arithmetic spec; used by bench.py so the timed CPU baseline is not handicapped by the
# gather-form PEG / materialised attention below.  tests/test_oracle.py checks both forms agree.
USE_LIBRARY_OPS = False

# Numerics-model hook (tests only): when set, every matrix product that the CUDA path runs on the tensor cores --
# the nn.Linear layers routed through omt_linear and the spatial attention core -- is computed by
# MATMUL_MODEL(a, b) instead of ``a @ b``; tests/test_oracle.py plugs in an emulation of the kernels' 3xTF32
# arithmetic to show on the CPU that it keeps the code indices bit-exact (DESIGN.md section 4).
MATMUL_MODEL = None


def _mm(a: Tensor, b: Tensor) -> Tensor:
    return a @ b if MATMUL_MODEL is None else MATMUL_MODEL(a, b)



@dataclass
class Config:
    """The subset of the reference's argparse Namespace that shapes the hot path
    (omnitokenizer.py:64-160, 695-768; base.py:246-269)."""
    resolution: int = 256
    sequence_length: int = 17
    image_channels: int = 3
    patch_size: int = 8
    temporal_patch_size: int = 4
    embedding_dim: int = 512
    dim_head: int = 64
    heads: int = 8
    ff_mult: float = 4.0
    enc_block: str = "ttww"
    dec_block: str = "tttt"
    temporal_depth: int = 4
    twod_window_size: int = 8
    causal_in_temporal_transformer: bool = True
    causal_in_peg: bool = True
    spatial_pos: str = "rope"
    n_codes: int = 8192
    codebook_dim: int = 8
    l2_code: bool = True
    use_vae: bool = False
    patch_embed: str = "linear"      # 'linear' (every shipped script) | 'cnn' (Conv3d + eval-mode BatchNorm)

    @property
    def ff_inner(self) -> int:  # modules/attention.py:161
        return int(self.ff_mult * (2 / 3) * self.embedding_dim)

    @staticmethod
    def from_args(args) -> "Config":
        c = Config()
        for k in c.__dataclass_fields__:
            if hasattr(args, k) and getattr(args, k) is not None:
                setattr(c, k, getattr(args, k))
        if not hasattr(args, "enc_block"):
            c.enc_block = "t" * args.spatial_depth
        if not hasattr(args, "dec_block"):
            c.dec_block = "t" * args.spatial_depth
        return c


# --------------------------------------------------------------------------------------
# row-wise pieces
# --------------------------------------------------------------------------------------

def layer_norm(x: Tensor, w: Tensor, b: Optional[Tensor], eps: float = 1e-5) -> Tensor:
    """modules/attention.py:73-80 (custom LayerNorm, beta buffer) and nn.LayerNorm; eps 1e-5."""
    if USE_LIBRARY_OPS:
        return F.layer_norm(x, x.shape[-1:], w, b, eps)
    mu = x.mean(dim=-1, keepdim=True)
    xc = x - mu
    var = (xc * xc).mean(dim=-1, keepdim=True)
    y = xc * torch.rsqrt(var + eps) * w
    return y + b if b is not None else y


def gelu_erf(x: Tensor) -> Tensor:
    if USE_LIBRARY_OPS:
        return F.gelu(x)
    return 0.5 * x * (1.0 + torch.erf(x * (1.0 / math.sqrt(2.0))))


def patchify(video: Tensor, p: int, pt: int) -> Tuple[Tensor, Optional[Tensor]]:
    """omnitokenizer.py:806-822 Rearrange patterns.  video (B,C,T,H,W) ->
    first (B,1,h,w,C*p*p) with feature order (c,p1,p2); rest (B,t,h,w,C*pt*p*p) order (c,pt,p1,p2)."""
    B, C, T, H, W = video.shape
    h, w = H // p, W // p
    f = video[:, :, :1].reshape(B, C, 1, h, p, w, p).permute(0, 2, 3, 5, 1, 4, 6).reshape(B, 1, h, w, C * p * p)
    if T == 1:
        return f, None
    t = (T - 1) // pt
    r = video[:, :, 1:].reshape(B, C, t, pt, h, p, w, p).permute(0, 2, 4, 6, 1, 3, 5, 7)
    return f, r.reshape(B, t, h, w, C * pt * p * p)


def unpatchify(first: Tensor, rest: Optional[Tensor], C: int, p: int, pt: int) -> Tensor:
    """omnitokenizer.py:1006-1017 inverse Rearranges; returns (B,C,T,H,W)."""
    B, _, h, w, _ = first.shape
    f = first.reshape(B, 1, h, w, C, p, p).permute(0, 4, 1, 2, 5, 3, 6).reshape(B, C, 1, h * p, w * p)
    if rest is None:
        return f
    t = rest.shape[1]
    r = rest.reshape(B, t, h, w, C, pt, p, p).permute(0, 4, 1, 5, 2, 6, 3, 7).reshape(B, C, t * pt, h * p, w * p)
    return torch.cat([f, r], dim=2)


def patch_embed(sd: SD, cfg: Config, video: Tensor) -> Tensor:
    """omnitokenizer.py:919-947 + 806-822: LN -> Linear -> LN per patch; returns X (B,T',N,C)."""
    p, pt = cfg.patch_size, cfg.temporal_patch_size
    assert (video.shape[2] - 1) % pt == 0, "number of frames minus one must be divisible by temporal patch size"
    if cfg.patch_embed == "cnn":
        return patch_embed_cnn(sd, cfg, video)
    first, rest = patchify(video, p, pt)

    def emb(x, pre):
        x = layer_norm(x, sd[pre + ".1.weight"], sd[pre + ".1.bias"])
        x = _mm(x, sd[pre + ".2.weight"].t()) + sd[pre + ".2.bias"]
        return layer_norm(x, sd[pre + ".3.weight"], sd[pre + ".3.bias"])

    tok = emb(first, "encoder.to_patch_emb_first_frame")
    if rest is not None:
        tok = torch.cat([tok, emb(rest, "encoder.to_patch_emb")], dim=1)
    B, T, h, w, C = tok.shape
    return tok.reshape(B, T, h * w, C)


def _bn_eval(x: Tensor, sd: SD, pre: str) -> Tensor:
    """base.py:272-277 Normalize(norm_type='batch') = SyncBatchNorm; in eval it is the running-stats affine."""
    return F.batch_norm(x, sd[pre + ".running_mean"], sd[pre + ".running_var"], sd[pre + ".weight"], sd[pre + ".bias"],
                        False, 0.0, 1e-5)


def patch_embed_cnn(sd: SD, cfg: Config, video: Tensor) -> Tensor:
    """omnitokenizer.py:823-838: strided Conv3d (kernel = stride = (1|pt, p, p)) + Normalize, no LayerNorms."""
    p, pt = cfg.patch_size, cfg.temporal_patch_size
    pre = "encoder.to_patch_emb_first_frame"
    tok = _bn_eval(F.conv3d(video[:, :, :1], sd[pre + ".0.weight"], sd[pre + ".0.bias"], stride=(1, p, p)), sd, pre + ".1")
    if video.shape[2] > 1:
        pre = "encoder.to_patch_emb"
        r = _bn_eval(F.conv3d(video[:, :, 1:], sd[pre + ".0.weight"], sd[pre + ".0.bias"], stride=(pt, p, p)), sd, pre + ".1")
        tok = torch.cat([tok, r], dim=2)
    B, C, T, h, w = tok.shape
    return tok.permute(0, 2, 3, 4, 1).reshape(B, T, h * w, C)


def to_pixels_cnn(sd: SD, cfg: Config, X: Tensor, hw: Tuple[int, int]) -> Tensor:
    """omnitokenizer.py:1019-1035: ConvTranspose3d (kernel = stride) + Normalize(image_channel)."""
    B, T, N, C = X.shape
    h, w = hw
    p, pt = cfg.patch_size, cfg.temporal_patch_size
    vol = X.reshape(B, T, h, w, C).permute(0, 4, 1, 2, 3)
    pre = "decoder.to_pixels_first_frame"
    out = _bn_eval(F.conv_transpose3d(vol[:, :, :1], sd[pre + ".1.weight"], sd[pre + ".1.bias"], stride=(1, p, p)), sd, pre + ".2")
    if T > 1:
        pre = "decoder.to_pixels"
        r = _bn_eval(F.conv_transpose3d(vol[:, :, 1:], sd[pre + ".1.weight"], sd[pre + ".1.bias"], stride=(pt, p, p)), sd, pre + ".2")
        out = torch.cat([out, r], dim=2)
    return out


def to_pixels(sd: SD, cfg: Config, X: Tensor, hw: Tuple[int, int]) -> Tensor:
    """omnitokenizer.py:1089-1094."""
    if cfg.patch_embed == "cnn":
        return to_pixels_cnn(sd, cfg, X, hw)
    B, T, N, C = X.shape
    h, w = hw
    tok = X.reshape(B, T, h, w, C)
    f = _mm(tok[:, :1], sd["decoder.to_pixels_first_frame.0.weight"].t()) + sd["decoder.to_pixels_first_frame.0.bias"]
    r = None
    if T > 1:
        r = _mm(tok[:, 1:], sd["decoder.to_pixels.0.weight"].t()) + sd["decoder.to_pixels.0.bias"]
    return unpatchify(f, r, cfg.image_channels, cfg.patch_size, cfg.temporal_patch_size)


# --------------------------------------------------------------------------------------
# PEG (modules/attention.py:298-338) as an explicit gather over the canonical buffer
# --------------------------------------------------------------------------------------

def peg_index_map(T: int, h: int, w: int, temporal: bool, causal: bool) -> Tuple[Tensor, Tensor]:
    """For every canonical row r=(tau,n) of one batch element returns the 27 neighbour
    canonical rows (or -1 for zero padding).

    spatial call: the reference tensor (b t)(h w) d reshaped to (b,t,h,w,d) IS the canonical
    order, flat position f = tau*N + n.
    temporal call: the reference tensor is (b h w) t d but is reshaped LITERALLY to
    (b,t,h,w,d) (attention.py:313-319, the '# TO FIX' comments): flat f = n*T + tau is
    unravelled over (T,h,w).  The stencil and zero padding live in that scrambled space.
    Returns (rows[T*N,27] int64, f_of_row[T*N])."""
    N = h * w
    tau = torch.arange(T).view(T, 1).expand(T, N).reshape(-1)
    n = torch.arange(N).view(1, N).expand(T, N).reshape(-1)
    f = (n * T + tau) if temporal else (tau * N + n)
    t2, rem = f // N, f % N
    h2, w2 = rem // w, rem % w
    rows = torch.full((T * N, 27), -1, dtype=torch.int64)
    k = 0
    for kt in range(3):
        for kh in range(3):
            for kw in range(3):
                tt = t2 + kt - (2 if causal else 1)
                hh, ww = h2 + kh - 1, w2 + kw - 1
                ok = (tt >= 0) & (tt < T) & (hh >= 0) & (hh < h) & (ww >= 0) & (ww < w)
                f2 = (tt * h + hh) * w + ww
                if temporal:
                    r2 = (f2 % T) * N + (f2 // T)      # (n', tau') = divmod(f', T) -> canonical row tau'*N+n'
                else:
                    r2 = f2
                rows[:, k] = torch.where(ok, r2, torch.full_like(r2, -1))
                k += 1
    return rows, f


def peg(X: Tensor, weight: Tensor, bias: Tensor, hw: Tuple[int, int], temporal: bool, causal: bool) -> Tensor:
    """Depthwise 3x3x3 cross-correlation + bias (no residual).  X (B,T',N,C); weight (C,1,3,3,3)."""
    B, T, N, C = X.shape
    if USE_LIBRARY_OPS:     # the reference's own formulation: literal reshape + pad + conv3d (attention.py:319-326)
        h, w = hw
        src = X.permute(0, 2, 1, 3).contiguous() if temporal else X          # '(b h w) t d' vs '(b t) (h w) d'
        vol = src.reshape(B, T, h, w, C).permute(0, 4, 1, 2, 3)
        vol = F.pad(vol, (1, 1, 1, 1) + ((2, 0) if causal else (1, 1)))
        out = F.conv3d(vol, weight, bias, groups=C).permute(0, 2, 3, 4, 1)
        if temporal:
            return out.reshape(B, N, T, C).permute(0, 2, 1, 3).contiguous()
        return out.reshape(B, T, N, C)
    rows, _ = peg_index_map(T, hw[0], hw[1], temporal, causal)
    Xf = X.reshape(B, T * N, C)
    Xz = torch.cat([Xf, torch.zeros(B, 1, C, dtype=X.dtype)], dim=1)          # row -1 -> zeros
    wk = weight.reshape(C, 27)
    out = bias.view(1, 1, C).expand(B, T * N, C).clone()
    for k in range(27):
        out = out + Xz[:, rows[:, k]] * wk[:, k]
    return out.reshape(B, T, N, C)


# --------------------------------------------------------------------------------------
# attention blocks
# --------------------------------------------------------------------------------------

def rope_table(N: int, dim_head: int = 64, theta: float = 10000.0) -> Tuple[Tensor, Tensor]:
    """modules/attention.py:28-44 in closed form: (cos,sin) of shape (N, dim_head/2).
    pair j: i=j//2, f_i = theta^(-4i/dim_head); angle = (p%H if j even else p//H) * f_i."""
    H = int(N ** 0.5)
    pos = torch.arange(N)
    xp, yp = pos % H, pos // H
    freqs = 1.0 / (theta ** (torch.arange(0, dim_head, 4)[: dim_head // 4].float() / dim_head))
    xa = torch.outer(xp, freqs).float()
    ya = torch.outer(yp, freqs).float()
    ang = torch.stack([xa, ya], dim=-1).reshape(N, -1)                          # (N, 32): x0,y0,x1,y1,...
    cis = torch.polar(torch.ones_like(ang), ang)                                # same op as attention.py:37-38
    return cis.real.contiguous(), cis.imag.contiguous()


def apply_rope(t: Tensor, cos: Tensor, sin: Tensor) -> Tensor:
    """modules/attention.py:59-70.  t (..., N, heads, 64); pairs (2j, 2j+1)."""
    a, b = t[..., 0::2], t[..., 1::2]
    c, s = cos.unsqueeze(1), sin.unsqueeze(1)                                   # (N,1,32)
    return torch.stack([a * c - b * s, a * s + b * c], dim=-1).flatten(-2)


def l2norm(t: Tensor) -> Tensor:
    return t / t.norm(dim=-1, keepdim=True).clamp_min(1e-12)                    # F.normalize eps


def attention_t(sd: SD, pre: str, cfg: Config, X: Tensor, temporal: bool, causal: bool) -> Tensor:
    """modules/attention.py:395-486, SDPA branch (:439-451): NO additive bias, scale=8,
    k/v from the UN-normalised input (:407 vs :409).  X (B,T',N,C) -> attn(x) (no residual)."""
    B, T, N, C = X.shape
    H, D = cfg.heads, cfg.dim_head
    xn = layer_norm(X, sd[pre + ".norm.gamma"], sd[pre + ".norm.beta"])
    q = _mm(xn, sd[pre + ".to_q.weight"].t())
    kv = _mm(X, sd[pre + ".to_kv.weight"].t())
    k, v = kv[..., : H * D], kv[..., H * D:]
    q, k, v = (t.reshape(B, T, N, H, D) for t in (q, k, v))
    if (not temporal) and cfg.spatial_pos == "rope":
        cos, sin = rope_table(N, D)
        q, k = apply_rope(q, cos, sin), apply_rope(k, cos, sin)
    q = l2norm(q) * sd[pre + ".q_scale"]
    k = l2norm(k) * sd[pre + ".k_scale"]
    if temporal:        # sequences run over T' for each (b,n)
        q, k, v = (t.permute(0, 2, 3, 1, 4) for t in (q, k, v))               # (B,N,H,T,D)
    else:               # sequences run over N for each (b,t)
        q, k, v = (t.permute(0, 1, 3, 2, 4) for t in (q, k, v))               # (B,T,H,N,D)
    if USE_LIBRARY_OPS:
        o = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=causal, scale=8)
    else:
        tc_core = (not temporal) and N % 128 == 0        # the shapes attn_tc3_kernel takes (tensor-core core)
        mm = _mm if tc_core else torch.matmul
        s = mm(q, k.transpose(-1, -2)) * 8.0
        if causal:
            L = s.shape[-1]
            mask = torch.ones(L, L, dtype=torch.bool).triu(1)
            s = s.masked_fill(mask, float("-inf"))
        o = mm(torch.softmax(s, dim=-1), v)
    o = o.permute(0, 3, 1, 2, 4) if temporal else o.permute(0, 1, 3, 2, 4)      # -> (B,T,N,H,D)
    return _mm(o.reshape(B, T, N, H * D), sd[pre + ".to_out.weight"].t())


def window_rows(h: int, w: int, ws: int) -> Tensor:
    """modules/attention.py:170-183: canonical token index n for (window, slot): (nW, ws*ws)."""
    n = torch.arange(h * w).reshape(h // ws, ws, w // ws, ws).permute(0, 2, 1, 3)
    return n.reshape(-1, ws * ws)


def window_attention(sd: SD, pre: str, cfg: Config, X: Tensor, hw: Tuple[int, int]) -> Tensor:
    """modules/attention.py:254-293.  X (B,T',N,C) -> (no residual)."""
    B, T, N, C = X.shape
    H, D, ws = cfg.heads, C // cfg.heads, cfg.twod_window_size
    xn = layer_norm(X, sd[pre + ".norm.gamma"], sd[pre + ".norm.beta"])
    rows = window_rows(hw[0], hw[1], ws)                                        # (nW, 64)
    xw = xn[:, :, rows]                                                         # (B,T,nW,64,C)
    qkv = _mm(xw, sd[pre + ".qkv.weight"].t()).reshape(B, T, rows.shape[0], ws * ws, 3, H, D)
    q, k, v = (qkv[..., i, :, :].permute(0, 1, 2, 4, 3, 5) for i in range(3))   # (B,T,nW,H,64,D)
    s = (q * (D ** -0.5)) @ k.transpose(-1, -2)
    bias = sd[pre + ".relative_position_bias_table"][sd[pre + ".relative_position_index"].reshape(-1)]
    s = s + bias.reshape(ws * ws, ws * ws, H).permute(2, 0, 1)
    o = (torch.softmax(s, dim=-1) @ v).permute(0, 1, 2, 4, 3, 5).reshape(B, T, rows.shape[0], ws * ws, C)
    o = _mm(o, sd[pre + ".proj.weight"].t()) + sd[pre + ".proj.bias"]
    out = torch.empty_like(X)
    out[:, :, rows] = o
    return out


def feed_forward(sd: SD, pre: str, cfg: Config, X: Tensor) -> Tensor:
    """modules/attention.py:153-168: LN -> Linear(512,2730) -> gelu(gate)*x -> Linear(1365,512)."""
    inner = sd[pre + ".4.weight"].shape[1]
    y = _mm(layer_norm(X, sd[pre + ".0.weight"], sd[pre + ".0.bias"]), sd[pre + ".1.weight"].t())
    u = gelu_erf(y[..., inner:]) * y[..., :inner]
    return _mm(u, sd[pre + ".4.weight"].t())


def transformer(sd: SD, pre: str, cfg: Config, X: Tensor, hw: Tuple[int, int], block: str,
                temporal: bool, taps: Optional[dict] = None) -> Tensor:
    """modules/attention.py:655-689: x=peg(x)+x; x=attn(x)+x; x=ff(x)+x per layer; final norm_out."""
    causal_attn = temporal and cfg.causal_in_temporal_transformer
    for i, blk in enumerate(block):
        lp = f"{pre}.layers.{i}"
        if blk == "t":
            X = peg(X, sd[lp + ".0.dsconv.weight"], sd[lp + ".0.dsconv.bias"], hw, temporal, cfg.causal_in_peg) + X
            if taps is not None:
                taps[lp + ".peg"] = X
            X = attention_t(sd, lp + ".1", cfg, X, temporal, causal_attn) + X
        elif blk == "w":
            X = window_attention(sd, lp + ".1", cfg, X, hw) + X
        else:
            raise NotImplementedError(f"block type {blk!r} is outside the shipped configs (SURVEY.md 2)")
        if taps is not None:
            taps[lp + ".attn"] = X
        X = feed_forward(sd, lp + ".3", cfg, X) + X
        if taps is not None:
            taps[lp + ".ff"] = X
    return layer_norm(X, sd[pre + ".norm_out.gamma"], sd[pre + ".norm_out.beta"])


# --------------------------------------------------------------------------------------
# encoder / codebook / decoder
# --------------------------------------------------------------------------------------

def encoder(sd: SD, cfg: Config, x: Tensor, taps: Optional[dict] = None) -> Tuple[Tensor, Tuple[int, int]]:
    """omnitokenizer.py:881-947 then pre_vq_conv (:144-154).  Returns h (B,T',N,cd) channels-last."""
    video = x.unsqueeze(2) if x.ndim == 4 else x
    hw = (video.shape[3] // cfg.patch_size, video.shape[4] // cfg.patch_size)
    X = patch_embed(sd, cfg, video)
    if taps is not None:
        taps["patch_embed"] = X
    X = transformer(sd, "encoder.enc_spatial_transformer", cfg, X, hw, cfg.enc_block, False, taps)
    X = transformer(sd, "encoder.enc_temporal_transformer", cfg, X, hw, "t" * cfg.temporal_depth, True, taps)
    if taps is not None:
        taps["encoder_out"] = X
    h = X @ sd["pre_vq_conv.1.weight"].t() + sd["pre_vq_conv.1.bias"]
    return h, hw


def codebook(E: Tensor, z: Tensor) -> Dict[str, Tensor]:
    """modules/codebook.py:76-143 eval branch.  z (M, cd) flat rows.  d = (sum z^2 - 2 z E^T) + sum E^2
    in that association; argmin takes the first minimum."""
    d = (z ** 2).sum(dim=1, keepdim=True) - (2 * z) @ E.t() + (E.t() ** 2).sum(dim=0, keepdim=True)
    idx = torch.argmin(d, dim=1)
    e = E[idx]
    n_codes = E.shape[0]
    counts = torch.bincount(idx, minlength=n_codes).float()
    usage = counts / idx.numel()
    perplexity = torch.exp(-torch.sum(usage * torch.log(usage + 1e-10)))
    commitment = 0.25 * F.mse_loss(z, e)
    return dict(idx=idx, e=e, st=(e - z) + z, batch_usage=usage, perplexity=perplexity,
                commitment_loss=commitment)


def encode(sd: SD, cfg: Config, x: Tensor, include_embeddings: bool = False, noise: Optional[Tensor] = None):
    """omnitokenizer.py:247-266.  VQ: LongTensor (B,T',h,w) [+ straight-through embeddings (B,cd,T',h,w)].
    VAE: z (B,cd,T',h,w) (squeezed for images) with ``noise`` standing in for torch.randn (vae.py:16)."""
    is_image = x.ndim == 4
    h, hw = encoder(sd, cfg, x)
    B, T, N, cd = h.shape
    if not cfg.use_vae:
        z = h.reshape(-1, cd)
        if cfg.l2_code:
            z = z / z.norm(dim=1, keepdim=True).clamp_min(1e-12)
        out = codebook(sd["codebook.embeddings"], z)
        idx = out["idx"].reshape(B, T, hw[0], hw[1])
        if include_embeddings:
            return out["st"].reshape(B, T, hw[0], hw[1], cd).permute(0, 4, 1, 2, 3).contiguous(), idx
        return idx
    c = cd // 2
    mean, logvar = h[..., :c], h[..., c:].clamp(-30.0, 20.0)
    if noise is None:
        noise = torch.randn(B, c, T, hw[0], hw[1])
    z = mean.reshape(B, T, hw[0], hw[1], c).permute(0, 4, 1, 2, 3) + \
        torch.exp(0.5 * logvar).reshape(B, T, hw[0], hw[1], c).permute(0, 4, 1, 2, 3) * noise
    return z.squeeze(2) if is_image else z.contiguous()


def decoder(sd: SD, cfg: Config, zc: Tensor, hw: Tuple[int, int], is_image: bool,
            taps: Optional[dict] = None) -> Tensor:
    """post_vq_conv (:156-160) + OmniTokenizer_Decoder (:1059-1118).  zc (B,T',N,cd) channels-last."""
    X = zc @ sd["post_vq_conv.1.weight"].t() + sd["post_vq_conv.1.bias"]
    X = transformer(sd, "decoder.dec_temporal_transformer", cfg, X, hw, "t" * cfg.temporal_depth, True, taps)
    X = transformer(sd, "decoder.dec_spatial_transformer", cfg, X, hw, cfg.dec_block, False, taps)
    if taps is not None:
        taps["decoder_out"] = X
    vid = to_pixels(sd, cfg, X, hw)
    return vid.squeeze(2) if is_image else vid


def decode(sd: SD, cfg: Config, enc: Tensor, is_image: bool) -> Tensor:
    """omnitokenizer.py:268-317 including the flat-index and VAE layout conventions."""
    if not cfg.use_vae:
        z = sd["codebook.embeddings"][enc]
        if z.ndim == 3:                       # flat (B, T'hw)
            if is_image:
                h = int(math.sqrt(z.shape[1])); w = h; T = 1
            else:
                h = w = cfg.resolution // cfg.patch_size; T = z.shape[1] // (h * w)
            B = z.shape[0]
        else:
            B, T, h, w, _ = z.shape
        zc = z.reshape(B, T, h * w, -1)
    else:
        z = enc
        if is_image:
            if z.ndim == 3:
                B = z.shape[0]; h = int(math.sqrt(z.shape[1])); w = h; T = 1
                zc = z.reshape(B, 1, h * w, -1)
            else:                             # b c h w
                B, c, h, w = z.shape; T = 1
                zc = z.permute(0, 2, 3, 1).reshape(B, 1, h * w, c)
        else:
            if z.ndim == 3:
                B = z.shape[0]; h = w = cfg.resolution // cfg.patch_size; T = z.shape[1] // (h * w)
                zc = z.reshape(B, T, h * w, -1)
            else:                             # b t h w c  (channels-LAST, omnitokenizer.py:313)
                B, T, h, w, c = z.shape
                zc = z.reshape(B, T, h * w, c)
    return decoder(sd, cfg, zc, (h, w), is_image)


def forward_log_image(sd: SD, cfg: Config, x: Tensor, frame_idx: Optional[Tensor] = None,
                      noise: Optional[Tensor] = None, usage_state: Optional[dict] = None):
    """omnitokenizer.py:330-413 with log_image=True.  The decoder is fed the straight-through
    tensor (e - z) + z (codebook.py:120).  ``frame_idx`` stands in for torch.randint(0,T,[B]) (:401)."""
    is_image = x.ndim == 4
    h, hw = encoder(sd, cfg, x)
    B, T, N, cd = h.shape
    vq_output = None
    if not cfg.use_vae:
        z = h.reshape(-1, cd)
        if cfg.l2_code:
            z = z / z.norm(dim=1, keepdim=True).clamp_min(1e-12)
        out = codebook(sd["codebook.embeddings"], z)
        x_recon = decoder(sd, cfg, out["st"].reshape(B, T, N, cd), hw, is_image)
        usage = out["batch_usage"]
        if usage_state is None:
            usage_state = {"call_cnt": 0, "codebook_usage": torch.zeros_like(usage)}
        if usage_state["call_cnt"] == 0:                                           # codebook.py:133-138
            usage_state["codebook_usage"] = usage
        else:
            usage_state["codebook_usage"] = 0.99 * usage_state["codebook_usage"] + (1 - 0.99) * usage
        usage_state["call_cnt"] += 1
        n_codes = usage.numel()
        vq_output = dict(
            embeddings=out["st"].reshape(B, T, hw[0], hw[1], cd).permute(0, 4, 1, 2, 3).contiguous(),
            encodings=out["idx"].reshape(B, T, hw[0], hw[1]),
            commitment_loss=out["commitment_loss"], perplexity=out["perplexity"],
            avg_usage=(usage_state["codebook_usage"] > (1 / n_codes)).sum() / n_codes,
            batch_usage=usage)
    else:
        c = cd // 2
        if noise is None:
            noise = torch.randn(B, c, T, hw[0], hw[1])
        nz = noise.permute(0, 2, 3, 4, 1).reshape(B, T, N, c)
        z = h[..., :c] + torch.exp(0.5 * h[..., c:].clamp(-30.0, 20.0)) * nz
        x_recon = decoder(sd, cfg, z, hw, is_image)
    if is_image:
        frames, frames_recon = x, x_recon
    else:
        Tin = x.shape[2]
        if frame_idx is None:
            frame_idx = torch.randint(0, Tin, [B])
        ar = torch.arange(B)
        frames, frames_recon = x[ar, :, frame_idx], x_recon[ar, :, frame_idx]
    return frames, frames_recon, x, x_recon, vq_output


# ---- consumers either side of encode / decode (SURVEY.md section 8f) -----------------------------------------------------
LATENT_SCALE = 0.18215


def to_u8(video: Tensor, mul: float = 1.0, add: float = 0.5, lo: float = 0.0, hi: float = 1.0, post: float = 255.0) -> Tensor:
    """(B,C,T,H,W) fp32 -> (B,T,H,W,C) uint8.  Defaults: vqgan_eval.py:139,147-148  shift_dim(clamp(x + 0.5, 0, 1) * 255, 1, -1)
    .byte()  (also Latte sample_ddp.py:206); (255, 128, 0, 255, 1): DiT sample_ddp.py:163  clamp(255 * x + 128.0, 0, 255)."""
    t = torch.clamp(video * mul + add, lo, hi) * post
    return t.permute(0, 2, 3, 4, 1).contiguous().to(torch.uint8)


def encode_to_z(sd: SD, cfg: Config, x: Tensor, is_image: bool, sample_every_n_latent_frames: int = 0):
    """lm_transformer.py:258-268 (vtokens False): embeddings channels-last + flat targets, every n-th latent frame."""
    emb, targets = encode(sd, cfg, x, include_embeddings=True)
    if sample_every_n_latent_frames > 0:
        emb = emb[:, :, ::sample_every_n_latent_frames]
        targets = targets[:, ::sample_every_n_latent_frames]
    return emb.permute(0, 2, 3, 4, 1).contiguous(), targets.reshape(targets.shape[0], -1)


def decode_tokens(sd: SD, cfg: Config, ix: Tensor, is_image: bool, cond_stage_vocab_size: int = 0) -> Tensor:
    """lm_transformer.py:433-434: clamp(ix - cond_vocab, 0, first_vocab - 1).squeeze(-1) -> decode (flat indices)."""
    n_codes = sd["codebook.embeddings"].shape[0]
    index = torch.clamp(ix - cond_stage_vocab_size, min=0, max=n_codes - 1)
    if index.ndim == 3:
        index = index.squeeze(-1)
    return decode(sd, cfg, index, is_image)


def dit_roundtrip(sd: SD, cfg: Config, x: Tensor, noise: Tensor):
    """DiT/train.py:242 then DiT/sample_ddp.py:162-163 on the same latent: (scaled latents, uint8 images (B,H,W,3))."""
    z = encode(sd, cfg, x, noise=noise) * LATENT_SCALE
    img = decode(sd, cfg, z / LATENT_SCALE, True)
    return z, to_u8(img.unsqueeze(2), 255.0, 128.0, 0.0, 255.0, 1.0)[:, 0]


def latte_roundtrip(sd: SD, cfg: Config, x_bfchw: Tensor, noise: Tensor):
    """Latte/train.py:215-217 then sample_ddp.py:201-206: (scaled latents 'b f c h w', video 'b f c h w', uint8 'b f h w c')."""
    z = encode(sd, cfg, x_bfchw.permute(0, 2, 1, 3, 4).contiguous(), noise=noise) * LATENT_SCALE
    z = z.permute(0, 2, 1, 3, 4).contiguous()
    video = decode(sd, cfg, z.permute(0, 1, 3, 4, 2) / LATENT_SCALE, False)
    return z, video.permute(0, 2, 1, 3, 4).contiguous(), to_u8(video)
