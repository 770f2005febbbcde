"""Kernel orchestration for OmniTokenizer_VQGAN.encode / decode / forward on one B200.

The engine owns (a) the packed device copies of the checkpoint in kernel layouts and (b) the
per-shape workspace; every arithmetic step is a call into libomnitok_b200.so (see
include/omnitok_b200.h).  torch is used for device memory, streams and a handful of
O(codebook)-sized reductions (usage statistics) -- never for the per-token math.

Activations stay in ONE canonical buffer X[B][T'][N][C] for the whole network.  The reference's
four rearrange copies between spatial and temporal blocks (omnitokenizer.py:891,902,907,1072,1081)
do not exist here: spatial kernels read rows contiguously, temporal kernels stride by N, window
attention and both PEG variants go through index maps.
"""
from __future__ import annotations

import math
import os
from typing import Dict, Optional, Tuple

import torch

from . import _cabi
from . import layout as L

MATH_MODES = {"fp32": _cabi.MATH_FP32, "3xtf32": _cabi.MATH_3XTF32, "f16x3": _cabi.MATH_F16X3}
DEFAULT_MATH = "f16x3"


def default_math() -> str:
    return os.environ.get("OMT_MATH", DEFAULT_MATH).lower()


class Planes:
    """fp16 hi / lo operand planes of an [M, ld] fp32 matrix (the A operands of the f16x3 GEMMs; layout.split_f16)."""

    def __init__(self, device, M: int, ld: int, row_scaled: bool = False):
        self.buf = torch.empty(2, M, ld, device=device, dtype=torch.int16)
        self.hi, self.lo, self.ld = self.buf[0], self.buf[1], ld
        # row-scaled form (written by producers that see whole rows): inverse per-row scales; None = the 2^11-scaled lo form
        self.rs = torch.empty(M, device=device, dtype=torch.float32) if row_scaled else None


class PackedLinear:
    """nn.Linear weight in GEMM layout: rows padded to 128, K padded, optional tf32 hi/lo split."""

    def __init__(self, weight: torch.Tensor, bias: Optional[torch.Tensor], device, math: int,
                 k_pad: Optional[int] = None, geglu: Optional[Tuple[int, int]] = None, row_scaled: bool = False):
        w = weight.detach().to(device=device, dtype=torch.float32)
        if geglu is not None:
            inner, ku = geglu
            w = L.pack_geglu(w, inner, ku)
        self.n = w.shape[0]
        if k_pad is not None:
            w = L.pad_cols(w, k_pad)
        self.k = w.shape[1]
        w = L.pad_rows(w, 256 if math == _cabi.MATH_F16X3 else 128)
        if math == _cabi.MATH_3XTF32:
            hi = L.tf32_round(w)
            self.w, self.w_lo = hi, (w - hi).contiguous()
        elif math == _cabi.MATH_F16X3 and row_scaled:
            self.w, self.w_lo, self.w_scale = L.split_f16_rs(w)      # fp16 planes, one scale per matrix (single-accumulator GEMM)
        elif math == _cabi.MATH_F16X3:
            self.w, self.w_lo = L.split_f16(w)          # fp16 operand planes, lo scaled by 2^11 (two-accumulator GEMM)
        else:
            self.w, self.w_lo = w, None
        self.bias = None if bias is None else bias.detach().to(device=device, dtype=torch.float32).contiguous()
        self.math = math
        self.row_scaled = row_scaled and math == _cabi.MATH_F16X3


class Workspace:
    def __init__(self, device, M: int, C: int, ku: int, kmax: int, cd: int, planes: bool):
        f = dict(device=device, dtype=torch.float32)
        self.M = M
        self.buf0 = torch.empty(M, C, **f)
        self.buf1 = torch.empty(M, C, **f)
        self.X, self.Y = self.buf0, self.buf1
        self.QKV = torch.empty(M, 3 * C, **f)
        self.P = torch.empty(M, kmax, **f)       # patch matrix (pixels side), rows x K
        if planes:     # f16x3: every GEMM A operand lives as fp16 hi / lo planes written by its producer
            self.XNp, self.XSp = Planes(device, M, C, True), Planes(device, M, C, True)     # LayerNorm sees whole rows
            self.Op, self.Up = Planes(device, M, C), Planes(device, M, ku)                  # attention heads / GEGLU tiles do not
            self.Pp = Planes(device, M, kmax, True)
            self.QKVp = Planes(device, M, 3 * C)     # q | k | v operand planes for the f16 attention core (QKV GEMM epilogue)
            self.vinv = torch.empty(C // 64, M, device=device, dtype=torch.float32)   # inverse (row, head) scales of the v planes
        else:
            self.XN = torch.empty(M, C, **f)
            self.O = torch.empty(M, C, **f)
            self.U = torch.empty(M, ku, **f)
        self.z = torch.empty(M, cd, **f)
        self.idx = torch.empty(M, device=device, dtype=torch.int64)
        self.counts = torch.zeros(8192, device=device, dtype=torch.int32)
        # static I/O buffers + captured CUDA graphs of this shape
        self.x_in = None
        self.video_u8 = None
        self.idx_in = torch.empty(M, device=device, dtype=torch.int64)
        self.zc_in = torch.empty(M, cd, **f)
        self.zq = torch.empty(M, cd, **f)
        self.video = None
        self.graphs = {}

    def reset(self):
        self.X, self.Y = self.buf0, self.buf1


class Engine:
    def __init__(self, model, device: torch.device, math: Optional[str] = None):
        _cabi.load()
        _cabi.set_option("pdl", int(os.environ.get("OMT_PDL", "0")))     # programmatic dependent launch between kernels
        # process-wide kernel selectors (tuning knobs; see omt_set_option): the environment or the library default
        for env, opt in (("OMT_PEG_KERNEL", "peg_kernel"),        # 4 (cp.async gather, default) | 3
                         ("OMT_ATTN_CTAS", "attn_f16_ctas"),      # CTAs per SM of the f16 attention core
                         ("OMT_F16_BN", "f16_bn")):               # 0 (by shape) | 128 | 256: tile N of the two-accumulator GEMM form
            _cabi.set_option(opt, int(os.environ.get(env) or _cabi.DEFAULT_OPTIONS[opt]))
        self.device = device
        self.math_name = (math or default_math()).lower()
        if self.math_name not in MATH_MODES:
            raise ValueError(f"unknown OMT_MATH mode {self.math_name!r}; choose from {sorted(MATH_MODES)}")
        self.math = MATH_MODES[self.math_name]
        a = model.args
        self.C = a.embedding_dim
        self.heads, self.dh = a.heads, a.dim_head
        if self.C != 512 or self.dh != 64 or self.heads * self.dh != self.C:
            raise NotImplementedError("omnitok_b200 kernels are specialised for embedding_dim=512, heads x dim_head = 8 x 64")
        self.p, self.pt, self.cin = a.patch_size, a.temporal_patch_size, a.image_channels
        self.ws = a.twod_window_size
        self.causal_attn = bool(a.causal_in_temporal_transformer)
        self.causal_peg = bool(a.causal_in_peg)
        self.rope = a.spatial_pos == "rope"
        self.use_vae = bool(model.use_vae)
        self.cd = a.codebook_dim
        self.l2 = bool(a.l2_code)
        if not self.use_vae and self.cd != 8:
            raise NotImplementedError(f"--codebook_dim {self.cd}: the VQ search / post_vq kernels are specialised for "
                                      "codebook_dim 8 (every shipped config); VAE mode takes 8 latent channels as well")
        self.planes = self.math == _cabi.MATH_F16X3
        # spatial attention core on fp16 operand planes (attention_f16.cu, default); OMT_ATTN_F16=0 = the 3xTF32 core on the fp32 QKV buffer
        self.attn_f16 = self.planes and os.environ.get("OMT_ATTN_F16", "1") == "1"
        # GEGLU output planes with a static (pack-time) scale -> the second FF GEMM takes the single-accumulator form (default).
        # The bound |U| <= (|LN(x)|_2 max|W1_n|_2)^2 is structural (|LN(x)|_2 <= max|gamma| sqrt(C) + |beta|_2), at most ~2^10
        # above typical values, so the planes keep 22 significant bits; OMT_STATIC_U=0 = per-element 2^11 form, two accumulators
        self.static_u = self.planes and os.environ.get("OMT_STATIC_U", "1") == "1"
        if a.attn_dropout != 0 or a.ff_dropout != 0:
            raise NotImplementedError("non-zero dropout reaches SDPA even in eval in the reference (attention.py:451); rejected")
        self._ws: Dict[Tuple, Workspace] = {}
        self._tables: Dict[Tuple, torch.Tensor] = {}
        sd = {k: v for k, v in model.state_dict().items()}
        self._pack(sd, a)

    # ------------------------------------------------------------------ packing
    def _pack(self, sd, a):
        dev, m = self.device, self.math
        f32 = lambda t: t.detach().to(device=dev, dtype=torch.float32).contiguous()
        self.inner = sd["encoder.enc_spatial_transformer.layers.0.3.4.weight"].shape[1]
        self.ku = L.round_up(self.inner, 64 if self.planes else 32)     # K of the second FF GEMM: whole k-blocks

        def PL(weight, bias, **kw):
            return PackedLinear(weight, bias, dev, m, **kw)

        def lin(name, bias=True, **kw):
            return PL(sd[name + ".weight"], sd.get(name + ".bias") if bias else None, **kw)

        def t_layer(lp):
            d = {"kind": "t"}
            d["peg_w"] = f32(sd[lp + ".0.dsconv.weight"].reshape(self.C, 27).t())      # [27, C]
            d["peg_b"] = f32(sd[lp + ".0.dsconv.bias"])
            ap = lp + ".1"
            d["norm_g"], d["norm_b"] = f32(sd[ap + ".norm.gamma"]), f32(sd[ap + ".norm.beta"])
            d["q_scale"], d["k_scale"] = f32(sd[ap + ".q_scale"]), f32(sd[ap + ".k_scale"])
            # after l2norm every |q_d| <= |q_scale_d|: one exact power of two per layer puts the q / k planes in fp16 range
            d["q_ps"], d["k_ps"] = L.pow2_scale(float(d["q_scale"].abs().max())), L.pow2_scale(float(d["k_scale"].abs().max()))
            # [Wq; Wkv] stacked: one dual-A GEMM writes q | k | v into the QKV buffer
            d["to_qkv"] = PL(torch.cat([sd[ap + ".to_q.weight"], sd[ap + ".to_kv.weight"]], dim=0), None, row_scaled=True)
            d["to_out"] = lin(ap + ".to_out", bias=False)
            ff(d, lp + ".3")
            return d

        def w_layer(lp):
            d = {"kind": "w"}
            ap = lp + ".1"
            d["norm_g"], d["norm_b"] = f32(sd[ap + ".norm.gamma"]), f32(sd[ap + ".norm.beta"])
            d["bias"] = L.window_bias(sd[ap + ".relative_position_bias_table"].detach().float().cpu(),
                                      sd[ap + ".relative_position_index"].cpu(), self.ws).to(dev)
            d["qkv"] = lin(ap + ".qkv", bias=False, row_scaled=True)
            d["proj"] = lin(ap + ".proj")
            ff(d, lp + ".3")
            return d

        def ff(d, fp):
            d["ff_g"], d["ff_b"] = f32(sd[fp + ".0.weight"]), f32(sd[fp + ".0.bias"])
            d["ff1"] = PL(sd[fp + ".1.weight"], None, geglu=(self.inner, self.ku), row_scaled=True)
            # |U| = |gelu(g) a| <= |g| |a| <= (|LN(x)|_2 max_n |W1_n|_2)^2 with |LN(x)|_2 <= max|gamma| sqrt(C) + |beta|_2: a bound
            # known at pack time, so the U planes take ONE static power-of-two scale (single-accumulator FF2, no overflow possible)
            w1 = sd[fp + ".1.weight"].detach().float()
            ln_bound = float(d["ff_g"].abs().max()) * math.sqrt(self.C) + float(d["ff_b"].norm())
            u_bound = (ln_bound * float(w1[:self.inner].norm(dim=1).max())) * (ln_bound * float(w1[self.inner:].norm(dim=1).max()))
            d["u_scale"] = L.pow2_scale(u_bound) if self.static_u else 0.0
            d["ff2"] = PL(sd[fp + ".4.weight"], None, k_pad=self.ku, row_scaled=self.static_u)

        def transformer(pre, block):
            layers = []
            for i, blk in enumerate(block):
                if blk == "t":
                    layers.append(t_layer(f"{pre}.layers.{i}"))
                elif blk == "w":
                    layers.append(w_layer(f"{pre}.layers.{i}"))
                else:
                    raise NotImplementedError(f"block type {blk!r}: pooling/upsampling blocks are outside the shipped configs")
            return {"layers": layers, "out_g": f32(sd[pre + ".norm_out.gamma"]), "out_b": f32(sd[pre + ".norm_out.beta"])}

        tb = "t" * a.temporal_depth
        self.enc_spatial = transformer("encoder.enc_spatial_transformer", a.enc_block)
        self.enc_temporal = transformer("encoder.enc_temporal_transformer", tb)
        self.dec_temporal = transformer("decoder.dec_temporal_transformer", tb)
        self.dec_spatial = transformer("decoder.dec_spatial_transformer", a.dec_block)

        self.has_window = "w" in (a.enc_block + a.dec_block)
        self.pe = {}
        self.cnn = getattr(a, "patch_embed", "linear") == "cnn"
        if self.cnn:
            # patch_embed='cnn' (omnitokenizer.py:823-838, 1019-1035): a Conv3d with kernel == stride is a GEMM over
            # the same (c, pt, p1, p2) patch vectors as the linear variant, and eval-mode (Sync)BatchNorm is a
            # per-channel affine -> both fold into ONE packed weight/bias; no LayerNorms in this variant.
            def bn_affine(pre):
                g, b = sd[pre + ".weight"].float(), sd[pre + ".bias"].float()
                rm, rv = sd[pre + ".running_mean"].float(), sd[pre + ".running_var"].float()
                s_ = g / torch.sqrt(rv + 1e-5)
                return s_, b - rm * s_
            for key, pre in (("first", "encoder.to_patch_emb_first_frame"), ("rest", "encoder.to_patch_emb")):
                w = sd[pre + ".0.weight"].float().reshape(self.C, -1)                 # (dim, c*pt*p*p)
                s_, t_ = bn_affine(pre + ".1")
                self.pe[key] = dict(ln1_g=None, ln1_b=None, ln2_g=None, ln2_b=None,
                                    lin=PL(w * s_[:, None], sd[pre + ".0.bias"].float() * s_ + t_, row_scaled=True))
            self.px = {}
            for key, pre in (("first", "decoder.to_pixels_first_frame"), ("rest", "decoder.to_pixels")):
                wt = sd[pre + ".1.weight"].float()                                    # (dim, channels, pt, p, p)
                per_c = wt[0, 0].numel()
                s_, t_ = bn_affine(pre + ".2")
                w = wt.reshape(self.C, -1).t() * s_.repeat_interleave(per_c)[:, None]  # (channels*pt*p*p, dim)
                bias = (sd[pre + ".1.bias"].float() * s_ + t_).repeat_interleave(per_c)
                self.px[key] = PL(w.contiguous(), bias, row_scaled=True)
        else:
            for key, pre in (("first", "encoder.to_patch_emb_first_frame"), ("rest", "encoder.to_patch_emb")):
                self.pe[key] = dict(ln1_g=f32(sd[pre + ".1.weight"]), ln1_b=f32(sd[pre + ".1.bias"]), lin=lin(pre + ".2", row_scaled=True),
                                    ln2_g=f32(sd[pre + ".3.weight"]), ln2_b=f32(sd[pre + ".3.bias"]))
            self.px = {"first": lin("decoder.to_pixels_first_frame.0", row_scaled=True),
                       "rest": lin("decoder.to_pixels.0", row_scaled=True)}
        self.pre_w, self.pre_b = f32(sd["pre_vq_conv.1.weight"]), f32(sd["pre_vq_conv.1.bias"])
        self.post_w, self.post_b = f32(sd["post_vq_conv.1.weight"]), f32(sd["post_vq_conv.1.bias"])
        E = sd["codebook.embeddings"].detach().float()
        self.E = E.to(dev).contiguous()
        # sum E^2 with the reference's own expression (modules/codebook.py:84), evaluated on the host
        self.e2 = (E.cpu().t() ** 2).sum(dim=0).to(dev).contiguous()
        self.n_codes = E.shape[0]

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def fuse_qkprep(M: int) -> bool:
        """rope + l2norm + scale ride in the QKV GEMM epilogue.  The choice must NOT depend on the batch size: the
        fused epilogue and the stand-alone kernel round differently (x * (1/|x|) vs x / |x|, different reduction
        trees), and a shard of a batch has to reproduce the full batch bit for bit (tests/test_gpu_fullsize.py)."""
        return os.environ.get("OMT_FUSE_QKPREP", "1") != "0"

    def _workspace(self, M: int) -> Workspace:
        ws = self._ws.get(M)
        if ws is None:
            kmax = self.cin * self.pt * self.p * self.p
            ws = Workspace(self.device, M, self.C, self.ku, kmax, max(self.cd, 16), self.planes)
            if ws.counts.numel() < self.n_codes:
                ws.counts = torch.zeros(self.n_codes, device=self.device, dtype=torch.int32)
            while len(self._ws) >= 3:  # keep a few shapes (and their graphs) resident
                self._ws.pop(next(iter(self._ws)))
            self._ws[M] = ws
        return ws

    def _table(self, key, fn):
        t = self._tables.get(key)
        if t is None:
            t = fn()
            t = tuple(x.to(self.device) for x in t) if isinstance(t, tuple) else t.to(self.device)
            self._tables[key] = t
        return t

    def _linear(self, A, lda, lin: PackedLinear, C, ldc, M, *, a_map=(0, 0, 0), c_map=(0, 0, 0), residual=None,
                ldr=0, epi=_cabi.EPI_NONE, bias=True):
        """nn.Linear on the fp32-operand paths (CUDA-core fp32 / tcgen05 3xTF32)."""
        _cabi.call("omt_linear", A, lda, a_map[0], a_map[1], a_map[2], lin.w, lin.w_lo, C, ldc, c_map[0], c_map[1],
                   c_map[2], M, lin.n, lin.k, lin.bias if bias else None, residual, ldr, epi, lin.math)

    def _linear_h(self, A: Planes, lin: PackedLinear, M, *, C=None, ldc=0, U: Optional[Planes] = None, A2: Optional[Planes] = None,
                  n_split=0, a_map=(0, 0, 0), c_map=(0, 0, 0), residual=None, ldr=0, epi=_cabi.EPI_NONE, qk=None,
                  planes=None, a_uniform=0.0, u_scale=0.0):
        """nn.Linear on operand planes (tcgen05 f16x3).  U: GEGLU output planes; qk: (q_scale, k_scale, cos, sin, qk_cols, tokens)."""
        if ((A.rs is not None) or a_uniform > 0.0) != lin.row_scaled:
            raise RuntimeError("operand planes and weight planes are in different f16x3 forms (row-scaled vs 2^11-scaled lo)")
        kw = dict(a_hi=A.hi, a_lo=A.lo, lda=A.ld, a_seg=a_map[0], a_seg_stride=a_map[1], a_seg_off=a_map[2],
                  w_hi=lin.w, w_lo=lin.w_lo, c=C, ldc=ldc, c_seg=c_map[0], c_seg_stride=c_map[1], c_seg_off=c_map[2],
                  M=M, N=lin.n, K=lin.k, bias=lin.bias, residual=residual, ldr=ldr, epilogue=epi)
        if A.rs is not None:
            kw.update(a_rs=A.rs, w_scale=lin.w_scale)
        elif a_uniform > 0.0:
            kw.update(a_rs_uniform=a_uniform, w_scale=lin.w_scale)
        if u_scale > 0.0:
            kw.update(u_scale=u_scale)
        if A2 is not None:
            kw.update(a2_hi=A2.hi, a2_lo=A2.lo, a2_rs=A2.rs, n_split=n_split)
        if U is not None:
            kw.update(u_hi=U.hi, u_lo=U.lo, ldu=U.ld)
        if qk is not None:
            kw.update(q_scale=qk[0], k_scale=qk[1], rope_cos=qk[2], rope_sin=qk[3], qk_cols=qk[4], tokens=qk[5])
        if planes is not None:      # EPI_QKV_PLANES: U = the q | k | v planes, (q plane scale, k plane scale, vinv)
            kw.update(q_plane_scale=planes[0], k_plane_scale=planes[1], vinv=planes[2])
        _cabi.linear_h(**kw)

    def _ln(self, x, y, g, b, M, C=None, seg=(0, 0, 0)):
        C = C or self.C
        _cabi.call("omt_layernorm", x, C, y, C, g, b, M, C, 1e-5, seg[0], seg[1], seg[2])

    def _ln_h(self, x, yp: Planes, g, b, M, xp: Optional[Planes] = None):
        """LayerNorm straight into the operand planes of the consuming GEMM (+ planes of the raw row for to_kv)."""
        C = self.C
        _cabi.call("omt_layernorm_h", x, C, None, 0, yp.hi, yp.lo, yp.rs, None if xp is None else xp.hi,
                   None if xp is None else xp.lo, None if xp is None else xp.rs, yp.ld, g, b, M, C, 1e-5, 0, 0, 0)

    # ------------------------------------------------------------------ transformer
    def _transformer(self, tr, ws: Workspace, B, T, h, w, temporal: bool, out_planes: Optional[Planes] = None):
        """modules/attention.py:655-689.  out_planes: norm_out goes to operand planes (decoder -> to_pixels GEMMs)."""
        C, N, M = self.C, h * w, ws.M
        H = self.planes
        q_ptr = ws.QKV.data_ptr()
        k_ptr, v_ptr = q_ptr + C * 4, q_ptr + 2 * C * 4
        ld3 = 3 * C
        o, o_hi, o_lo = (None, ws.Op.hi, ws.Op.lo) if H else (ws.O, None, None)
        for lyr in tr["layers"]:
            if lyr["kind"] == "t":
                _cabi.call("omt_peg_volume", ws.X, ws.Y, lyr["peg_w"], lyr["peg_b"], B, T, h, w, C, int(temporal),
                           int(self.causal_peg))
                ws.X, ws.Y = ws.Y, ws.X
                # q from the normalised input, k / v from the RAW input (attention.py:407-412), one launch;
                # rope (spatial blocks) + l2norm + q/k scale ride in the same launch (fused GEMM epilogue)
                wq = lyr["to_qkv"]
                cos = sin = None
                if (not temporal) and self.rope:
                    cos, sin = self._table(("rope", N), lambda: L.rope_tables(N, self.dh))
                f16_core = H and self.attn_f16 and (not temporal) and N % 128 == 0
                if f16_core:
                    self._ln_h(ws.X, ws.XNp, lyr["norm_g"], lyr["norm_b"], M, xp=ws.XSp)
                    self._linear_h(ws.XNp, wq, M, U=ws.QKVp, A2=ws.XSp, n_split=C, epi=_cabi.EPI_QKV_PLANES,
                                   qk=(lyr["q_scale"], lyr["k_scale"], cos, sin, 2 * C, N),
                                   planes=(lyr["q_ps"], lyr["k_ps"], ws.vinv))
                elif H:
                    self._ln_h(ws.X, ws.XNp, lyr["norm_g"], lyr["norm_b"], M, xp=ws.XSp)
                    self._linear_h(ws.XNp, wq, M, C=q_ptr, ldc=ld3, A2=ws.XSp, n_split=C, epi=_cabi.EPI_QKV,
                                   qk=(lyr["q_scale"], lyr["k_scale"], cos, sin, 2 * C, N))
                else:
                    self._ln(ws.X, ws.XN, lyr["norm_g"], lyr["norm_b"], M)
                    if self.fuse_qkprep(M):
                        _cabi.call("omt_linear2", ws.XN, ws.X, C, C, wq.w, wq.w_lo, q_ptr, ld3, M, wq.n, wq.k, wq.math,
                                   lyr["q_scale"], lyr["k_scale"], cos, sin, 2 * C, N)
                    else:
                        _cabi.call("omt_linear2", ws.XN, ws.X, C, C, wq.w, wq.w_lo, q_ptr, ld3, M, wq.n, wq.k, wq.math,
                                   None, None, None, None, 0, 0)
                        _cabi.call("omt_qk_prep", q_ptr, ld3, k_ptr, ld3, lyr["q_scale"], lyr["k_scale"], cos, sin, M, N,
                                   self.heads)
                if f16_core:
                    ph, pl = ws.QKVp.hi.data_ptr(), ws.QKVp.lo.data_ptr()
                    _cabi.call("omt_attn_spatial_h", ph, pl, ld3, ph + 2 * C, pl + 2 * C, ld3, ph + 4 * C, pl + 4 * C, ld3,
                               ws.vinv, lyr["q_ps"] * lyr["k_ps"], None, o_hi, o_lo, C, B * T, N, self.heads, 8.0)
                elif temporal:
                    _cabi.call("omt_attn_temporal", q_ptr, ld3, k_ptr, ld3, v_ptr, ld3, o, o_hi, o_lo, C, B, T, N,
                               self.heads, 8.0, int(self.causal_attn))
                else:
                    _cabi.call("omt_attn_spatial", q_ptr, ld3, k_ptr, ld3, v_ptr, ld3, o, o_hi, o_lo, C, B * T, N,
                               self.heads, 8.0)
                proj = lyr["to_out"]
            else:
                if H:
                    self._ln_h(ws.X, ws.XNp, lyr["norm_g"], lyr["norm_b"], M)
                    self._linear_h(ws.XNp, lyr["qkv"], M, C=q_ptr, ldc=ld3)
                else:
                    self._ln(ws.X, ws.XN, lyr["norm_g"], lyr["norm_b"], M)
                    self._linear(ws.XN, C, lyr["qkv"], q_ptr, ld3, M)
                _cabi.call("omt_attn_window", q_ptr, ld3, k_ptr, ld3, v_ptr, ld3, o, o_hi, o_lo, C, lyr["bias"], B * T, h,
                           w, self.ws, self.heads, float(self.dh) ** -0.5)
                proj = lyr["proj"]
            if H:
                self._linear_h(ws.Op, proj, M, C=ws.X, ldc=C, residual=ws.X, ldr=C)
                self._ln_h(ws.X, ws.XNp, lyr["ff_g"], lyr["ff_b"], M)
                us = lyr["u_scale"]
                self._linear_h(ws.XNp, lyr["ff1"], M, U=ws.Up, epi=_cabi.EPI_GEGLU, u_scale=us)
                self._linear_h(ws.Up, lyr["ff2"], M, C=ws.X, ldc=C, residual=ws.X, ldr=C, a_uniform=(1.0 / us if us > 0 else 0.0))
            else:
                self._linear(ws.O, C, proj, ws.X, C, M, residual=ws.X, ldr=C)
                self._ln(ws.X, ws.XN, lyr["ff_g"], lyr["ff_b"], M)
                self._linear(ws.XN, C, lyr["ff1"], ws.U, self.ku, M, epi=_cabi.EPI_GEGLU)
                self._linear(ws.U, self.ku, lyr["ff2"], ws.X, C, M, residual=ws.X, ldr=C)
        if out_planes is not None:
            self._ln_h(ws.X, out_planes, tr["out_g"], tr["out_b"], M)
        else:
            self._ln(ws.X, ws.X, tr["out_g"], tr["out_b"], M)

    # ------------------------------------------------------------------ shapes / graphs
    def _shape(self, shape):
        B, Cin, T, H, W = shape
        if Cin != self.cin:
            raise ValueError(f"expected {self.cin} channels, got {Cin}")
        assert (T - 1) % self.pt == 0, (f"number of frames ({T}) minus one ({T - 1}) must be divisible by temporal "
                                        f"patch size ({self.pt})")
        if H != W or H % self.p != 0:
            raise ValueError(f"frames must be square with side a multiple of the patch size {self.p} (got {H}x{W})")
        if self.has_window and (self.ws * self.ws != 64 or (H // self.p) % self.ws != 0):
            raise ValueError(f"window blocks need twod_window_size 8 and a token grid divisible by it (got window "
                             f"{self.ws}, grid {H // self.p}x{W // self.p}): omt_attn_window is specialised for 8x8 windows")
        if ((H // self.p) * (W // self.p)) % 64 != 0:
            raise ValueError(f"tokens per frame ({(H // self.p) * (W // self.p)}) must be a multiple of 64 (attention tiles)")
        dims = B, T, H, W, 1 + (T - 1) // self.pt, H // self.p, W // self.p
        self._check_size(*dims[4:], B)
        return dims

    # Shape limit.  Kernels index rows (and the TMA maps row coordinates) with 32-bit integers, so every buffer of a shape
    # -- the widest is QKV at 3C fp32 per row, the video B*C*T*H*W -- must hold fewer than 2^31 elements; the spatial
    # attention grid also takes at most 65535 frames (B*T').  Beyond that a shape is refused before anything is allocated.
    MAX_ELEMS = 2 ** 31 - 1
    MAX_FRAMES = 65535

    def _max_batch(self, Tp: int, h: int, w: int) -> int:
        """largest batch of T' latent frames on an h x w token grid within the shape limit"""
        kmax = self.cin * self.pt * self.p * self.p
        per_sample = max(Tp * h * w * max(3 * self.C, self.ku, kmax),                          # workspace rows
                         self.cin * (1 + (Tp - 1) * self.pt) * h * self.p * w * self.p)        # the video
        return min(self.MAX_ELEMS // per_sample, self.MAX_FRAMES // Tp)

    def _check_size(self, Tp: int, h: int, w: int, B: int):
        bmax = self._max_batch(Tp, h, w)
        if B > bmax:
            T, H = 1 + (Tp - 1) * self.pt, h * self.p
            raise ValueError(f"{B} clips of {T} frames at {H}x{w * self.p} exceed the supported shape (every buffer below "
                             f"2^31 elements, at most {self.MAX_FRAMES} latent frames per call): at most {bmax} clips of "
                             f"this size fit; split the batch")

    @staticmethod
    def graphs_enabled() -> bool:
        return os.environ.get("OMT_CUDA_GRAPH", "1") != "0"

    def _run(self, ws: Workspace, key, body):
        """Run ``body`` (a fixed launch sequence over static buffers): the first call of a shape runs eagerly
        (sets function attributes, builds tables), the second captures a CUDA graph, later calls replay it --
        ~170 launches per encode+decode collapse into one submission."""
        if not self.graphs_enabled():
            return body()
        g = ws.graphs.get(key)
        if g is None:
            body()
            ws.graphs[key] = "warm"
        elif g == "warm":
            graph = torch.cuda.CUDAGraph()
            torch.cuda.synchronize(self.device)
            n0 = _cabi.launch_count
            with torch.cuda.graph(graph):
                body()
            ws.graphs[key] = (graph, _cabi.launch_count - n0)
            graph.replay()
        else:
            g[0].replay()
            _cabi.launch_count += g[1]        # kernels inside the replayed graph (bench.py accounting)

    # ------------------------------------------------------------------ encoder side
    def _encode_body(self, ws: Workspace, x, dims, mode: str):
        """patch embed -> spatial -> temporal -> pre_vq [-> VQ search].  omnitokenizer.py:881-947, 247-258."""
        B, T, H, W, Tp, h, w = dims
        N, C = h * w, self.C
        ws.reset()
        k1 = self.cin * self.p * self.p

        def embed(pe, first, rows, K, cmap):
            if self.planes:
                Pp = Planes.__new__(Planes)          # dense [rows, K] view at the start of the patch planes
                Pp.hi, Pp.lo, Pp.ld, Pp.rs = ws.Pp.hi, ws.Pp.lo, K, ws.Pp.rs
                _cabi.call("omt_patchify_ln", x, None, Pp.hi, Pp.lo, Pp.rs, pe["ln1_g"], pe["ln1_b"], B, self.cin, T, H, W,
                           self.p, self.pt, first, 1e-5)
                self._linear_h(Pp, pe["lin"], rows, C=ws.X, ldc=C, c_map=cmap)
            else:
                _cabi.call("omt_patchify_ln", x, ws.P, None, None, None, pe["ln1_g"], pe["ln1_b"], B, self.cin, T, H, W, self.p,
                           self.pt, first, 1e-5)
                self._linear(ws.P, K, pe["lin"], ws.X, C, rows, c_map=cmap)
            if not self.cnn:
                self._ln(ws.X, ws.X, pe["ln2_g"], pe["ln2_b"], rows, seg=cmap)

        embed(self.pe["first"], 1, B * N, k1, (N, Tp * N, 0))
        if Tp > 1:
            embed(self.pe["rest"], 0, B * (Tp - 1) * N, k1 * self.pt, ((Tp - 1) * N, Tp * N, N))
        self._transformer(self.enc_spatial, ws, B, Tp, h, w, temporal=False)
        self._transformer(self.enc_temporal, ws, B, Tp, h, w, temporal=True)
        cd = self.pre_w.shape[0]
        z = ws.z.view(-1)[: ws.M * cd].view(ws.M, cd)
        if mode == "vq":      # pre_vq + l2norm + modules/codebook.py:82-86 in one cluster kernel
            ws.counts.zero_()
            _cabi.call("omt_vq_fused", ws.X, C, self.pre_w, self.pre_b, C, int(self.l2), z, self.E, self.e2, ws.M,
                       self.n_codes, ws.idx, ws.counts)
        else:
            _cabi.call("omt_pre_vq", ws.X, C, self.pre_w, self.pre_b, z, ws.M, C, cd, 0)

    def encode(self, x: torch.Tensor, mode: str):
        """x (B,C,T,H,W) fp32 on the device.  mode 'vq': returns (ws, dims) with ws.z (l2-normalised z),
        ws.idx, ws.counts filled; mode 'raw': ws.z = pre_vq output (VAE moments).  Results live in the
        workspace until the next call of the same shape."""
        dims = self._shape(tuple(x.shape))
        B, T, H, W, Tp, h, w = dims
        ws = self._workspace(B * Tp * h * w)
        if ws.x_in is None or ws.x_in.shape != x.shape:
            ws.x_in = torch.empty_like(x, memory_format=torch.contiguous_format)
            ws.graphs = {k: v for k, v in ws.graphs.items() if not k[0].startswith("enc")}
        ws.x_in.copy_(x)
        self._run(ws, ("enc:" + mode, tuple(x.shape)), lambda: self._encode_body(ws, ws.x_in, dims, mode))
        return ws, (B, Tp, h, w)

    def z_view(self, ws: Workspace) -> torch.Tensor:
        return self._dense(ws.z, ws.M, self.pre_w.shape[0])

    @staticmethod
    def _dense(buf: torch.Tensor, M: int, cols: int) -> torch.Tensor:
        """Dense [M, cols] view at the start of a wider scratch buffer (kernels take packed rows)."""
        return buf.view(-1)[: M * cols].view(M, cols)

    def zq_view(self, ws: Workspace) -> torch.Tensor:
        return self._dense(ws.zq, ws.M, self.post_w.shape[1])

    # ------------------------------------------------------------------ decoder side
    def _decode_body(self, ws: Workspace, dims, mode: str, u8=None):
        """[gather +] post_vq -> temporal -> spatial -> to_pixels.  omnitokenizer.py:268-317, 1059-1118.
        u8 = (mul, add, lo, hi, post): the pixels leave as uint8 (B,T,H,W,C) = trunc(clamp(x*mul+add, lo, hi)*post)."""
        B, Tp, h, w = dims
        N, M, C = h * w, ws.M, self.C
        ws.reset()
        cdp = self.post_w.shape[1]
        if mode == "idx":
            _cabi.call("omt_post_vq", ws.idx_in, self.E, None, None, None, self.post_w, self.post_b, ws.X, M, C, cdp)
        elif mode == "idx_st":    # forward(): decoder sees (E[idx] - z) + z, codebook.py:120
            _cabi.call("omt_post_vq", ws.idx_in, self.E, None, self.z_view(ws), self.zq_view(ws), self.post_w,
                       self.post_b, ws.X, M, C, cdp)
        else:
            _cabi.call("omt_post_vq", None, None, self._dense(ws.zc_in, M, cdp), None, None, self.post_w, self.post_b,
                       ws.X, M, C, cdp)
        self._transformer(self.dec_temporal, ws, B, Tp, h, w, temporal=True)
        self._transformer(self.dec_spatial, ws, B, Tp, h, w, temporal=False, out_planes=ws.XNp if self.planes else None)
        T = 1 + (Tp - 1) * self.pt
        H, W = h * self.p, w * self.p
        k1 = self.cin * self.p * self.p

        def pixels(px, first, rows, K, amap):
            if self.planes:
                self._linear_h(ws.XNp, px, rows, C=ws.P, ldc=K, a_map=amap)
            else:
                self._linear(ws.X, C, px, ws.P, K, rows, a_map=amap)
            if u8 is None:
                _cabi.call("omt_unpatchify", ws.P, ws.video, B, self.cin, T, H, W, self.p, self.pt, first)
            else:
                _cabi.call("omt_unpatchify_u8", ws.P, ws.video_u8, B, self.cin, T, H, W, self.p, self.pt, first, *u8)

        pixels(self.px["first"], 1, B * N, k1, (N, Tp * N, 0))
        if Tp > 1:
            pixels(self.px["rest"], 0, B * (Tp - 1) * N, k1 * self.pt, ((Tp - 1) * N, Tp * N, N))

    def decode(self, dims, *, idx=None, zc=None, straight_through=False, u8=None) -> torch.Tensor:
        """dims (B,T',h,w).  idx: int64 [M] codes | zc: fp32 [M, cd] latents (VAE).  With straight_through
        the rows are (E[idx] - z) + z using the z left in the workspace by encode(); ws.zq receives them.
        Returns a fresh (B,C,T,H,W) tensor (the reference's decoder ends in .clone(), omnitokenizer.py:1116);
        with u8 = (mul, add, lo, hi, post) a fresh uint8 (B,T,H,W,C) tensor (fused consumer conversion)."""
        B, Tp, h, w = dims
        self._check_size(Tp, h, w, B)
        ws = self._workspace(B * Tp * h * w)
        vshape = (B, self.cin, 1 + (Tp - 1) * self.pt, h * self.p, w * self.p)
        if ws.video is None or tuple(ws.video.shape) != vshape:
            ws.video = torch.empty(vshape, device=self.device, dtype=torch.float32)
            ws.video_u8 = torch.empty((B, vshape[2], vshape[3], vshape[4], self.cin), device=self.device, dtype=torch.uint8)
            ws.graphs = {k: v for k, v in ws.graphs.items() if not k[0].startswith("dec")}
        if idx is not None:
            ws.idx_in.copy_(idx.reshape(-1))
            mode = "idx_st" if straight_through else "idx"
        else:
            self._dense(ws.zc_in, ws.M, zc.shape[1]).copy_(zc)
            mode = "zc"
        u8 = None if u8 is None else tuple(float(v) for v in u8)
        self._run(ws, ("dec:" + mode, dims, u8), lambda: self._decode_body(ws, dims, mode, u8))
        return ws.video.clone() if u8 is None else ws.video_u8.clone()
