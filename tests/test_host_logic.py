"""CPU tests of the host-side conventions of OmniTokenizer_VQGAN.decode / encode with a stub engine
(no kernels run): the index / flat-index / VAE layout rules of omnitokenizer.py:268-317."""
import os
import types

import pytest
import torch

import omnitokenizer_b200 as ob


class _StubEngine:
    """Records what the module asks the engine to do; returns zeros of the right shape."""

    def __init__(self, model):
        a = model.args
        self.p, self.pt, self.cin = a.patch_size, a.temporal_patch_size, a.image_channels
        self.calls = []

    def decode(self, dims, *, idx=None, zc=None, straight_through=False, u8=None):
        B, Tp, h, w = dims
        self.calls.append(dict(dims=dims, idx=None if idx is None else idx.clone(), zc=None if zc is None else zc.clone(),
                               u8=u8))
        T = 1 + (Tp - 1) * self.pt
        if u8 is not None:
            return torch.zeros(B, T, h * self.p, w * self.p, self.cin, dtype=torch.uint8)
        return torch.zeros(B, self.cin, T, h * self.p, w * self.p)


def _model(extra=()):
    m = ob.OmniTokenizer_VQGAN(ob.canonical_args(list(extra)))
    stub = _StubEngine(m)
    m.engine = types.MethodType(lambda self: stub, m)
    # the real module refuses CPU; the stub path needs a device context-free call
    torch.cuda.device = lambda *_a, **_k: __import__("contextlib").nullcontext()
    return m, stub


@pytest.fixture(autouse=True)
def _restore_cuda_device():
    orig = torch.cuda.device
    yield
    torch.cuda.device = orig


def test_decode_index_conventions():
    m, stub = _model()
    codes = torch.randint(0, 8192, (2, 5, 32, 32))
    out = m.decode(codes, False)
    assert stub.calls[-1]["dims"] == (2, 5, 32, 32) and tuple(out.shape) == (2, 3, 17, 256, 256)
    assert torch.equal(stub.calls[-1]["idx"], codes.reshape(-1))
    # flat video indices use resolution // patch_size for h = w (omnitokenizer.py:284-286)
    m.decode(codes.reshape(2, -1), False)
    assert stub.calls[-1]["dims"] == (2, 5, 32, 32)
    # flat image indices: h = w = sqrt(hw) (omnitokenizer.py:271-275); result squeezed to 4-D
    img = torch.randint(0, 8192, (3, 64))
    out = m.decode(img, True)
    assert stub.calls[-1]["dims"] == (3, 1, 8, 8) and tuple(out.shape) == (3, 3, 64, 64)
    out = m.decode(torch.randint(0, 8192, (3, 1, 16, 16)), True)
    assert tuple(out.shape) == (3, 3, 128, 128)
    # fused uint8 form: same conventions, channels-last bytes, the eval script's affine by default
    out = m.decode_u8(codes.reshape(2, -1), False)
    assert stub.calls[-1]["dims"] == (2, 5, 32, 32) and stub.calls[-1]["u8"] == (1.0, 0.5, 0.0, 1.0, 255.0)
    assert tuple(out.shape) == (2, 17, 256, 256, 3) and out.dtype == torch.uint8


def test_decode_vae_layouts():
    m, stub = _model(["--use_vae"])
    z4 = torch.randn(2, 8, 16, 16)                       # image: 'b c h w'
    m.decode(z4, True)
    c = stub.calls[-1]
    assert c["dims"] == (2, 1, 16, 16)
    assert torch.equal(c["zc"], z4.permute(0, 2, 3, 1).reshape(-1, 8))
    z5 = torch.randn(1, 5, 32, 32, 8)                    # video: channels-LAST 'b t h w c' (omnitokenizer.py:313)
    m.decode(z5, False)
    c = stub.calls[-1]
    assert c["dims"] == (1, 5, 32, 32) and torch.equal(c["zc"], z5.reshape(-1, 8))
    zf = torch.randn(1, 5 * 32 * 32, 8)                  # flat video latents at the configured resolution
    m.decode(zf, False)
    assert stub.calls[-1]["dims"] == (1, 5, 32, 32)


def test_cnn_decoder_is_pinned_to_the_configured_resolution():
    m, stub = _model(["--patch_embed", "cnn"])
    m.decode(torch.zeros(1, 5, 32, 32, dtype=torch.long), False)          # 256 // 8 = 32: fine
    with pytest.raises(ValueError, match="configured resolution"):
        m.decode(torch.zeros(1, 5, 8, 8, dtype=torch.long), False)       # the reference's Rearrange raises here too


def test_unsupported_configurations_say_why():
    for extra, msg in ((["--use_external_codebook"], "external"), (["--defer_temporal_pool"], "multi-resolution"),
                       (["--enc_block", "ttaa"], "pooling"), (["--patch_embed", "pixelshuffle"], "linear / cnn")):
        with pytest.raises(NotImplementedError, match=msg):
            ob.OmniTokenizer_VQGAN(ob.canonical_args(extra))
    a = ob.canonical_args(["--attn_dropout", "0.1"])
    m = ob.OmniTokenizer_VQGAN(a)          # constructing is fine (training flag); the engine rejects it on first use
    assert m.args.attn_dropout == 0.1


def test_f16x3_split_is_tight():
    """Host-side operand split of the f16x3 path (layout.split_f16 == the device-side rule in csrc/omt_common.cuh):
    |x - (hi + lo * 2^-11)| <= 2^-22 |x|; hi saturates instead of overflowing and lo carries what it can of the rest."""
    from omnitokenizer_b200 import layout as L
    x = (torch.rand(4096, generator=torch.Generator().manual_seed(1)) - 0.5) * 60.0
    hi, lo = L.split_f16(x)
    assert hi.dtype == torch.float16 and lo.dtype == torch.float16
    assert ((L.join_f16(hi, lo) - x).abs() <= 2.0 ** -22 * x.abs() + 1e-30).all()
    tiny = torch.tensor([3e-6, -7e-8, 1e-9])                    # below fp16's normal range: lo rescues the precision
    hi, lo = L.split_f16(tiny)
    assert ((L.join_f16(hi, lo) - tiny).abs() <= 2.0 ** -36).all()
    big = torch.tensor([1e6, -3e5, 65504.0])
    hi, lo = L.split_f16(big)
    assert torch.isfinite(hi.float()).all() and torch.isfinite(lo.float()).all()        # saturates, never inf / nan


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the arm the driver runs next to the GPU arm) on a 2-image slice of cfg-2: one JSON line with
    the contract's keys, the metric / unit / config of the GPU arm, and a cpu_baseline describing the run."""
    import json, subprocess, sys
    env = dict(os.environ, OMT_BENCH_BATCH="2", OMT_REF_WORKERS="2")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--workload", "cfg2", "--steps", "1", "--warmup", "1"],
                         cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "video_frames_per_sec_encode_decode" and line["unit"] == "frames/s"
    assert line["higher_is_better"] is True and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["config"]["global_batch"] == 2 and line["config"]["workload"].startswith("cfg2")
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] > 0 and "full batch" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_dump_outputs_format(tmp_path):
    """`bench.py --dump-outputs DIR`: integer codes as exact float64 in their own shape; a float32 output above DUMP_SAMPLE
    elements as a sample at seeded flat positions (written next to it), the same positions on every run; 64 MB at most."""
    import numpy as np
    import bench
    codes = torch.randint(0, 8192, (2, 5, 4, 4))
    rec = torch.randn(2, bench.DUMP_SAMPLE // 2 + 1)
    dumps = []
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), {"codes": codes, "reconstruction": rec, "absent": None})
        dumps.append({f: np.load(tmp_path / d / f) for f in sorted(os.listdir(tmp_path / d))})
    a, b = dumps
    assert sorted(a) == ["codes.npy", "reconstruction.npy", "reconstruction_index.npy"]
    assert all(np.array_equal(a[f], b[f]) for f in a)
    assert a["codes.npy"].dtype == np.float64 and np.array_equal(a["codes.npy"], codes.numpy())
    pos = a["reconstruction_index.npy"]
    assert a["reconstruction.npy"].dtype == np.float32 and a["reconstruction.npy"].shape == pos.shape == (bench.DUMP_SAMPLE,)
    assert np.array_equal(a["reconstruction.npy"], rec.reshape(-1).numpy()[pos.astype(np.int64)])
    # the largest possible dump: two sampled arrays, one of them integer codes
    bench.write_outputs(str(tmp_path / "c"), {"codes": torch.zeros(bench.DUMP_SAMPLE + 1, dtype=torch.long), "reconstruction": rec})
    assert sum(os.path.getsize(tmp_path / "c" / f) for f in os.listdir(tmp_path / "c")) <= 64 << 20
