"""Long-clip measurements on one GPU (profiles/r03_long_clips.*).

    python scripts/bench_long.py --out DIR              # encode -> decode steps + temporal attention alone
    python scripts/bench_long.py --out DIR --profile    # torch.profiler kernel breakdown of one 257-frame step

Steps: encode -> decode through the public API (shipped default math and kernels) on a seeded input already on the device;
CUDA events around each step, a 256 MiB L2 flush before it, warm-up that covers the eager run and the CUDA-graph capture,
median of --steps.  Temporal attention alone: omt_attn_temporal at the model's shapes (N = 1024 tokens per frame, B = 1,
8 heads, causal, output as fp16 operand planes as in the default math), events around single launches with the L2 flushed
between them.  The card's name, power limit and the SM clock during the attention loop are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_BPS = 7.7e12                 # HGX B200 data sheet, per GPU
FFMA_LANES_PER_CLK_SM = 125      # profiles/r02_alu_issue_rates.md
SMS = 148
HEADS, DH = 8, 64


def attn_work(B, T, N, causal=True):
    """algorithmic FLOP and HBM bytes of temporal attention: q.k and p.v are 2 * 64 FMA per (query, visible key, head);
    q, k, v are read and o written once (fp32 in, fp16 hi / lo planes out: 4 + 4 + 4 + 2 + 2 bytes per element)"""
    pairs = T * (T + 1) // 2 if causal else T * T
    flop = B * N * HEADS * pairs * 2 * DH * 2
    bytes_ = B * T * N * HEADS * DH * (3 * 4 + 2 * 2)
    return flop, bytes_


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                          "-i", "0"], capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"name": out[0], "power_limit_w": float(out[1]), "max_sm_clock_mhz": float(out[2])}


def sm_clock_mhz():
    out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return float(out)


def model(dev):
    import omnitokenizer_b200 as ob
    from oracle import omni_oracle as oo
    from oracle import weights as W
    cfg = oo.Config()
    m = ob.OmniTokenizer_VQGAN(ob.canonical_args())
    m.load_state_dict(W.make_state_dict(cfg, 0), strict=False)
    m.codebook._need_init = False
    return m.to(dev).eval(), W


def steps(dev, n_steps, warmup):
    m, W = model(dev)
    flush = torch.empty(64 * 1024 * 1024, device=dev)           # 256 MiB, twice the L2
    res = []
    for B, T in ((8, 17), (1, 17), (1, 65), (1, 129), (1, 257)):
        x = W.synthetic_input((B, 3, T, 256, 256), 4000 + T).to(dev)
        ts = []
        for i in range(warmup + n_steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            idx = m.encode(x, False)
            rec = m.decode(idx, False)
            b.record()
            torch.cuda.synchronize()
            if i >= warmup:
                ts.append(a.elapsed_time(b))
        ms = statistics.median(ts)
        Tp = 1 + (T - 1) // 4
        res.append({"clip": f"{B}x{T}x256x256", "B": B, "T": T, "latent_frames": Tp, "rows": B * Tp * 1024,
                    "ms_per_step": ms, "ms_min": min(ts), "ms_max": max(ts), "steps": n_steps,
                    "frames_per_s": B * T / ms * 1e3, "latent_tokens_per_s": B * Tp * 1024 / ms * 1e3,
                    "us_per_latent_token": ms * 1e3 / (B * Tp * 1024), "finite": bool(torch.isfinite(rec).all())})
        print(json.dumps(res[-1]), flush=True)
        del x, idx, rec
    return res


def attention(dev, reps=20):
    from omnitokenizer_b200 import _cabi
    _cabi.load()
    flush = torch.empty(64 * 1024 * 1024, device=dev)
    N, B = 1024, 1
    res = []
    for T in (17, 18, 33, 65, 129):
        M = B * T * N
        qkv = (torch.rand((M, 1536), generator=torch.Generator().manual_seed(T)) - 0.5).to(dev)
        planes = torch.empty((2, M, 512), dtype=torch.int16, device=dev)
        p = qkv.data_ptr()

        def call():
            _cabi.call("omt_attn_temporal", p, 1536, p + 2048, 1536, p + 4096, 1536, None, planes[0], planes[1], 512, B, T, N,
                       HEADS, 8.0, 1)
        for _ in range(3):
            call()
        ts = []
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); call(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        # the SM clock while the kernel runs: enqueue ~0.3 s of back-to-back launches, sample, then wait
        us = statistics.median(ts)
        for _ in range(max(1, int(3e5 / us))):
            call()
        clk = sm_clock_mhz()
        torch.cuda.synchronize()
        flop, nbytes = attn_work(B, T, N)
        t_hbm = nbytes / HBM_BPS * 1e6
        t_ffma = flop / (SMS * FFMA_LANES_PER_CLK_SM * 2 * clk * 1e6) * 1e6
        bound = "hbm" if t_hbm >= t_ffma else "ffma"
        res.append({"T_latent": T, "kernel": "attn_temporal_kernel<17>" if T <= 17 else "attn_temporal_long_kernel",
                    "us": us, "us_min": min(ts), "flop": flop, "bytes": nbytes, "sm_clock_mhz": clk,
                    "hbm_bound_us": t_hbm, "ffma_bound_us": t_ffma, "binding_bound": bound,
                    "fraction_of_bound": max(t_hbm, t_ffma) / us,
                    "achieved_tflops": flop / us * 1e-6, "achieved_tbps": nbytes / us * 1e-6})
        print(json.dumps(res[-1]), flush=True)
        del qkv, planes
    return res


def profile(dev, out):
    """one 257-frame encode -> decode step under torch.profiler (eager launches, so every kernel is listed)"""
    os.environ["OMT_CUDA_GRAPH"] = "0"
    m, W = model(dev)
    x = W.synthetic_input((1, 3, 257, 256, 256), 4257).to(dev)
    for _ in range(2):
        m.decode(m.encode(x, False), False)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile as tprof
    with tprof(activities=[ProfilerActivity.CUDA]) as prof:
        m.decode(m.encode(x, False), False)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            k = kernels.setdefault(e.name, [0, 0.0])
            k[0] += 1
            k[1] += e.device_time
    total = sum(v[1] for v in kernels.values())
    rows = sorted(({"kernel": n, "calls": c, "us": t, "share": t / total} for n, (c, t) in kernels.items()),
                  key=lambda r: -r["us"])
    res = {"clip": "1x257x256x256", "total_kernel_us": total, "kernels": rows}
    for r in rows[:15]:
        print(f"{r['share']:6.1%} {r['us']:10.1f} us {r['calls']:4d}x  {r['kernel'][:110]}")
    with open(os.path.join(out, "r03_long_clips_kernels.json"), "w") as f:
        json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_long.py measures on a GPU; no CUDA device found")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda:0")
    if a.profile:
        return profile(dev, a.out)
    res = {"card": card(), "steps": steps(dev, a.steps, a.warmup), "temporal_attention": attention(dev)}
    res["card_after"] = card()
    with open(os.path.join(a.out, "r03_long_clips.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
