#!/usr/bin/env python
"""bench.py -- video-frames/s of OmniTokenizer_VQGAN encode -> codes -> decode (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg4|cfg5]
                    [--math f16x3|3xtf32|fp32] [--dump-outputs DIR]

Workload (config.workload): cfg3 = batch of 8 synthetic videos 17x256x256 (the configuration the
metric is quoted on, BASELINE.json configs[2]); under torchrun the batch is split over ranks
(strong scaling), each rank encodes its shard, ONE all-gather of code indices, decode of the shard.
cfg2 (64 images), cfg4 (4 videos 33x512x512: ranks beyond the batch idle, "replicas only beyond B") and
cfg5 (cfg3 in VAE mode: no codes, hence no collective) are BASELINE.json's other configurations.
A "step" is one pass of that path over the batch.  Prints ONE JSON line (rank 0).

--impl reference: the CPU baseline arm -- the oracle port of the reference's PyTorch path
(oracle/omni_oracle.py; the reference tree itself does not travel to the GPU box) on the host
threads, every step the SAME full batch and the same weights as the GPU arm.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg3": dict(shape=(8, 3, 17, 256, 256), desc="batch=8 videos 17x256x256 (UCF-shaped synthetic), VQVAE"),
    "cfg2": dict(shape=(64, 3, 256, 256), desc="batch=64 images 256x256, VQVAE"),
    "cfg4": dict(shape=(4, 3, 33, 512, 512), desc="batch=4 videos 33x512x512 (long-sequence stress), VQVAE"),
    "cfg5": dict(shape=(8, 3, 17, 256, 256), desc="batch=8 videos 17x256x256, VAE mode (use_vae, KL path, no codebook argmin)", vae=True),
}
# algorithmic FLOPs per batch (SURVEY.md 8d): enc+dec, un-padded dims
TFLOP = {"cfg3": 4.729, "cfg2": 7.500, "cfg4": 22.615, "cfg5": 4.724}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_ev = index, [], threading.Event()

    def run(self):
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_ev.wait(0.2)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=5)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = max([int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()] or [0])
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(self.rows)}


def make_model(dev, vae=False):
    import omnitokenizer_b200 as ob
    torch.manual_seed(0)
    m = ob.OmniTokenizer_VQGAN(ob.canonical_args(["--use_vae"] if vae else []))
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():      # move scales / LN gains off their ones init (SURVEY.md 8d)
        for n, p in m.named_parameters():
            if n.endswith(("q_scale", "k_scale", "gamma")) or (p.ndim == 1 and n.endswith(".weight")):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
    m.codebook._need_init = False
    return m.to(dev).eval()


def pick_cpu_threads(sd, x_small, vae=False):
    """The oracle's many small torch ops do not scale to every core of a 100+-core host (128 threads is
    ~30x SLOWER than 16 on the B200 box), so take the best of a short sweep; `cores` reports that count."""
    cores = os.cpu_count() or 1
    best, best_t = None, None
    for nt in sorted({min(c, cores) for c in (8, 16, 32, 64)}):
        torch.set_num_threads(nt)
        cpu_oracle_run(sd, x_small, vae=vae)
        dt, _, _ = cpu_oracle_run(sd, x_small, vae=vae)
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    torch.set_num_threads(best)
    return best


def cpu_oracle_run(sd, x, reps=1, vae=False):
    from oracle import omni_oracle as oo
    oo.USE_LIBRARY_OPS = True      # same torch library calls as the reference (conv3d PEG, SDPA)
    cfg = oo.Config(use_vae=vae)
    is_image = x.ndim == 4
    best = None
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            if vae:      # encode draws the posterior noise on the CPU generator (vae.py:16); decode takes 'b t h w c' (:313)
                idx = oo.encode(sd, cfg, x, noise=torch.randn((x.shape[0], 8) + ((1,) if is_image else (1 + (x.shape[2] - 1) // 4,))
                                                              + (x.shape[-2] // 8, x.shape[-1] // 8)))
                rec = oo.decode(sd, cfg, idx if is_image else idx.permute(0, 2, 3, 4, 1), is_image)
            else:
                idx = oo.encode(sd, cfg, x)
                rec = oo.decode(sd, cfg, idx, is_image)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return best, idx, rec


def near_tie_report(sd, x, idx_o, idx_g, z_gpu):
    """Explain every code index that differs from the oracle's.  Both sides compute the pre-quantisation vector z in fp32
    with different summation orders (|z_gpu - z_oracle| ~ 1e-6 after 12 layers); a change dz moves the distance gap
    between two codes e_a, e_b by 2 dz.(e_b - e_a).  An index may therefore differ only where the float64 gap at the
    oracle's z is no larger than that bound (+ a few fp32 ulps of the O(1) distances): a tie at fp32 resolution of z,
    which the reference's own GPU and CPU runs would break differently as well."""
    from oracle import omni_oracle as oo
    cfg = oo.Config()
    oo.USE_LIBRARY_OPS = True
    with torch.no_grad():
        h, _ = oo.encoder(sd, cfg, x)
    z = h.reshape(-1, h.shape[-1]).double()
    z = z / z.norm(dim=1, keepdim=True).clamp_min(1e-12)
    E = sd["codebook.embeddings"].double()
    ig, io = idx_g.reshape(-1), idx_o.reshape(-1)
    bad = (ig != io).nonzero().flatten()
    rep = []
    for i in bad.tolist():
        gap = float(((z[i] - E[ig[i]]) ** 2).sum() - ((z[i] - E[io[i]]) ** 2).sum())
        dz = z_gpu[i].double().cpu() - z[i]
        bound = float(2.0 * dz.norm() * (E[ig[i]] - E[io[i]]).norm()) + 4 * 1.2e-7
        rep.append({"row": i, "f64_distance_gap": float(f"{gap:.3e}"), "abs_dz": float(f"{float(dz.abs().max()):.3e}"),
                    "tie_bound": float(f"{bound:.3e}"), "within_bound": bool(abs(gap) <= bound)})
    return {"rows": rep[:8], "all_within_fp32_resolution_of_z": bool(all(r["within_bound"] for r in rep)),
            "max_abs_dz_all_rows": float(f"{float((z_gpu.double().cpu() - z).abs().max()):.3e}")}


def _ref_worker(threads, sd, vae, q_in, q_out):
    """one host worker of the reference arm: samples in, code indices (or VAE latents) out"""
    torch.set_num_threads(threads)
    while True:
        item = q_in.get()
        if item is None:
            return
        i, x = item
        _, idx, rec = cpu_oracle_run(sd, x, vae=vae)
        q_out.put((i, idx, float(rec.double().sum())))


def run_reference(args):
    """CPU arm: the oracle port of the reference path on the host cores, the FULL batch of the workload every step with the GPU
    arm's weights; rank 0 only.  One torch process does not scale past ~32 threads on this op mix, so the samples of a batch
    are spread over host_cores // best_threads worker processes (all the host threads the port can use)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch.multiprocessing as mp
    wl = dict(WORKLOADS[args.workload])
    if os.environ.get("OMT_BENCH_BATCH"):        # diagnostic (same knob as the GPU arm): a smaller batch of the workload
        wl["shape"] = (int(os.environ["OMT_BENCH_BATCH"]),) + wl["shape"][1:]
    vae = bool(wl.get("vae"))
    m = make_model(torch.device("cpu"), vae)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    shape = wl["shape"]
    B = shape[0]
    x = torch.rand(shape, generator=torch.Generator().manual_seed(1234)) - 0.5
    threads = pick_cpu_threads(sd, x[:1], vae)
    host = os.cpu_count() or 1
    workers = max(1, min(B, host // threads, int(os.environ.get("OMT_REF_WORKERS", "64"))))
    frames = B * (shape[2] if len(shape) == 5 else 1)
    ctx = mp.get_context("spawn")
    q_in, q_out = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=_ref_worker, args=(threads, sd, vae, q_in, q_out), daemon=True) for _ in range(workers)]
    for p in procs:
        p.start()
    per = max(1, B // (workers * 4))              # samples per work item
    items = [x[i:i + per] for i in range(0, B, per)]

    def step(conc):
        """one pass over the batch with at most `conc` work items in flight (= `conc` busy worker processes)"""
        sent, done = 0, 0
        while done < len(items):
            while sent < len(items) and sent - done < conc:
                q_in.put((sent, items[sent]))
                sent += 1
            q_out.get(timeout=1800)
            done += 1

    # how many workers to keep busy: more processes share the host's memory bandwidth, so calibrate once (untimed; this is
    # also the warm pass) and keep the fastest setting
    best_c, best_t = workers, None
    for c in sorted({1, max(1, workers // 2), workers}):
        t0 = time.perf_counter()
        step(c)
        t = time.perf_counter() - t0
        if best_t is None or t < best_t:
            best_c, best_t = c, t
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(best_c)
    dt = time.perf_counter() - t0
    for _ in procs:
        q_in.put(None)
    for p in procs:
        p.join(timeout=30)
    v = frames * args.steps / dt
    sample = (f"the full batch ({'x'.join(map(str, shape))}) every step, same weights as the GPU arm; {best_c} busy worker processes "
              f"(best of 1 / {max(1, workers // 2)} / {workers} on this host) x {threads} torch threads (best of a sweep), {per} sample(s) "
              f"per work item; the calibration passes double as warm-up")
    print(json.dumps({
        "impl": "reference", "metric": "video_frames_per_sec_encode_decode", "value": round(v, 3), "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 2),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload + ": " + wl["desc"], "global_batch": B, "frames": frames},
        "cpu_baseline": {"value": round(v, 3), "unit": "frames/s", "cores": best_c * threads, "host_cores": host, "kind": "port",
                         "sample": sample},
        "e2e": {"value": round(v, 3), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def _event_time(fn, flush, reps=10):
    """median CUDA-event time of fn() in ms, L2 flushed before every repetition"""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for i in range(reps + 2):
        flush.add_(1.0)
        if i >= 2:
            evs[i - 2][0].record()
        fn()
        if i >= 2:
            evs[i - 2][1].record()
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in evs)[reps // 2]


def time_dominant_kernel(m, M, dev, flush):
    """CUDA-event timing of the dominant kernel (FeedForward first Linear + GEGLU, 16 launches per
    enc+dec) alone, same shapes as in the step: achieved algorithmic TFLOP/s."""
    from omnitokenizer_b200 import _cabi
    eng = m.engine()
    lyr = eng.enc_spatial["layers"][0]
    ws = eng._workspace(M)
    if eng.planes:
        x = torch.randn(M, eng.C, device=dev)
        eng._ln_h(x, ws.XNp, lyr["ff_g"], lyr["ff_b"], M)
        fn = lambda: eng._linear_h(ws.XNp, lyr["ff1"], M, U=ws.Up, epi=_cabi.EPI_GEGLU)
    else:
        ws.XN.normal_()
        fn = lambda: eng._linear(ws.XN, eng.C, lyr["ff1"], ws.U, eng.ku, M, epi=_cabi.EPI_GEGLU)
    ms = _event_time(fn, flush)
    flops = 2.0 * M * (2 * eng.inner) * eng.C          # un-padded algorithmic FLOPs of Linear(512 -> 2730)
    return ms, flops


def time_vq_lookup(m, M, dev, flush):
    """The codebook nearest-neighbour search alone (BASELINE.json's "VQ-lookup HBM GB/s"): algorithmic bytes =
    z (M x 8 fp32) + the 8192 x 8 table + int64 indices; FLOPs = 2 * 8 * n_codes per row (SURVEY.md 8d)."""
    from omnitokenizer_b200 import _cabi
    eng = m.engine()
    ws = eng._workspace(M)
    z = torch.nn.functional.normalize(torch.randn(M, 8, device=dev), dim=1)

    def fn():
        ws.counts.zero_()
        _cabi.call("omt_vq_search", z, eng.E, eng.e2, M, eng.n_codes, ws.idx, ws.counts)
    ms = _event_time(fn, flush)
    bytes_ = M * 8 * 4 + eng.n_codes * 8 * 4 + M * 8
    flops = 2.0 * 8 * eng.n_codes * M
    sms, _, _ = _cabi.device_info()
    fp32_peak = sms * 128 * 2 * 1.965e9 / 1e12          # FFMA lanes x 2 flop x max SM clock
    return {"us": round(ms * 1e3, 1), "hbm_gbs": round(bytes_ / (ms * 1e-3) / 1e9, 2), "algorithmic_bytes": bytes_,
            "fma_tflops": round(flops / (ms * 1e-3) / 1e12, 2), "fp32_peak_tflops": round(fp32_peak, 1),
            "frac_fma": round(flops / (ms * 1e-3) / 1e12 / fp32_peak, 3),
            "note": "FP32-FMA-bound (3.3 kFLOP/B): the HBM figure is reported because the metric names it, the FMA fraction binds"}


DUMP_SAMPLE = 1 << 21      # elements: a larger output is dumped as this many seeded picks (<= 32 MB with their positions)


def write_outputs(dirname, arrays):
    """--dump-outputs: every tensor as DIR/<name>.npy, float32 (integer code indices as float64, exact).  A tensor of more
    than DUMP_SAMPLE elements is written as DUMP_SAMPLE elements at flat (C-order) positions drawn with a fixed seed; the
    positions go to DIR/<name>_index.npy.  Two arrays stay within 64 MB."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        if t is None:
            continue
        if t.numel() > DUMP_SAMPLE:
            pos = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            np.save(os.path.join(dirname, name + "_index.npy"), pos.double().numpy())
            t = t.reshape(-1)[pos.to(t.device)]
        t = t.detach().cpu()
        np.save(os.path.join(dirname, name + ".npy"), t.numpy().astype(np.float32 if t.is_floating_point() else np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--math", default=None, help="f16x3 | 3xtf32 | fp32 (default: OMT_MATH or the engine default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (code indices "
                    "or VAE latents, and the reconstruction) as DIR/<name>.npy; inputs and weights are seeded, so two builds "
                    "can be compared output for output (see write_outputs).  Under torchrun rank 0 writes its own shard")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    if args.impl == "reference":
        return run_reference(args)
    if args.math:
        os.environ["OMT_MATH"] = args.math
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    import omnitokenizer_b200 as ob
    from omnitokenizer_b200 import _cabi, dist as od
    from omnitokenizer_b200.engine import default_math

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = dict(WORKLOADS[args.workload])
    if os.environ.get("OMT_BENCH_BATCH"):        # diagnostic: per-GPU load of an N-GPU strong-scaling run on one GPU
        wl["shape"] = (int(os.environ["OMT_BENCH_BATCH"]),) + wl["shape"][1:]
        wl["desc"] += f" [batch overridden to {wl['shape'][0]}]"
    shape = wl["shape"]
    B = shape[0]
    is_image = len(shape) == 4
    vae = bool(wl.get("vae"))
    frames_per_sample = 1 if is_image else shape[2]
    s, e = od.shard_bounds(B, rank, world)
    x_full = torch.rand(shape, generator=torch.Generator().manual_seed(1234)) - 0.5
    x_host = x_full[s:e].contiguous().pin_memory()
    x_dev = x_host.to(dev)
    m = make_model(dev, vae)
    m.prepare()
    flush = torch.zeros(64 * 1024 * 1024, device=dev)      # 256 MiB > 126 MB L2
    gathered = {}

    def step(x, u8=False):
        """One pass of the path; returns what its caller receives: (code indices, or VAE latents; reconstruction).
        u8: the reconstruction leaves as uint8 frames (vqgan_eval.py's clamp / 255 / byte conversion fused into the last kernel)"""
        dec = (lambda c: m.decode_u8(c, is_image)) if u8 else (lambda c: m.decode(c, is_image))
        if vae:      # KL path: no code indices, hence no collective; decode takes the channels-last latent (omnitokenizer.py:313)
            if x.shape[0] == 0:
                return None, None
            z = m.encode(x, is_image)
            return z, dec(z if is_image else z.permute(0, 2, 3, 4, 1))
        codes = m.encode(x, is_image)                       # an empty shard (B < world) returns an empty, right-shaped tensor
        pending = None
        if world > 1 and not os.environ.get("OMT_BENCH_NO_GATHER"):
            pending = od.all_gather_codes_async(codes, B)   # the single collective, overlapped with the local decode
        rec = None if x.shape[0] == 0 else dec(codes)
        if pending is not None:
            gathered["codes"] = pending.wait()              # every rank now holds the full (B,T',h,w) index tensor
        return codes, rec

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(x_dev)
    barrier()
    # ---- device-timed region: K steps, L2 flushed (untimed) between steps ----
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    n0 = _cabi.launch_count
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in evs:
        out = None                   # release the previous step's outputs first: the allocator reuses their blocks
        flush.add_(1.0)
        a.record()
        out = step(x_dev)
        b.record()
    barrier()
    launches = _cabi.launch_count - n0
    t_ms = sum(a.elapsed_time(b) for a, b in evs)
    if args.dump_outputs and rank == 0:          # codes / latents and reconstruction of the same samples: rank 0's shard
        first, rec = out
        write_outputs(args.dump_outputs, {"latents" if vae else "codes": first, "reconstruction": rec})
    out = None
    # the gathered codes of the last step must be the single-GPU codes of the full batch (checked once, untimed)
    gather_ok = None
    if world > 1 and not vae and "codes" in gathered:
        ok = torch.ones(1, device=dev)
        if rank == 0:
            full = m.encode(x_full.to(dev), is_image)
            ok[0] = float(torch.equal(full, gathered["codes"]))
        dist.broadcast(ok, 0)
        gather_ok = bool(ok.item())
    # ---- e2e: pinned host input -> H2D -> encode -> decode -> D2H of the reconstruction, every step ----
    # Serving-style pipeline through the public API: the H2D copy of step i+1 and the D2H copy of step i-1 run on
    # their own streams (separate DMA engines) while step i computes; all copies are inside the timed region
    # (one event pair around the K steps, the end event waits for the last D2H).
    out_host = [torch.empty((e - s,) + shape[1:], dtype=torch.float32).pin_memory() for _ in range(2)]
    out_host_u8 = [torch.empty((e - s, 1 if is_image else shape[2], shape[-2], shape[-1], shape[1]), dtype=torch.uint8).pin_memory()
                   for _ in range(2)]
    e2e_steps = args.steps
    main = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    xd = [torch.empty_like(x_dev) for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_used = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    keep = []

    def e2e_run(nsteps, u8=False):
        oh = out_host_u8 if u8 else out_host
        for i in range(nsteps):
            sl = i & 1
            with torch.cuda.stream(s_in):
                if i >= 2:
                    s_in.wait_event(ev_used[sl])            # step i-2 has consumed this input buffer
                xd[sl].copy_(x_host, non_blocking=True)
                ev_in[sl].record(s_in)
            main.wait_event(ev_in[sl])
            rec = step(xd[sl], u8)[1]
            ev_used[sl].record(main)
            if rec is not None:
                rec.record_stream(s_out)                     # allocator: the tensor is still read by the copy stream
                keep.append(rec)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_used[sl])
                    oh[sl].copy_(rec, non_blocking=True)         # oh[sl] of step i-2 was drained on this same stream
                    ev_out[sl].record(s_out)
            if len(keep) > 3:
                keep.pop(0)
        for sl in range(2):
            main.wait_event(ev_out[sl])                      # the end event below is ordered after the last D2H

    barrier()
    # link speed of THIS box (untimed, explains e2e - value: boxes differ by several x in host copy bandwidth)
    c_a, c_b, c_c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    c_a.record(main)
    xd[0].copy_(x_host, non_blocking=True)
    c_b.record(main)
    out_host[0].copy_(xd[0], non_blocking=True)
    c_c.record(main)
    barrier()
    link = {"h2d_GBps": round(x_host.numel() * 4 / c_a.elapsed_time(c_b) / 1e6, 1) if x_host.numel() else None,
            "d2h_GBps": round(x_host.numel() * 4 / c_b.elapsed_time(c_c) / 1e6, 1) if x_host.numel() else None}
    e2e_run(6)                                               # warm the pipeline (untimed): the caching allocator needs a few
                                                             # steps until the per-step output tensors stop costing a cudaMalloc
    barrier()
    flush.add_(1.0)
    t_a, t_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_a.record(main)
    e2e_run(e2e_steps)
    t_b.record(main)
    barrier()
    s_in.synchronize(); s_out.synchronize()
    clocks = sampler.stop() if sampler else None
    t2_ms = t_a.elapsed_time(t_b)
    # same pipeline with the uint8 epilogue: D2H is a quarter of the bytes (what vqgan_eval.py's metrics consume)
    e2e_run(4, u8=True)
    barrier()
    flush.add_(1.0)
    u_a, u_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u_a.record(main)
    e2e_run(e2e_steps, u8=True)
    u_b.record(main)
    barrier()
    s_in.synchronize(); s_out.synchronize()
    t3_ms = u_a.elapsed_time(u_b)
    tt = torch.tensor([t_ms, t2_ms, t3_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_ms, t2_ms, t3_ms = tt.tolist()
    frames = B * frames_per_sample
    value = frames * args.steps / (t_ms / 1e3)
    e2e = frames * e2e_steps / (t2_ms / 1e3)

    if rank == 0:
        pk, pk_src = peaks()
        h, w = shape[-2] // 8, shape[-1] // 8
        Tp = 1 if is_image else 1 + (shape[2] - 1) // 4
        M_local = (e - s) * Tp * h * w
        k_ms, k_flops = time_dominant_kernel(m, M_local, dev, flush)
        math = default_math()
        tf32_peak = pk["bf16_tflops"] / 2.0
        achieved = k_flops / (k_ms * 1e-3) / 1e12
        traffic = None
        try:      # dram__bytes_read+write of this launch from the committed `ncu --set full` capture (cfg-3, N=1)
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_ff1_traffic.json")))
            if world == 1 and args.workload in ("cfg3", "cfg5") and not os.environ.get("OMT_BENCH_BATCH") and math in tj:
                traffic = tj[math]["dram_bytes"]
        except Exception:
            pass
        kname = {"3xtf32": "gemm_tc2_kernel", "f16x3": "gemm_f16_kernel", "fp32": "gemm_fp32_kernel"}[math]
        own = {"3xtf32": "3xTF32 issues 3 tf32 MMAs per product: its own ceiling is 1/3 of this",
               "f16x3": "f16x3 issues 3 kind::f16 MMAs (2x the tf32 rate) per product: its own ceiling is 2/3 of this",
               "fp32": "CUDA-core FFMA kernel: bounded by the fp32 pipe, not the tensor pipe"}[math]
        roof = {"bound": "tensor", "kernel": f"{kname}[{math}] FF1+GEGLU M={M_local} N=2730 K=512",
                "achieved": round(achieved, 2), "peak": round(tf32_peak, 1), "unit": "TFLOP/s",
                "frac": round(achieved / tf32_peak, 4), "traffic": traffic,
                "algorithmic_bytes": int(M_local * 512 * 4 + 2 * 2730 * 512 * 4 + M_local * 1365 * 4),
                "ms_per_launch": round(k_ms, 4),
                "peak_note": f"tf32 dense = 0.5 x {pk_src} bf16 burst {pk['bf16_tflops']} TF/s; FLOPs are algorithmic fp32 "
                             f"(2MNK); {own}",
                "whole_path": {"tflop_per_batch": TFLOP[args.workload],
                               "achieved_tflops": round(TFLOP[args.workload] * args.steps / (t_ms / 1e3), 2)}}
        line = {
            "metric": "video_frames_per_sec_encode_decode", "value": round(value, 2), "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t_ms / args.steps, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload + ": " + wl["desc"], "global_batch": B, "frames": frames,
                       "parallelism": (f"batch-shard dp{world}, no collective (VAE latents stay local)" if vae else
                                       f"batch-shard dp{world}, 1 all-gather of code indices")
                                      + (f"; {world - B} ranks idle (replicas only beyond B)" if world > B else ""),
                       "math": math,
                       "l2": "256 MiB flush between timed steps (untimed); activations >> L2"},
            "e2e": {"value": round(e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": out_host[0].numel() * 4, "ms_per_step": round(t2_ms / e2e_steps, 3),
                    "steps": e2e_steps, "pipeline": "H2D / compute / D2H of consecutive steps overlap on 3 streams",
                    "host_link": link,
                    "u8": {"value": round(frames * e2e_steps / (t3_ms / 1e3), 2), "unit": "frames/s",
                           "d2h_bytes_per_step": out_host_u8[0].numel(), "ms_per_step": round(t3_ms / e2e_steps, 3),
                           "what": "reconstruction fetched as uint8 frames (decode_u8: clamp(x+0.5,0,1)*255 fused into un-patchify)"}},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof,
        }
        if gather_ok is not None:
            line["gathered_codes_equal_single_gpu"] = gather_ok
        if not vae and M_local > 0:
            line["vq_lookup"] = time_vq_lookup(m, M_local, dev, flush)
        if not args.no_cpu_baseline and world == 1:
            sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
            xs = x_full[:1]
            cores = pick_cpu_threads(sd, xs, vae)
            cpu_oracle_run(sd, xs, vae=vae)                     # warm-up
            torch.manual_seed(7)
            dt, idx_o, rec_o = cpu_oracle_run(sd, xs, reps=1, vae=vae)
            torch.manual_seed(7)                                # VAE: the same CPU-generator noise draw on both sides
            idx_g = m.encode(xs.to(dev), is_image)
            rec_g = m.decode(idx_g if (is_image or not vae) else idx_g.permute(0, 2, 3, 4, 1), is_image)
            line["cpu_baseline"] = {"value": round(frames_per_sample / dt, 3), "unit": "frames/s", "cores": cores, "host_cores": os.cpu_count(),
                                    "kind": "port",
                                    "sample": f"1 of {B} samples ({'x'.join(map(str, xs.shape))}), one pass after warm-up"}
            if vae:
                line["parity"] = {"max_abs_latent_err": float((idx_g.cpu() - idx_o).abs().max()),
                                  "max_abs_pixel_err": float((rec_g.cpu() - rec_o).abs().max())}
            else:
                mism = int((idx_g.cpu() != idx_o).sum())
                line["parity"] = {"idx_mismatch": mism, "n_idx": idx_o.numel(),
                                  "max_abs_pixel_err": float((rec_g.cpu() - rec_o).abs().max())}
                if mism:     # explain every differing index, and compare the decoder on the oracle's own indices
                    eng = m.engine()
                    z_gpu = eng.z_view(eng._workspace(idx_o.numel())).clone()       # z of the encode() just above
                    line["parity"]["near_tie"] = near_tie_report(sd, xs, idx_o, idx_g.cpu(), z_gpu)
                    line["parity"]["max_abs_pixel_err_same_codes"] = float(
                        (m.decode(idx_o.to(dev), is_image).cpu() - rec_o).abs().max())
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
