"""On-hardware multi-GPU correctness (SURVEY.md section 4 item 4): 2 NCCL ranks, batch-sharded encode -> ONE all-gather of
the code indices -> local decode; the gathered codes equal the single-GPU codes of the full batch bit for bit and each
rank's decoded shard equals the rows of the single-GPU decode.  Skipped on a box with fewer than 2 GPUs."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, q):
    import torch.distributed as dist
    import omnitokenizer_b200 as ob
    from omnitokenizer_b200 import dist as od
    from oracle import omni_oracle as oo
    from oracle import weights as W
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    cfg = oo.Config()
    sd = W.make_state_dict(cfg, 3)
    m = ob.OmniTokenizer_VQGAN(ob.canonical_args())
    m.load_state_dict(sd, strict=False)
    m.codebook._need_init = False
    m = m.to(dev).eval()
    res = {}
    for B in (3, 1):                                  # ragged split (2 + 1) and world > B (one rank idles)
        x = W.synthetic_input((B, 3, 5, 64, 64), 17)
        allc, local = od.encode_sharded(m, x, False)
        full = m.encode(x.to(dev), False)
        s, e = od.shard_bounds(B, rank, world)
        ok = torch.equal(allc, full) and torch.equal(local, full[s:e])
        if e > s:
            ok = ok and torch.equal(m.decode(local, False), m.decode(full, False)[s:e])
        res[B] = bool(ok)
    q.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_equals_single_gpu_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
    assert all(all(r.values()) for _, r in res), res
