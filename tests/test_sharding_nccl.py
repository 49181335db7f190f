"""The multi-GPU path with the real engine: world size 2, NCCL, one process per GPU.  Each rank runs
Engine.count_reads on its catalog partition and the per-read results are gathered on rank 0 (sharding.py); the
gathered rows must equal the CPU port's.  Needs two GPUs: skipped on a one-GPU box."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, q):
    import torch
    import torch.distributed as dist

    import strkit_b200 as sb
    from strkit_b200 import synth

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        batch = synth.generate(synth.CONFIGS[2], 3000, seed=5).to_host()   # every rank: the same catalog description
        eng = sb.Engine(device=rank)
        params = sb.RepeatCountParams("repalign", 50, 3, 1)
        uploaded = []

        def compute(b):
            uploaded.append(b.arena.nbytes)
            return eng.count_reads(b.to_nibble(), params)

        res = sb.count_reads_sharded(batch, compute, rank, world)
        assert uploaded and uploaded[0] < 0.7 * batch.arena.nbytes     # a rank holds its partition's bytes only
        if rank == 0:
            q.put(res)
        else:
            assert res is None
        eng.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_sharded_engine_nccl_world2(oracle):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from strkit_b200 import synth

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    sharded = q.get(timeout=500)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    b = synth.generate(synth.CONFIGS[2], 3000, seed=5).to_host()
    oracle.set_simd(True)
    want, _ = oracle.count_loci(b.arena, b.seq_off, b.lens, b.est_cn, b.read_begin, b.motif_off, b.motif_len, n_threads=16)
    oracle.set_simd(False)
    assert sharded.shape == want.shape and np.array_equal(sharded, want)
