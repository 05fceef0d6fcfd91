"""N>1 host logic on CPU: two gloo ranks, rank 0 scatters packed pyramids, each rank computes its
frames (the oracle stands in for the GPU engine), rank 0 gathers -- result must equal the
single-process result frame for frame."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_frames_partition():
    from of_dis_b200.sharding import shard_frames

    for n in (0, 1, 5, 8, 64, 67):
        for world in (1, 2, 3, 8):
            blocks = [shard_frames(n, world, r) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(blocks, blocks[1:]))
            sizes = [b - a for a, b in blocks]
            assert max(sizes) - min(sizes) <= 1
    assert shard_frames(64, 8, 3) == (24, 32)  # BASELINE configs[3]: 8 pairs per GPU


def _worker(rank, world, port, nfr, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    from of_dis_b200 import params, preprocess, sharding, synth
    from oracle import port_driver

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    prm = params.from_cli_numbers("3 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split())
    H, W = 64, 96

    def unpack(vec):
        """(img0 | img1) uint8 values stored as float32 -> PairPyramids"""
        a = vec[:H * W].reshape(H, W).astype(np.uint8)
        b = vec[H * W:].reshape(H, W).astype(np.uint8)
        return preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s)

    def compute(local):
        outs = [port_driver.port_run(unpack(v.numpy()), prm).reshape(-1) for v in local]
        return torch.from_numpy(np.stack(outs)) if outs else torch.empty((0, flow_elems))

    flow_elems = (H >> prm.sc_l) * (W >> prm.sc_l) * 2
    packed = None
    if rank == 0:
        rows = []
        for s in range(nfr):
            i0, i1, _ = synth.synthetic_pair(H, W, 1, seed=40 + s, amp=3.0)
            rows.append(np.concatenate([i0.reshape(-1), i1.reshape(-1)]).astype(np.float32))
        packed = torch.from_numpy(np.stack(rows))
    out = sharding.run_sharded(packed, nfr, 2 * H * W, flow_elems, compute, torch.device("cpu"))
    if rank == 0:
        ref = compute(packed)
        q.put(bool(torch.equal(out, ref)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("nfr", [5])
def test_scatter_compute_gather_world2_gloo(nfr):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000) + nfr
    procs = [ctx.Process(target=_worker, args=(r, 2, port, nfr, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    assert q.get(timeout=5) is True


def _nccl_worker(rank, world, port, nfr, io, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    from of_dis_b200 import api, params, preprocess, sharding, synth

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    prm = params.from_cli_numbers("3 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split())
    H, W = 120, 200
    stream = torch.cuda.Stream()
    eng = sharding.ShardedEngine(prm, nfr, W, H, io, dev, stream)
    host_in = host_out = None
    pairs = []
    if rank == 0:
        pairs = [synth.synthetic_pair(H, W, 1, seed=40 + s, amp=3.0)[:2] for s in range(nfr)]
        pyrs = [preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s) for a, b in pairs]
        if io == "cli":
            arr = np.stack([np.stack([a, b]).reshape(-1) for a, b in pairs])
        else:
            P, l = pyrs[0].imgpadding, prm.sc_l
            arr = np.stack([np.stack([p.i0[l][P:-P, P:-P], p.i1[l][P:-P, P:-P]]).reshape(-1) for p in pyrs])
        host_in = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
        host_out = torch.empty((nfr, eng.out_elems), dtype=torch.float32).pin_memory()
    for _ in range(2):  # second pass: graph replay
        eng.step(host_in, host_out)
    torch.cuda.synchronize()
    if rank == 0:
        # the same pairs on this GPU alone through the plain context
        ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr, device=0)
        for f, p in enumerate(pyrs):
            ctx.upload_pyramids(f, p)
        ctx.run(nfr)
        ok = True
        for f, p in enumerate(pyrs):
            lvl = ctx.get_flow(f, prm.sc_l)
            exp = preprocess.postprocess(lvl, prm.sc_l, p.padw, p.padh, W, H) if io == "cli" else lvl
            ok = ok and np.array_equal(host_out[f].numpy().view(np.uint32), np.ascontiguousarray(exp).reshape(-1).view(np.uint32))
        ctx.close()
        q.put(bool(ok))
    eng.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("io,nfr", [("cli", 6), ("ofclass", 5)])
def test_sharded_engine_on_nccl_with_the_real_engine(io, nfr):
    """BASELINE configs[3] in miniature on two GPUs: rank 0 scatters the pairs over NCCL, both ranks run the
    CUDA engine, rank 0 gathers -- bitwise equal to the single-GPU result (equal and unequal blocks)."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + (os.getpid() % 2000) + nfr
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, nfr, io, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    assert q.get(timeout=5) is True
