"""The peer-memory observation path (K2 of every rank stores into rank 0's buffer; one-way stream-ordered
completion flags instead of a per-step collective) returns exactly what the NCCL gather and a single-process run
return.  Two variants: two ranks on two GPUs over NVLink (skipped with < 2 GPUs), and two ranks sharing ONE GPU
(CUDA IPC between processes, gloo for the set-up exchange) so that the path is exercised on any box."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, total, steps, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from miniworld_b200.dist import ShardedMiniWorld
    acts_all = np.random.default_rng(5).integers(0, 3, size=(steps, total), dtype=np.int32)
    results = {}
    for mode in ("nccl", "peer"):
        env = ShardedMiniWorld("MiniWorld-FourRooms-v0", total, dist=dist, device=rank)
        env.reset(1000)
        ok = mode == "nccl" or env.enable_peer_obs()
        frames = []
        for t in range(steps):
            mine = torch.as_tensor(acts_all[t, env.start:env.start + env.count], device="cuda")
            if mode == "peer" and ok:
                obs = env.step_peer(mine)
            else:
                obs = env.step(mine)[0]
            torch.cuda.synchronize()
            dist.barrier()
            if rank == 0:
                frames.append(obs.cpu().numpy().copy())
        results[mode] = (ok, frames)
        env.close()
    if rank == 0:
        q.put({k: (v[0], np.stack(v[1])) for k, v in results.items()})
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("total,steps", [(64, 5), (4096, 2)])
def test_peer_observation_buffer_equals_gather(libmwb_path, total, steps):
    """total = 64: frames split over several blocks, 8-byte row-segment peer stores; total = 4096 (2048 per
    rank): one block per frame, whole-frame shared-memory stage written to the peer as 16-byte stores."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, total, steps, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert res["peer"][0], "CUDA IPC peer buffer could not be established"
    assert np.array_equal(res["nccl"][1], res["peer"][1])
    from miniworld_b200.batched import BatchedMiniWorld
    env = BatchedMiniWorld("MiniWorld-FourRooms-v0", total)
    env.reset(seed=1000)
    acts_all = np.random.default_rng(5).integers(0, 3, size=(steps, total), dtype=np.int32)
    for t in range(steps):
        obs = env.step(torch.as_tensor(acts_all[t], device="cuda"))[0]
        assert np.array_equal(obs.cpu().numpy(), res["peer"][1][t])
    env.close()


def _worker_one_gpu(rank, world, port, total, steps, q, flag_mode, level="MiniWorld-FourRooms-v0", size=(80, 60), staged=False):
    """Two processes on cuda:0: the peer buffer crosses a process boundary (CUDA IPC), not a GPU boundary."""
    sys.path.insert(0, ROOT)
    os.environ["MWB_FLAG_MODE"] = flag_mode
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from miniworld_b200.dist import ShardedMiniWorld
    acts_all = np.random.default_rng(5).integers(0, 3, size=(steps, total), dtype=np.int32)
    env = ShardedMiniWorld(level, total, dist=dist, device=0, obs_width=size[0], obs_height=size[1])
    acts_all = np.random.default_rng(5).integers(0, env.local.action_space.n, size=(steps, total), dtype=np.int32)
    env.reset(1000)
    ok = env.enable_peer_obs()
    frames = []
    if ok:
        if staged:
            env.local.engine.set_obs_peer(True)   # stage frames as for another GPU although the destination is local
        for t in range(steps):              # no synchronisation between the ranks inside the loop: the flags order it
            obs = env.step_peer(torch.as_tensor(acts_all[t, env.start:env.start + env.count], device="cuda"))
            if rank == 0:
                frames.append(obs.clone())  # stream-ordered after the completion waits
        torch.cuda.synchronize()
    mode = env._lib.mwb_flag_mode() if ok else -1
    env.close()
    if rank == 0:
        q.put((ok, mode, np.stack([f.cpu().numpy() for f in frames]) if ok else None))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("flag_mode", ["memop", "kernel"])
@pytest.mark.parametrize("total,steps", [(64, 6), (2048, 4)])
def test_peer_observation_buffer_two_processes_one_gpu(libmwb_path, total, steps, flag_mode):
    import torch
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker_one_gpu, args=(r, 2, port, total, steps, q, flag_mode)) for r in range(2)]
    for p in procs:
        p.start()
    ok, mode, frames = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert ok, "CUDA IPC peer buffer could not be established"
    assert mode == (1 if flag_mode == "kernel" else mode)      # "memop" may fall back to kernels on an old driver
    from miniworld_b200.batched import BatchedMiniWorld
    env = BatchedMiniWorld("MiniWorld-FourRooms-v0", total)
    env.reset(seed=1000)
    acts_all = np.random.default_rng(5).integers(0, 3, size=(steps, total), dtype=np.int32)
    for t in range(steps):
        obs = env.step(torch.as_tensor(acts_all[t], device="cuda"))[0]
        assert np.array_equal(obs.cpu().numpy(), frames[t]), "step %d" % t
    env.close()


@pytest.mark.parametrize("level,size,total", [("MiniWorld-FourRooms-v0", (80, 60), 64), ("MiniWorld-FourRooms-v0", (80, 60), 2048),
                                              ("MiniWorld-PickupObjects-v0", (160, 120), 24)])
def test_staged_peer_stores_on_one_gpu(libmwb_path, level, size, total):
    """The store shape K2 uses towards another GPU -- the frame, or the block's band of whole half-tile rows when a
    frame is cut into several blocks (80x60 at small N: 3-row bands; 160x120: 8-row bands), collected in shared memory
    and written as address-ordered 16-byte stores -- forced on for a local destination, so that a one-GPU box
    exercises it: two ranks on cuda:0 must reproduce the single-process frames."""
    import torch
    import torch.multiprocessing as mp
    steps = 4
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29750 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker_one_gpu, args=(r, 2, port, total, steps, q, "memop", level, size, True)) for r in range(2)]
    for p in procs:
        p.start()
    ok, mode, frames = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert ok
    from miniworld_b200.batched import BatchedMiniWorld
    env = BatchedMiniWorld(level, total, obs_width=size[0], obs_height=size[1])
    env.reset(seed=1000)
    acts_all = np.random.default_rng(5).integers(0, env.action_space.n, size=(steps, total), dtype=np.int32)
    for t in range(steps):
        obs = env.step(torch.as_tensor(acts_all[t], device="cuda"))[0]
        assert np.array_equal(obs.cpu().numpy(), frames[t]), "step %d" % t
    env.close()
