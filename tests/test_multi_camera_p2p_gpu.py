"""Config 5 over peer memory (reid.match_cameras_p2p): two processes (one camera each), galleries published through CUDA
IPC handles and read IN PLACE by the distance GEMM's operand conversion of the rank that owns the camera pair.  On a box
with >= 2 GPUs the two ranks sit on two GPUs and the read crosses NVLink (`gpurun --gpus 2`); on a single-GPU box both
ranks share device 0 -- the same IPC / mapping / barrier-before-free path, minus the link."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, q, golden_path):
    import torch
    import torch.distributed as dist
    from object_detection_tracking_b200 import reid
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)       # host-side channel for handles / metadata
    g = np.load(golden_path)
    name = ("c1", "c2")[rank]
    cam = {int(t): (g["%s_t%d_rows" % (name, t)], g["%s_t%d_feat" % (name, t)]) for t in g[name + "_ids"]}
    res = reid.match_cameras_p2p(cam, device=dev, frame_offsets={(0, 1): 4}, tol=50,
                                 ignore_pairs={(0, 1): ([int(v) for v in g["ignore0"]], [int(v) for v in g["ignore1"]])})
    q.put((rank, {k: v for k, v in res.items()}))
    dist.barrier()
    dist.destroy_process_group()


def test_two_cameras_peer_memory(golden_dir):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    path = os.path.join(golden_dir, "reid_pairs.npz")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, path)) for r in range(2)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    g = np.load(path)
    ids1, ids2 = sorted(int(t) for t in g["c1_ids"]), sorted(int(t) for t in g["c2_ids"])
    ref = [(ids1[i], ids2[int(j)]) for i, j in enumerate(g["x"]) if j >= 0]
    assert out[0] == {(0, 1): ref} and out[1] == {}


def _worker_allgather(rank, world, port, q, golden_path):
    import torch
    import torch.distributed as dist
    from object_detection_tracking_b200 import reid
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g = np.load(golden_path)
    name = ("c1", "c2")[rank]
    ids = sorted(int(t) for t in g[name + "_ids"])
    feats = [g["%s_t%d_feat" % (name, t)] for t in ids]
    rows_cap = 4096
    gallery = torch.zeros((rows_cap, feats[0].shape[1]), dtype=torch.float32, device="cuda")
    allf = np.concatenate(feats, 0)
    gallery[:len(allf)] = torch.from_numpy(allf).cuda()
    meta = {t: (g["%s_t%d_rows" % (name, t)], len(f)) for t, f in zip(ids, feats)}
    timing = {}
    res = reid.match_cameras_allgather(meta, gallery, rows_cap, device=rank, frame_offsets={(0, 1): 4}, tol=50, timing=timing,
                                       ignore_pairs={(0, 1): ([int(v) for v in g["ignore0"]], [int(v) for v in g["ignore1"]])})
    q.put((rank, dict(res), timing))
    dist.barrier()
    dist.destroy_process_group()


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


# NCCL cannot place two ranks on one GPU; on a single-GPU machine the same pair-cost kernels are covered by the p2p form
# above and tests/test_widen_gpu.py.
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs: NCCL cannot place two ranks on one GPU")
def test_two_cameras_nccl_allgather_device_resident(golden_dir):
    """Device-resident form of config 5: galleries in HBM, ONE all_gather_into_tensor over NCCL, pair cost on the
    gathered device pointers; ids pinned by the reference-generated reid_pairs.npz (multi_video_reid.py:260-324,512)."""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    path = os.path.join(golden_dir, "reid_pairs.npz")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker_allgather, args=(r, 2, port, q, path)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    out = {r: m for r, m, _ in got}
    g = np.load(path)
    ids1, ids2 = sorted(int(t) for t in g["c1_ids"]), sorted(int(t) for t in g["c2_ids"])
    ref = [(ids1[i], ids2[int(j)]) for i, j in enumerate(g["x"]) if j >= 0]
    assert out[0] == {(0, 1): ref} and out[1] == {}
    assert all(t["allgather_ms"] > 0 for _, _, t in got)
