"""Landmark-sharded window solve (SURVEY.md 8e, BASELINE cfg 4) on the GPUs of one box vs the single-process CPU oracle.

One process per GPU (torch.multiprocessing spawn, NCCL rendezvous on 127.0.0.1); every rank uploads the camera-side problem and ITS
block of landmarks, the ranks solve together, rank 0 merges the landmark results and compares with the oracle's solution of the
whole window: same LM trajectory, solution within 1e-6 relative.  Skipped on boxes with fewer than 2 GPUs; the same sharded code path
runs with two ranks on ONE GPU in tests/test_ba_gpu.py (peer-memory transport, in-process)."""
import copy
import ctypes as C
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _worker(rank, world, port, cfg, transport, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
        import oracle
        from datagen import synth_ba
        from ic_gvins_b200.ba import WindowSolver, connect_shards, shard_window
        from tests import oracle_api as oa
        olib = C.CDLL(oracle.build())
        oa.declare(olib)
        oa.declare_ba(olib)
        K, L, nwin = cfg
        probs = []
        for w in range(nwin):
            p, _ = synth_ba.make_window(lambda *a: oa.preintegrate(olib, *a), K=K, L=L, seed=2040 + w, with_marg=(w % 2 == 1))
            if w % 3 == 2:
                p["ext_const"], p["td_const"] = 1, 1
            probs.append(p)
        shards = [shard_window(p, rank, world) for p in probs]
        s = WindowSolver(max_windows=nwin, max_K=K, max_L=max(1, max(sh["L"] for sh in shards)), max_F=max(1, max(sh["F"] for sh in shards)),
                         max_gnss=16, max_marg_r=64, device=rank)
        connect_shards(s, rank, world, transport, dist)
        summ = s.solve(shards, 20)
        parts = [None] * world
        dist.all_gather_object(parts, [(sh["lm_lo"], sh["lm_hi"], sh["invdepth"], sh["pose"], sh["mix"], sh["ext"]) for sh in shards])
        if rank == 0:
            rel = lambda a, b: float(np.abs(a - b).max() / max(1e-300, np.abs(b).max()))
            for w, p in enumerate(probs):
                full = copy.deepcopy(p)
                for r in range(world):
                    lo, hi, rho, pose, mix, ext = parts[r][w]
                    full["invdepth"][lo:hi] = rho
                    assert np.array_equal(pose, parts[0][w][3]) and np.array_equal(mix, parts[0][w][4]) and np.array_equal(ext, parts[0][w][5]), \
                        "camera-side blocks differ between shards"
                po = copy.deepcopy(p)
                so = oa.ba_solve(olib, po, 20)
                assert summ[w]["iterations"] == so["iterations"] and summ[w]["num_successful_steps"] == so["num_successful_steps"], (w, summ[w], so)
                assert abs(summ[w]["final_cost"] - so["final_cost"]) <= 1e-7 * so["final_cost"]
                assert rel(parts[0][w][3], po["pose"]) <= 1e-6 and rel(full["invdepth"], po["invdepth"]) <= 1e-6, w
                assert rel(parts[0][w][5], po["ext"]) <= 1e-6
        s.close()
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok"))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, "FAIL: " + repr(e) + "\n" + traceback.format_exc()))


def _run(world, cfg, transport):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cfg, transport, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = []
    for _ in procs:
        res.append(q.get(timeout=600))
    for p in procs:
        p.join(60)
        if p.is_alive():
            p.kill()
    bad = [r for r in res if r[1] != "ok"]
    assert not bad, bad


@pytest.mark.skipif(_ngpu() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("world", [2, 0])  # 0 = min(8, all GPUs of the box)
def test_sharded_cfg4_matches_oracle(world):
    """cfg 4 (20 KF / 2000 landmarks): the reduced camera system does not fit one CTA, so the handle runs the split pipeline and the shards talk
    over peer memory (CUDA IPC, transport p2p)."""
    n = _ngpu()
    world = world or min(8, n)
    _run(world, (20, 2000, 3), "p2p")


@pytest.mark.skipif(_ngpu() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("transport", ["p2p"])
def test_sharded_cfg3_matches_oracle(transport):
    _run(2, (10, 300, 2), transport)
