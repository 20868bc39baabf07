"""GPU, world_size 2 over NCCL/NVLink (skipped with fewer than 2 devices): the scene-parallel step with the
fused one-shot all-reduce + clamp + Adam kernel (spg_allreduce_clamp_adam over symmetric memory) against
the torch.distributed.all_reduce + spg_clamp_adam_dev path, and replica consistency."""
import os
import socket
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from superpoint_graph_b200 import ops, workloads
    from superpoint_graph_b200.trainer import HostBatch, Trainer, create_model
    w = workloads.get("s3dis_train", nodes=256)
    w["margs"].model_config = "gru_3_1_1_1_0,f_13"
    batch = workloads.batch(w, 1 + 1000 * rank)
    results = {}
    for fused in (True, False):
        ops.USE_FUSED_ALLREDUCE[0] = fused
        torch.manual_seed(1)
        model = create_model(w["margs"]).to(dev)
        tr = Trainer(model, w["margs"], process_group=dist.group.WORLD, world_size=world)
        assert (tr._fused_ar is not None) == fused
        db = HostBatch(batch).to_device(dev)
        losses = []
        for _ in range(3):
            loss, _ = tr.train_step(db)
            losses.append(float(loss[0]))
        key = tr.capture(db, warmup=1)
        for _ in range(2):
            loss, _ = tr.replay(key)
            losses.append(float(loss[0]))
        torch.cuda.synchronize()
        gathered = [torch.empty_like(tr.flat) for _ in range(world)]
        dist.all_gather(gathered, tr.flat)
        same = all(torch.equal(gathered[0], g) for g in gathered)
        results[fused] = (tr.flat.clone(), losses, same, int(tr.step_dev.item()))
    pf, lf, same_f, steps_f = results[True]
    pn, ln, same_n, steps_n = results[False]
    # sums of `world` float32 numbers in rank order vs NCCL's order differ in the last bit; Adam turns the sign
    # of a noise-level gradient element (e.g. the analytically zero pre-BatchNorm biases) into a +-lr step,
    # so a few elements may sit 2*lr apart: compare the fraction of agreeing elements and the losses
    d = (pf - pn).abs()
    rel = float((d > 1e-4 * pn.abs().max()).float().mean())
    if rank == 0:
        q.put(dict(same_f=same_f, same_n=same_n, rel=rel, lf=lf, ln=ln, steps=(steps_f, steps_n)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_fused_allreduce_adam_matches_nccl_path_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0
    res = q.get()
    assert res["same_f"], "replicas drifted apart on the fused path"
    assert res["same_n"]
    assert res["steps"] == (5, 5)  # 3 eager steps + 2 replays (the capture warm-up runs on a snapshot)
    assert res["rel"] < 0.02, res  # fraction of parameter elements that differ by more than 1e-4 of the scale
    for a, b in zip(res["lf"], res["ln"]):
        assert abs(a - b) <= 2e-4 * abs(b), (res["lf"], res["ln"])
