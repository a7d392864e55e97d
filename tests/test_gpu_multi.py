"""Multi-GPU plumbing on real hardware (needs >= 2 visible GPUs; skipped otherwise): NCCL gather of the packed game
records to rank 0 (parallel.gather_records) and the generation's weight hand-over — the trainer rank folds, the FOLDED
blob is NCCL-broadcast into every other rank's weight arena and adopted without folding (kv_net_folded_* /
kv_net_adopt_folded) — checked by bit-identical network outputs on every rank.  The CPU-side logic of the same calls is
covered under gloo in tests/test_distributed_cpu.py."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    try:
        from knightvision_b200 import layout as L
        from knightvision_b200 import parallel as P
        from knightvision_b200.engine import Engine, lines_to_device
        from knightvision_b200.model import ChessNet
        eng = Engine(rank)
        # ---- weights: rank 0 has the real net, the others a different one; after the hand-over all agree bit for bit
        torch.manual_seed(100 + rank)
        net = ChessNet().eval().attach(eng, max_batch=64)
        lines = lines_to_device(np.stack([L.start_line()] * 3), eng.device)
        before = eng.net_forward(lines)[0].clone()
        dist.broadcast(eng.net_folded_tensor(), src=0)
        if rank != 0:
            eng.net_adopt_folded()
        pol, val = eng.net_forward(lines)
        ref = [torch.zeros_like(pol) for _ in range(world)]
        dist.all_gather(ref, pol)
        assert all(torch.equal(r, ref[0]) for r in ref)
        assert rank == 0 or not torch.equal(before, pol)
        # ---- records: G games per rank with the hash evaluator, gathered on rank 0 in global game order
        G, sims, plies = 24 + 8 * rank, 8, 6
        eng.mcts_create(G, sims, max_plies=plies, temp_plies=2, seed=7, eval_mode=0)
        base = 0 if rank == 0 else 24
        eng.mcts_reset(None, game_id_base=base)
        for _ in range(plies):
            eng.mcts_run_move()
        l, m, r, g = eng.mcts_records()
        out = P.gather_records(l, m, r, base, g, dst=0)
        mine = (l.cpu(), m.cpu(), r.cpu(), (g.to(torch.int64) + base).cpu())
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        if rank == 0:
            L_, M_, R_, G_ = (t.cpu() for t in out)
            assert torch.equal(L_, torch.cat([x[0] for x in gathered])) and torch.equal(M_, torch.cat([x[1] for x in gathered]))
            assert torch.equal(R_, torch.cat([x[2] for x in gathered])) and torch.equal(G_, torch.cat([x[3] for x in gathered]))
            assert G_.tolist() == sorted(G_.tolist()) and int(G_.max()) == 24 + 32 - 1
            ret.put(("ok", int(L_.shape[0])))
        else:
            assert out is None
        eng.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_nccl_weight_handover_and_record_gather():
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = 29600 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    tag, n = ret.get(timeout=5)
    assert tag == "ok" and 0 < n <= (24 + 32) * 6
