"""The per-step exchange of a sharded log (include/fpx.h, fpx_exchange_*): every engine's watermark
publication is stored into all shards' frontier tables from inside the publishing kernel; the global
executable prefix is the minimum (S/multipaxos/Replica.scala:397-402).  One GPU: engines of one process
attached locally.  Two GPUs: one process per GPU, IPC handles, peer stores over NVLink."""
import os
import sys

import numpy as np
import pytest

import harness as H
from frankenpaxos_b200 import Engine
from frankenpaxos_b200 import traces as T
from oracle import fpx_oracle_py as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("hole", [None, 1234])
def test_three_shards_on_one_gpu_publish_to_each_other(hole, fused):
    import torch
    cfg, _ = T.config_by_name("cfg2")
    n_slots, P = 6000, 3
    a, p, b = T.workload(21, cfg, n_slots)
    if hole is not None:
        b = b[b["slot"] != hole]
    ora = O.MultiPaxos(2, 1, 5, False, 3, 3)
    ora.arm(a); ora.acceptor_phase2a(p)
    _, _, oc = ora.proxyleader_phase2b(b)
    ora.replica_chosen(oc)
    engs = [Engine(slot_capacity=n_slots, max_batch=1 << 16, shard_index=g, shard_count=P, **cfg) for g in range(P)]
    for e in engs:
        for g, peer in enumerate(engs):
            e.exchange_attach_local(g, peer)
    dev = torch.device("cuda", 0)
    td = lambda x: torch.from_numpy(x.view(np.int32).reshape(len(x), -1).copy()).to(dev)
    for g, e in enumerate(engs):
        mine = lambda r: r[r["slot"] % P == g]
        if fused:
            da, dp, db = td(mine(a)), td(mine(p)), td(mine(b))
            o1 = torch.zeros((len(dp), 4), dtype=torch.int32, device=dev); o2 = torch.zeros((len(dp), 2), dtype=torch.int32, device=dev)
            o3 = torch.zeros((len(db), 2), dtype=torch.int32, device=dev); wm = torch.zeros(1, dtype=torch.int32, device=dev)
            e.step_dev(da.data_ptr(), len(da), dp.data_ptr(), len(dp), o1.data_ptr(), o2.data_ptr(), db.data_ptr(), len(db),
                       o3.data_ptr(), wm.data_ptr())
            e.sync()
        else:
            e.proxyleader_arm(mine(a))
            e.acceptor_phase2a(mine(p))
            e.replica_chosen(e.proxyleader_phase2b(mine(b)))
            e.chosen_watermark()
        assert e.exchange_epoch == 1
    for e in engs:
        g_wm, fr = e.global_watermark(epoch=1)
        assert g_wm == ora.executed_watermark() == (hole if hole is not None else n_slots)
        for g in range(P):   # every shard's first unchosen GLOBAL slot
            if hole is not None and hole % P == g:
                assert fr[g] == hole
            else:
                assert fr[g] >= n_slots and fr[g] % P == g
    # waiting for a publication that never comes is an error, not a hang
    from frankenpaxos_b200 import FpxError
    with pytest.raises(FpxError) as ei:
        engs[0].global_watermark(epoch=5, timeout_ms=20)
    assert ei.value.status == -16
    [e.close() for e in engs]


def _ipc_worker(rank, world, q_in, q_out, n_slots):
    sys.path.insert(0, ROOT)
    import torch
    torch.cuda.set_device(rank)
    from frankenpaxos_b200 import Engine
    from frankenpaxos_b200 import traces as T
    cfg, _ = T.config_by_name("cfg2")
    eng = Engine(slot_capacity=n_slots, max_batch=1 << 16, device=rank, shard_index=rank, shard_count=world, **cfg)
    q_out.put((rank, eng.exchange_export()))
    handles = q_in.get(timeout=120)
    for g, h in handles.items():
        if g != rank:
            eng.exchange_attach(g, h)
    q_out.put((rank, "attached"))
    assert q_in.get(timeout=120) == "go"
    a, p, b = T.workload(33, cfg, n_slots)
    mine = lambda r: r[r["slot"] % world == rank]
    for step in range(3):            # three publications: votes of the last third of the slots arrive last
        lo, hi = step * n_slots // 3, (step + 1) * n_slots // 3
        sel = lambda r: mine(r)[(mine(r)["slot"] >= lo) & (mine(r)["slot"] < hi)]
        eng.proxyleader_arm(sel(a))
        eng.acceptor_phase2a(sel(p))
        eng.replica_chosen(eng.proxyleader_phase2b(sel(b)))
        eng.chosen_watermark()
    g_wm, fr = eng.global_watermark(epoch=3, timeout_ms=20000)
    q_out.put((rank, int(g_wm), fr.tolist()))
    assert q_in.get(timeout=120) == "done"
    eng.close()


def test_two_processes_two_gpus_exchange_over_ipc():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (peer stores over NVLink)")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    world, n_slots = 2, 6000
    q_out = ctx.Queue()
    q_in = [ctx.Queue() for _ in range(world)]
    procs = [ctx.Process(target=_ipc_worker, args=(r, world, q_in[r], q_out, n_slots)) for r in range(world)]
    [p.start() for p in procs]
    handles = dict(q_out.get(timeout=300) for _ in range(world))
    [q.put(handles) for q in q_in]
    assert sorted(q_out.get(timeout=120)[0] for _ in range(world)) == [0, 1]
    [q.put("go") for q in q_in]
    res = sorted(q_out.get(timeout=300) for _ in range(world))
    [q.put("done") for q in q_in]
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    for rank, g_wm, fr in res:
        assert g_wm == n_slots and fr[0] >= n_slots and fr[1] >= n_slots and fr[0] % 2 == 0 and fr[1] % 2 == 1
