"""N > 1: nodes sharded in contiguous ranges over the GPUs of one box, one process per GPU, one exchange of
the constraint counters per ApplyState. The union of the per-rank outputs must equal the oracle's result on
the unsharded cluster, bit for bit — including the ordered slot allocation across the shard boundary and
abort semantics whose abort point lives on another rank."""
import os

import numpy as np
import pytest

import helpers
from helpers import abi
from ust import synth

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, cases, q, mode):
    import torch
    import torch.distributed as dist
    from ust import lib as ustlib
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    h = ustlib.Handle(rank)
    uid = [ustlib.get_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    h.comm_init(rank, world, uid[0])
    h.comm_set_mode(mode)  # 0 = NCCL all-reduce between two kernels, 1 = fused NVLink mailbox exchange
    results = []
    for (n, seed, p_err, pol_kwargs) in cases:
        with_pods = pol_kwargs.get("evaluate_actuators", False)
        pol = abi.make_policy(**pol_kwargs)
        soa = synth.make_nodes(n, seed, start=rank * n, error_pct=p_err)
        pods = synth.make_pods(n, seed, start=rank * n) if with_pods else None   # CSR split at the shard boundary
        rc, nxt, act, oc, cnt = h.apply_state(pol, soa, pods)
        results.append((rc, nxt, act, oc, cnt))
    gathered = [None] * world
    dist.all_gather_object(gathered, results)
    if rank == 0:
        q.put(gathered)
    h.close()
    dist.destroy_process_group()


CASES = [
    (300_000, 0x5EED0005, 0.0, dict(max_parallel_upgrades=100, max_unavailable="25%")),      # C5 policy
    (300_000, 0x5EED0005, 0.0, dict(max_parallel_upgrades=0)),                                # everything granted
    (300_000, 0x5EED0005, 0.0, dict(max_parallel_upgrades=0, max_unavailable="30%")),         # cut inside rank 0 / 1
    (300_000, 0x5EED0005, 0.0, dict(max_parallel_upgrades=250_000)),                          # cut on rank 1
    (150_001, 0x5EED0007, 0.001, dict(max_parallel_upgrades=5, max_unavailable=7)),           # aborts
    (100_000, 0x5EED0008, 0.0, dict(max_parallel_upgrades=3, use_maintenance_operator=True)), # requestor mode
    (120_000, 0x5EED0004, 0.0, dict(synth.CONFIGS["C4"]["policy"])),                          # C4: pod lists per shard
]


@pytest.mark.parametrize("mode", [0, 1], ids=["nccl", "fused-nvlink"])
def test_two_ranks_match_unsharded_oracle(mode):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs in one machine")
    world = min(int(os.environ.get("UST_TEST_WORLD", "2")), torch.cuda.device_count())
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, world, port + mode, CASES, q, mode)) for r in range(world)]
    for p in procs:
        p.start()
    gathered = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for ci, (n, seed, p_err, pol_kwargs) in enumerate(CASES):
        whole = synth.make_nodes(world * n, seed, error_pct=p_err)
        pol = abi.make_policy(**pol_kwargs)
        pods = synth.make_pods(world * n, seed) if pol_kwargs.get("evaluate_actuators", False) else None
        ref = helpers.oracle_apply(pol, whole, pods, variant=1)
        rcs = [gathered[r][ci][0] for r in range(world)]
        nxt = np.concatenate([gathered[r][ci][1] for r in range(world)])
        act = np.concatenate([gathered[r][ci][2] for r in range(world)])
        oc = np.concatenate([gathered[r][ci][3] for r in range(world)])
        assert all(rc == ref[0] for rc in rcs), (ci, rcs, ref[0])
        for r in range(world):
            assert gathered[r][ci][4] == ref[4], (ci, r, gathered[r][ci][4], ref[4])  # every rank reports cluster-wide counters
        helpers.assert_same((ref[0], nxt, act, oc, ref[4]), ref, f"case {ci}")
