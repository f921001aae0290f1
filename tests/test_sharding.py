"""Node sharding: host-side range arithmetic and digest composition on CPU (gloo, world_size 2),
and the real NCCL path when the box has >= 2 GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_ranges_partition(egs):
    for n in [1, 100, 128, 129, 1000, 50000, 100000, 1 << 20]:
        for world in [1, 2, 3, 4, 8]:
            edges = [egs.shard_range(n, r, world) for r in range(world)]
            assert edges[0][0] == 0 and edges[-1][1] == n
            for (lo, hi), (lo2, _) in zip(edges, edges[1:]):
                assert hi == lo2 and lo <= hi
            assert all(lo % 128 == 0 for lo, _ in edges)


def _gloo_worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import torch
        import torch.distributed as dist
        import egs_b200
        import oracle_c
        dist.init_process_group("gloo", rank=rank, world_size=world)
        # the id exchange bench.py uses (broadcast of a 128-byte token from rank 0)
        box = [bytes(range(128)) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        assert box[0] == bytes(range(128))
        # each rank filters ITS node range with the oracle; per-shard digests must add up (mod 2^64)
        w = egs_b200.workloads.config(1, n_nodes=1000, n_pods=4)
        o = oracle_c.OracleC(w.policy)
        for n in range(w.n_nodes):
            o.add_node(800, 8 * w.mem_total)
            o.set_rows(n, w.core[n], w.mem[n])
        lo, hi = egs_b200.capi.shard_range(w.n_nodes, rank, world)
        req = [tuple(int(x) for x in w.units[0])]
        ids = np.arange(lo, hi, dtype=np.int32)
        fit = o.filter(ids, req)
        _, sc = o.score(ids[fit.astype(bool)], req)
        L = oracle_c.lib()
        fd = sum(L.egso_mix64(2 * int(i) + 1) for i in ids[fit.astype(bool)]) & (2**64 - 1)
        sd = sum(L.egso_mix64(2 * int(i) + 2) * (2 * (int(s) & 0xFFFFFFFF) + 1)
                 for i, s in zip(ids[fit.astype(bool)], sc)) & (2**64 - 1)
        t = torch.tensor([int(fit.sum()), fd - (1 << 64) if fd >= 1 << 63 else fd, sd - (1 << 64) if sd >= 1 << 63 else sd],
                         dtype=torch.int64)
        dist.all_reduce(t)                      # int64 wrap-around == addition mod 2^64
        o2 = oracle_c.OracleC(w.policy)
        for n in range(w.n_nodes):
            o2.add_node(800, 8 * w.mem_total)
            o2.set_rows(n, w.core[n], w.mem[n])
        full = o2.schedule_batch(w.c_off[:2], w.units64()[:1])
        assert int(t[0]) == int(full["fit_count"][0])
        assert int(t[1]) & (2**64 - 1) == int(full["fit_digest"][0])
        assert int(t[2]) & (2**64 - 1) == int(full["score_digest"][0])
        dist.destroy_process_group()
        q.put((rank, "ok"))
    except Exception as ex:  # pragma: no cover
        q.put((rank, repr(ex)))


def test_gloo_world2_digest_composition():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res


@pytest.mark.gpu
def test_nccl_sharded_rounds_equal_unsharded():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (NCCL across devices)")
    world = 2 if n < 4 else 4
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29731",
                        os.path.join(ROOT, "tools", "multi_gpu_check.py")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "MULTI_GPU_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_engine_in_process_equals_unsharded(world):
    """The sharded rounds engine at world sizes 2 / 4 / 8 on whatever GPUs exist (all shards on device 0 of a
    single-GPU box): an in-process shard group (egs_comm_init_local) replaces NCCL by device-to-device copies of the
    same candidate buffers; kernels, buffers and the replicated resolver are those of the NCCL path.  Every rank's
    outputs must equal the unsharded run bit for bit, and every shard's rows the unsharded rows."""
    import threading
    import egs_b200
    cap = egs_b200.capi
    F = ["node", "status", "alloc_mask", "fit_count", "fit_digest", "score_digest"]
    # config 4 at full node count, long enough that nearly every round ends on a dry per-shard list (at 8 shards each
    # contributes only 32 candidates per shape): the replicated resolvers must stop at the SAME pod on every rank
    cases = [(4, None, 200000 if world == 8 else 60000, None), (1, None, None, None), (2, 3000, 6000, None), (3, 300, 2000, 0),
             (4, 1000, 3000, 0)]
    for cfg, nn, npods, pol in cases:
        w = egs_b200.workloads.config(cfg, n_nodes=nn, n_pods=npods, policy=pol)
        e0 = egs_b200.Egs(w.policy, w.n_nodes)
        e0.state_load_bulk(0, w.gpus, w.mem_total, w.core, w.mem)
        ref = e0.schedule_batch(w.c_off, w.units, mode=cap.EGS_MODE_ROUNDS)
        ref_core, ref_mem, _, _ = e0.state_dump()
        e0.close()
        hs = []
        for r in range(world):
            e = egs_b200.Egs(w.policy, w.n_nodes)
            e.shard_set(r, world)
            hs.append(e)
        cap.comm_init_local(hs)
        for e in hs:
            e.state_load_bulk(0, w.gpus, w.mem_total, w.core, w.mem)
        outs, errs = [None] * world, []

        def run(r):
            try:
                outs[r] = hs[r].schedule_batch(w.c_off, w.units, mode=cap.EGS_MODE_ROUNDS)
            except Exception as ex:   # pragma: no cover
                errs.append(repr(ex))
        th = [threading.Thread(target=run, args=(r,)) for r in range(world)]
        for t_ in th:
            t_.start()
        for t_ in th:
            t_.join(timeout=600)
        assert not errs, errs
        for r in range(world):
            for f in F:
                assert np.array_equal(ref[f], outs[r][f]), f"cfg{cfg} world {world} rank {r}: {f} differs"
            lo, hi = cap.shard_range(w.n_nodes, r, world)
            core, mem, _, _ = hs[r].state_dump(lo, hi - lo)
            assert np.array_equal(core, ref_core[lo:hi]) and np.array_equal(mem, ref_mem[lo:hi]), f"rows of shard {r}"
        for e in hs:
            e.close()
