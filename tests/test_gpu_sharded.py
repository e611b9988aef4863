"""GPU tests of the sharded store: CudaBackend (the product) under the same protocol."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as O  # noqa: E402
from util import assert_close, oracle_state  # noqa: E402

pytestmark = pytest.mark.gpu
capi = pytest.importorskip("difacto_b200.capi")

STATE_TOL = dict(rtol=1e-3, atol=1e-5)


def make_batch(rank, step, valued, S, dev, B=96, ids=500, max_nnz=24):
    from difacto_b200.sharded import shard_bounds_np
    rng = np.random.default_rng(100 * rank + step)
    nnzr = rng.integers(0, max_nnz, B)
    off = np.concatenate([[0], np.cumsum(nnzr)]).astype(np.uint64)
    n = int(off[-1])
    idx = rng.integers(0, ids, n).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    val = rng.random(n).astype(np.float32) if valued else None
    lab = np.where(rng.random(B) < 0.4, 1.0, -1.0).astype(np.float32)
    lidx, keys, cnt = O.localize(off, idx)
    host = dict(off=off, lab=lab, lidx=lidx, keys=keys, cnt=cnt, val=val, idx=idx)
    d = dict(nrows=B, nnz=n, U=len(keys), bounds=shard_bounds_np(keys, S),
             off=torch.from_numpy(off.view(np.int64).copy()).to(dev), lab=torch.from_numpy(lab).to(dev),
             lidx=torch.from_numpy(lidx.view(np.int32).copy()).to(dev),
             keys=torch.from_numpy(keys.view(np.int64).copy()).to(dev), cnt=torch.from_numpy(cnt).to(dev),
             val=torch.from_numpy(val).to(dev) if valued else None)
    return d, host


@pytest.mark.parametrize("V_dim,scatter", [(16, "sorted"), (16, "atomic"), (6, "sorted"), (0, "sorted"), (16, "p2p")])
def test_single_rank_sharded_equals_fused_and_oracle(V_dim, scatter):
    from difacto_b200.sharded import CudaBackend, PeerShardedStore, ShardedStore
    p2p = scatter == "p2p"
    if p2p:
        scatter = "sorted"
    dev = torch.device("cuda", 0)
    kw = dict(V_dim=V_dim, l1=0.05, l2=0.01, lr=0.2, V_lr=0.1, V_threshold=1, V_l2=0.01, V_init_scale=0.2, seed=3)
    E1 = capi.Engine(table_capacity=1 << 14, scatter=scatter, **kw)     # behind the sharded protocol (S = 1)
    E2 = capi.Engine(table_capacity=1 << 14, scatter=scatter, **kw)     # fused single-engine step
    M = O.Oracle(**kw)
    be = CudaBackend(E1, dev)
    store = PeerShardedStore(be, max_keys=4096) if p2p else ShardedStore(be)
    allkeys = []
    with torch.cuda.stream(be.stream):
        for step in range(8):
            d, h = make_batch(0, step, step % 2 == 0, 1, dev)
            store.step(d, True, push_cnt=step < 2)
            pr1 = E1.read_progress()
            pr2 = E2.train_step(h["off"], h["lidx"], h["val"], h["lab"], h["keys"], h["cnt"] if step < 2 else None, True)
            ref = M.sgd_step(h["off"], h["idx"], h["val"], h["lab"], True, step < 2)
            assert abs(pr1.loss - ref[0]) <= 1e-4 * abs(ref[0]) + 1e-4
            assert abs(pr1.penalty - ref[1]) <= 1e-4 * abs(ref[1]) + 1e-5
            assert abs(pr1.loss - pr2.loss) <= 1e-5 * abs(pr2.loss) + 1e-5
            allkeys.append(h["keys"])
    keys = np.unique(np.concatenate(allkeys))
    s1, s2 = E1.read_entries(keys), E2.read_entries(keys)
    assert np.array_equal(s1[1], s2[1])
    for a, b in zip(s1, s2):
        assert_close(a, b, what="sharded(S=1) vs fused", rtol=1e-5, atol=1e-6)
    oscal, ohasv, oV, ocg = oracle_state(M, keys)
    assert np.array_equal(s1[1], ohasv)
    assert_close(s1[0][:, 1:], oscal[:, 1:], what="w/sqrt_g/z", **STATE_TOL)
    assert_close(s1[2], oV, what="V", **STATE_TOL)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


KW2 = dict(V_dim=16, l1=0.05, l2=0.01, lr=0.2, V_lr=0.1, V_threshold=1, V_l2=0.01, V_init_scale=0.2, seed=3)
STEPS2 = 6


def _worker(rank, world, port, out, p2p):
    import torch.distributed as dist
    from difacto_b200 import capi as C2
    from difacto_b200.sharded import CudaBackend, PeerShardedStore, ShardedStore, key_owner_np
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    E = C2.Engine(device=rank, table_capacity=1 << 14, **KW2)
    be = CudaBackend(E, dev)
    store = PeerShardedStore(be, max_keys=4096) if p2p else ShardedStore(be)
    prog = np.zeros(2)
    with torch.cuda.stream(be.stream):
        for step in range(STEPS2):
            d, _ = make_batch(rank, step, step % 2 == 0, world, dev)
            store.step(d, True, push_cnt=step < 2)
            pr = E.read_progress()
            prog += [pr.loss, pr.penalty]
    allkeys = np.unique(np.concatenate([make_batch(r, st, False, world, torch.device("cpu"))[1]["keys"]
                                        for r in range(world) for st in range(STEPS2)]))
    mine = allkeys[key_owner_np(allkeys, world) == rank]
    scal, hasv, V, cg = E.read_entries(mine)
    np.savez(out.format(rank=rank), scal=scal, hasv=hasv, V=V, cg=cg, prog=prog, nkeys=E.table_stats()["n_keys"])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("p2p", [False, True])
def test_two_gpu_nccl_sharded_vs_oracle_simulation(tmp_path, p2p):
    import torch.multiprocessing as mp
    from difacto_b200.sharded import key_owner_np
    from oracle_backend import OracleBackend
    world = 2
    out = str(tmp_path / "shard{rank}.npz")
    mp.spawn(_worker, args=(world, _free_port(), out, p2p), nprocs=world, join=True)
    # sequential simulation with oracle shards (same protocol semantics)
    cpu = torch.device("cpu")
    shards = [OracleBackend(**KW2) for _ in range(world)]
    workers = [OracleBackend(**KW2) for _ in range(world)]
    for step in range(STEPS2):
        batches = [make_batch(r, step, step % 2 == 0, world, cpu)[0] for r in range(world)]
        owners = [key_owner_np(b["keys"].numpy().view(np.uint64), world) for b in batches]
        if step < 2:
            for s in range(world):
                for r in range(world):
                    m = owners[r] == s
                    shards[s].feacnt(batches[r]["keys"][m], batches[r]["cnt"][m])
        pulled, grads = [], []
        for r in range(world):
            b = batches[r]
            U, ks = b["U"], shards[0].ks
            w, hasv, V = torch.zeros(U), torch.zeros(U, dtype=torch.int32), torch.zeros(U, ks)
            for s in range(world):
                m = np.nonzero(owners[r] == s)[0]
                ws, hs, Vs = torch.zeros(len(m)), torch.zeros(len(m), dtype=torch.int32), torch.zeros(len(m), ks)
                shards[s].pull_rows(b["keys"][m], ws, hs, Vs)
                w[m], hasv[m], V[m] = ws, hs, Vs
            pulled.append((w, hasv, V))
            gw, gV = torch.zeros(U), torch.zeros(U, ks)
            workers[r].fm_step(b, w, hasv, V, True, gw, gV)
            grads.append((gw, gV))
        for s in range(world):
            for r in range(world):
                m = np.nonzero(owners[r] == s)[0]
                shards[s].push_rows(batches[r]["keys"][m], grads[r][0][m], pulled[r][1][m], grads[r][1][m])
    allkeys = np.unique(np.concatenate([make_batch(r, st, False, world, cpu)[1]["keys"]
                                        for r in range(world) for st in range(STEPS2)]))
    own = key_owner_np(allkeys, world)
    for s in range(world):
        got = np.load(out.format(rank=s))
        oscal, ohasv, oV, ocg = oracle_state(shards[s].M, allkeys[own == s])
        assert np.array_equal(got["hasv"], ohasv)
        assert np.array_equal(got["scal"][:, 0], oscal[:, 0])
        assert_close(got["scal"][:, 1:], oscal[:, 1:], what=f"shard {s} w/sqrt_g/z", **STATE_TOL)
        assert_close(got["V"], oV, what=f"shard {s} V", **STATE_TOL)
        assert_close(got["cg"], ocg, what=f"shard {s} cg", **STATE_TOL)
        assert got["nkeys"] == shards[s].M.size()
        assert abs(got["prog"][0] - workers[s].progress[0]) <= 1e-4 * abs(workers[s].progress[0])
