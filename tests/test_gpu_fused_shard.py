"""GPU parity tests of the NVLink-sharded store behind the C-ABI (dfb_shard_*): the product's multi-GPU path.

Every test compares the CUDA path with a sequential simulation of the same parameter-server semantics built
on oracle shards (tests/shard_sim.py).  The protocol is exercised
  * with one rank (events only),
  * with 2 and 3 ranks that live in ONE process on ONE GPU (peer pointers are plain device pointers; the step
    counters are polled exactly as between GPUs) -- so the driver's single-GPU test box runs the whole protocol,
  * with one process per GPU over CUDA IPC when 2 GPUs are visible.
Tolerances as in test_gpu_parity.py: model state after T steps rel 1e-3 / abs 1e-5 (fp32, different summation
order over k and over the owners' partials); keys, has-V flags, feature counts bit-exact."""
import os
import socket
import sys

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # several engines on one GPU: one hardware queue per stream

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from shard_sim import all_keys, key_owner_np, raw_batch, simulate  # noqa: E402
from util import assert_close, oracle_state  # noqa: E402

pytestmark = pytest.mark.gpu
capi = pytest.importorskip("difacto_b200.capi")

STATE_TOL = dict(rtol=1e-3, atol=1e-5)
KW = dict(V_dim=16, l1=0.05, l2=0.01, lr=0.2, V_lr=0.1, V_threshold=1, V_l2=0.01, V_init_scale=0.2, seed=3)
STEPS = 6


def batch_fn(rank, step):
    return raw_batch(rank, step, valued=(step % 2 == 0))


def check_shard(E, shard, keys, what):
    scal, hasv, V, cg = E.read_entries(keys)
    oscal, ohasv, oV, ocg = oracle_state(shard.M, keys)
    assert np.array_equal(hasv, ohasv), what
    assert np.array_equal(scal[:, 0], oscal[:, 0]), what                     # feature counts: exact
    assert_close(scal[:, 1:], oscal[:, 1:], what=f"{what} w/sqrt_g/z", **STATE_TOL)
    assert_close(V, oV, what=f"{what} V", **STATE_TOL)
    assert_close(cg, ocg, what=f"{what} cg", **STATE_TOL)
    assert E.table_stats()["n_keys"] == shard.M.size(), what


def check_progress(pr, ref, what):
    # ref = [loss, penalty, auc, nnz_w, nrows]
    assert abs(pr.loss - ref[0]) <= 1e-4 * abs(ref[0]) + 1e-4, (what, pr.loss, ref[0])
    assert abs(pr.penalty - ref[1]) <= 1e-4 * abs(ref[1]) + 1e-5, (what, pr.penalty, ref[1])
    # AUC * n: predictions that are tied in exact arithmetic (rows whose only active feature is the same) are
    # ordered by rounding; each flipped pair moves AUC * n by n / (n_pos * n_neg) <= ~0.05 at these sizes
    if ref[4] > 0:     # (the reference never evaluates an empty batch; a worker without one contributes nothing)
        assert abs(pr.auc - ref[2]) <= 1e-4 * abs(ref[2]) + 0.3, (what, pr.auc, ref[2])
    assert pr.nrows == ref[4], (what, pr.nrows, ref[4])


def run_local(S, kw, steps, fn, train_fn=None, devices=None, **shard_kw):
    from difacto_b200.sharded import FusedShardedStore
    engines = [capi.Engine(device=devices[r] if devices else 0, table_capacity=1 << 14, shard_timeout_ms=8000, **kw)
               for r in range(S)]
    shard_kw.setdefault("max_rows", 128)
    shard_kw.setdefault("max_nnz", 4096)
    FusedShardedStore.connect_local(engines, **shard_kw)
    prog = [[] for _ in range(S)]
    for step in range(steps):
        is_train = True if train_fn is None else train_fn(step)
        # one host thread, several engines on one device: interleave the five enqueue phases (see difacto_b200.h)
        for r in range(S):
            off, idx, val, lab = fn(r, step)
            engines[r].shard_begin_async(len(lab), off, idx, val, lab, push_cnt=step < 2, is_train=is_train)
        for phase in range(5):
            for r in range(S):
                engines[r].shard_phase(phase)
        for r in range(S):
            prog[r].append(engines[r].wait_step())
    return engines, prog


@pytest.mark.parametrize("S", [1, 2, 3])
def test_fused_shard_local_ranks_vs_oracle_simulation(S):
    engines, prog = run_local(S, KW, STEPS, batch_fn)
    shards, workers, per_step = simulate(S, STEPS, KW, batch_fn)
    for step in range(STEPS):
        for r in range(S):
            check_progress(prog[r][step], per_step[step][r], f"S={S} step {step} worker {r}")
    keys = all_keys(S, STEPS, batch_fn)
    own = key_owner_np(keys, S)
    for s in range(S):
        assert (own == s).sum() > 10
        check_shard(engines[s], shards[s], keys[own == s], f"S={S} shard {s}")
        # nothing leaked to the wrong shard
        if S > 1:
            _, hasv, _, _ = engines[s].read_entries(keys[own != s][:64])
            assert np.all(hasv == -1)
    for E in engines:
        E.close()


def test_fused_shard_equals_single_engine_raw_step():
    """S = 1 through the shard path == the fused single-GPU raw step, same inputs"""
    engines, prog = run_local(1, KW, STEPS, batch_fn)
    E2 = capi.Engine(device=0, table_capacity=1 << 14, **KW)
    for step in range(STEPS):
        off, idx, val, lab = batch_fn(0, step)
        pr2 = E2.train_step_raw(off, idx, val, lab, push_cnt=step < 2, is_train=True)
        assert abs(prog[0][step].loss - pr2.loss) <= 1e-5 * abs(pr2.loss) + 1e-5
        assert abs(prog[0][step].penalty - pr2.penalty) <= 1e-5 * abs(pr2.penalty) + 1e-6
    keys = all_keys(1, STEPS, batch_fn)
    for a, b in zip(engines[0].read_entries(keys), E2.read_entries(keys)):
        assert_close(a, b, what="shard(S=1) vs fused raw step", rtol=1e-5, atol=1e-6)
    assert engines[0].rng_state() == E2.rng_state()


def test_fused_shard_validation_steps_do_not_touch_the_model():
    S = 2
    train_fn = lambda step: step % 3 != 2      # noqa: E731  every third batch is a validation batch
    engines, prog = run_local(S, KW, STEPS, batch_fn, train_fn=train_fn)
    shards, workers, per_step = simulate(S, STEPS, KW, batch_fn, train_fn=train_fn)
    for step in range(STEPS):
        for r in range(S):
            check_progress(prog[r][step], per_step[step][r], f"step {step} worker {r}")
    keys = all_keys(S, STEPS, batch_fn)
    own = key_owner_np(keys, S)
    for s in range(S):
        # a validation batch must not insert its unseen keys (the oracle's Get() default-constructs them: compare values)
        scal, hasv, V, cg = engines[s].read_entries(keys[own == s])
        oscal, ohasv, oV, ocg = oracle_state(shards[s].M, keys[own == s])
        seen = hasv >= 0
        assert np.array_equal(hasv[seen], ohasv[seen])
        assert_close(scal[seen][:, 1:], oscal[seen][:, 1:], what="w/sqrt_g/z", **STATE_TOL)
        assert_close(V[seen], oV[seen], what="V", **STATE_TOL)
        assert np.all(oscal[~seen] == 0)


def test_fused_shard_hot_shared_keys_and_v64():
    """few distinct ids: every key is held by every worker in every step (the pull-time V of a key another
    worker's push already updated must be used), V_dim = 64, long column lists"""
    kw = dict(KW, V_dim=64, V_threshold=0)
    fn = lambda rank, step: raw_batch(rank, step, valued=(step % 2 == 1), B=128, ids=40, max_nnz=30)   # noqa: E731
    S, steps = 3, 5
    engines, prog = run_local(S, kw, steps, fn)
    shards, workers, per_step = simulate(S, steps, kw, fn)
    for step in range(steps):
        for r in range(S):
            check_progress(prog[r][step], per_step[step][r], f"step {step} worker {r}")
    keys = all_keys(S, steps, fn)
    own = key_owner_np(keys, S)
    for s in range(S):
        check_shard(engines[s], shards[s], keys[own == s], f"shard {s}")


def test_fused_shard_mixed_binary_valued_and_empty_batches():
    """the workers of one step hold a binary batch, a valued one and none at all (the last round of an epoch whose
    file parts have unequal lengths): on the wire every batch is valued, so an owner never has to know"""
    def fn(rank, step):
        if rank == 1 and step in (2, 5):
            return raw_batch(rank, step, valued=False, B=0)
        if rank == 2 and step == 5:
            return raw_batch(rank, step, valued=True, B=0)
        return raw_batch(rank, step, valued=(rank + step) % 2 == 0)
    S = 3
    engines, prog = run_local(S, KW, STEPS, fn)
    shards, workers, per_step = simulate(S, STEPS, KW, fn)
    for step in range(STEPS):
        for r in range(S):
            check_progress(prog[r][step], per_step[step][r], f"step {step} worker {r}")
    keys = all_keys(S, STEPS, fn)
    own = key_owner_np(keys, S)
    for s in range(S):
        check_shard(engines[s], shards[s], keys[own == s], f"shard {s}")
    for E in engines:
        E.close()


def test_fused_shard_segment_capacity_is_reported():
    from difacto_b200.sharded import FusedShardedStore
    engines = [capi.Engine(device=0, table_capacity=1 << 14, shard_timeout_ms=8000, **KW) for _ in range(2)]
    FusedShardedStore.connect_local(engines, max_rows=128, max_nnz=4096, seg_keys=8, seg_nnz=16)
    for r in range(2):
        off, idx, val, lab = batch_fn(r, 0)
        engines[r].shard_begin_async(len(lab), off, idx, val, lab, push_cnt=False, is_train=True)
    for phase in range(5):
        for r in range(2):
            engines[r].shard_phase(phase)
    with pytest.raises(capi.DfbError) as ei:
        for r in range(2):
            engines[r].wait_step()
    assert ei.value.code == capi.DFB_ERR_CAPACITY


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("big", [False, True])
def test_fused_shard_two_gpus_one_process_vs_oracle_simulation(big):
    """two engines on two devices inside ONE process, driven by ONE host thread (peer access instead of CUDA IPC; the
    C++ CLI's num_gpus mode).  The enqueue phases are interleaved over the ranks as on one device: a monolithic
    dfb_shard_step_async per rank would leave rank 0's pollers waiting for work the host has not enqueued yet, and any
    blocking driver call in between (a lazily loaded kernel, for one) then never returns.  big = the CLI's capacities"""
    S = 2
    shard_kw = dict(max_rows=65536, max_nnz=65536 * 64) if big else {}
    engines, prog = run_local(S, KW, STEPS, batch_fn, devices=[0, 1], **shard_kw)
    shards, workers, per_step = simulate(S, STEPS, KW, batch_fn)
    for step in range(STEPS):
        for r in range(S):
            check_progress(prog[r][step], per_step[step][r], f"step {step} worker {r}")
    keys = all_keys(S, STEPS, batch_fn)
    own = key_owner_np(keys, S)
    for s in range(S):
        check_shard(engines[s], shards[s], keys[own == s], f"shard {s}")
    for E in engines:
        E.close()


# ---------------------------------------------------------------------------------------------------------
# one process per GPU, mailboxes shared through CUDA IPC
# ---------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from difacto_b200 import capi as C2
    from difacto_b200.sharded import FusedShardedStore
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    E = C2.Engine(device=rank, table_capacity=1 << 14, **KW)
    store = FusedShardedStore(E, max_rows=128, max_nnz=4096)
    prog = []
    for step in range(STEPS):
        off, idx, val, lab = batch_fn(rank, step)
        store.step_host(len(lab), off, idx, val, lab, is_train=True, push_cnt=step < 2)
        pr = E.wait_step()
        prog.append([pr.loss, pr.penalty, pr.auc, 0.0, pr.nrows])
    keys = all_keys(world, STEPS, batch_fn)
    mine = keys[key_owner_np(keys, world) == rank]
    scal, hasv, V, cg = E.read_entries(mine)
    np.savez(out.format(rank=rank), scal=scal, hasv=hasv, V=V, cg=cg, prog=np.array(prog), nkeys=E.table_stats()["n_keys"])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_fused_shard_two_gpus_ipc_vs_oracle_simulation(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    out = str(tmp_path / "shard{rank}.npz")
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    shards, workers, per_step = simulate(world, STEPS, KW, batch_fn)
    keys = all_keys(world, STEPS, batch_fn)
    own = key_owner_np(keys, world)
    for s in range(world):
        got = np.load(out.format(rank=s))
        oscal, ohasv, oV, ocg = oracle_state(shards[s].M, keys[own == s])
        assert np.array_equal(got["hasv"], ohasv)
        assert np.array_equal(got["scal"][:, 0], oscal[:, 0])
        assert_close(got["scal"][:, 1:], oscal[:, 1:], what=f"shard {s} w/sqrt_g/z", **STATE_TOL)
        assert_close(got["V"], oV, what=f"shard {s} V", **STATE_TOL)
        assert_close(got["cg"], ocg, what=f"shard {s} cg", **STATE_TOL)
        assert got["nkeys"] == shards[s].M.size()
        for step in range(STEPS):
            ref = per_step[step][s]
            assert abs(got["prog"][step][0] - ref[0]) <= 1e-4 * abs(ref[0]) + 1e-4
            assert abs(got["prog"][step][1] - ref[1]) <= 1e-4 * abs(ref[1]) + 1e-5
