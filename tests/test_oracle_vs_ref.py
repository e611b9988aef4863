"""Bit-for-bit check of the C restatement against the compiled reference on random inputs.  The reference's
outputs on these inputs are stored in tests/golden/ref_checks.npz (written by tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest

from oracle import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_checks.npz")
LOSS_CASES = [(0, True), (3, False), (8, True), (64, False)]
UPDATER_KW = dict(V_dim=6, l1=0.6, l2=0.02, lr=0.3, V_lr=0.07, V_threshold=12, V_l2=0.05,
                  V_init_scale=0.3, lr_beta=0.5, V_lr_beta=2.0, seed=99)
UPDATER_STEPS = 40


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLDEN))


def rand_batch(rng, B, max_nnz, id_space, valued):
    nnzr = rng.integers(0, max_nnz + 1, B)
    off = np.concatenate([[0], np.cumsum(nnzr)]).astype(np.uint64)
    n = int(off[-1])
    idx = rng.integers(0, id_space, n).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    val = (rng.random(n).astype(np.float32) * 2 - 0.5) if valued else None
    lab = np.where(rng.random(B) < 0.4, 1.0, -1.0).astype(np.float32)
    return off, lab, idx, val


def loss_case(V_dim, valued, U):
    """inputs of one loss case: a batch, then weights for its U distinct keys (70% of them with a V row)"""
    rng = np.random.default_rng(V_dim * 2 + int(valued))
    off, lab, idx, val = rand_batch(rng, 200, 30, 500, valued)
    if V_dim == 0:
        W = rng.standard_normal(U).astype(np.float32) * 0.1
        w_pos = V_pos = None
    else:
        lens = np.where(rng.random(U) < 0.7, V_dim + 1, 1).astype(np.int32)
        w_pos, V_pos = O.get_pos(lens)
        W = rng.standard_normal(int(lens.sum())).astype(np.float32) * 0.1
    return off, lab, idx, val, W, w_pos, V_pos


def updater_batches():
    rng = np.random.default_rng(123)
    return [rand_batch(rng, 50, 15, 250, step % 3 == 0) for step in range(UPDATER_STEPS)]


def updater_flags(step):
    """(is_train, push_cnt) of every step of the trajectory"""
    return step % 7 != 6, step < 12


@pytest.mark.parametrize("V_dim,valued", LOSS_CASES)
def test_loss_bit_exact(V_dim, valued, gold):
    tag = f"loss_v{V_dim}_{int(valued)}_"
    rk = gold[tag + "keys"]
    off, lab, idx, val, W, w_pos, V_pos = loss_case(V_dim, valued, len(rk))
    lidx, keys, cnt = O.localize(off, idx)
    assert np.array_equal(lidx, gold[tag + "lidx"]) and np.array_equal(keys, rk) and np.array_equal(cnt, gold[tag + "cnt"])
    op = O.fm_predict(V_dim, off, lidx, val, W, w_pos, V_pos)
    assert np.array_equal(op, gold[tag + "pred"])
    og = O.fm_calc_grad(V_dim, off, lidx, val, lab, W, op, w_pos, V_pos)
    assert np.array_equal(og, gold[tag + "grad"])
    objv = float(gold[tag + "objv"])
    assert O.evaluate(lab, op) == pytest.approx(objv, rel=1e-6)
    assert abs(O.evaluate(lab, op) - objv) == 0.0  # 2-thread chunked sum mirrored


def test_updater_trajectory_bit_exact(gold):
    M = O.Oracle(**UPDATER_KW)
    seen = []
    for step, (off, lab, idx, val) in enumerate(updater_batches()):
        is_train, push_cnt = updater_flags(step)
        p1 = M.sgd_step(off, idx, val, lab, is_train, push_cnt)
        p2 = gold["updater_progress"][step]
        assert abs(p1[0] - p2[0]) <= 2e-5 * abs(p2[0]) and p1[1] == p2[1] and p1[4] == p2[4]
        seen.append(O.reverse_bytes_np(idx))
    keys = np.unique(np.concatenate(seen))
    assert np.array_equal(keys, gold["updater_keys"])
    a, b = M.get(keys), (gold["updater_vals"], gold["updater_lens"])
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])
    assert (a[1] > 1).sum() > 20 and (a[1] == 1).sum() > 0
