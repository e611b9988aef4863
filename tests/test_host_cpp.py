"""The host-side C++ mirror of the reference's Learner/Loss/Updater/Store API (difacto_b200/host):
the reference's own gtest cases re-expressed against it (host_tests.cc) and the CLI/.conf surface."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "difacto_b200", "host", "bin")
GOLDEN_REF_CHECKS = os.path.join(ROOT, "tests", "golden", "ref_checks.npz")


@pytest.fixture(scope="session")
def host_bin():
    sys.path.insert(0, ROOT)
    from difacto_b200 import build as eb
    from difacto_b200.host import build as hb
    eb.build()
    hb.build()
    return BIN


def write_libsvm(rcv1, path):
    """the reference's 100-row fixture as libsvm text (%.9g round-trips float32 exactly)"""
    off, lab, idx, val = rcv1["offset"], rcv1["label"], rcv1["index"], rcv1["value"]
    with open(path, "w") as f:
        for r in range(len(lab)):
            feats = " ".join(f"{int(idx[j])}:{val[j]:.9g}" for j in range(int(off[r]), int(off[r + 1])))
            f.write(f"{int(lab[r])} {feats}\n")


@pytest.fixture(scope="session")
def libsvm_fixture(tmp_path_factory, rcv1):
    path = tmp_path_factory.mktemp("data") / "rcv1_100.libsvm"
    write_libsvm(rcv1, path)
    return str(path)


def test_host_unit_cases_cpu(host_bin, libsvm_fixture):
    env = dict(os.environ, DFB_TEST_DATA=libsvm_fixture)
    out = subprocess.run([os.path.join(host_bin, "host_tests"), "-Gpu"], env=env, capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "Localizer.Base" in out.stdout and "BatchReader.PartRead" in out.stdout and "0 failed" in out.stdout
    assert "BatchReader.StreamedChunks" in out.stdout


# (part, nparts, batch_size, shuffle window, negative sampling, batches); the reference's batches of every case are
# stored in tests/golden/ref_checks.npz (tests/golden/make_golden.py)
READER_CASES = [(0, 1, 10, 30, 1.0, 5), (1, 2, 7, 21, 0.5, 4)]


def reader_tag(part, nparts, bs, shuf, neg, nb):
    return f"reader_{part}_{nparts}_{bs}_{shuf}_{neg:g}_{nb}"


@pytest.mark.parametrize("part,nparts,bs,shuf,neg,nb", READER_CASES)
def test_shuffled_batches_equal_the_reference_reader(host_bin, libsvm_fixture, part, nparts, bs, shuf, neg, nb):
    """shuffle window + negative down-sampling: the host BatchReader in its reference order (libstdc++'s
    std::random_shuffle on rand(), persistent permutation, rand_r seed 0: src/reader/batch_reader.cc:8-78) yields the
    very batches of the reference's BatchReader, row for row: per batch its index, rows, nnz, a hash of the ids, a hash
    of the labels and whether it carries values, as the compiled reference printed them."""
    ours = subprocess.run([os.path.join(host_bin, "batch_dump"), libsvm_fixture, str(part), str(nparts), str(bs), str(shuf),
                           str(neg), str(nb), "reference"], capture_output=True, text=True)
    assert ours.returncode == 0, ours.stderr
    ref = [str(r) for r in np.load(GOLDEN_REF_CHECKS)[reader_tag(part, nparts, bs, shuf, neg, nb)]]
    assert len(ref) >= 3
    assert ours.stdout.strip().split("\n") == ref
    # the seeded order (num_gpus > 1: concurrent readers) is a different permutation of the same rows
    seeded = subprocess.run([os.path.join(host_bin, "batch_dump"), libsvm_fixture, str(part), str(nparts), str(bs), str(shuf),
                             "1.0", str(nb), "seeded"], capture_output=True, text=True)
    assert seeded.returncode == 0 and len(seeded.stdout.strip().split("\n")) == nb


def test_cli_conf_surface(host_bin, tmp_path, libsvm_fixture):
    conf = tmp_path / "sgd.conf"
    conf.write_text(f"# data\ndata_in = {libsvm_fixture}\nl1 = 1\nlr = .1\nlearner = sgd\n"
                    "max_num_epochs = 10\nbatch_size = 100\n\n# embedding term\nV_dim = 0\n")
    exe = os.path.join(host_bin, "difacto_b200")
    out = subprocess.run([exe, f"argfile={conf}", "V_dim=16", "dry_run=1"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    kv = dict(line.split(" = ") for line in out.stdout.strip().split("\n"))
    assert kv["learner"] == "sgd" and kv["batch_size"] == "100" and kv["lr"] == ".1"
    assert kv["V_dim"] == "0"        # dmlc::Config: the last occurrence wins and the argfile comes last
    # batch_size is a required field (src/sgd/sgd_param.h:58): the README quick-start line fails the same way
    out = subprocess.run([exe, f"data_in={libsvm_fixture}", "V_dim=2", "dry_run=1"], capture_output=True, text=True)
    assert out.returncode != 0 and "batch_size" in out.stderr
    out = subprocess.run([exe, "task=predict", f"data_in={libsvm_fixture}", "batch_size=1", "dry_run=1"],
                         capture_output=True, text=True)
    assert out.returncode == 0 and "task = predict" in out.stdout
    out = subprocess.run([exe, "task=convert", f"data_in={libsvm_fixture}", "batch_size=1"], capture_output=True, text=True)
    assert out.returncode != 0 and "convert" in out.stderr


@pytest.mark.gpu
def test_host_unit_cases_gpu(host_bin, libsvm_fixture):
    env = dict(os.environ, DFB_TEST_DATA=libsvm_fixture)
    out = subprocess.run([os.path.join(host_bin, "host_tests"), "Gpu"], env=env, capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "GpuSGDLearner.Basic" in out.stdout and "0 failed" in out.stdout


@pytest.mark.gpu
def test_cli_trains_like_the_reference(host_bin, libsvm_fixture, refout):
    exe = os.path.join(host_bin, "difacto_b200")
    out = subprocess.run([exe, f"data_in={libsvm_fixture}", "V_dim=0", "l1=1", "l2=1", "lr=1", "batch_size=100",
                          "num_jobs_per_epoch=1", "max_num_epochs=20", "stop_rel_objv=0", "table_capacity=8192",
                          "foo=bar"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "Unrecognized keyword argument" in out.stderr and "foo = bar" in out.stderr
    losses = [float(l.split("loss = ")[1].split(",")[0]) for l in out.stdout.split("\n") if "Training: loss" in l]
    gold = refout["sgd_v0_trace"][:, 0]
    assert len(losses) == 20
    # printed with 6 significant digits, like the reference's log line (sgd_utils.h:47-51)
    assert np.allclose(losses, gold, rtol=2e-5, atol=1e-3)


@pytest.mark.gpu
def test_cli_model_out_then_model_in(host_bin, libsvm_fixture, tmp_path):
    """model_out / model_in (sgd_param.h:53-54; declared but never acted on by the reference):
    10 epochs + save, then load + 10 more epochs == 20 epochs in one run"""
    exe = os.path.join(host_bin, "difacto_b200")
    common = [f"data_in={libsvm_fixture}", "V_dim=8", "l1=0.1", "lr=0.5", "V_threshold=1", "batch_size=100",
              "num_jobs_per_epoch=1", "stop_rel_objv=0", "table_capacity=8192", "shuffle=0"]
    model = str(tmp_path / "model.dfb")

    def losses(args):
        out = subprocess.run([exe] + common + args, capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        return [float(l.split("loss = ")[1].split(",")[0]) for l in out.stdout.split("\n") if "Training: loss" in l], out.stdout

    full, _ = losses(["max_num_epochs=20"])
    first, so = losses(["max_num_epochs=10", f"model_out={model}"])
    assert "Saved model" in so and os.path.getsize(model) > 1000
    assert first == full[:10]
    # the resumed run does not re-push feature counts of "epoch 0"? it does (epoch numbering restarts), exactly
    # like re-running the reference binary would; compare against the loss level instead of bit equality
    second, so2 = losses(["max_num_epochs=10", f"model_in={model}"])
    assert "Loaded model" in so2
    assert second[0] < first[0] and abs(second[0] - full[10]) < 0.05 * full[10]


def _write_synthetic_libsvm(path, rows, nnz, id_space, seed, binary):
    rng = np.random.default_rng(seed)
    batches = []
    with open(path, "w") as f:
        for r in range(rows):
            n = int(rng.integers(1, nnz + 1))
            ids = np.unique(rng.zipf(1.3, n) % id_space)
            lab = 1 if rng.random() < 0.3 else -1
            if binary:
                f.write(f"{lab} " + " ".join(f"{int(i)}:1" for i in ids) + "\n")
            else:
                vals = (rng.random(len(ids)).astype(np.float32) + 0.1)
                f.write(f"{lab} " + " ".join(f"{int(i)}:{v:.9g}" for i, v in zip(ids, vals)) + "\n")


def _oracle_epoch_losses(path, conf, batch_size, epochs):
    """replay of SGDLearner::IterateData with the oracle: file order batches (shuffle=0), 1 job per epoch"""
    from oracle import oracle as O
    rows = [l.split() for l in open(path).read().strip().split("\n")]
    M = O.Oracle(**conf)
    losses = []
    for ep in range(epochs):
        prog = np.zeros(5, np.float32)
        for b0 in range(0, len(rows), batch_size):
            chunk = rows[b0:b0 + batch_size]
            lab = np.array([float(r[0]) for r in chunk], np.float32)
            idx, val, off = [], [], [0]
            for r in chunk:
                for t in r[1:]:
                    i, v = t.split(":")
                    idx.append(int(i))
                    val.append(np.float32(v))
                off.append(len(idx))
            val = np.array(val, np.float32)
            if np.all(val == 1):
                val = None          # BatchReader drops all-ones values (batch_reader.cc:71-73)
            M.sgd_step(np.array(off, np.uint64), np.array(idx, np.uint64), val, lab, True, ep == 0, progress=prog)
        losses.append(float(prog[0]))
    return losses


@pytest.mark.gpu
@pytest.mark.parametrize("name,conf,binary", [
    # BASELINE.json configs: rcv1_sgd.conf + V_dim=16; criteo_sgd.conf as shipped (V_dim=10: generic kernels);
    # criteo l1-regularised FTRL with V_dim=32
    ("rcv1_v16", dict(l1=1, lr=.1, V_dim=16, V_threshold=2), False),
    ("criteo_v10", dict(l1=10, l2=10, V_dim=10, V_threshold=10, V_l2=10), True),
    ("criteo_ftrl_v32", dict(l1=2, l2=1, lr=.5, V_dim=32, V_threshold=5, V_l2=1), True),
])
def test_cli_conf_runs_match_oracle(host_bin, tmp_path, name, conf, binary):
    data = str(tmp_path / f"{name}.libsvm")
    _write_synthetic_libsvm(data, rows=1500, nnz=30, id_space=3000, seed=11, binary=binary)
    conffile = tmp_path / f"{name}.conf"
    conffile.write_text("# generated\n" + f"data_in = {data}\nlearner = sgd\ntask = train\nmax_num_epochs = 4\n"
                        "batch_size = 500\nnum_jobs_per_epoch = 1\nshuffle = 0\nstop_rel_objv = 0\ntable_capacity = 16384\n"
                        + "".join(f"{k} = {v}\n" for k, v in conf.items()))
    exe = os.path.join(host_bin, "difacto_b200")
    ref = _oracle_epoch_losses(data, conf, 500, 4)
    for fused in ("1", "0"):
        out = subprocess.run([exe, f"argfile={conffile}", f"fused={fused}"], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        got = [float(l.split("loss = ")[1].split(",")[0]) for l in out.stdout.split("\n") if "Training: loss" in l]
        assert len(got) == 4
        assert np.allclose(got, ref, rtol=2e-4, atol=1e-3), (name, fused, got, ref)


@pytest.mark.gpu
def test_cli_validation_epochs(host_bin, libsvm_fixture, tmp_path):
    """data_val: every epoch runs a validation pass (Pull + Predict only, sgd_learner.cc:41-44,158-171);
    with data_val == data_in the validation loss of epoch k equals the training loss of epoch k+1's forward
    only if the model did not change -- so compare against the oracle's predict-only replay instead"""
    from oracle import oracle as O
    exe = os.path.join(host_bin, "difacto_b200")
    conf = dict(V_dim=8, l1=0.1, lr=0.5, V_threshold=1)
    out = subprocess.run([exe, f"data_in={libsvm_fixture}", f"data_val={libsvm_fixture}", "batch_size=100", "shuffle=0",
                          "num_jobs_per_epoch=1", "max_num_epochs=5", "stop_rel_objv=0", "stop_val_auc=-1",
                          "table_capacity=8192"] + [f"{k}={v}" for k, v in conf.items()], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    tr = [float(l.split("loss = ")[1].split(",")[0]) for l in out.stdout.split("\n") if "Training: loss" in l]
    va = [float(l.split("loss = ")[1].split(",")[0]) for l in out.stdout.split("\n") if "Validation: loss" in l]
    auc = [float(l.split("AUC = ")[1]) for l in out.stdout.split("\n") if "Validation: loss" in l]
    assert len(tr) == 5 and len(va) == 5
    d = np.load(os.path.join(ROOT, "tests", "golden", "rcv1_100.npz"))
    M = O.Oracle(**conf)
    for ep in range(5):
        pt = M.sgd_step(d["offset"], d["index"], d["value"], d["label"], True, ep == 0)
        pv = M.sgd_step(d["offset"], d["index"], d["value"], d["label"], False, False)
        assert abs(tr[ep] - float(pt[0])) <= 2e-4 * abs(float(pt[0])) + 1e-3
        assert abs(va[ep] - float(pv[0])) <= 2e-4 * abs(float(pv[0])) + 1e-3
        assert abs(auc[ep] - float(pv[2]) / 100.0) < 5e-3


@pytest.mark.gpu
def test_cli_task_predict(host_bin, libsvm_fixture, tmp_path, rcv1):
    """task=predict (TODO in the reference, main.cc:61-62): forward pass of a saved model"""
    from oracle import oracle as O
    exe = os.path.join(host_bin, "difacto_b200")
    conf = ["V_dim=8", "l1=0.1", "lr=0.5", "V_threshold=1", "batch_size=100", "num_jobs_per_epoch=1", "shuffle=0",
            "stop_rel_objv=0", "table_capacity=8192"]
    model, preds = str(tmp_path / "m.dfb"), str(tmp_path / "pred.txt")
    out = subprocess.run([exe, f"data_in={libsvm_fixture}", "max_num_epochs=6", f"model_out={model}"] + conf,
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    out = subprocess.run([exe, "task=predict", f"data_in={libsvm_fixture}", f"model_in={model}", f"pred_out={preds}"] + conf,
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    got = np.loadtxt(preds, dtype=np.float32)
    assert got.shape == (100,)
    M = O.Oracle(V_dim=8, l1=0.1, lr=0.5, V_threshold=1)
    for ep in range(6):
        M.sgd_step(rcv1["offset"], rcv1["index"], rcv1["value"], rcv1["label"], True, ep == 0)
    lidx, keys, _ = O.localize(rcv1["offset"], rcv1["index"])
    vals, lens = M.get(keys)
    w_pos, V_pos = O.get_pos(lens)
    ref = O.fm_predict(8, rcv1["offset"], lidx, rcv1["value"], vals, w_pos, V_pos)
    assert np.allclose(got, ref, rtol=2e-3, atol=2e-3)
    loss = float(out.stdout.split("loss = ")[1].split(",")[0])
    assert abs(loss - O.evaluate(rcv1["label"], ref)) <= 2e-3 * abs(loss) + 1e-2


def _synthetic_libsvm(path, rows, seed):
    rng = np.random.default_rng(seed)
    w = rng.normal(0, 1, 400)
    with open(path, "w") as f:
        for _ in range(rows):
            ids = np.unique(rng.integers(1, 400, rng.integers(5, 25)))
            x = rng.random(len(ids)).astype(np.float32)
            y = 1 if (w[ids] * x).sum() + rng.normal(0, 0.3) > 0 else -1
            f.write(f"{y} " + " ".join(f"{int(i) * 7919}:{float(v):.6g}" for i, v in zip(ids, x)) + "\n")


@pytest.mark.gpu
def test_cli_two_gpus_sharded_store(host_bin, tmp_path):
    """num_gpus=2: the C++ learner drives the NVLink-sharded store (dfb_shard_*) from one host thread that interleaves the enqueue phases of all GPUs,
    the worker/server split SGDLearner::RunEpoch was written for (sgd_learner.cc:78-89).  The run must learn like the
    one-GPU run (same data, same hyper-parameters; batch composition per step differs), save one snapshot per shard,
    and a reloaded model must reproduce the validation loss it was saved with."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    exe = os.path.join(host_bin, "difacto_b200")
    data, val = str(tmp_path / "train.libsvm"), str(tmp_path / "val.libsvm")
    _synthetic_libsvm(data, 4000, 1)
    _synthetic_libsvm(val, 1000, 2)
    common = [f"data_in={data}", f"data_val={val}", "V_dim=16", "l1=0.01", "l2=0.01", "lr=0.1", "V_lr=0.05", "V_threshold=2",
              "batch_size=200", "shuffle=0", "num_jobs_per_epoch=1", "max_num_epochs=4", "stop_rel_objv=0", "stop_val_auc=-1e9",
              "table_capacity=65536"]

    def losses(out, tag):
        return [float(l.split("loss = ")[1].split(",")[0]) for l in out.stdout.split("\n") if f"{tag}: loss" in l]

    one = subprocess.run([exe] + common, capture_output=True, text=True, timeout=300)
    assert one.returncode == 0, one.stderr[-2000:]
    model = str(tmp_path / "model")
    two = subprocess.run([exe] + common + ["num_gpus=2", f"model_out={model}"], capture_output=True, text=True, timeout=300)
    assert two.returncode == 0, two.stderr[-2000:]
    t1, t2, v1, v2 = losses(one, "Training"), losses(two, "Training"), losses(one, "Validation"), losses(two, "Validation")
    assert len(t2) == 4 and len(v2) == 4
    assert t2[0] == pytest.approx(t1[0], rel=0.1)                  # same rows, same start; two workers step together
    assert all(b < a for a, b in zip(t2[:-1], t2[1:]))             # it learns
    assert v2[-1] == pytest.approx(v1[-1], rel=0.05)               # like the one-GPU run (two half-size streams of batches)
    assert os.path.exists(model + "_part-0") and os.path.exists(model + "_part-1")
    # the saved shards, reloaded and scored by two GPUs again (task=predict): the validation loss they were saved with
    again = subprocess.run([exe, "task=predict", f"data_in={val}", f"model_in={model}", "num_gpus=2", "V_dim=16",
                            "batch_size=200", "table_capacity=65536"], capture_output=True, text=True, timeout=300)
    assert again.returncode == 0, again.stderr[-2000:]
    assert losses(again, "Prediction")[0] == pytest.approx(v2[-1], rel=1e-4)
