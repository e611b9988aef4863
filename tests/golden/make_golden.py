"""Generate the committed golden fixtures from the UNMODIFIED reference.

Needs the reference's sources, from which `make -C oracle ref` builds oracle/_ref (see oracle/Makefile):

    python tests/golden/make_golden.py               # all three files
    python tests/golden/make_golden.py ref_checks    # only ref_checks.npz

Writes tests/golden/rcv1_100.npz  -- the reference's own 100-row fixture
(/root/reference/tests/data, tests/README.md:5-7) as parsed by the reference's
BatchReader + dmlc LibSVMParser (so values carry the reference's float parsing), and
tests/golden/ref_outputs.npz -- outputs of the compiled reference (FMLoss, SGDUpdater,
Localizer, SGDLearner) on that fixture and on small seeded synthetic batches, and
tests/golden/ref_checks.npz -- the reference's outputs on the random inputs of
tests/test_oracle_vs_ref.py and the batches its BatchReader yields in the cases of
tests/test_host_cpp.py::test_shuffled_batches_equal_the_reference_reader.
Tests read only these files: they need neither the reference nor oracle/_ref.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DATA = "/root/reference/tests/data"

# one batch of the reference's BatchReader, read from the start in a fresh interpreter: it shuffles with rand(),
# process-wide state.  Prints: batch index, rows, nnz, hash of the ids, hash of the labels, has values
_REF_BATCH = r"""
import sys
sys.path.insert(0, sys.argv[1])
from oracle import oracle as O
path, part, nparts, bs, shuf, neg, which = sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]), int(sys.argv[6]), float(sys.argv[7]), int(sys.argv[8])
r = O.ref_read_batch(path, "libsvm", part, nparts, bs, shuf, neg, which)
if r is None:
    print("END")
else:
    off, lab, idx, val = r
    hi = hl = 0
    for x in idx.tolist():
        hi = (hi * 1000003 + x) & 0xFFFFFFFFFFFFFFFF
    for y in lab.tolist():
        hl = (hl * 1000003 + (1 if y > 0 else 2)) & 0xFFFFFFFFFFFFFFFF
    print(which, len(lab), len(idx), hi, hl, 1 if val is not None else 0)
"""


def synth_batches(seed, nbatch, B, max_nnz, id_space, with_values):
    rng = np.random.default_rng(seed)
    out = []
    for b in range(nbatch):
        nnzr = rng.integers(0, max_nnz + 1, B)
        off = np.concatenate([[0], np.cumsum(nnzr)]).astype(np.uint64)
        n = int(off[-1])
        idx = (rng.integers(0, id_space, n).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(3)
        val = rng.random(n).astype(np.float32) if (with_values and b % 2 == 0) else None
        lab = np.where(rng.random(B) < 0.35, 1.0, -1.0).astype(np.float32)
        out.append((off, lab, idx, val))
    return out


def fixtures():
    off, lab, idx, val = O.ref_read_batch(REF_DATA, "libsvm", 0, 1, 100)
    np.savez_compressed(os.path.join(HERE, "rcv1_100.npz"), offset=off, label=lab, index=idx, value=val)

    out = {}
    # --- Localizer (tests/cpp/localizer_test.cc) ---
    lidx, keys, cnt, _ = O.ref_localize(off, idx, val, lab)
    out["loc_lidx"], out["loc_keys"], out["loc_cnt"] = lidx, keys, cnt
    l2, k2, c2, _ = O.ref_localize(off, idx, val, lab, max_index=1000)
    out["loc1000_lidx"], out["loc1000_keys"], out["loc1000_cnt"] = l2, k2, c2
    uidx = O.reverse_bytes_np(keys)

    # --- FMLoss.NoV / FMLoss.HasV (tests/cpp/fm_loss_test.cc:12-83) ---
    R0 = O.RefOracle(V_dim=0)
    w = (uidx.astype(np.float64) / 5e4).astype(np.float32)
    p0 = R0.predict(off, lidx, val, w, None, None, lab)
    g0 = R0.calc_grad(off, lidx, val, lab, w, p0)
    out["nov_w"], out["nov_pred"], out["nov_grad"] = w, p0, g0
    out["nov_objv"] = np.float32(R0.evaluate(lab, p0))
    k = 5
    U = len(uidx)
    W = np.zeros((U, k + 1), np.float32)
    W[:, 0] = w
    for j in range(1, k + 1):
        W[:, j] = (uidx.astype(np.int64) * j / 5e5).astype(np.float32)
    w_pos = (np.arange(U) * (k + 1)).astype(np.int32)
    V_pos = w_pos + 1
    R5 = O.RefOracle(V_dim=k)
    p5 = R5.predict(off, lidx, val, W.ravel(), w_pos, V_pos, lab)
    g5 = R5.calc_grad(off, lidx, val, lab, W.ravel(), p5, w_pos, V_pos)
    out["hasv_w"], out["hasv_pred"], out["hasv_grad"] = W.ravel(), p5, g5
    out["hasv_objv"] = np.float32(R5.evaluate(lab, p5))

    # --- SGDLearner.Basic (tests/cpp/sgd_learner_test.cc), all 20 epochs (stop_rel_objv=0) ---
    tr = O.ref_sgd_learner_run(data_in=REF_DATA, V_dim=0, l2=1, l1=1, lr=1, num_jobs_per_epoch=1,
                               batch_size=100, max_num_epochs=20, stop_rel_objv=0)
    out["sgd_v0_trace"] = tr

    # --- the reference's own SGDLearner with V_dim > 0 and a validation set (unpinned by reference tests): the
    #     trace the GPU-plugged learner of integration/ must reproduce (tests/test_gpu_reference_binding.py) ---
    kwl = dict(data_in=REF_DATA, data_val=REF_DATA, V_dim=8, l1=0.05, l2=0.01, lr=0.1, V_lr=0.05, V_threshold=1,
               V_l2=0.01, V_init_scale=0.1, seed=3, num_jobs_per_epoch=1, batch_size=100, max_num_epochs=12,
               stop_rel_objv=0, stop_val_auc=-1e9)
    out["sgd_v8_learner_kwargs"] = np.array([f"{a}={b}" for a, b in kwl.items() if a not in ("data_in", "data_val")])
    out["sgd_v8_learner_trace"] = O.ref_sgd_learner_run(**kwl)

    # --- V_dim>0 SGD on the fixture through the reference step (unpinned by reference tests) ---
    kw = dict(V_dim=8, l1=0.05, l2=0.01, lr=0.1, V_lr=0.05, V_threshold=1, V_l2=0.01,
              V_init_scale=0.1, seed=3)
    Rv = O.RefOracle(**kw)
    prog = []
    for ep in range(12):
        pr = Rv.sgd_step(off, idx, val, lab, True, ep == 0)
        prog.append(pr.copy())
    out["sgd_v8_kwargs"] = np.array([f"{a}={b}" for a, b in kw.items()])
    out["sgd_v8_trace"] = np.array(prog)
    vals, lens = Rv.get(keys)
    out["sgd_v8_final_vals"], out["sgd_v8_final_lens"] = vals, lens

    # --- seeded synthetic batches: binary + valued, ragged, empty rows, duplicate ids ---
    kw2 = dict(V_dim=16, l1=0.02, l2=0.0, lr=0.2, V_lr=0.1, V_threshold=2, V_l2=0.001,
               V_init_scale=0.2, seed=11)
    Rs = O.RefOracle(**kw2)
    batches = synth_batches(5, 6, 96, 24, 400, True)
    prog = []
    for ep in range(3):
        for b, (o, l, i, v) in enumerate(batches):
            pr = Rs.sgd_step(o, i, v, l, True, ep == 0)
            prog.append(pr.copy())
    out["syn_kwargs"] = np.array([f"{a}={b}" for a, b in kw2.items()])
    out["syn_trace"] = np.array(prog)
    allkeys = np.unique(np.concatenate([O.reverse_bytes_np(i) for (_, _, i, _) in batches]))
    vals, lens = Rs.get(allkeys)
    out["syn_keys"], out["syn_final_vals"], out["syn_final_lens"] = allkeys, vals, lens
    for b, (o, l, i, v) in enumerate(batches):
        out[f"syn{b}_offset"], out[f"syn{b}_label"], out[f"syn{b}_index"] = o, l, i
        if v is not None:
            out[f"syn{b}_value"] = v
    # AUC on an untied prediction vector
    rng = np.random.default_rng(9)
    pa = rng.standard_normal(500).astype(np.float32)
    la = np.where(rng.random(500) < 0.3, 1.0, -1.0).astype(np.float32)
    out["auc_pred"], out["auc_label"] = pa, la
    out["auc_value"] = np.float32(O.ref_auc(la, pa))
    np.savez_compressed(os.path.join(HERE, "ref_outputs.npz"), **out)
    print("wrote", {k: getattr(v, "shape", None) for k, v in out.items()})


def ref_checks():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_host_cpp as H
    import test_oracle_vs_ref as T
    out = {}
    # --- FMLoss / Localizer on random batches (test_oracle_vs_ref.py::test_loss_bit_exact) ---
    for V_dim, valued in T.LOSS_CASES:
        tag = f"loss_v{V_dim}_{int(valued)}_"
        # the batch alone first: the weights loss_case draws after it need its number of distinct keys
        rng = np.random.default_rng(V_dim * 2 + int(valued))
        off, lab, idx, val = T.rand_batch(rng, 200, 30, 500, valued)
        lidx, keys, cnt, _ = O.ref_localize(off, idx, val, lab)
        off, lab, idx, val, W, w_pos, V_pos = T.loss_case(V_dim, valued, len(keys))
        R = O.RefOracle(V_dim=V_dim)
        pred = R.predict(off, lidx, val, W, w_pos, V_pos, lab)
        out[tag + "lidx"], out[tag + "keys"], out[tag + "cnt"] = lidx, keys, cnt
        out[tag + "pred"] = pred
        out[tag + "grad"] = R.calc_grad(off, lidx, val, lab, W, pred, w_pos, V_pos)
        out[tag + "objv"] = np.float32(R.evaluate(lab, pred))
    # --- SGDUpdater trajectory (test_oracle_vs_ref.py::test_updater_trajectory_bit_exact) ---
    R = O.RefOracle(**T.UPDATER_KW)
    prog, seen = [], []
    for step, (off, lab, idx, val) in enumerate(T.updater_batches()):
        prog.append(R.sgd_step(off, idx, val, lab, *T.updater_flags(step)).copy())
        seen.append(O.reverse_bytes_np(idx))
    keys = np.unique(np.concatenate(seen))
    out["updater_progress"], out["updater_keys"] = np.array(prog), keys
    out["updater_vals"], out["updater_lens"] = R.get(keys)
    # --- BatchReader shuffle + negative sampling (test_host_cpp.py::test_shuffled_batches_equal_the_reference_reader) ---
    d = np.load(os.path.join(HERE, "rcv1_100.npz"))
    with tempfile.TemporaryDirectory() as tmp:
        data = os.path.join(tmp, "rcv1_100.libsvm")
        H.write_libsvm(d, data)
        for case in H.READER_CASES:
            lines = []
            for b in range(case[-1]):
                r = subprocess.run([sys.executable, "-c", _REF_BATCH, ROOT, data] + [str(x) for x in case[:-1]] + [str(b)],
                                   capture_output=True, text=True, check=True)
                lines.append(r.stdout.strip().split("\n")[-1])
            out[H.reader_tag(*case)] = np.array([x for x in lines if x != "END"])
    np.savez_compressed(os.path.join(HERE, "ref_checks.npz"), **out)
    print("wrote", {k: getattr(v, "shape", None) for k, v in out.items()})


if __name__ == "__main__":
    O.build(ref=True)
    which = sys.argv[1:] or ["fixtures", "ref_checks"]
    if "fixtures" in which:
        fixtures()
    if "ref_checks" in which:
        ref_checks()
