#!/usr/bin/env python
"""bench.py -- FM-SGD examples/sec on synthetic Criteo-shaped CSR minibatches (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one minibatch through the whole hot path of SGDLearner::IterateData
(src/sgd/sgd_learner.cc:138-177 of the reference): Pull -> FM forward -> logloss/AUC/penalty ->
FM backward -> Push (FTRL on w, AdaGrad on V).  Workload (default): B=65536 rows x 100 nnz,
feature ids uniform over [0, 1e9), binary values, V_dim=64, V_threshold=0 and l1=0 so that every
key owns a V row (the bandwidth worst case of SURVEY.md 8d, config "S").

Printed JSON line (rank 0):
  value        examples/s, inputs already resident in HBM, CUDA-event timed, max over ranks
  e2e          same metric through the C-ABI call a user makes, every step's inputs copied
               host->device from pinned memory and every step's Progress read back
  roofline     dominant kernel (fused FM forward+backward): algorithmic bytes / event-timed
               duration vs the measured HBM peak in MEASURED_PEAKS.json
  cpu_baseline the reference's own CPU SGD path (oracle/_ref) on a bounded sample, host cores

--dump-outputs DIR (one GPU) writes what the timed steps left behind as DIR/<name>.npy, so that two builds can be
compared output for output on the same seeded inputs (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--nnz", type=int, default=100)
    ap.add_argument("--vdim", type=int, default=64)
    ap.add_argument("--id-space", type=int, default=10 ** 9)
    ap.add_argument("--workload", default="synthetic", choices=["synthetic", "criteo39", "gisette", "rcv1"])
    ap.add_argument("--hyper", default="allV", choices=["allV", "criteo_conf", "ftrl_l1", "rcv1_conf"])
    ap.add_argument("--no-sweep", action="store_true", help="skip the short runs of the other named configs")
    ap.add_argument("--cold", action="store_true", help="cold table: every timed batch brings only new keys")
    ap.add_argument("--working-set", type=int, default=8, help="distinct batches cycled (per rank)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-overlap-auc", action="store_true", help="keep everything on one stream (profiler runs)")
    ap.add_argument("--cpu-rows", type=int, default=0,
                    help="rows per CPU batch (0: 4096 for the in-run cpu_baseline sample, the full batch for --impl reference)")
    ap.add_argument("--engine-kw", default="", help="extra engine kwargs k=v,k=v (tuning experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the model entries of a seeded sample of the last batch's keys "
                         "and the progress counters as DIR/<name>.npy (one GPU only)")
    return ap.parse_args()


# --------------------------------------------------------------------------------------
# workload
# --------------------------------------------------------------------------------------
def reverse_bytes_np(x):
    """nibble reversal of a uint64 array (include/difacto/base.h:39-51 of the reference)"""
    x = x.astype(np.uint64, copy=True)
    x = (x << np.uint64(32)) | (x >> np.uint64(32))
    x = ((x & np.uint64(0x0000FFFF0000FFFF)) << np.uint64(16)) | ((x & np.uint64(0xFFFF0000FFFF0000)) >> np.uint64(16))
    x = ((x & np.uint64(0x00FF00FF00FF00FF)) << np.uint64(8)) | ((x & np.uint64(0xFF00FF00FF00FF00)) >> np.uint64(8))
    x = ((x & np.uint64(0x0F0F0F0F0F0F0F0F)) << np.uint64(4)) | ((x & np.uint64(0xF0F0F0F0F0F0F0F0)) >> np.uint64(4))
    return x


GISETTE_NNZ = 5000      # gisette: 5000 dense features per example (SURVEY.md 5, the "long row" shape)
RCV1_NNZ, RCV1_IDS = 74, 47236      # rcv1.binary: ~74 tf-idf features per document out of 47236 (SURVEY.md 8d, config R)


def nnz_of(args):
    return {"synthetic": args.nnz, "criteo39": 39, "gisette": GISETTE_NNZ, "rcv1": RCV1_NNZ}[args.workload]


def gen_raw_batch(args, seed, rows=None):
    """raw (un-localized) CSR<u64> minibatch of the named shape: (offset, label, ids[, values])"""
    rng = np.random.default_rng(seed)
    B = rows or args.batch
    if args.workload == "gisette":
        # every example holds all 5000 features, real-valued (gisette's pixel features scaled to [0, 1))
        nnz = GISETTE_NNZ
        ids = np.tile(np.arange(1, nnz + 1, dtype=np.uint64), B)
        off = (np.arange(B + 1, dtype=np.uint64) * np.uint64(nnz))
        lab = np.where(rng.random(B) < 0.5, 1.0, -1.0).astype(np.float32)
        return off, lab, ids, (rng.random(B * nnz, dtype=np.float32) * np.float32(0.02))
    if args.workload == "rcv1":
        # BASELINE.json configs[1] stand-in: 74 real-valued (tf-idf-like, U(0, 0.3)) features per row, ids over 47236
        nnz = RCV1_NNZ
        ids = rng.integers(1, RCV1_IDS + 1, B * nnz).astype(np.uint64)
        off = (np.arange(B + 1, dtype=np.uint64) * np.uint64(nnz))
        lab = np.where(rng.random(B) < 0.5, 1.0, -1.0).astype(np.float32)
        return off, lab, ids, (rng.random(B * nnz, dtype=np.float32) * np.float32(0.3))
    if args.workload == "criteo39":
        # 13 "integer" + 26 "categorical" groups, id = (hash << 12) | group (criteo_parser.h:68-88), Zipf-ish hashes
        nnz = 39
        gid = np.tile(np.arange(nnz, dtype=np.uint64), B)
        z = rng.zipf(1.05, B * nnz).astype(np.uint64) % np.uint64(1 << 26)
        ids = (z << np.uint64(12)) | gid
    else:
        nnz = args.nnz
        ids = rng.integers(0, args.id_space, B * nnz).astype(np.uint64)
    off = (np.arange(B + 1, dtype=np.uint64) * np.uint64(nnz))
    lab = np.where(rng.random(B) < 0.25, 1.0, -1.0).astype(np.float32)
    return off, lab, ids, None


def localize_np(ids):
    """host restatement of Localizer::Compact (src/data/localizer.cc:11-103) with numpy:
    reversed keys, ascending unique, occurrence counts, rank of every nnz"""
    rk = reverse_bytes_np(ids)
    keys, lidx, cnt = np.unique(rk, return_inverse=True, return_counts=True)
    return lidx.astype(np.uint32), keys.astype(np.uint64), cnt.astype(np.float32)


def hyper(args):
    """hyper-parameters by --hyper (other values are the defaults of src/sgd/sgd_param.h:94-106):
       allV         V_threshold=0, l1=0: every key owns a V row (the bandwidth worst case of SURVEY.md 8d, config S)
       criteo_conf  the regularisation of example/criteo_sgd.conf:10-17 (l1=l2=V_l2=10, V_threshold=10)
       ftrl_l1      the defaults (l1=1, V_threshold=10): l1-regularised FTRL, most keys have w == 0 and therefore no V
       rcv1_conf    example/rcv1_sgd.conf (l1=1, lr=.1), the other values at their defaults"""
    base = dict(V_dim=args.vdim, l1=0.0, l2=0.0, lr=0.01, lr_beta=1.0, V_l2=0.01, V_lr=0.01, V_lr_beta=1.0,
                V_init_scale=0.01, V_threshold=0, seed=0)
    if args.hyper == "criteo_conf":
        base.update(l1=10.0, l2=10.0, V_l2=10.0, V_threshold=10)
    elif args.hyper == "ftrl_l1":
        base.update(l1=1.0, l2=0.0, V_threshold=10)
    elif args.hyper == "rcv1_conf":        # example/rcv1_sgd.conf: l1 = 1, lr = .1 (+ V_dim given on the command line)
        base.update(l1=1.0, lr=0.1, V_threshold=10)
    return base


# --------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md)
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.05:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1]))
                smax = max(smax, float(f[2]))
                for n, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------
# the reference arm / cpu baseline: the reference's own CPU SGD path (oracle/_ref), bounded sample
# --------------------------------------------------------------------------------------
def cpu_reference_run(args, steps, warmup, nthreads=None, rows=None):
    """the reference's own CPU SGD path through oracle/_ref (the UNMODIFIED reference compiled here), else the
    oracle port: Localizer::Compact -> Update(kFeaCount) -> Get -> GetPos -> Predict -> Evaluate -> penalty -> AUC ->
    CalcGrad -> Update(kGradient) on raw batches of the same shape and hyper-parameters"""
    from oracle import oracle as O   # test infrastructure: allowed here as the CPU baseline only
    cores = os.cpu_count() or 1
    if nthreads is None:
        nthreads = max(2, min(48, cores))     # loss.h:80-83 caps nthreads at < 50
    kind = "reference" if O.have_ref() else "port"
    kw = hyper(args)
    rows = rows or args.cpu_rows or 4096
    nb = 2
    batches = [gen_raw_batch(args, 10_000 + b, rows=rows) for b in range(nb)]
    eng = O.RefOracle(nthreads=nthreads, **kw) if kind == "reference" else O.Oracle(**kw)
    # table warm-up: two passes so that every key of the sample has reached its steady state (as on the GPU arm)
    for p in range(2):
        for (off, lab, ids, val) in batches:
            eng.sgd_step(off, ids, val, lab, True, p == 0)
    for t in range(warmup):
        off, lab, ids, val = batches[t % nb]
        eng.sgd_step(off, ids, val, lab, True, False)
    secs = np.zeros(6, np.float64)
    t0 = time.perf_counter()
    for t in range(steps):
        off, lab, ids, val = batches[t % nb]
        if kind == "reference":
            eng.sgd_step(off, ids, val, lab, True, False, seconds=secs)
        else:
            eng.sgd_step(off, ids, val, lab, True, False)
    dt = time.perf_counter() - t0
    ex_s = steps * rows / dt
    sample = (f"{steps} steps x {rows} rows x {nnz_of(args)} nnz "
              f"(same shape/hyper-parameters, table warmed, Localizer::Compact included)")
    return dict(value=ex_s, unit="examples/s", cores=int(nthreads if kind == "reference" else 1), kind=kind,
                sample=sample, ms_per_step=dt / steps * 1e3, host_cores=cores, rows=rows,
                stage_seconds=dict(zip(["localize", "feacnt", "get", "predict", "calcgrad", "update"],
                                       [float(x) for x in secs])))


def main_reference(args, rank, world):
    """--impl reference: the reference's CPU path on the box's host cores, SAME config as the B200 arm: every step
    is one full batch (args.batch rows) unless --cpu-rows bounds it"""
    if rank != 0:
        return
    rows = args.cpu_rows or args.batch
    res = cpu_reference_run(args, args.steps, args.warmup, rows=rows)
    line = {
        "impl": "reference", "metric": metric_name(args), "value": res["value"], "unit": "examples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, None),
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "host_cores": res["host_cores"], "stage_seconds": res["stage_seconds"],
        "rows_per_step": res["rows"],
    }
    print(json.dumps(line))


def metric_name(args):
    return f"FM-SGD examples/sec, synthetic Criteo-shape CSR, V_dim={args.vdim}"


def workload_config(args, extra):
    nnz = nnz_of(args)
    cfg = {"workload": (f"synthetic CSR (BASELINE.json configs[4] / SURVEY 8d 'S'): batch {args.batch} x {nnz} nnz/row, "
                        f"ids uniform over [0,{args.id_space}), binary values, V_dim={args.vdim}"
                        + (", every key owns a V row" if args.hyper == "allV" else f", hyper={args.hyper}")
                        if args.workload == "synthetic" else
                        f"gisette-shaped CSR: batch {args.batch} x {GISETTE_NNZ} dense real-valued features, V_dim={args.vdim}, "
                        f"hyper={args.hyper}" if args.workload == "gisette" else
                        f"rcv1-shaped CSR (BASELINE.json configs[1] stand-in): batch {args.batch} x {RCV1_NNZ} real-valued nnz/row over "
                        f"{RCV1_IDS} ids, V_dim={args.vdim}, hyper={args.hyper}" if args.workload == "rcv1" else
                        f"criteo-shaped CSR: batch {args.batch} x 39 nnz/row, Zipf ids with 12-bit group id, "
                        f"V_dim={args.vdim}, hyper={args.hyper}"),
           "global_batch": args.batch * args.gpus, "batch_per_gpu": args.batch, "nnz_per_row": nnz, "V_dim": args.vdim,
           "id_space": args.id_space, "hyper": hyper(args),
           "l2_policy": "inputs_exceed_l2 (each step gathers/updates >1 GB of distinct table rows; "
                        "the working set of batches is cycled, never the same batch twice in a row)"}
    if extra:
        cfg.update(extra)
    return cfg


# --------------------------------------------------------------------------------------
# the B200 arm
# --------------------------------------------------------------------------------------
def load_peaks():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", FALLBACK_HBM_GBS))
    src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    return peak, src


def byte_model(B, N, U, k):
    """algorithmic bytes per launch (DESIGN.md section 4), every key owning a V row:
       K1 gather+interaction (SURVEY.md 8d): N(4k+8) + 16B; the emit variant used in training adds the p*XV rows
       (4kB + 4B); K2+K3 fused per-key reduce + FTRL/AdaGrad: per key read {entry 16, V|cg 8k, slot/vrow/col 16},
       write {entry 16, V|cg 8k}; per nnz read {p*XV row 4k, p 4, payload 4}"""
    fwd = N * (4 * k + 8) + 16 * B
    emit = fwd + B * (4 * k + 4)
    upd = U * (2 * (8 * k + 16) + 16) + N * (4 * k + 8)
    # BASELINE.md section 3 full-step model (the reference's dataflow: gradient buffer + second gather)
    step = (fwd + (N * (4 * k + 8) + 16 * B + N * 4 * (k + 1)) + U * (4 * (k + 1) + 8 * k + 12) + U * (8 * k + 12))
    return fwd, emit, upd, step


def gen_raw_set(args, nb, seed0, torch, rows=None):
    out = []
    for b in range(nb):
        off, lab, ids, val = gen_raw_batch(args, seed0 + b, rows=rows)
        out.append(dict(off=torch.from_numpy(off.view(np.int64)).pin_memory(), lab=torch.from_numpy(lab).pin_memory(),
                        ids=torch.from_numpy(ids.view(np.int64)).pin_memory(), nnz=len(ids), nrows=len(lab),
                        val=torch.from_numpy(val).pin_memory() if val is not None else None))
    return out


DUMP_MAX_BYTES = 64 << 20
DUMP_MAX_KEYS = 1 << 16


def dump_outputs(E, d, args, last_batch, prog):
    """what a caller of the timed path receives after its last step, as float arrays in d/<name>.npy:
       progress                  [loss, penalty, auc, nnz_w, nrows] of dfb_read_progress, summed over the warm-up and
                                 timed steps
       fea_cnt, w, sqrt_g, z     per key, the model entry after the last step (dfb_read_entries) ...
       has_V, V, V_cg            ... for a fixed, seeded sample of the distinct keys of the last timed batch (ascending
                                 reversed keys; every one of them was updated by that step).  has_V: 1 V row, 0 none.
    The sample is bounded so that all files together stay under DUMP_MAX_BYTES."""
    _, keys, _ = localize_np(last_batch["ids"].numpy().view(np.uint64))
    k = args.vdim
    n = min(len(keys), DUMP_MAX_KEYS, (DUMP_MAX_BYTES - (1 << 16)) // (4 * (5 + 2 * k)))
    sel = np.sort(np.random.default_rng(0).choice(len(keys), n, replace=False))
    scal, hasv, V, cg = E.read_entries(keys[sel])
    arrays = {"progress": np.array([prog.loss, prog.penalty, prog.auc, prog.nnz_w, prog.nrows], np.float64),
              "fea_cnt": scal[:, 0], "w": scal[:, 1], "sqrt_g": scal[:, 2], "z": scal[:, 3],
              "has_V": hasv.astype(np.float32), "V": V, "V_cg": cg}
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(a))


def run_single(args, local_rank, full, sampler=None):
    """one configuration on one GPU.  Batches are the reader's raw CSR<uint64> (ids not localized): every step runs
    Localizer::Compact on the GPU, then the fused minibatch.  full: also e2e, localizer check, clocks."""
    import torch
    from difacto_b200 import capi
    dev = torch.device("cuda", local_rank)
    kw = hyper(args)
    nnz_row = nnz_of(args)
    B, k = args.batch, args.vdim
    N = B * nnz_row
    steps, warm = args.steps, args.warmup
    cold = args.cold
    nb = (steps + warm + 2) if cold else args.working_set
    t_gen = time.perf_counter()
    if cold:
        # disjoint id ranges per batch: every batch brings only keys the table has never seen
        a2 = argparse.Namespace(**vars(args))
        host = []
        for b in range(nb):
            hb = gen_raw_set(a2, 1, 1 + b, torch)[0]
            hb["ids"] += b * args.id_space
            host.append(hb)
    else:
        host = gen_raw_set(args, nb, 1, torch)
    t_gen = time.perf_counter() - t_gen
    extra = dict(kv.split("=") for kv in args.engine_kw.split(",") if kv)
    # capacity: unique keys of one batch (measured with the product's own localizer) x batches
    probe = capi.Engine(device=local_rank, table_capacity=1024, V_dim=k)
    ids0 = host[0]["ids"].numpy().view(np.uint64)
    off0 = host[0]["off"].numpy().view(np.uint64)
    gl, gk, gc = probe.localize(off0, ids0)
    U0 = len(gk)
    localizer_check = None
    if full:     # the product's localizer must agree bit for bit with the harness's numpy restatement of Localizer::Compact
        nl, nk, nc = localize_np(ids0)
        localizer_check = bool(np.array_equal(gl, nl) and np.array_equal(gk, nk) and np.array_equal(gc, nc))
    probe.close()
    cap = int(nb * U0 * 1.05) + 4096
    id_bits = int(np.ceil(np.log2(float(max(args.id_space * (nb if cold else 1), 2))))) if args.workload == "synthetic" else {"gisette": 13, "rcv1": 16}.get(args.workload, 64)
    E = capi.Engine(device=local_rank, table_capacity=cap, V_capacity=cap, id_bits=min(id_bits, 64),
                    overlap_auc=0 if args.no_overlap_auc else 1, **extra, **kw)
    devb = [dict(off=h["off"].to(dev), lab=h["lab"].to(dev), ids=h["ids"].to(dev),
                 val=h["val"].to(dev) if h["val"] is not None else None) for h in host]
    torch.cuda.synchronize()

    def step_dev(b, push_cnt=False, train=True):
        d = devb[b]
        E.train_step_raw_dev(B, N, d["off"], d["ids"], d["val"], d["lab"], push_cnt, train)

    if not cold:
        # table warm-up (untimed): two passes, after which every key has reached its steady state
        for p in range(2):
            for b in range(nb):
                step_dev(b, push_cnt=(p == 0))
        E.read_progress()
    st = E.table_stats()
    if args.hyper == "allV" and not cold:
        assert st["n_vrows"] == st["n_keys"], st      # every key owns a V row

    # ---- value: raw batches resident in HBM, CUDA events over all streams of the engine ----
    order = list(range(nb)) if cold else None
    bi = (lambda t: order[t]) if cold else (lambda t: t % nb)
    for t in range(warm):
        step_dev(bi(t))
    E.sync()
    launches0 = E.launch_count()
    wall0 = time.time()
    E.time_mark(0)
    for t in range(steps):
        step_dev(bi(warm + t))
    E.time_mark(1)
    ms = E.time_elapsed_ms()
    E.sync()
    wall1 = time.time()
    launches = E.launch_count() - launches0
    prog = E.read_progress()
    value = steps * B / (ms * 1e-3)
    st2 = E.table_stats()
    if full and args.dump_outputs:
        dump_outputs(E, args.dump_outputs, args, host[bi(warm + steps - 1)], prog)

    out = {"value": value, "ms_per_step": ms / steps, "gpu_launches": int(launches),
           "loss_per_example": prog.loss / max(prog.nrows, 1), "unique_keys_per_batch": int(U0),
           "table_keys": int(st2["n_keys"]), "table_vrows": int(st2["n_vrows"]), "wall": (wall0, wall1)}
    if cold:
        out["new_keys_per_step"] = (st2["n_keys"] - st["n_keys"]) / max(steps + warm, 1)
        E.close()
        return out

    # ---- the same steps with per-stage CUDA events (kernel durations for the roofline) ----
    E.profile(True)
    for t in range(steps):
        step_dev(bi(warm + t))
    E.sync()
    stages = E.profile_read()
    E.profile(False)
    E.read_progress()
    # ---- forward-only launches (validation batches): the pure gather+interaction kernel K1 ----
    E.profile(True)
    for t in range(max(4, steps // 2)):
        step_dev(t % nb, train=False)
    E.sync()
    stages_fwd = E.profile_read()
    E.profile(False)
    E.read_progress()
    per = lambda sd, n: sd[n]["ms"] / max(sd[n]["count"], 1)      # noqa: E731
    out["stages_ms_per_step"] = {n: per(stages, n) for n in ("localize", "lookup", "fm", "auc", "update")}
    out["k1_predict_ms"] = per(stages_fwd, "fm")

    # ---- e2e: raw uint64 CSR in pinned host memory through the C-ABI, Progress of every step read back ----
    if full and not args.no_e2e:
        def submit_raw(b, nxt=None):
            r = host[b]
            E.train_step_raw_async(B, r["off"], r["ids"], r["val"], r["lab"], False, True)
            if nxt is not None:       # start the H2D of the next batch while this step runs
                n_ = host[nxt]
                E.prefetch_raw(B, n_["off"], n_["ids"], n_["val"], n_["lab"])
        for t in range(warm):
            submit_raw(t % nb)
        E.read_progress()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss_sum = 0.0
        for t in range(steps):
            submit_raw((warm + t) % nb, (warm + t + 1) % nb if t + 1 < steps else None)
            if t >= 1:
                loss_sum += E.wait_step().loss          # D2H read of step t-1's result while step t runs
        loss_sum += E.wait_step().loss
        E.sync()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out["e2e"] = {"value": steps * B / dt, "unit": "examples/s",
                      "h2d_bytes_per_step": int((B + 1) * 8 + N * 8 + B * 4 + (N * 4 if host[0]["val"] is not None else 0)), "d2h_bytes_per_step": 64,
                      "ms_per_step": dt / steps * 1e3, "mean_loss_per_step": loss_sum / steps,
                      "api": "dfb_train_step_raw_async (+ dfb_prefetch_raw) + dfb_wait_step: raw uint64 CSR from pinned "
                             "host memory, Localizer::Compact on the GPU, then the fused step; nothing else is "
                             "synchronised with the host"}
        out["wall"] = (wall0, time.time())
    out["localizer_check"] = localizer_check
    out["datagen_s"] = t_gen
    E.close()
    return out


def roofline_of(args, res, peak):
    nnz_row = nnz_of(args)
    B, k = args.batch, args.vdim
    N, U = B * nnz_row, res["unique_keys_per_batch"]
    fwd, emit, upd, step = byte_model(B, N, U, k)
    sm = res["stages_ms_per_step"]
    ach = lambda by, ms: by / (ms * 1e-3) / 1e9 if ms > 0 else 0.0      # noqa: E731
    return {"update": {"kernel_ms": sm["update"], "achieved": ach(upd, sm["update"]), "frac": ach(upd, sm["update"]) / peak,
                       "algorithmic_bytes": int(upd)},
            "k1_predict": {"kernel_ms": res["k1_predict_ms"], "achieved": ach(fwd, res["k1_predict_ms"]),
                           "frac": ach(fwd, res["k1_predict_ms"]) / peak, "algorithmic_bytes": int(fwd)},
            "k1_train": {"kernel_ms": sm["fm"], "achieved": ach(emit, sm["fm"]), "frac": ach(emit, sm["fm"]) / peak,
                         "algorithmic_bytes": int(emit)},
            "step_model_bytes": int(step),
            "step": {"achieved": ach(step, res["ms_per_step"]), "frac": ach(step, res["ms_per_step"]) / peak}}


def sweep_configs(args):
    """the other configurations BASELINE.json names, one short run each"""
    def cfg(**kw):
        a = argparse.Namespace(**vars(args))
        a.steps, a.warmup, a.working_set, a.engine_kw = 6, 3, 4, args.engine_kw
        for k_, v_ in kw.items():
            setattr(a, k_, v_)
        return a
    return [("synthetic_V8", cfg(vdim=8)), ("synthetic_V16", cfg(vdim=16)), ("synthetic_V128", cfg(vdim=128)),
            ("criteo39_V64_conf", cfg(workload="criteo39", vdim=64, hyper="criteo_conf")),
            ("criteo39_V64_allV", cfg(workload="criteo39", vdim=64, hyper="allV")),
            ("criteo39_V32_ftrl_l1", cfg(workload="criteo39", vdim=32, hyper="ftrl_l1")),
            ("synthetic_V64_cold_table", cfg(vdim=64, cold=True)),
            # long rows: 1024 examples x 5000 dense features (5.1 M nnz per step); CTA-per-row forward vs warp-per-row
            ("gisette_V64_long_rows", cfg(workload="gisette", batch=1024, vdim=64)),
            ("gisette_V64_warp_per_row", cfg(workload="gisette", batch=1024, vdim=64,
                                             engine_kw=",".join(x for x in (args.engine_kw, "long_row_nnz=0") if x))),
            # BASELINE.json configs[1]: rcv1_sgd.conf + V_dim=16 (74 real-valued nnz per row over 47236 ids: every key is
            # hot); at the batch this bench uses and at the conf's own batch_size = 100 (launch-bound)
            ("rcv1_V16_conf_batch65536", cfg(workload="rcv1", vdim=16, hyper="rcv1_conf")),
            ("rcv1_V16_conf_batch100", cfg(workload="rcv1", vdim=16, hyper="rcv1_conf", batch=100, steps=20))]


def main_b200(args, rank, world, local_rank):
    import torch
    if world > 1:
        from difacto_b200 import sharded
        return sharded.bench_main(args, rank, world, local_rank, sys.modules[__name__])

    torch.cuda.set_device(local_rank)
    peak, peak_src = load_peaks()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    res = run_single(args, local_rank, full=True)
    clocks = sampler.summary(res["wall"][0], res["wall"][1])
    nnz_row = nnz_of(args)
    B, k = args.batch, args.vdim
    rf = roofline_of(args, res, peak)
    traffic = None
    try:   # DRAM bytes per launch from the committed ncu --set full capture of the same kernel/config (not measured in this run)
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")))
        if args.batch == 65536 and nnz_row == 100 and args.workload == "synthetic" and args.hyper == "allV":
            e_ = tr.get(f"k_bwd_update<{k}>")
            if e_:
                traffic = e_["dram_read_bytes"] + e_["dram_write_bytes"]
    except Exception:
        pass
    roofline = {"bound": "hbm",
                "kernel": f"k_bwd_update<{k}> (per-key gradient reduce fused with FTRL/AdaGrad; dominant kernel of the step; "
                          "the timed stage also contains the small InitV-pass kernels)",
                "achieved": rf["update"]["achieved"], "peak": peak, "unit": "GB/s", "frac": rf["update"]["frac"],
                "traffic": traffic, "traffic_source": "profiles/ncu_traffic_r2.json (committed ncu --set full capture, per launch)",
                "peak_source": peak_src, "kernel_ms": rf["update"]["kernel_ms"],
                "algorithmic_bytes": rf["update"]["algorithmic_bytes"],
                "bytes_model": "DESIGN.md section 4 (the fused design has no gradient buffer and no second gather, so its bytes "
                               "are fewer than SURVEY 8d's K2+K3; 4kN of them are p*XV rows that stay in L2 by design)",
                "gather_interaction": dict(rf["k1_predict"], kernel=f"k_fm_fast<{k},predict> (gather+interaction, K1 of SURVEY 8d; "
                                                                    "validation launches)"),
                "gather_interaction_train": dict(rf["k1_train"], kernel=f"k_fm_fast<{k},emit> (K1 + p*XV rows)")}
    step_roof = {"model_bytes": rf["step_model_bytes"], "achieved": rf["step"]["achieved"], "frac": rf["step"]["frac"],
                 "note": "BASELINE.md section 3 full-step byte model / whole step time (the step also runs Localizer::Compact)"}

    sweep = None
    if not args.no_sweep and not args.cold:
        sweep = {}
        for name, a2 in sweep_configs(args):
            try:
                r2 = run_single(a2, local_rank, full=False)
                ent = {"value": r2["value"], "unit": "examples/s", "ms_per_step": r2["ms_per_step"],
                       "unique_keys_per_batch": r2["unique_keys_per_batch"], "table_keys": r2["table_keys"],
                       "table_vrows": r2["table_vrows"], "steps": a2.steps, "warmup": a2.warmup,
                       "hyper": a2.hyper, "V_dim": a2.vdim, "workload": a2.workload}
                if "stages_ms_per_step" in r2:
                    ent["stages_ms_per_step"] = r2["stages_ms_per_step"]
                    if a2.hyper == "allV":       # the byte model assumes a V row per key
                        rr = roofline_of(a2, r2, peak)
                        ent["k1_predict_frac"] = rr["k1_predict"]["frac"]
                        ent["k1_predict_ms"] = rr["k1_predict"]["kernel_ms"]
                        ent["update_frac"] = rr["update"]["frac"]
                if "new_keys_per_step" in r2:
                    ent["new_keys_per_step"] = r2["new_keys_per_step"]
                sweep[name] = ent
            except Exception as e:      # a sweep entry must never take the headline down with it
                sweep[name] = {"error": repr(e)}

    cpu = None
    if not args.no_cpu_baseline:
        try:
            res_c = cpu_reference_run(args, steps=3, warmup=1, rows=args.cpu_rows or 4096)
            cpu = {k2: res_c[k2] for k2 in ("value", "unit", "cores", "kind", "sample")}
            cpu["host_cores"] = res_c["host_cores"]
            res2 = cpu_reference_run(args, steps=2, warmup=1, nthreads=2, rows=args.cpu_rows or 4096)
            cpu["value_reference_default_2_threads"] = res2["value"]
        except Exception as e:   # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": "examples/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}
    sampler.stop()

    line = {
        "metric": metric_name(args), "value": res["value"], "unit": "examples/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, {"unique_keys_per_batch": res["unique_keys_per_batch"],
                                         "working_set_batches": args.working_set, "table_keys": res["table_keys"],
                                         "input": "raw CSR<uint64> resident in HBM; every step = Localizer::Compact on the GPU "
                                                  "+ the fused minibatch (SGDLearner::IterateData minus file I/O)",
                                         "parallelism": "1 gpu, table resident in HBM"}),
        "roofline": roofline, "step_roofline": step_roof, "cpu_baseline": cpu, "e2e": res.get("e2e"),
        "gpu_launches": res["gpu_launches"], "clocks": clocks, "stages_ms_per_step": res["stages_ms_per_step"],
        "loss_per_example": res["loss_per_example"], "datagen_s": res["datagen_s"],
        "gpu_localizer_equals_numpy_localizer": res["localizer_check"], "sweep": sweep,
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    args.warmup = max(args.warmup, 3)      # timing hygiene: never fewer than 3 untimed warm-up steps
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (world > 1 or args.impl != "b200"):
        sys.exit("--dump-outputs: only for the B200 arm on one GPU")
    if args.impl == "reference":
        return main_reference(args, rank, world)
    return main_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
