#!/usr/bin/env python
"""bench.py — the driver contract (see DESIGN.md §Measurement).

A "step" is one pass of hot path (i) over one batch: the fused on-device negative sampler + triple scoring
forward/backward kernel + the row optimiser on both tables (what one session.run([loss, optimizer]) of
models/basic_model.py:224-230 does in the reference).  Default workload = the shape BASELINE.json's north-star target
is quoted on (BootEA, D_W_100K_V1 shape, dim 100, batch 20000, 10 ε-truncated negatives; it fits one GPU); the
BASELINE.json configs[1] shape (D_W_15K_V1, batch 5000) is measured in the same run and reported as the
`bootea_15k` block of the same JSON line (N = 1 only).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload bootea_100k|bootea_15k]
                    [--dump-outputs DIR]

Prints ONE JSON line on rank 0.  With --dump-outputs, rank 0 also writes what the last timed step left for its caller
(see dump_outputs) as DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments can be compared
array for array.
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

WORKLOADS = {
    # BASELINE.json configs[1]; args from the reference's run/args/bootea_args_15K.json
    "bootea_15k": dict(shape="15K", dim=100, batch=5000, k=10, eps=0.9, lr=0.01, margin=0.01, neg_margin=2.0,
                       balance=0.2, name="BootEA D_W_15K_V1 shape (synthetic), dim=100, batch=5000, 10 eps-truncated negatives"),
    # the shape the north-star target is quoted on; args from bootea_args_100K.json
    "bootea_100k": dict(shape="100K", dim=100, batch=20000, k=10, eps=0.98, lr=0.01, margin=0.01, neg_margin=2.0,
                        balance=0.2, name="BootEA D_W_100K_V1 shape (synthetic), dim=100, batch=20000, 10 eps-truncated negatives"),
}
L2_FLUSH_BYTES = 512 << 20
SHAPE_ENTITIES = {"15K": 15000, "100K": 100000}      # entities per KG (openea_b200/synth.py SHAPES)
# --dump-outputs keeps under 64 MB: at dim 100 this many entity rows of weights + Adagrad slots are 52 MB
DUMP_ENTITY_ROWS = 65536
DUMP_ROW_SEED = 7


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def build_workload(wl, rank, device, world=1):
    """Synthetic KG of the workload's shape, resident on the device, plus tables and the trainer."""
    import torch
    from openea_b200 import engine as eng
    from openea_b200.synth import synth_id_arrays
    cfg = WORKLOADS[wl]
    arr = synth_id_arrays(cfg["shape"], seed=20200901)
    n_triples_global = len(arr["triples1"]) + len(arr["triples2"])
    if world > 1:   # every rank trains on the triples whose head row it owns (openea_b200/parallel.py)
        from openea_b200 import parallel as par
        arr = dict(arr)
        arr["triples1"] = np.ascontiguousarray(par.shard_triples(arr["triples1"], rank, world))
        arr["triples2"] = np.ascontiguousarray(par.shard_triples(arr["triples2"], rank, world))
    g = torch.Generator(device="cpu").manual_seed(1234)      # replicas start identical
    d = cfg["dim"]
    # init='normal': truncated normal σ = 1/√d (initializers.py:29-34); plain clamp-resampled normal here
    ent0 = torch.nn.init.trunc_normal_(torch.empty(arr["n_ent"], d), std=d ** -0.5, a=-2 * d ** -0.5, b=2 * d ** -0.5, generator=g)
    rel0 = torch.nn.init.trunc_normal_(torch.empty(arr["n_rel"], d), std=d ** -0.5, a=-2 * d ** -0.5, b=2 * d ** -0.5, generator=g)
    ent = eng.EmbeddingTable(ent0, True, "Adagrad", device)
    rel = eng.EmbeddingTable(rel0, True, "Adagrad", device)
    kg1 = eng.DeviceKG(arr["triples1"], arr["entities1"], arr["n_ent"], device)
    kg2 = eng.DeviceKG(arr["triples2"], arr["entities2"], arr["n_ent"], device)
    # ε-truncated candidate lists: k_c = int((1-ε)·N_kg) ids per entity (basic_model.py:270-271).  For the
    # benchmark the lists are random same-KG ids (the access pattern of the sampler does not depend on which).
    for kg, ents in ((kg1, arr["entities1"]), (kg2, arr["entities2"])):
        n_kg = len(ents)
        n_cand = int((1 - cfg["eps"]) * n_kg)
        idx = torch.randint(0, n_kg, (n_kg, n_cand), generator=g, dtype=torch.int32)
        cand = torch.from_numpy(ents)[idx.long()].to(torch.int32).to(device)
        kg.set_candidates(cand, ents)
    tset = eng.DeviceTripleSet([kg1.triples, kg2.triples], arr["n_ent"], arr["n_rel"], device)
    loss = eng.loss_cfg("limited", "L2", cfg["margin"], cfg["neg_margin"], cfg["balance"])
    trainer = eng.TripleTrainer(ent, rel, loss, cfg["lr"])
    T = kg1.triples.shape[0] + kg2.triples.shape[0]
    steps_per_epoch = int(np.ceil(T / cfg["batch"]))
    return dict(cfg=cfg, arr=arr, ent=ent, rel=rel, kg1=kg1, kg2=kg2, tset=tset, trainer=trainer,
                steps_per_epoch=steps_per_epoch, n_triples=T, n_triples_global=n_triples_global)


def dump_outputs(out_dir, tr, last_step_loss):
    """Writes what a caller of the timed path holds after its last step: that step's loss and the trained variables with
    their Adagrad accumulators (raw, unnormalised rows).  Entity tables larger than DUMP_ENTITY_ROWS rows are sampled:
    the same seeded, sorted row set on every run."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    ent, rel = tr.ent, tr.rel
    n = min(DUMP_ENTITY_ROWS, ent.rows)
    rows = np.sort(np.random.default_rng(DUMP_ROW_SEED).choice(ent.rows, n, replace=False))
    idx = torch.from_numpy(rows).to(ent.weight.device)
    arrays = {"last_step_loss": np.array([last_step_loss], dtype=np.float64),
              "entity_embeddings_sampled": ent.weight[idx, :ent.dim].cpu().numpy(),
              "entity_adagrad_sampled": ent.state1[idx, :ent.dim].cpu().numpy(),
              "relation_embeddings": rel.weight[:, :rel.dim].cpu().numpy(),
              "relation_adagrad": rel.state1[:, :rel.dim].cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def decode_dbg(dbg, n, t1, t2, k):
    """Host (pos, neg) [3, n] index arrays of the batch the fused kernel sampled (vectorised)."""
    rows = dbg[:n]
    tri = rows[:, 0].astype(np.int64)
    q = (tri >> 30) & 1
    idx = tri & ((1 << 30) - 1)
    hrt = np.where(q[:, None] == 0, t1[np.minimum(idx, len(t1) - 1)], t2[np.minimum(idx, len(t2) - 1)])
    pos = np.ascontiguousarray(hrt.T.astype(np.int32))
    mask = rows[:, 1].astype(np.int64)
    e = rows[:, 2:2 + k].astype(np.int32)
    head = ((mask[:, None] >> np.arange(k)[None, :]) & 1).astype(bool)
    nh = np.where(head, e, hrt[:, 0:1]).reshape(-1)
    nr = np.repeat(hrt[:, 1], k)
    nt = np.where(head, hrt[:, 2:3], e).reshape(-1)
    neg = np.ascontiguousarray(np.stack([nh, nr, nt]).astype(np.int32))
    return pos, neg


def cpu_reference_run(wl, steps, warmup, batches=None, budget_s=25.0):
    """Times the CPU oracle port of the TF step (dense normalise + dense grads + dense Adagrad) with all host
    threads on a bounded sample of the workload's batches.  Returns (pos_triples_per_s, info)."""
    from oracle import triple as orc
    from openea_b200.synth import synth_id_arrays
    cfg = WORKLOADS[wl]
    arr = synth_id_arrays(cfg["shape"], seed=20200901)
    rng = np.random.default_rng(4321)
    d = cfg["dim"]
    ent = (rng.standard_normal((arr["n_ent"], d)) / np.sqrt(d)).astype(np.float32)
    rel = (rng.standard_normal((arr["n_rel"], d)) / np.sqrt(d)).astype(np.float32)
    st = orc.DenseState(ent, rel, "Adagrad")
    if batches is None:  # host-side uniform corruption, same batch geometry (used by --impl reference)
        batches = []
        tri = np.concatenate([arr["triples1"], arr["triples2"]])
        for _ in range(4):
            sel = rng.integers(0, len(tri), size=cfg["batch"])
            pos = np.ascontiguousarray(tri[sel].T)
            neg = np.repeat(pos, cfg["k"], axis=1)
            side = rng.random(neg.shape[1]) < 0.5
            par = neg[0] & 1
            repl = (rng.integers(0, arr["n_ent"] // 2, size=neg.shape[1]) * 2 + par).astype(np.int32)
            neg[0, side] = repl[side]; neg[2, ~side] = repl[~side]
            batches.append((pos, np.ascontiguousarray(neg)))
    kw = dict(margin=cfg["margin"], neg_margin=cfg["neg_margin"], balance=cfg["balance"])
    # give the CPU arm its best thread count (OpenMP over all cores is not always the fastest on many-core hosts):
    # per candidate 2 untimed + 5 timed steps, MEDIAN; the whole sweep is reported.  One noisy sample used to pick a
    # slow setting and swing the baseline several-fold between boxes (VERDICT r01).
    ncpu = os.cpu_count() or 1
    sweep = {}
    for nt in sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, 16), min(ncpu, 8)}):
        orc.set_num_threads(nt)
        ts = []
        for rep in range(7):
            t0 = time.perf_counter()
            orc.step(st, *batches[rep % len(batches)], "limited", "L2", True, True, cfg["lr"], **kw)
            if rep >= 2:
                ts.append(time.perf_counter() - t0)
        sweep[nt] = float(np.median(ts))
    best_t = min(sweep, key=sweep.get)
    orc.set_num_threads(best_t)
    for i in range(max(1, warmup)):
        orc.step(st, *batches[i % len(batches)], "limited", "L2", True, True, cfg["lr"], **kw)
    t0 = time.perf_counter()
    done, n_pos = 0, 0
    while done < steps:
        pos, neg = batches[done % len(batches)]
        orc.step(st, pos, neg, "limited", "L2", True, True, cfg["lr"], **kw)
        n_pos += pos.shape[1]
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    info = dict(cores=best_t, steps=done, seconds=dt, thread_sweep_ms={str(k): 1e3 * v for k, v in sorted(sweep.items())},
                omp_env={k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES")},
                sample="%d steps of %d positives + %d negatives (dense TF-style step, C/OpenMP port)" % (done, batches[0][0].shape[1], batches[0][1].shape[1]))
    return n_pos / dt, info


def bench_csls(shape, device, reps=3):
    """CSLS pairs/sec: the full greedy_alignment(csls_k=10, accurate=True) equivalent (row k-means, column
    k-means, rank pass: three similarity passes + gold pre-pass) on test-link-sized inputs, device-timed."""
    import torch
    from openea_b200 import finding as F
    from openea_b200.synth import SHAPES
    n = SHAPES[shape]["links"][2]
    d = 100
    g = torch.Generator(device="cpu").manual_seed(99)
    e2 = torch.randn(n, d, generator=g)
    e1 = e2 + 0.5 * torch.randn(n, d, generator=g)
    d1, _ = F.to_device_rows(e1.to(device), False)
    d2, _ = F.to_device_rows(e2.to(device), False)
    times = []
    for i in range(reps + 1):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        top1, rk, hits, mr, mrr = F.eval_alignment(d1, d2, [1, 5, 10, 50], "inner", False, 10)
        ev1.record()
        torch.cuda.synchronize()
        if i:
            times.append(ev0.elapsed_time(ev1))
    ms = float(np.median(times))
    pairs = float(n) * n
    flops = 2.0 * pairs * d              # ONE FP32 contraction pass (matrix stored once), then 3 streaming passes
    # the same evaluation through the reference-facing call (modules/finding/alignment.greedy_alignment): NumPy
    # embeddings in, Python set of pairs + Hits / MR / MRR out, host<->device copies and the result lines included
    try:
        import contextlib
        import io
        a1, a2 = e1.numpy(), e2.numpy()
        wall = []
        for i in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                F.greedy_alignment(a1, a2, [1, 5, 10, 50], 4, "inner", False, 10, True)
            wall.append(time.perf_counter() - t0)
        e2e_ms = 1e3 * float(np.median(wall[1:]))
        e2e = {"value": pairs / (e2e_ms * 1e-3), "unit": "pairs/s", "ms": e2e_ms, "h2d_bytes": 8 * n * d, "d2h_bytes": 8 * n,
               "api": "finding.greedy_alignment(embeds1, embeds2, top_k, threads, 'inner', False, csls_k=10, accurate=True)"}
    except Exception as exc:       # informational: never lose the bench line over it
        e2e = {"value": None, "note": "failed: %r" % (exc,)}
    # the reference's CPU path for the same evaluation: the NumPy restatement of similarity.py / alignment.py with the
    # reference's task split over `nums_threads` workers (oracle/finding.greedy_alignment_mt; BLAS threads for the
    # contraction) on a bounded 8000 x 8000 sub-problem (a few seconds); pairs/s is size-normalised
    try:
        from oracle import finding as orf
        m = min(n, 8000)
        nthreads = min(os.cpu_count() or 1, 32)
        orf.greedy_alignment_mt(e1[:1000].numpy(), e2[:1000].numpy(), [1, 5, 10, 50], "inner", False, 10, nthreads)   # warm-up
        t0 = time.perf_counter()
        orf.greedy_alignment_mt(e1[:m].numpy(), e2[:m].numpy(), [1, 5, 10, 50], "inner", False, 10, nthreads)
        cpu = {"value": float(m) * m / (time.perf_counter() - t0), "unit": "pairs/s", "cores": nthreads, "kind": "port",
               "sample": "%d x %d sub-problem, inner + CSLS(k=10), accurate ranks, %d worker threads + BLAS threads" % (m, m, nthreads)}
    except Exception as exc:
        cpu = {"value": None, "note": "failed: %r" % (exc,)}
    return {"metric": "CSLS pairs/sec", "value": pairs / (ms * 1e-3), "unit": "pairs/s", "n1": n, "n2": n, "dim": d, "e2e": e2e,
            "cpu_baseline": cpu,
            "ms": ms, "contraction_passes": 1, "streaming_passes": 3, "matrix_bytes": 4.0 * pairs,
            "fp32_tflops_whole_eval": flops / (ms * 1e-3) / 1e12, "hits1": hits[0],
            "note": "inner + CSLS(k=10), exact ranks (greedy_alignment accurate=True equivalent); includes the host-side "
                    "reduction of the rank vector"}


def bench_csls_sharded(shape, device, reps=3):
    """CSLS evaluation with E1's rows block-sharded over the ranks (E2 replicated, one all-gather of partial
    column top-k lists).  Time = max over ranks (device events)."""
    import torch
    import torch.distributed as dist
    from openea_b200 import finding as F
    from openea_b200.synth import SHAPES
    n, d = SHAPES[shape]["links"][2], 100
    g = torch.Generator(device="cpu").manual_seed(99)
    e2 = torch.randn(n, d, generator=g)
    e1 = (e2 + 0.5 * torch.randn(n, d, generator=g)).to(device)
    e2 = e2.to(device)
    times = []
    for i in range(reps + 1):
        dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        hits, mr, mrr, _ = F.eval_alignment_sharded(e1, e2, [1, 5, 10, 50], "inner", False, 10)
        ev1.record()
        torch.cuda.synchronize()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if i:
            times.append(float(t.item()))
    ms = float(np.median(times))
    return {"metric": "CSLS pairs/sec", "value": float(n) * n / (ms * 1e-3), "unit": "pairs/s", "n1": n, "n2": n, "dim": d,
            "ms": ms, "hits1": hits[0], "sharding": "E1 row blocks per rank, E2 replicated, all-gather of partial column top-k"}


_T0 = time.perf_counter()


def _phase(msg):
    sys.stderr.write("[bench %7.1fs] %s\n" % (time.perf_counter() - _T0, msg))
    sys.stderr.flush()


def probe_pipelined_e2e(args):
    """The same host-index steps through the depth-2 pipeline (oea_triple_step_fed_host_submit / _collect): first the
    losses of 6 steps are checked against the synchronous API from identical tables, then K steps are timed back to back
    (H2D of every step's index vectors and D2H of every step's loss inside the timed region; no L2 flush is possible
    between overlapping steps, the tables are 12–80 MB).  Runs in its own process under the parent's time limit, so a
    fault here cannot take the bench line with it.  Informational: not the headline e2e."""
    import torch
    from openea_b200 import engine as eng
    torch.cuda.set_device(0)
    device = torch.device("cuda", 0)
    cfg = WORKLOADS[args.workload]
    B, k = cfg["batch"], cfg["k"]

    W = build_workload(args.workload, 0, device, 1)
    tr = W["trainer"]
    snap = [(t, t.weight.clone(), t.state1.clone()) for t in (tr.ent, tr.rel)]

    def restore():       # both APIs start from the same variables and Adagrad accumulators
        for t, w, a in snap:
            t.weight.copy_(w); t.state1.copy_(a); t.grad.zero_(); t.touched.zero_()
        tr.read_loss()
        torch.cuda.synchronize()
    t1, t2 = W["arr"]["triples1"], W["arr"]["triples2"]
    dbg = torch.empty(B, 2 + k, dtype=torch.int32, device=device)
    npos_dev = torch.zeros(1, dtype=torch.int32, device=device)
    batches = []
    for i in range(8):
        tr.score_sampled(W["kg1"], W["kg2"], W["tset"], B, k, i % max(1, W["steps_per_epoch"] - 1), 0xE2E + i, dbg=dbg,
                         n_pos_out=npos_dev)
        torch.cuda.synchronize()
        pos, neg = decode_dbg(dbg.cpu().numpy(), int(npos_dev.item()), t1, t2, k)
        batches.append((torch.from_numpy(pos).pin_memory(), torch.from_numpy(neg).pin_memory()))
    restore()
    want = [tr.step_fed_host(*batches[i]) for i in range(6)]
    restore()
    pipe = eng.FedHostPipeline(tr, 3 * (batches[0][0].shape[1] + batches[0][1].shape[1]) + 64)
    got = []
    for i in range(6):
        pipe.submit(i % 2, *batches[i])
        if i >= 1:
            got.append(pipe.collect((i - 1) % 2))
    got.append(pipe.collect(5 % 2))
    rel = max(abs(a - b) / max(1e-12, abs(b)) for a, b in zip(got, want))
    K = args.steps
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        pipe.submit(i % 2, *batches[i % 8])
        if i >= 1:
            pipe.collect((i - 1) % 2)
    pipe.collect((K - 1) % 2)
    dt = time.perf_counter() - t0
    n_pos_h, n_neg_h = batches[0][0].shape[1], batches[0][1].shape[1]
    res = {"value": n_pos_h * K / dt, "unit": "positive triples/s", "ms_per_step": 1e3 * dt / K, "steps": K,
           "h2d_bytes_per_step": 12 * (n_pos_h + n_neg_h), "d2h_bytes_per_step": 8,
           "loss_max_rel_diff_vs_sync_api": rel, "losses_agree": bool(rel <= 1e-4),
           "api": "oea_triple_step_fed_host_submit / _collect (depth-2 pipeline, steps back to back, L2 not flushed)"}
    try:     # the same pipeline with OEA_FED_GROUPED=1: one warp per positive and its negatives (oea_triple_grouped.cu)
        os.environ["OEA_FED_GROUPED"] = "1"
        restore()
        got = []
        for i in range(6):
            pipe.submit(i % 2, *batches[i])
            if i >= 1:
                got.append(pipe.collect((i - 1) % 2))
        got.append(pipe.collect(5 % 2))
        rel_g = max(abs(a - b) / max(1e-12, abs(b)) for a, b in zip(got, want))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(K):
            pipe.submit(i % 2, *batches[i % 8])
            if i >= 1:
                pipe.collect((i - 1) % 2)
        pipe.collect((K - 1) % 2)
        dt = time.perf_counter() - t0
        res["grouped_scorer"] = {"value": n_pos_h * K / dt, "ms_per_step": 1e3 * dt / K,
                                 "loss_max_rel_diff_vs_sync_api": rel_g, "losses_agree": bool(rel_g <= 1e-4)}
    except Exception as exc:
        res["grouped_scorer"] = {"value": None, "note": "failed: %r" % (exc,)}
    finally:
        os.environ.pop("OEA_FED_GROUPED", None)
    try:     # and with OEA_FED_FUSED=1: grouped scoring + row optimiser as one cooperative launch per step
        os.environ["OEA_FED_FUSED"] = "1"
        restore()
        got = []
        for i in range(6):
            pipe.submit(i % 2, *batches[i])
            if i >= 1:
                got.append(pipe.collect((i - 1) % 2))
        got.append(pipe.collect(5 % 2))
        rel_f = max(abs(a - b) / max(1e-12, abs(b)) for a, b in zip(got, want))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(K):
            pipe.submit(i % 2, *batches[i % 8])
            if i >= 1:
                pipe.collect((i - 1) % 2)
        pipe.collect((K - 1) % 2)
        dt = time.perf_counter() - t0
        res["one_launch_step"] = {"value": n_pos_h * K / dt, "ms_per_step": 1e3 * dt / K,
                                  "loss_max_rel_diff_vs_sync_api": rel_f, "losses_agree": bool(rel_f <= 1e-4)}
    except Exception as exc:
        res["one_launch_step"] = {"value": None, "note": "failed: %r" % (exc,)}
    finally:
        os.environ.pop("OEA_FED_FUSED", None)
    print(json.dumps(res))
    return 0


def bench_triples(args, wl, rank, local_rank, world, device, full):
    """Device-timed K steps of workload `wl` (+ roofline); with `full` also the e2e leg, the epoch graph and the clocks.
    Returns the fields of the JSON line that describe this workload."""
    import torch
    import torch.distributed as dist
    cfg = WORKLOADS[wl]
    unit = "positive triples/s"
    W = build_workload(wl, rank, device, world)
    _phase("%s: workload resident" % wl)
    tr, kg1, kg2, tset = W["trainer"], W["kg1"], W["kg2"], W["tset"]
    B, k, d = cfg["batch"], cfg["k"], cfg["dim"]
    spe = W["steps_per_epoch"]
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=device)
    npos_dev = torch.zeros(1, dtype=torch.int32, device=device)
    full_steps = max(1, spe - 1) if spe > 1 else 1   # full batches per pass over the local shard (the ragged last step is skipped)

    # ---- multi-GPU: seed-row exchange on a GLOBAL cadence (identical on every rank by construction) -------------------
    xchg = None
    epoch_steps = None
    if world > 1:
        from openea_b200 import parallel as par
        seeds = np.concatenate([W["arr"]["train_links"][:, 0], W["arr"]["train_links"][:, 1]])
        xchg = par.SeedRowSync(W["ent"].weight, seeds, rank, world, mode=os.environ.get("OEA_XCHG_MODE", "auto"))
        # one global epoch = every triple of the UNSHARDED lists once = ceil(T / (G·B)) steps on every rank
        epoch_steps = max(1, int(np.ceil(W["n_triples_global"] / float(world * B))))
    gstep = [0]          # steps issued with the exchange enabled: drives the cadence, the same sequence on every rank
    pulled = [0]

    def one_step(i, ev=None, split=False, exchange=True):
        # weak scaling: every rank steps through ITS shard with the full per-GPU batch.  After the last step of a global
        # epoch the owners publish their seed-pair rows (push); one step later every replica applies them (pull), so the
        # NVLink transfer overlaps a training step.
        step = i % full_steps
        seed = 0xB007EA + 1000003 * (i // full_steps) + rank
        if ev:
            ev[0].record()
        if xchg is not None and exchange:
            g = gstep[0]
            gstep[0] += 1
            if g > 0 and g % epoch_steps == 1 % epoch_steps and xchg.epoch > pulled[0]:
                xchg.pull()
                pulled[0] = xchg.epoch
            if g > 0 and g % epoch_steps == 0:
                xchg.push()
        if ev and split:
            ev[3].record()          # kernel-only interval starts after the (rare) exchange
            tr.score_sampled(kg1, kg2, tset, B, k, step, seed)
            ev[1].record()
            tr.apply()
            ev[2].record()
        elif ev:
            ev[3].record()
            tr.step_sampled(kg1, kg2, tset, B, k, step, seed)      # ONE cooperative launch: score + optimiser
            ev[2].record()
        else:
            # n_pos_out costs a small H2D copy in front of the kernel: asked for once, outside the timed region
            tr.step_sampled(kg1, kg2, tset, B, k, step, seed, n_pos_out=npos_dev if i == 0 else None)

    n_warm = max(3, args.warmup)
    for i in range(n_warm):
        one_step(i)
    if xchg is not None:      # first use of a transport pays lazy set-up (NCCL channels / first peer mapping touch): untimed
        for _ in range(2):
            xchg.sync()
        pulled[0] = xchg.epoch
    torch.cuda.synchronize()
    n_pos_step = int(npos_dev.item())
    tr.read_loss()

    # ---- device-timed region: EXACTLY K steps, CUDA events on the launching stream --------------------------
    K = args.steps
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n_push0 = 0 if xchg is None else xchg.epoch
    dump = full and rank == 0 and args.dump_outputs
    with ClockSampler(local_rank) as clocks:
        t_wall0 = time.perf_counter()
        for i in range(K):
            if not args.no_flush:
                flush.fill_(float(i))   # L2 flush (not timed: outside the event pairs)
            if dump and i == K - 1:
                loss_before_last = tr.loss_dev.clone()      # outside the event pair, like the flush
            one_step(n_warm + i, evs[i])
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
    n_push = 0 if xchg is None else xchg.epoch - n_push0
    if world > 1:
        dist.barrier()
    kern_ms = np.array([e[3].elapsed_time(e[2]) for e in evs])
    step_ms = np.array([e[0].elapsed_time(e[2]) for e in evs])
    total_ms = float(step_ms.sum())
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    if dump:          # before anything below steps the tables again
        dump_outputs(args.dump_outputs, tr, float((tr.loss_dev - loss_before_last).item()))
    loss_val = tr.read_loss()
    value = world * n_pos_step * K / (total_ms * 1e-3)

    # ---- roofline of the dominant kernel: k_step_sampled_duo = the whole step in one launch --------------------
    # SURVEY §8(d): 24·d bytes per scored triple (3 row reads + 3 row-gradient writes); frac is computed on THOSE bytes.
    # The row optimiser the same launch runs moves another 24·d per touched row (read g, x, acc; write x, acc, g := 0):
    # reported separately (`optimiser_bytes`), not part of `achieved`.
    pk, pk_kind = peaks()
    touched = []
    for i in range(4):
        tr.score_sampled(kg1, kg2, tset, B, k, (n_warm + i) % full_steps, 0xB007EA + rank)
        touched.append(int((tr.ent.touched != 0).sum().item()) + int((tr.rel.touched != 0).sum().item()))
        tr.apply()
    n_touched = float(np.mean(touched))
    score_bytes = 24.0 * d * (1 + k) * n_pos_step
    opt_bytes = 24.0 * d * n_touched
    kern_med_ms = float(np.median(kern_ms))
    achieved = score_bytes / (kern_med_ms * 1e-3) / 1e9
    traffic = score_traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic_%s.json" % wl)
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        traffic = tj.get("k_step_sampled_dram_bytes_per_launch", tj.get("k_step_sampled_oct_dram_bytes_per_launch"))
        score_traffic = tj.get("k_score_sampled_dram_bytes_per_launch")
    # the same steps as two launches (score kernel, optimiser kernel) with an event between them: what the score
    # kernel alone achieves against the same bytes
    evs2 = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    for i in range(K):
        if not args.no_flush:
            flush.fill_(float(i))
        one_step(n_warm + K + i, evs2[i], split=True)
    if xchg is not None and xchg.epoch > pulled[0]:      # the last publication is applied on every rank (matched)
        xchg.pull()
        pulled[0] = xchg.epoch
    torch.cuda.synchronize()
    score_med_ms = float(np.median([e[3].elapsed_time(e[1]) for e in evs2]))
    split_step_ms = float(np.mean([e[0].elapsed_time(e[2]) for e in evs2]))
    roofline = {"bound": "hbm", "kernel": "k_step_sampled_duo", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "peak_kind": pk_kind + " (burst copy)",
                "algorithmic_bytes_per_launch": score_bytes, "bytes_model": "SURVEY 8(d): 24*d per scored triple",
                "optimiser_bytes": opt_bytes, "achieved_incl_optimiser": (score_bytes + opt_bytes) / (kern_med_ms * 1e-3) / 1e9,
                "touched_rows_per_step": n_touched,
                "kernel_ms_median": kern_med_ms, "kernel_share_of_step": float(kern_ms.sum() / step_ms.sum()),
                "score_kernel_alone": {"kernel": "k_score_sampled_duo", "ms_median": score_med_ms,
                                       "achieved": score_bytes / (score_med_ms * 1e-3) / 1e9,
                                       "frac": score_bytes / (score_med_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                                       "two_launch_ms_per_step": split_step_ms, "traffic": score_traffic}}
    _phase("%s: device-timed region done" % wl)
    out = {"value": value, "unit": unit, "ms_per_step": total_ms / K, "positives_per_step": n_pos_step,
           "scored_triples_per_s": value * (1 + k), "roofline": roofline, "wall_s_timed_region": t_wall, "last_loss_sum": loss_val,
           "workload": cfg["name"]}
    if xchg is not None:
        out["collective"] = {"kind": {"p2p": "own kernels: peer-memory stores over NVLink + release/acquire flags (oea_seed_push / oea_seed_pull)",
                                      "nccl": "oea_seed_pack + ncclAllGather (async) + oea_seed_unpack",
                                      "torch": "torch ops + all_gather"}[xchg.mode],
                             "mode": xchg.mode, "bytes_per_exchange": xchg.bytes_per_sync, "exchanges_in_timed_region": n_push,
                             "epoch_steps": epoch_steps, "time_to_global_epoch_ms": epoch_steps * total_ms / K,
                             "status": xchg.status(),
                             "accuracy_note": "this is the north-star's stale-replica scheme: fast, but measured to lose Hits@1 "
                                              "(15K shape, 100 epochs: 36.4 on one GPU, 19.7 at N=2, 9.2 at N=8); the exact and "
                                              "delta-sum modes keep it (DESIGN.md section 6, scripts/bench_multi_modes.py)"}
    if not full:
        if xchg is not None:
            xchg.close()
        return out, None

    # ---- e2e: the session.run(feed_dict) boundary with HOST index buffers -------------------------------------
    n_b = min(K, 8)
    t1, t2 = W["arr"]["triples1"], W["arr"]["triples2"]
    host_batches = []
    dbg = torch.empty(B, 2 + k, dtype=torch.int32, device=device)
    for i in range(n_b):
        tr.score_sampled(kg1, kg2, tset, B, k, i % full_steps, 0xE2E + i + rank, dbg=dbg, n_pos_out=npos_dev)
        torch.cuda.synchronize()
        pos, neg = decode_dbg(dbg.cpu().numpy(), int(npos_dev.item()), t1, t2, k)
        host_batches.append((torch.from_numpy(pos).pin_memory(), torch.from_numpy(neg).pin_memory()))
        tr.ent.grad.zero_(); tr.rel.grad.zero_(); tr.ent.touched.zero_(); tr.rel.touched.zero_()
    tr.read_loss()
    n_pos_h, n_neg_h = host_batches[0][0].shape[1], host_batches[0][1].shape[1]
    # (a) synchronous call, L2 flushed between steps: one session.run at a time
    for i in range(3):
        tr.step_fed_host(*host_batches[i % n_b])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e2e_s = 0.0
    for i in range(K):
        flush.fill_(float(i)); torch.cuda.synchronize()
        pos, neg = host_batches[i % n_b]
        t0 = time.perf_counter()
        tr.step_fed_host(pos, neg)          # H2D of 6 index vectors, score, optimiser, D2H loss, sync
        e2e_s += time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    sync_e2e = {"value": world * n_pos_h * K / e2e_s, "ms_per_step": 1e3 * e2e_s / K,
                "api": "oea_triple_step_fed_host (host index buffers, tables resident, synchronous, L2 flushed between steps)"}
    # (b) the same steps through the depth-2 pipelined entry points (the copy of step i+1 overlaps the kernels of step i,
    # every step's indices still cross PCIe and every step's loss still comes back inside the timed region).  Steps run
    # back to back, so L2 cannot be flushed between them: see config["l2_e2e"].
    from openea_b200 import engine as eng
    os.environ["OEA_FED_FUSED"] = "1"       # grouped scorer + row optimiser as one cooperative launch per step
    pipe = eng.FedHostPipeline(tr, 3 * (n_pos_h + n_neg_h) + 64)
    for rep in range(2):                    # rep 0 = warm-up
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(K):
            pipe.submit(i % 2, *host_batches[i % n_b])
            if i >= 1:
                pipe.collect((i - 1) % 2)
        pipe.collect((K - 1) % 2)
        pipe_s = time.perf_counter() - t0
    os.environ.pop("OEA_FED_FUSED", None)
    if world > 1:
        t = torch.tensor([pipe_s], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pipe_s = float(t.item())
    e2e = {"value": world * n_pos_h * K / pipe_s, "unit": unit, "h2d_bytes_per_step": 12 * (n_pos_h + n_neg_h),
           "d2h_bytes_per_step": 8, "ms_per_step": 1e3 * pipe_s / K, "steps": K,
           "api": "oea_triple_step_fed_host_submit / _collect (pinned host index buffers, depth-2 pipeline, one cooperative launch per step)",
           "synchronous": sync_e2e}
    _phase("%s: e2e done" % wl)

    # ---- informational: the same steps as ONE CUDA graph per epoch, L2 warm (how the training loop really runs) ----
    graph_info = None
    if world == 1:
        eg = tr.capture_epoch(kg1, kg2, tset, B, k, full_steps)
        for e in range(3):
            eg.replay(1234 + e)
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        g0.record()
        for e in range(reps):
            eg.replay(99 + e)
        g1.record()
        torch.cuda.synchronize()
        g_ms = g0.elapsed_time(g1) / (reps * full_steps)
        graph_info = {"ms_per_step": g_ms, "positives_per_s": n_pos_step / (g_ms * 1e-3), "steps_per_graph": full_steps,
                      "note": "one CUDA graph per epoch, L2 NOT flushed between steps: informational, not the bench value"}
        tr.read_loss()
    # clocks: the timed region is a few ms, shorter than nvidia-smi's sampling period; continue the SAME step loop
    # untimed under the sampler until it has >= 5 samples so the clocks line reflects this load.  The continuation runs a
    # wall-clock-bounded, rank-dependent number of steps, so it issues NO exchange and no collective (exchange=False).
    clk = clocks.summary()
    if clk["samples"] < 5:
        with ClockSampler(local_rank) as clocks2:
            t_end = time.perf_counter() + 1.0
            i = 0
            while time.perf_counter() < t_end:
                flush.fill_(0.0); one_step(i, exchange=False); i += 1
                if i % 64 == 0:
                    torch.cuda.synchronize()
            torch.cuda.synchronize()
        clk = clocks2.summary()
        clk["note"] = "timed region shorter than the sampling period: sampled over an untimed 1 s continuation of the same step loop (no exchange inside)"
        tr.read_loss()
    out.update({"e2e": e2e, "clocks": clk, "epoch_graph": graph_info})
    if xchg is not None:
        out["collective"]["status"] = xchg.status()
        xchg.close()
    return out, W


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="bootea_100k", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the bootea_15k block and the CSLS block (profiling runs)")
    ap.add_argument("--no-flush", action="store_true", help="diagnostic only: keep L2 warm between timed steps (the number is NOT a valid bench value)")
    ap.add_argument("--probe-pipelined-e2e", action="store_true",
                    help="internal: measure the depth-2 pipelined host-index step in this process and print its JSON")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss and the trained tables (entity rows: a fixed "
                         "seeded sample) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.probe_pipelined_e2e:
        return probe_pipelined_e2e(args)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = WORKLOADS[args.workload]
    unit = "positive triples/s"
    config = {"workload": cfg["name"], "batch_size": cfg["batch"], "neg_per_pos": cfg["k"], "dim": cfg["dim"],
              "sharding": ("triples sharded by head-row owner (id mod G), replicated tables, seed-pair rows exchanged once per "
                           "global epoch over NVLink peer memory") if world > 1 else "single",
              "l2": "flushed between timed steps (512 MiB write)",
              "l2_e2e": "pipelined e2e steps run back to back (no flush possible); per-step working set = tables + gradients + "
                        "Adagrad slots (%d MB) + candidate lists, vs 126 MB of L2" % (3 * 4 * cfg["dim"] * 2 * SHAPE_ENTITIES.get(cfg["shape"], 0) // 1000000)}

    if args.no_flush:
        config["l2"] = "NOT flushed (diagnostic run, invalid as a bench value)"
    if args.impl == "reference":
        if rank != 0:
            return 0
        val, info = cpu_reference_run(args.workload, args.steps, args.warmup)
        line = {"impl": "reference", "metric": "training triples/sec", "value": val, "unit": unit, "n_gpus": args.gpus,
                "steps": info["steps"], "warmup": args.warmup, "ms_per_step": 1e3 * info["seconds"] / max(1, info["steps"]),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": val, "unit": unit, "cores": info["cores"], "kind": "port", "sample": info["sample"],
                                 "thread_sweep_ms_per_step": info["thread_sweep_ms"], "omp_env": info["omp_env"]},
                "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    os.environ.setdefault("NCCL_DEBUG", "WARN")     # no version banner on stdout: the JSON line must stand alone
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _phase("cuda ready; building workload")
    main_blk, W = bench_triples(args, args.workload, rank, local_rank, world, device, full=True)
    K = args.steps
    k = cfg["k"]

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the CPU port is timed in a fresh process (the same command as `--impl reference`): inside this process
        # the OpenMP runtime shares cores with torch's thread pools and runs up to 2× slower
        try:
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload",
                                  args.workload, "--steps", "40", "--warmup", "2"], capture_output=True, text=True,
                                 timeout=300, env=reference_env())
            cpu_base = json.loads(res.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as exc:   # never lose the GPU line because the CPU leg failed
            cpu_base = {"value": None, "unit": unit, "cores": None, "kind": "port", "sample": "failed: %r" % (exc,)}
    _phase("cpu baseline done")
    del W
    torch.cuda.empty_cache()
    secondary = None
    if world == 1 and not args.no_secondary and args.workload == "bootea_100k":
        try:
            secondary, _ = bench_triples(args, "bootea_15k", rank, local_rank, world, device, full=False)
            secondary["note"] = "BASELINE.json configs[1] shape, same run, device-timed (same rules: L2 flushed, CUDA events)"
        except Exception as exc:
            secondary = {"value": None, "note": "failed: %r" % (exc,)}
        torch.cuda.empty_cache()
    csls = None
    if not args.no_secondary:
        if world == 1:
            csls = bench_csls(cfg["shape"], device)
        else:
            csls = bench_csls_sharded(cfg["shape"], device)
    _phase("csls done")
    if rank == 0:
        line = {"metric": "training triples/sec", "value": main_blk["value"], "unit": unit, "n_gpus": world, "steps": K,
                "warmup": max(3, args.warmup), "ms_per_step": main_blk["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "scored_triples_per_s": main_blk["scored_triples_per_s"], "positives_per_step": main_blk["positives_per_step"],
                "gpu_launches": K, "kernels": ["k_step_sampled_duo (fused sampler + duo scorer, grid barrier, row optimiser: one cooperative launch)"],
                "roofline": main_blk["roofline"], "e2e": main_blk["e2e"], "cpu_baseline": cpu_base, "clocks": main_blk["clocks"],
                "bootea_15k": secondary, "csls": csls, "epoch_graph": main_blk["epoch_graph"],
                "wall_s_timed_region": main_blk["wall_s_timed_region"], "last_loss_sum": main_blk["last_loss_sum"],
                "collective": main_blk.get("collective")}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def reference_env():
    """Environment of the CPU reference arm: threads pinned to cores in order (a migrating OpenMP team was one source
    of the 5.6x box-to-box swing of the r01 baseline)."""
    env = dict(os.environ)
    env.setdefault("OMP_PROC_BIND", "close")
    env.setdefault("OMP_PLACES", "cores")
    return env


if __name__ == "__main__":
    if "--impl" in sys.argv and "reference" in sys.argv and "OMP_PROC_BIND" not in os.environ:
        # libgomp reads its binding policy at load time: re-exec once with the pinned environment
        os.execve(sys.executable, [sys.executable] + sys.argv, reference_env())
    sys.exit(main())
