"""CPU: bench.py's and smoke()'s Python logic (argument plumbing, the JSON contract of the bench line, the pipelined
probe's choreography and its three variants) executed in a subprocess whose CUDA surface is faked and whose liboea entry
points are the kernels' sources on the warp emulator (tests/emu/fake_cuda.py).  The numbers are not measurements."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.emu import build_emu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "tests", "emu", "fake_cuda.py")


def run(*args, timeout=600):
    if build_emu.build() is None:
        pytest.skip("no CUDA headers for the emulator build")
    res = subprocess.run([sys.executable, RUNNER] + list(args), capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stdout.strip().splitlines()


def test_bench_line_contract_on_the_emulator(tmp_path):
    line = json.loads(run("bench", "--workload", "micro", "--steps", "3", "--warmup", "3", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path / "out"))[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "e2e", "cpu_baseline", "clocks", "gpu_launches"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 3 and line["higher_is_better"] is True and line["dtype"] == "f32"
    assert line["value"] > 0 and line["gpu_launches"] == 3 and "workload" in line["config"]
    roof = line["roofline"]
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(roof) and roof["bound"] == "hbm"
    e2e = line["e2e"]
    assert e2e["value"] > 0 and e2e["h2d_bytes_per_step"] == 12 * 48 * 4 and e2e["d2h_bytes_per_step"] == 8
    assert e2e["steps"] == 3
    dumped = {f[:-4]: np.load(tmp_path / "out" / f) for f in os.listdir(tmp_path / "out")}
    assert set(dumped) == {"last_step_loss", "entity_embeddings_sampled", "entity_adagrad_sampled", "relation_embeddings",
                           "relation_adagrad"}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in dumped.values())
    assert dumped["last_step_loss"].shape == (1,) and dumped["last_step_loss"][0] > 0
    assert dumped["entity_embeddings_sampled"].shape == dumped["entity_adagrad_sampled"].shape
    assert sum(a.nbytes for a in dumped.values()) <= 64 << 20
    csls = line["csls"]
    assert csls["value"] > 0 and csls["e2e"]["value"] > 0 and csls["cpu_baseline"]["value"] > 0 and csls["hits1"] > 0


def test_pipelined_probe_variants_agree_with_the_synchronous_step():
    out = json.loads(run("probe")[-1])
    assert out["losses_agree"] and out["value"] > 0
    assert out["grouped_scorer"]["losses_agree"] and out["one_launch_step"]["losses_agree"]


def test_smoke_passes_on_the_emulator():
    assert any(line.startswith("smoke ok") for line in run("smoke", timeout=900))


LIFECYCLES = ["TransE", "TransH", "TransD", "DistMult", "SimplE", "MTransE", "AlignE", "BootEA", "BootEA_TransH", "GCN_Align",
              "AliNet", "RDGCN", "IPTransE", "SEA", "IMUSE", "AttrE", "JAPE"]


def test_every_model_class_runs_its_lifecycle_on_the_emulator(tmp_path):
    """set_args / set_kgs / init / run (two epochs, one validation) / test / save of all 17 model classes on the micro
    synthetic dataset, kernels on the emulator: every Python line of the lifecycles — evaluation, result lines, files on
    disk, bootstrapping, graph builders — executes without a GPU (several processes side by side)."""
    import concurrent.futures
    if build_emu.build() is None:
        pytest.skip("no CUDA headers for the emulator build")

    def one(name):
        folder = str(tmp_path / name)
        os.makedirs(folder)
        res = subprocess.run([sys.executable, RUNNER, "lifecycle", name, folder], capture_output=True, text=True, timeout=900,
                             cwd=ROOT)
        return name, res.returncode, res.stdout[-300:] + res.stderr[-1500:]
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(17, max(2, (os.cpu_count() or 4) // 4))) as pool:
        results = list(pool.map(one, LIFECYCLES))
    failed = [(name, tail) for name, rc, tail in results if rc != 0 or "lifecycle ok: " + name not in tail]
    assert not failed, failed


@pytest.mark.parametrize("world", [2, 8])        # 8 ranks on the micro KG: a global epoch is ONE step (pull and push every step)
def test_bench_two_ranks_issue_matched_collectives_on_the_emulator(world):
    """bench.py's N > 1 path as two processes on the CPU (gloo instead of NCCL, kernels on the emulator, the exchange in its
    torch transport): the exchange cadence is a global step count, the wall-clock-bounded clock continuation issues no
    collective, so both ranks finish — round 1's N = 8 run deadlocked in exactly this code — and rank 0 prints one line."""
    import socket
    if build_emu.build() is None:
        pytest.skip("no CUDA headers for the emulator build")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for rank in range(world):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   OMP_NUM_THREADS="1")
        procs.append(subprocess.Popen([sys.executable, RUNNER, "bench", "--workload", "micro", "--gpus", str(world), "--steps", "9", "--warmup", "3",
                                       "--no-cpu-baseline"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, env=env))
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-1500:] for o in outs]
    lines = outs[0][0].strip().splitlines()
    line = json.loads(lines[-1])
    assert all(o[0].strip() == "" for o in outs[1:]), "only rank 0 prints"
    assert line["n_gpus"] == world and line["steps"] == 9 and line["value"] > 0 and line["scaling"] == "weak"
    coll = line["collective"]
    assert coll["mode"] == "torch" and coll["exchanges_in_timed_region"] >= 1 and coll["epoch_steps"] >= 1 and coll["status"] == 0
    if world == 8:
        assert coll["epoch_steps"] == 1 and coll["exchanges_in_timed_region"] == 9
    assert line["csls"]["value"] > 0 and "sharding" in line["csls"]
    assert line["e2e"]["value"] > 0


@pytest.mark.parametrize("mode", ["exact", "seed"])
def test_bootea_lifecycle_as_two_ranks_on_the_emulator(tmp_path, mode):
    """The reference lifecycle of BootEA as two gloo ranks on the CPU (kernels on the emulator) in both multi-GPU modes of
    DESIGN.md §6: 'exact' (batch sharded, gradients all-reduced) and 'seed' (head-owner shards + seed-row exchange) — replica
    sync before validation / bootstrapping / test, sharded evaluation, rank 0 writes the results; every rank prints the same
    accurate-results line."""
    import re
    import socket
    if build_emu.build() is None:
        pytest.skip("no CUDA headers for the emulator build")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for rank in range(2):
        folder = str(tmp_path / ("r%d" % rank))
        os.makedirs(folder)
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   OEA_MULTI_MODE=mode, OMP_NUM_THREADS="1")
        procs.append(subprocess.Popen([sys.executable, RUNNER, "lifecycle", "BootEA", folder], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                                      text=True, cwd=ROOT, env=env))
    outs = [p.communicate(timeout=900) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1][-1500:] for o in outs]
    lines = [re.findall(r"accurate results: hits@.*?mrr = [0-9.]+", o[0]) for o in outs]
    assert lines[0] and lines[0][-1] == lines[1][-1], (lines[0][-1:], lines[1][-1:])
    assert all("lifecycle ok: BootEA" in o[0] for o in outs)
