"""CPU: bench.py's reference arm prints ONE JSON line with the contract's keys (a tiny sample, a couple of seconds)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-seconds", "0.2"], capture_output=True, text=True, check=True, cwd=ROOT).stdout.strip().splitlines()
    assert len(out) == 1
    line = json.loads(out[0])
    assert line["impl"] == "reference" and line["unit"] == "agent-steps/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["e2e"] == {"value": line["value"], "unit": "agent-steps/s", "h2d_bytes_per_step": 0,
                                                 "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == (os.cpu_count() or 1) and "sample" in cb and cb["value"] == line["value"]
    assert set(line["config"]) >= {"workload", "baseline_config", "instances_per_gpu", "agents", "iters_per_step"}
    assert line["vs_baseline"] is None and line["scaling"] == "weak" and line["dtype"] == "f32" and line["data"] == "synthetic"


def test_other_ranks_of_the_reference_arm_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_every_bench_workload_compiles_and_is_described():
    """bench.py's workload table: every entry builds a scenario that compiles to device tables (on the host, no GPU), names its
    dominant kernel and bound, and the committed ncu-derived traffic file only refers to known workloads and existing captures."""
    import json

    sys.path.insert(0, ROOT)
    import bench

    import multiagent_rlrm_b200 as P

    for name, (desc, base, n, iters, bytes_per, kernel) in bench.WORKLOADS.items():
        sc = bench.scenario(name)
        c = P.compile_scenario(sc)
        assert c.n_agents == len(sc.starts) and n > 0 and iters > 0 and kernel and desc and base, name
        assert name in bench.BOUND, f"{name}: no entry in bench.BOUND"
        assert bytes_per is None or bytes_per > 0
    traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    for name, entry in traffic.items():
        if name.startswith("_"):
            continue
        assert name in bench.WORKLOADS, name
        assert entry["dram_bytes_per_active_step"] > 0 and os.path.exists(os.path.join(ROOT, entry["source"])), name


@pytest.mark.parametrize("layout", ["per_slot", "per_agent_rm", "shared"])
def test_dump_outputs_writes_a_fixed_float_sample_within_budget(layout, tmp_path):
    """bench.py --dump-outputs on each table layout the engine has — one table per agent slot (N*A, S, 4), per-agent machines
    concatenated per instance (N, rows, 4), one shared table per agent index (A, S, 4), written whole and charged to the budget
    first — with a stand-in engine on host tensors (the dump only reads the state arrays): float32 / float64 files under the
    byte budget, the same seeded instance sample every time, and every array equal to the engine's own at every sampled
    instance, the slot words decoded with the header's field layout."""
    import types

    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    from multiagent_rlrm_b200.engine import STATS_DTYPE

    N, A = (8192, 4) if layout == "shared" else (2048, 2)
    q_shape = {"per_slot": (N * A, 100, 4), "per_agent_rm": (N, 300, 4), "shared": (A, 100, 4)}[layout]
    rng = np.random.default_rng(3)
    fields = {"cell": rng.integers(0, 1 << 16, N * A), "agent_steps": rng.integers(0, 1 << 16, N * A),
              "timestep": rng.integers(0, 1 << 16, N * A), "rm_state": rng.integers(0, 1 << 8, N * A), "flags": rng.integers(0, 1 << 8, N * A)}
    words = (fields["cell"] | fields["agent_steps"] << 16 | fields["timestep"] << 32 | fields["rm_state"] << 48
             | fields["flags"] << 56).astype(np.uint64)  # include/rlrm_b200.h: slot word bit layout
    stats = np.zeros(N * A, dtype=STATS_DTYPE)
    for name in STATS_DTYPE.names:
        stats[name] = rng.integers(0, 1 << 20, N * A).astype(stats.dtype[name]) / (1 if stats.dtype[name].kind == "u" else 8)
    eng = types.SimpleNamespace(N=N, A=A, cfg=types.SimpleNamespace(shared_q=int(layout == "shared")), sync_tables=lambda: None,
                                q=torch.from_numpy(rng.random(q_shape, dtype=np.float32)), slot=torch.from_numpy(words.view(np.int64)),
                                epsilon=torch.from_numpy(rng.random(N * A)), ep_return=torch.from_numpy(rng.random(N * A)),
                                stats=torch.from_numpy(stats.view(np.uint8).reshape(N * A, 32)))
    budget = 1 << 20
    for out in ("a", "b"):
        bench.dump_outputs(eng, str(tmp_path / out), budget=budget)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == sorted(p.name for p in (tmp_path / "b").iterdir())
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= budget
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert got[f[:-4]].dtype in (np.float32, np.float64) and np.array_equal(got[f[:-4]], np.load(tmp_path / "b" / f)), f
    idx = got.pop("instances").astype(np.int64)
    assert 0 < len(idx) < N and np.all(np.diff(idx) > 0)
    q = eng.q.numpy()
    want = {"q": q if layout == "shared" else q.reshape(N, -1, *q_shape[1:])[idx].reshape(-1, *q_shape[1:]),
            "epsilon": eng.epsilon.numpy().reshape(N, A)[idx], "ep_return": eng.ep_return.numpy().reshape(N, A)[idx]}
    want.update({"slot_" + k: v.reshape(N, A)[idx] for k, v in fields.items()})
    want.update({"stats_" + k: stats[k].reshape(N, A)[idx] for k in STATS_DTYPE.names})
    assert sorted(got) == sorted(want)
    for k, v in want.items():
        assert got[k].shape == v.shape and np.array_equal(got[k], v), k
