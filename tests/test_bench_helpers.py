"""CPU-side pieces of bench.py that the driver's runs depend on (no GPU): the CPU-oracle leg and the committed measurement of
the reference's own Python loop that the bench line quotes."""
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench  # noqa: E402


def test_cpu_port_rate_runs_a_sample_of_at_least_the_requested_length():
    rate, n_sample, seconds, steps = bench.cpu_port_rate(1 << 14, 4, 2, budget_s=2.0, min_wall_s=0.2)
    assert rate > 1e5 and n_sample == 1 << 14
    assert steps >= 4 and seconds >= 0.1           # more steps of the same batch until the sample is worth timing


def test_reference_python_loop_measurement_is_committed_and_quoted():
    """SURVEY 8(d) CPU baseline (i): the unmodified reference's own Python loop, measured where /root/reference exists
    (oracle/ref_python_rate.py) -- the GPU box cannot run it, so the bench line quotes the committed file."""
    d = json.load(open(os.path.join(REPO, "profiles", "r02", "ref_python_loop_rate.json")))
    procs = {r["procs"]: r["env_steps_per_s"] for r in d["runs"]}
    assert set(procs) == {1, 8} and 5e3 < procs[1] < 1e5 and procs[1] < procs[8] < 8 * procs[1] * 1.1
    q = bench.ref_python_loop()
    assert q["unit"] == bench.UNIT and [r["procs"] for r in q["runs"]] == [1, 8]
    assert abs(q["runs"][0]["value"] - procs[1]) < 1e-6


def test_engine_sections_cite_their_own_committed_ncu_capture():
    """bench.py's sawyer_door / sawyer_peg sections quote figures READ from the committed ncu captures (profiles/r02/), one per
    task; a renamed or missing file would silently drop the block."""
    import bench
    for task in ("sawyer_door", "sawyer_peg"):
        s = bench.ncu_engine_summary(task)
        assert s is not None and bench.ENGINE_CAPTURES[task][0] in s["source"] and task in s["source"]
        assert s["registers_per_thread"] == 128 and 20 < s["achieved_occupancy_pct"] <= 25.1
        assert 0 < s["executed_ipc"] < 4 and 16 < s["active_lanes_per_instruction"] <= 32
    k = bench.ncu_engine_summary("kitchen")
    assert k is not None and "kitchen" in k["source"] and k["registers_per_thread"] == 246 and 12 < k["achieved_occupancy_pct"] <= 12.6


def test_dump_outputs_writes_float32_and_a_fixed_sample_beyond_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch
    obs = torch.arange(40 * 12, dtype=torch.float32).reshape(40, 12)
    done = (torch.arange(40) % 3 == 0).to(torch.uint8)
    bench.dump_outputs(str(tmp_path / "all"), {"obs": obs, "done": done})
    assert sorted(os.listdir(tmp_path / "all")) == ["done.npy", "obs.npy"]
    o, d = np.load(tmp_path / "all" / "obs.npy"), np.load(tmp_path / "all" / "done.npy")
    assert o.dtype == d.dtype == np.float32 and np.array_equal(o, obs.numpy()) and np.array_equal(d, done.float().numpy())

    monkeypatch.setattr(bench, "DUMP_BYTES", 10 * (13 * 4 + 8) + 3 * bench.NPY_HEADER_BYTES)
    for run in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / run), {"obs": obs, "done": done})
    idx = np.load(tmp_path / "s1" / "env_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 10 and np.all(np.diff(idx) > 0)
    rows = idx.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "s1" / "obs.npy"), obs.numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "s1" / "done.npy"), done.float().numpy()[rows])
    assert sum(os.path.getsize(tmp_path / "s1" / f) for f in os.listdir(tmp_path / "s1")) <= bench.DUMP_BYTES
    for f in os.listdir(tmp_path / "s1"):
        assert np.array_equal(np.load(tmp_path / "s1" / f), np.load(tmp_path / "s2" / f))


def test_bench_names_the_host_data_path_it_measured(monkeypatch):
    import bench
    for k in ("LOCAL_WORLD_SIZE", "WORLD_SIZE", "EARL_TT_HOST_ZEROCOPY"):
        monkeypatch.delenv(k, raising=False)
    assert "one launch per step" in bench.host_path_note()
    monkeypatch.setenv("WORLD_SIZE", "4")
    assert "staged pipeline" in bench.host_path_note()
    monkeypatch.setenv("EARL_TT_HOST_ZEROCOPY", "1")
    assert "one launch per step" in bench.host_path_note()
