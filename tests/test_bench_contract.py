"""bench.py's reference arm (`--impl reference`: the staged Python reference and the C restatement on the host cores) runs
without a GPU, so its JSON contract is checked here; the GPU arm prints the same keys (profiles/r01_bench_*.json).
Its argument checks need no GPU either; `--dump-outputs` does."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                           "--warmup", "1", "--cpu-envs", "64", *args], capture_output=True, text=True, env=env,
                          timeout=300)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "agent_steps_per_sec" and d["unit"] == "agent-steps/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("c4:") and d["config"]["num_drones"] == 32
    cb = d["cpu_baseline"]
    # the unmodified Python reference where oracle/_ref (or /root/reference) is present, else the C port alone
    assert d["reference_kind"] in ("python_reference", "c_port")
    assert cb["kind"] == ("reference" if d["reference_kind"] == "python_reference" else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["port"]["kind"] == "port" and d["port"]["value"] > 0
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, ("--gpus", "2"))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_follows_the_workload_flag():
    r = _run(args=("--workload", "c2"))
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["config"]["num_drones"] == 8 and d["config"]["num_obstacles"] == 4


@pytest.mark.parametrize("args", [("--steps", "0"), ("--graph", "20", "--steps", "30"), ("--dump-outputs", "out")])
def test_arguments_that_would_not_time_or_dump_what_they_name_are_refused(args):
    """--steps is the exact number of timed steps (so a graph of T steps needs a multiple of T); the reference arm has
    no device outputs to dump."""
    r = _run(args=args)
    assert r.returncode == 2 and r.stdout == "", r.stderr[-2000:]


def _bench_dump(out_dir, envs, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "7", "--warmup", "3",
                        "--envs-per-gpu", str(envs), "--no-cpu", "--no-e2e", "--no-dr-off", "--dump-outputs", str(out_dir),
                        *extra], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_dump_outputs_is_a_bounded_reproducible_sample_of_the_last_timed_step(tmp_path):
    E = 16384   # C4 outputs of 16384 envs exceed the 64 MB budget: a sample
    d = _bench_dump(tmp_path / "a", E)
    assert d["steps"] == 7
    _bench_dump(tmp_path / "b", E)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == sorted(n + ".npy" for n in ("env_index", "obs", "reward", "dist", "terminated", "truncated", "reached",
                                                 "collision", "obs_valid", "all_terminated", "all_truncated",
                                                 "global_state"))
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64 * 10**6
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert 0 < len(idx) < E and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < E
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and a.shape[0] == len(idx), f
        assert np.array_equal(a, b, equal_nan=True), f
    obs, valid = np.load(tmp_path / "a" / "obs.npy"), np.load(tmp_path / "a" / "obs_valid.npy")
    assert obs.shape == (len(idx), 32, 37) and set(np.unique(valid)) <= {0.0, 1.0} and valid.any()


@pytest.mark.gpu
def test_dump_outputs_are_the_oracle_step_after_the_last_timed_step(tmp_path):
    """With randomisation off every env follows the C oracle bit for bit, so a slice of the dumped envs is replayed on
    the oracle: env e is seeded with e, and bench.py's schedule is a pre-warm call (W warm-up + 3 steps) and the timed
    call (W warm-up + K steps), each cycling from the first of its four seeded U(-1, 1) action tensors.  A dump of
    another step, or rows paired with the wrong env_index entries, differs."""
    import torch
    import swarm_oracle as so
    from parity_util import assert_biteq

    E, N, W, K = 16384, 32, 3, 7
    cfg = {"num_drones": N, "num_obstacles": 8}
    out = tmp_path / "d"
    _bench_dump(out, E, "--dr", "off")
    rows = np.arange(0, len(np.load(out / "env_index.npy")), 61)
    envs = np.load(out / "env_index.npy")[rows].astype(np.int64)
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(1234)
    acts = [(torch.rand((E, N, 3), generator=gen, device="cuda:0") * 2.0 - 1.0).cpu().numpy()[envs] for _ in range(4)]
    o = so.OracleSwarm(len(envs), cfg)
    o.seed(envs.astype(np.uint64))
    o.reset()
    for k in [*range(W), *range(3), *range(W), *range(K)]:
        o.step(acts[k % 4], auto_reset=True)
    got = {name: np.load(out / f"{name}.npy")[rows] for name in
           ("obs", "reward", "dist", "terminated", "truncated", "reached", "collision", "obs_valid", "all_terminated",
            "all_truncated", "global_state")}
    assert_biteq("reward", got.pop("reward"), o.reward.astype(np.float32), K)
    obs = got.pop("obs")
    for name, a in got.items():
        assert_biteq(name, a, getattr(o, name), K)
    valid = o.obs_valid.astype(bool)
    assert valid.any()
    assert_biteq("obs", obs[valid], o.obs[valid], K)
