"""GPU parity tests proper: the CUDA path, called through the C ABI, against (a) the golden
fixtures recorded from the unmodified reference and (b) the C oracle on seeded inputs.

Bar (BASELINE.json north_star): fp32 state / obs / reward within 1e-5 relative over 1000
steps, flags bit-exact up to counted 1-ulp threshold cases.  What is asserted here is
stronger: state, observations, float64 rewards, distances, flags, global_state and the reset
draws are BIT-EXACT.  Against the golden fixtures the order of exactly tied distances in the
k-nearest blocks is validated instead (np.argsort is not stable, SURVEY T5); against the C oracle
it is not: the oracle and the kernels both put the lowest index first on a tie.
"""
import numpy as np
import pytest

import parity_util as pu

pytestmark = pytest.mark.gpu


def _backend(*a, **k):
    from engine_backend import EngineBackend
    return EngineBackend(*a, **k)


@pytest.mark.parametrize("name", pu.golden_names())
def test_cuda_matches_reference_golden(name):
    g = pu.load_golden(name)
    m = g["meta"]
    b = _backend(len(g["seeds"]), m["config"], kind=m["kind"])
    assert b.D == m["D"]
    stats = pu.replay_and_compare(b, g)
    assert stats["steps"] == m["T"]
    # float32 reward output == float32(reference float64 reward)
    b2 = _backend(len(g["seeds"]), m["config"], kind=m["kind"], reward64=False)
    pu.replay_and_compare(b2, g, reward_dtype=np.float32, steps=200)


CASES = [
    # kind, cfg, E, T, action scale
    ("swarm", {"num_drones": 8, "num_obstacles": 4}, 4096, 60, 1.5),                      # C2 full size
    ("swarm", {"num_drones": 16, "num_obstacles": 8}, 2048, 40, 1.5),                     # C3 shape
    ("swarm", {"num_drones": 32, "num_obstacles": 8}, 1024, 40, 1.0),                     # C4 shape, world 20
    ("swarm", {"num_drones": 32, "num_obstacles": 8, "world_size": 44.0}, 512, 60, 1.5),  # C4 density-matched
    ("swarm", {"num_drones": 128, "num_obstacles": 8, "world_size": 70.0}, 64, 12, 1.0),  # C5 shape
    ("swarm", {"num_drones": 3, "num_obstacles": 0, "max_steps": 30}, 1000, 80, 1.0),     # ragged warp packing
    ("swarm", {"num_drones": 5, "num_obstacles": 8, "max_steps": 25, "world_size": 24.0}, 777, 60, 1.0),
    ("swarm", {"num_drones": 12, "num_obstacles": 3, "neighbor_k": 5, "sensed_obstacles": 2}, 333, 40, 1.2),
    ("swarm", {"num_drones": 20, "num_obstacles": 6, "neighbor_k": 8, "sensed_obstacles": 8}, 100, 40, 1.2),
    ("swarm", {"num_drones": 40, "num_obstacles": 5, "world_size": 50.0}, 50, 30, 1.2),   # two slots, ragged
    ("swarm", {"num_drones": 64, "num_obstacles": 4, "world_size": 40.0, "max_steps": 25}, 200, 40, 1.2),  # wide rotation kernel, 2 slots
    ("swarm", {"num_drones": 128, "num_obstacles": 8, "world_size": 20.0}, 100, 10, 1.0),  # C5 as BASELINE names it: resets every step
    ("swarm", {"num_drones": 128, "num_obstacles": 12, "world_size": 120.0, "max_steps": 15}, 60, 40, 1.5),
    ("swarm", {"num_drones": 1, "num_obstacles": 2, "max_steps": 20}, 500, 50, 1.0),
    # the four stage env_configs of the reference's configs/curriculum_v1.yaml:12-55
    ("swarm", {"num_drones": 3, "num_obstacles": 0, "max_steps": 300, "world_size": 20.0}, 512, 50, 1.0),
    ("swarm", {"num_drones": 3, "num_obstacles": 4, "max_steps": 350, "world_size": 20.0}, 512, 50, 1.0),
    ("swarm", {"num_drones": 5, "num_obstacles": 8, "max_steps": 400, "world_size": 24.0}, 512, 50, 1.0),
    ("swarm", {"num_drones": 8, "num_obstacles": 12, "max_steps": 450, "world_size": 28.0}, 512, 50, 1.0),
    ("single", {"num_obstacles": 8, "max_steps": 50}, 5000, 120, 1.5),                    # C1 batched
    ("single", {"num_obstacles": 0, "max_steps": 10}, 33, 30, 1.0),
]


@pytest.fixture(autouse=True)
def _wide_kernel_everywhere(monkeypatch):
    """N = 64 / 128 run on the wide rotation-pass kernel (csrc/swarm_step_rotx.cu) at every batch size; pin the
    threshold knob to its default so an inherited environment variable cannot move these tests to the general kernel."""
    monkeypatch.setenv("SWARM_B200_ROTX_MIN_ENVS", "0")


def test_wide_and_general_kernels_agree(monkeypatch):
    """N = 128: the wide rotation-pass kernel and the general kernel step the same batch to the same bits."""
    import torch
    import swarm_b200
    cfg = {"num_drones": 128, "num_obstacles": 8, "world_size": 60.0, "max_steps": 20}
    E, T = 300, 30
    engines = []
    for min_envs in ("0", "1000000000"):
        monkeypatch.setenv("SWARM_B200_ROTX_MIN_ENVS", min_envs)
        e = swarm_b200.SwarmEngine(E, cfg, device="cuda:0", reward64=True)
        e.seed(np.arange(E, dtype=np.uint64))
        e.reset()
        engines.append(e)
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(11)
    for t in range(T):
        act = torch.rand((E, 128, 3), generator=gen, device="cuda:0") * 2.4 - 1.2
        for e in engines:
            e.step(act)
        a, b = engines
        for name in ("pos4", "vel4", "goal4", "obs", "reward64", "dist", "terminated", "truncated", "reached", "collision",
                     "obs_valid", "all_terminated", "all_truncated", "global_state", "rng", "step_count"):
            assert torch.equal(getattr(a, name), getattr(b, name)), (name, t)
    assert engines[0].launch_count != engines[1].launch_count   # two launches per step vs one


@pytest.mark.parametrize("N,M", [(8, 4), (16, 8), (32, 12)])
def test_rotation_and_general_kernels_agree_under_randomisation(monkeypatch, N, M):
    """Same batch, same actions, domain randomisation incl. the control-delay ring: the rotation-pass kernels and the
    general kernel (SWARM_B200_NO_ROT=1) write the same bits, ring and per-episode constants included."""
    import torch
    import swarm_b200
    from test_domain_randomization import DR_DELAY
    cfg = {"num_drones": N, "num_obstacles": M, "max_steps": 30}
    E, T = 700, 45
    engines = []
    for no_rot in ("0", "1"):
        monkeypatch.setenv("SWARM_B200_NO_ROT", no_rot)
        e = swarm_b200.SwarmEngine(E, cfg, device="cuda:0", reward64=True, domain_randomization=DR_DELAY, dr_seed=9)
        e.seed(np.arange(E, dtype=np.uint64))
        e.reset()
        engines.append(e)
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(3)
    for t in range(T):
        act = torch.rand((E, N, 3), generator=gen, device="cuda:0") * 2.4 - 1.2
        for e in engines:
            e.step(act)
        a, b = engines
        for name in ("pos4", "vel4", "goal4", "obst4", "obs", "reward64", "dist", "terminated", "truncated", "reached",
                     "collision", "obs_valid", "all_terminated", "all_truncated", "global_state", "rng", "step_count",
                     "dr_params", "act_hist"):
            assert torch.equal(getattr(a, name).view(torch.uint8), getattr(b, name).view(torch.uint8)), (name, t)
    assert engines[0].launch_count <= engines[1].launch_count   # rotation pass: auto-reset fused into the step launch


@pytest.mark.parametrize("N,world,dr", [(64, 60.0, False), (128, 90.0, False), (32, 40.0, False), (16, 30.0, False),
                                        (8, 24.0, False), (32, 40.0, True), (8, 24.0, True), (128, 90.0, True)])
def test_parked_drones_masked_rotation_pass(N, world, dr):
    """Envs with parked drones (they reached the goal earlier) stay on the rotation-pass kernels: neighbour blocks
    see every drone, formation error and collisions only the ACTIVE ones (drone_swarm_env.py:185-224).  Injected
    states: random subsets parked, parked drones sitting inside an active drone's collision sphere, and an active
    drone whose three nearest are all parked-and-touching with / without an active one just behind them."""
    import swarm_oracle as so
    from parity_util import assert_biteq

    cfg = {"num_drones": N, "num_obstacles": 8, "world_size": world, "max_steps": 50}
    E, T = 96, 10
    dr_cfg = None
    if dr:   # the DR instantiations carry the same masked pass (sensor noise: rows must then agree exactly)
        from test_domain_randomization import DR_DELAY
        dr_cfg = DR_DELAY
    b = _backend(E, cfg, **(dict(domain_randomization=dr_cfg, dr_seed=11) if dr else {}))
    o = so.OracleSwarm(E, cfg, dr=dr_cfg, dr_seed=11)
    seeds = np.arange(50, 50 + E, dtype=np.uint64)
    b.seed(seeds); o.seed(seeds)
    b.reset(); o.reset()
    rng = np.random.default_rng(5)
    active = (rng.random((E, N)) > rng.uniform(0.0, 0.4, (E, 1))).astype(np.uint8)
    active[0] = 1                      # nobody parked
    active[1] = 0; active[1, 7] = 1    # a single active drone
    active[:, 0] = 1
    pos = o.positions.copy()
    behind, touching = [], []
    for e in range(2, E):
        parked = np.flatnonzero(active[e] == 0)
        if e % 3 == 0 and len(parked) >= 3:   # three parked drones touching active drone 0 ...
            (behind if e % 6 == 0 else touching).append(e)
            for q, j in enumerate(parked[:3]):
                pos[e, j] = pos[e, 0] + np.float32(0.2 + 0.1 * q) * np.eye(3, dtype=np.float32)[q]
            if e % 6 == 0:                    # ... and an active one just behind them (the 4th nearest)
                j = 1 + int(np.flatnonzero(active[e, 1:])[0])
                pos[e, j] = pos[e, 0] - np.float32([0.0, 0.0, 0.7])
        elif e % 3 == 1 and len(parked) >= 1:  # one parked drone inside an active drone's collision sphere
            pos[e, parked[0]] = pos[e, 0] + np.float32([0.3, 0.0, 0.0])
    o.positions[:] = pos
    o.active[:] = active
    o.observe()
    b.eng.set_state(pos, o.velocities, o.goal, o.obstacles, alive=active)
    for t in range(-1, T):
        if t >= 0:
            act = rng.uniform(-0.3, 0.3, size=(E, N, 3)).astype(np.float32)
            b.step(act, auto_reset=True)
            o.step(act, auto_reset=True, num_threads=8)
        for name in ("positions", "velocities", "goal", "obstacles", "step_count", "dist", "obs_valid", "global_state",
                     "active") + (() if t < 0 else ("reward", "terminated", "truncated", "reached", "collision",
                                                    "all_terminated", "all_truncated")):
            assert_biteq(name, getattr(b, name), getattr(o, name), t)
        valid = o.obs_valid.astype(bool)
        assert_biteq("obs", b.obs[valid], o.obs[valid], t)
        if t == 0:   # the injected layouts did what they were built for
            assert len(behind) >= 3 and len(touching) >= 3
            assert (o.collision[behind, 0] == 1).all()       # the active 4th-nearest behind three parked ones counts
            assert (o.collision[touching, 0] == 0).sum() >= 3  # parked neighbours alone never collide
    assert int(o.active.sum()) < E * N


@pytest.mark.parametrize("kind,cfg,E,T,scale", CASES)
def test_cuda_matches_oracle_seeded(kind, cfg, E, T, scale):
    import swarm_oracle as so
    from parity_util import assert_biteq

    b = _backend(E, cfg, kind=kind)
    o = so.OracleSwarm(E, cfg, kind=kind)
    seeds = np.arange(1000, 1000 + E, dtype=np.uint64)
    b.seed(seeds)
    o.seed(seeds)
    b.reset()
    o.reset()
    rng = np.random.default_rng(42)
    N = o.N
    for t in range(-1, T):
        if t >= 0:
            if t % 3 == 2:  # goal seeking: parks drones, reaches goals
                d = o.goal[:, None, :] - o.positions
                d = d / np.maximum(np.linalg.norm(d, axis=2, keepdims=True), 1e-6)
                act = (d * 1.2 + rng.normal(0, 0.3, size=(E, N, 3))).astype(np.float32)
            else:
                act = rng.uniform(-scale, scale, size=(E, N, 3)).astype(np.float32)
            b.step(act, auto_reset=True)
            o.step(act, auto_reset=True, num_threads=8)
        for name in ("positions", "velocities", "goal", "obstacles", "step_count", "reward", "dist", "terminated",
                     "truncated", "reached", "collision", "obs_valid", "all_terminated", "all_truncated",
                     "global_state", "active"):
            assert_biteq(name, getattr(b, name), getattr(o, name), t)
        valid = o.obs_valid.astype(bool)
        assert_biteq("obs", b.obs[valid], o.obs[valid], t)
    print(f"{kind} {cfg}: E={E} T={T} bit-exact")


def test_no_auto_reset_and_dead_env_contract():
    """Without auto-reset an ended swarm episode leaves no active agent; further steps return
    terminated['__all__'] = True and nothing else (drone_swarm_env.py:94-95)."""
    import swarm_oracle as so
    from parity_util import assert_biteq

    cfg = {"num_drones": 4, "num_obstacles": 6, "max_steps": 12, "world_size": 10.0}
    E = 256
    b = _backend(E, cfg)
    o = so.OracleSwarm(E, cfg)
    seeds = np.arange(E, dtype=np.uint64)
    for x in (b, o):
        x.seed(seeds)
        x.reset()
    rng = np.random.default_rng(3)
    for t in range(30):
        act = rng.uniform(-1, 1, size=(E, 4, 3)).astype(np.float32)
        b.step(act, auto_reset=False)
        o.step(act, auto_reset=False)
        for name in ("positions", "velocities", "step_count", "reward", "terminated", "truncated", "obs_valid",
                     "all_terminated", "all_truncated", "active"):
            assert_biteq(name, getattr(b, name), getattr(o, name), t)
    assert o.all_terminated.all() and not o.active.any()
    # partial reset by mask, continuing each env's stream
    mask = (np.arange(E) % 3 == 0).astype(np.uint8)
    b.reset(mask)
    o.reset(mask)
    for name in ("positions", "velocities", "goal", "obstacles", "step_count", "obs_valid", "active", "dist"):
        assert_biteq(name, getattr(b, name), getattr(o, name), "masked reset")
    m = mask.astype(bool)
    assert np.array_equal(pu.bits(b.obs[m]), pu.bits(o.obs[m]))


def test_state_injection_and_observe():
    import swarm_oracle as so
    from parity_util import assert_biteq

    cfg = {"num_drones": 6, "num_obstacles": 5}
    E = 128
    b = _backend(E, cfg)
    o = so.OracleSwarm(E, cfg)
    rng = np.random.default_rng(11)
    o.positions[:] = rng.uniform(-10, 10, o.positions.shape).astype(np.float32)
    o.velocities[:] = rng.uniform(-2, 2, o.velocities.shape).astype(np.float32)
    o.goal[:] = rng.uniform(-10, 10, o.goal.shape).astype(np.float32)
    o.obstacles[:] = rng.uniform(-10, 10, o.obstacles.shape).astype(np.float32)
    o.active[:] = rng.integers(0, 2, o.active.shape)
    o.observe()
    b.eng.set_state(o.positions, o.velocities, o.goal, o.obstacles, alive=o.active)
    for name in ("obs", "dist", "obs_valid", "global_state"):
        assert_biteq(name, getattr(b, name), getattr(o, name), "observe")


def test_norm_mode_sequential_f32():
    """norm_mode=1 (BLAS builds whose sdot accumulates in float32) against the oracle's same switch."""
    import swarm_oracle as so
    from parity_util import assert_biteq

    cfg = {"num_drones": 8, "num_obstacles": 4}
    E = 200
    b = _backend(E, cfg, norm_mode=1)
    o = so.OracleSwarm(E, cfg, norm_mode=1)
    seeds = np.arange(E, dtype=np.uint64)
    for x in (b, o):
        x.seed(seeds)
        x.reset()
    rng = np.random.default_rng(5)
    for t in range(40):
        act = rng.uniform(-1.5, 1.5, size=(E, 8, 3)).astype(np.float32)
        b.step(act)
        o.step(act, auto_reset=True)
        for name in ("positions", "velocities", "reward", "terminated", "truncated", "obs_valid", "dist"):
            assert_biteq(name, getattr(b, name), getattr(o, name), t)


def test_step_host_matches_device_step():
    """The host-buffer (end-to-end) entry point returns what the device-resident step computes."""
    import torch
    import swarm_b200

    cfg = {"num_drones": 8, "num_obstacles": 4}
    E = 4096
    a = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    b = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    seeds = np.arange(E, dtype=np.uint64)
    for x in (a, b):
        x.seed(seeds)
        x.reset()
    rng = np.random.default_rng(9)
    for t in range(25):
        act = rng.uniform(-1.5, 1.5, size=(E, 8, 3)).astype(np.float32)
        a.step(torch.from_numpy(act).cuda())
        h = b.step_host(act)
        torch.cuda.synchronize()
        for name in ("obs", "reward", "dist", "terminated", "truncated", "reached", "collision", "obs_valid",
                     "all_terminated", "all_truncated", "global_state"):
            assert np.array_equal(pu.bits(h[name].numpy()), pu.bits(getattr(a, name).cpu().numpy())), (name, t)


@pytest.mark.parametrize("cfg,E", [({"num_drones": 32, "num_obstacles": 8, "max_steps": 9, "world_size": 60.0}, 2048),   # four pipelined chunks
                                   ({"num_drones": 5, "num_obstacles": 3, "max_steps": 12}, 333)])  # unaligned chunk
def test_step_host_packed_flags_and_output_sets(cfg, E):
    """ABI 5: `flags` is the five per-agent flag arrays in one byte, packed on the device behind the step; the
    "packed" / "lean" output sets copy it instead of them and leave the other host fields alone."""
    import torch
    import swarm_b200
    from swarm_b200 import _abi

    N = cfg["num_drones"]
    a = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    b = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    for x in (a, b):
        x.seed(np.arange(E, dtype=np.uint64))
        x.reset()
    rng = np.random.default_rng(4)
    names = ("terminated", "truncated", "reached", "collision", "obs_valid")
    assert names == _abi.FLAG_FIELDS
    seen = np.zeros(5, bool)
    for t in range(30):
        act = rng.uniform(-1.5, 1.5, size=(E, N, 3)).astype(np.float32)
        a.step(torch.from_numpy(act).cuda())
        mode = ("packed", "lean", ("flags", "terminated"))[t % 3]
        h = b.step_host(act, outputs=mode)
        want = sum((getattr(a, n).cpu().numpy().astype(np.uint8) & 1) << k for k, n in enumerate(names))
        assert np.array_equal(h["flags"].numpy(), want), (t, mode)
        un = swarm_b200.SwarmEngine.unpack_flags(h["flags"].numpy())
        for k, n in enumerate(names):
            assert np.array_equal(un[n], getattr(a, n).cpu().numpy().astype(bool)), (n, t)
            seen[k] |= un[n].any()
        for n in ("obs", "reward"):
            if mode != ("flags", "terminated"):
                assert np.array_equal(pu.bits(h[n].numpy()), pu.bits(getattr(a, n).cpu().numpy())), (n, t)
    assert seen.all()
    h2d, d2h = b.host_bytes_per_step("lean")
    assert h2d == E * N * 12 and d2h == E * N * (a.D * 4 + 4 + 1) + 2 * E


def test_engine_stats_and_episode_outputs():
    import torch
    import swarm_b200

    cfg = {"num_drones": 4, "num_obstacles": 8, "max_steps": 15, "world_size": 12.0}
    E, T = 512, 64
    eng = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    eng.seed(np.arange(E, dtype=np.uint64))
    eng.reset()
    rng = np.random.default_rng(1)
    eps = 0
    ret_sum = 0.0
    len_sum = 0
    running = np.zeros(E, np.float64)
    for t in range(T):
        act = torch.from_numpy(rng.uniform(-1, 1, size=(E, 4, 3)).astype(np.float32)).cuda()
        eng.step(act)
        done = (eng.all_terminated | eng.all_truncated).cpu().numpy().astype(bool)
        running += eng.reward.cpu().numpy().astype(np.float64).sum(axis=1)
        er = eng.episode_return.cpu().numpy()
        el = eng.episode_length.cpu().numpy()
        assert np.all(el[~done] == 0)
        np.testing.assert_allclose(er[done], running[done], rtol=1e-4, atol=1e-3)
        eps += int(done.sum())
        ret_sum += float(er[done].sum())
        len_sum += int(el[done].sum())
        running[done] = 0.0
    st = eng.stats()
    assert st["episodes"] == eps and st["length_sum"] == len_sum and st["env_steps"] == E * T
    assert st["success"] + st["collision"] + st["timeout"] == eps
    np.testing.assert_allclose(st["return_sum"], ret_sum, rtol=1e-5)


def test_sharding_invariance():
    """An env's trajectory depends on its GLOBAL index only, not on how the batch is split over
    ranks (SURVEY 8e): one engine with E envs == two engines with the halves."""
    import torch
    import swarm_b200
    from swarm_b200 import distributed as D

    cfg = {"num_drones": 8, "num_obstacles": 4, "max_steps": 30}
    E, T = 1024, 50
    whole = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    whole.seed(D.global_env_seeds(7, 0, E))
    parts = []
    for r in range(2):
        lo, hi = D.shard_range(E, r, 2)
        e = swarm_b200.SwarmEngine(hi - lo, cfg, device="cuda:0")
        e.seed(D.global_env_seeds(7, lo, hi))
        parts.append((lo, hi, e))
    whole.reset()
    for _, _, e in parts:
        e.reset()
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(3)
    for t in range(T):
        act = torch.rand((E, 8, 3), generator=gen, device="cuda:0") * 3 - 1.5
        whole.step(act)
        for lo, hi, e in parts:
            e.step(act[lo:hi].contiguous())
        for name in ("pos4", "vel4", "obs", "reward", "terminated", "truncated", "all_terminated", "global_state"):
            got = torch.cat([getattr(e, name) for _, _, e in parts])
            assert torch.equal(got, getattr(whole, name)), (name, t)
    s = D.stats_to_vector(whole.stats())
    s2 = sum(D.stats_to_vector(e.stats()) for _, _, e in parts)
    assert np.array_equal(s[[0, 1, 2, 3, 4, 6, 7]], s2[[0, 1, 2, 3, 4, 6, 7]])
    np.testing.assert_allclose(s[5], s2[5], rtol=1e-9)


@pytest.mark.parametrize("N,M", [(32, 8), (8, 4)])
def test_sharded_swarm_invariance_with_randomisation_and_delay(N, M):
    """`ShardedSwarm` (the repo's multi-GPU class) with domain randomisation AND the control-delay ring: one engine
    with E envs == two shards with the halves, bit for bit -- the randomisation streams are keyed by the GLOBAL env
    index (`env_index_base`), which the class must pass on.  Uses two devices when the box has them."""
    import torch
    import swarm_b200
    from swarm_b200 import distributed as D
    from test_domain_randomization import DR_DELAY

    cfg = {"num_drones": N, "num_obstacles": M, "max_steps": 25}
    E, T = 600, 60
    devs = ["cuda:0", "cuda:1" if torch.cuda.device_count() >= 2 else "cuda:0"]
    kw = dict(domain_randomization=DR_DELAY, dr_seed=41)
    whole = D.ShardedSwarm(E, cfg, base_seed=5, rank=0, world_size=1, device=torch.device("cuda:0"), **kw)
    parts = [D.ShardedSwarm(E, cfg, base_seed=5, rank=r, world_size=2, device=torch.device(devs[r]), **kw)
             for r in range(2)]
    assert [p.engine._c.env_index_base for p in parts] == [0, E // 2]
    for x in [whole] + parts:
        x.reset()
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(9)
    names = ("pos4", "vel4", "goal4", "obst4", "obs", "reward", "dist", "terminated", "truncated", "reached", "collision",
             "obs_valid", "all_terminated", "all_truncated", "global_state", "rng", "step_count", "dr_params", "act_hist")
    for t in range(-1, T):
        if t >= 0:
            act = torch.rand((E, N, 3), generator=gen, device="cuda:0") * 2.4 - 1.2
            whole.step(act)
            for p in parts:
                p.step(act[p.lo:p.hi].to(p.engine.device).contiguous())
        for name in names:
            got = torch.cat([getattr(p.engine, name).to("cuda:0") for p in parts])
            want = getattr(whole.engine, name)
            assert torch.equal(got.view(torch.uint8), want.view(torch.uint8)), (name, t)
    assert whole.engine.stats()["episodes"] > E   # the run went through resets (new per-episode constants)


@pytest.mark.parametrize("cfg,E,dr", [({"num_drones": 8, "num_obstacles": 4, "max_steps": 25}, 1000, False),
                                      ({"num_drones": 32, "num_obstacles": 8, "max_steps": 30}, 300, True),
                                      # more groups than resident warps: some warps own two groups (no resident state)
                                      ({"num_drones": 32, "num_obstacles": 8, "max_steps": 30}, 6000, False),
                                      ({"num_drones": 16, "num_obstacles": 4, "max_steps": 20}, 9001, True),
                                      ({"num_drones": 128, "num_obstacles": 8, "world_size": 60.0}, 64, False),
                                      ({"num_drones": 5, "num_obstacles": 3, "max_steps": 20}, 500, False)])
def test_step_many_and_graph_replay_match_the_step_loop(cfg, E, dr):
    """`swarm_step_many` (one host call for T steps) and a captured CUDA graph of it, replayed several times with an
    ODD number of steps per replay, leave every buffer exactly as a Python loop over `swarm_step` does: the library
    keeps no per-launch host state (the reset-list parity lives on the device)."""
    import torch
    import swarm_b200
    from test_domain_randomization import DR_DELAY

    N, T, R = cfg["num_drones"], 7, 3
    kw = dict(domain_randomization=DR_DELAY, dr_seed=5) if dr else {}
    engines = []
    for _ in range(3):
        e = swarm_b200.SwarmEngine(E, cfg, device="cuda:0", reward64=True, **kw)
        e.seed(np.arange(E, dtype=np.uint64))
        e.reset()
        engines.append(e)
    loop, many, graphed = engines
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(21)
    acts = [torch.rand((T, E, N, 3), generator=gen, device="cuda:0") * 2.4 - 1.2 for _ in range(R)]
    buf = acts[0].clone()
    graph = graphed.capture_steps(buf)      # (the capture's warm-up call already stepped once with buf[0])
    loop.step(acts[0][0]); many.step(acts[0][0])
    names = ["pos4", "vel4", "goal4", "obst4", "obs", "reward64", "dist", "terminated", "truncated", "reached", "collision",
             "obs_valid", "all_terminated", "all_truncated", "global_state", "rng", "step_count", "ep_return"]
    if dr:
        names += ["dr_params", "act_hist"]
    for r in range(R):
        for t in range(T):
            loop.step(acts[r][t])
        many.step_many(acts[r])
        buf.copy_(acts[r])
        graph.replay()
        for name in names:
            want = getattr(loop, name).view(torch.uint8)
            assert torch.equal(getattr(many, name).view(torch.uint8), want), ("step_many", name, r)
            assert torch.equal(getattr(graphed, name).view(torch.uint8), want), ("graph", name, r)
    assert loop.stats() == many.stats() == graphed.stats()


@pytest.mark.parametrize("auto_reset", [False, True])
def test_back_to_back_launches_without_host_sync(auto_reset):
    """Steps enqueued back to back with no host work in between (actions already on the device): the step launch
    does not wait at its top for the launch in front of it (programmatic dependent launch), so this is the case
    where a missing dependency would show -- with auto_reset off there is no reset launch between two step launches.
    Final state against the oracle, several rounds."""
    import os
    import torch
    import swarm_oracle as so
    cfg = {"num_drones": 32, "num_obstacles": 8, "max_steps": 12}
    E, T, R = 8192, 10, 3
    b = _backend(E, cfg)
    o = so.OracleSwarm(E, cfg)
    seeds = np.arange(E, dtype=np.uint64)
    for x in (b, o):
        x.seed(seeds)
        x.reset()
    rng = np.random.default_rng(8)
    threads = len(os.sched_getaffinity(0))
    for r in range(R):
        acts = rng.uniform(-1, 1, size=(T, E, 32, 3)).astype(np.float32)
        dev = torch.from_numpy(acts).to("cuda:0")
        torch.cuda.synchronize()
        for t in range(T):
            b.eng.step(dev[t], auto_reset=auto_reset)
        for t in range(T):
            o.step(acts[t], auto_reset=auto_reset, num_threads=threads)
        for fname in ("positions", "velocities", "goal", "obstacles", "step_count", "reward", "dist", "terminated",
                      "truncated", "obs_valid", "all_terminated", "all_truncated", "active"):
            pu.assert_biteq(fname, getattr(b, fname), getattr(o, fname), (r, auto_reset))
        if not auto_reset:   # (bring the dead envs back so that the next round has something to step)
            for x in (b, o):
                x.reset()


def test_step_accepts_a_misaligned_actions_view():
    """A float32 view at a 4-byte storage offset is a legal `actions` argument: the launch falls back to the general
    kernel, whose 16-byte copies must then be skipped too (it used to fault with a misaligned address)."""
    import torch
    import swarm_b200
    cfg = {"num_drones": 8, "num_obstacles": 4, "max_steps": 30}
    E = 256
    a, b = (swarm_b200.SwarmEngine(E, cfg, device="cuda:0") for _ in range(2))
    for e in (a, b):
        e.seed(np.arange(E, dtype=np.uint64))
        e.reset()
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(4)
    for t in range(12):
        act = torch.rand((E, 8, 3), generator=gen, device="cuda:0") * 2 - 1
        storage = torch.empty(act.numel() + 1, device="cuda:0")
        view = storage[1:].view(E, 8, 3)
        view.copy_(act)
        assert view.data_ptr() % 16 == 4
        a.step(act)
        b.step(view)
        for name in ("pos4", "vel4", "obs", "reward", "terminated", "all_terminated", "rng"):
            assert torch.equal(getattr(a, name), getattr(b, name)), (name, t)


def test_single_env_episode_statistics():
    """kind='single': success / collision / timeout counters partition the ended episodes (they used to stay 0)."""
    import torch
    import swarm_b200
    E, T = 2048, 120
    eng = swarm_b200.SwarmEngine(E, {"num_obstacles": 8, "max_steps": 40, "world_size": 8.0}, kind="single", device="cuda:0")
    eng.seed(np.arange(E, dtype=np.uint64))
    eng.reset()
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(1)
    succ = col = to = 0
    for t in range(T):
        # drive towards the goal so that all three endings occur
        act = (eng.obs[:, :, 6:9] * 0.5 + torch.randn((E, 1, 3), generator=gen, device="cuda:0") * 0.3).clamp(-1, 1)
        eng.step(act.contiguous())
        done = (eng.all_terminated | eng.all_truncated).bool()
        c = eng.collision[:, 0].bool() & done
        s = eng.reached[:, 0].bool() & done & ~c
        col += int(c.sum()); succ += int(s.sum()); to += int((done & ~c & ~s).sum())
    st = eng.stats()
    assert st["episodes"] == succ + col + to and st["episodes"] > 0
    assert (st["success"], st["collision"], st["timeout"]) == (succ, col, to)
    assert succ > 0 and col > 0 and to > 0


@pytest.mark.parametrize("kind,cfg", [("swarm", {"num_drones": 8, "num_obstacles": 4}),      # rotation-pass kernel
                                      ("swarm", {"num_drones": 5, "num_obstacles": 3}),      # general kernel
                                      ("swarm", {"num_drones": 64, "num_obstacles": 8, "world_size": 90.0}),   # wide kernel
                                      ("single", {"num_obstacles": 8})])
def test_nan_action_guard_counter(kind, cfg):
    """np.clip lets a NaN action through (drone_swarm_env.py:105) and so does the engine -- the env's state is NaN
    from then on, like the reference's; `stats()["nan_actions"]` counts the drones it was applied to (SURVEY 5.3)."""
    import torch
    import swarm_b200
    E = 64
    eng = swarm_b200.SwarmEngine(E, cfg, kind=kind, device="cuda:0")
    eng.seed(np.arange(E, dtype=np.uint64))
    eng.reset()
    N = eng.N
    act = torch.zeros((E, N, 3), device="cuda:0")
    eng.step(act, auto_reset=False)
    assert eng.stats()["nan_actions"] == 0
    alive = eng.alive.clone()
    live = torch.nonzero(alive.all(dim=1)).flatten().tolist()      # envs whose episode is still running
    assert len(live) >= 3
    e1, e2, e3 = live[:3]
    act[e1, 0, 1] = float("nan")
    act[e2, N - 1, :] = float("nan")
    eng.step(act, auto_reset=False)
    assert eng.stats()["nan_actions"] == 2
    assert bool(torch.isnan(eng.positions[e1, 0]).any()) and not bool(torch.isnan(eng.positions[e3]).any())


def test_state_dict_roundtrip_continues_bit_exact():
    import torch
    import swarm_b200

    cfg = {"num_drones": 5, "num_obstacles": 6, "max_steps": 20}
    E = 300
    a = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    a.seed(np.arange(E, dtype=np.uint64))
    a.reset()
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(0)
    acts = [torch.rand((E, 5, 3), generator=gen, device="cuda:0") * 2 - 1 for _ in range(40)]
    for t in range(15):
        a.step(acts[t])
    sd = a.state_dict()
    b = swarm_b200.SwarmEngine(E, cfg, device="cuda:0")
    b.load_state_dict(sd)
    for name in ("obs", "obs_valid", "reward", "terminated", "all_terminated", "global_state", "episode_return"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name     # outputs of the last call are restored too
    with pytest.raises(ValueError, match="max_steps"):                     # a different env config must not load
        swarm_b200.SwarmEngine(E, {**cfg, "max_steps": 21}, device="cuda:0").load_state_dict(sd)
    with pytest.raises(ValueError, match="domain_randomization"):
        from test_domain_randomization import DR_V1
        swarm_b200.SwarmEngine(E, cfg, device="cuda:0", domain_randomization=DR_V1).load_state_dict(sd)
    for t in range(15, 40):
        a.step(acts[t])
        b.step(acts[t])
        for name in ("pos4", "vel4", "goal4", "obs", "reward", "rng", "step_count", "all_terminated"):
            assert torch.equal(getattr(a, name), getattr(b, name)), (name, t)
    assert a.stats() == b.stats()


def test_batched_evaluator_matches_reference_loop_on_facade():
    """evaluate_batched(faithful=True) == the reference's per-episode loop
    (scripts/evaluate_protocol.py:237-331, restated here) driven through the façade env."""
    import math
    import torch
    import swarm_b200

    cfg = {"num_drones": 4, "num_obstacles": 6, "max_steps": 60, "world_size": 14.0}
    E, base = 24, 500

    def policy_np(obs):  # bang-bang goal seeking from the local observation (exactly reproducible)
        return np.sign(obs[6:9]).astype(np.float32)

    def policy_t(obs, valid):
        return torch.sign(obs[..., 6:9])

    def dist(a, b):
        return float(np.linalg.norm(a - b))

    ref = []
    for ep in range(E):
        env = swarm_b200.DroneSwarmEnv({**cfg, "seed": base + ep})
        obs, _ = env.reset()
        ids = list(obs)
        starts = {a: obs[a][0:3].copy() for a in ids}
        goals = {a: obs[a][0:3] + obs[a][6:9] for a in ids}
        last = {a: starts[a].copy() for a in ids}
        trav = {a: 0.0 for a in ids}
        rew_sum, step, any_col, reached_step, fes = 0.0, 0, False, None, []
        t_all = tr_all = False
        while not (t_all or tr_all):
            acts = {a: policy_np(o) for a, o in obs.items()}
            obs, rewards, term, trunc, infos = env.step(acts)
            step += 1
            rew_sum += float(np.mean(list(rewards.values()))) if rewards else 0.0
            pos_now, flag = {}, True
            for a, o in obs.items():
                p = o[0:3]
                trav[a] += dist(last[a], p)
                last[a] = p
                pos_now[a] = p
                if infos[a].get("collision"):
                    any_col = True
                if not infos[a].get("reached_goal"):
                    flag = False
            ks = list(pos_now)
            errs = []
            for a in ks:
                ds = [dist(pos_now[a], pos_now[b]) for b in ks if b != a]
                if ds:
                    errs.append(float(np.mean(np.abs(np.asarray(ds) - env.cfg.desired_spacing))))
            fes.append(float(np.mean(errs)) if len(ks) > 1 and errs else 0.0)
            if flag and reached_step is None:
                reached_step = step
            t_all, tr_all = term["__all__"], trunc["__all__"]
        pe = np.mean([dist(starts[a], goals[a]) / trav[a] if trav[a] > 1e-8 else 0.0 for a in ids])
        ref.append(dict(success=int(not any_col and reached_step is not None), ttg=reached_step, fe=np.mean(fes),
                        pe=pe, rew=rew_sum, length=step))
        env.close()

    eng = swarm_b200.SwarmEngine(E, cfg, device="cuda:0", reward64=True)
    eng.seed(np.arange(base, base + E, dtype=np.uint64))
    out = swarm_b200.evaluate_batched(eng, policy_t, faithful=True)
    pe_ = out["per_episode"]
    assert bool(pe_["finished"].all())
    assert pe_["length"].tolist() == [r["length"] for r in ref]
    assert pe_["success"].long().tolist() == [r["success"] for r in ref]
    assert [None if math.isnan(x) else int(x) for x in pe_["time_to_goal"].tolist()] == [r["ttg"] for r in ref]
    np.testing.assert_allclose(pe_["episode_reward"].cpu().numpy(), [r["rew"] for r in ref], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(pe_["formation_error"].cpu().numpy(), [r["fe"] for r in ref], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(pe_["path_efficiency"].cpu().numpy(), [r["pe"] for r in ref], rtol=1e-5, atol=1e-6)
    agg = out["aggregate"]
    assert agg["success_rate"] == 1.0  # the reference's scoring quirk: every finished episode is a "success"
    eng2 = swarm_b200.SwarmEngine(E, cfg, device="cuda:0", reward64=True)
    eng2.seed(np.arange(base, base + E, dtype=np.uint64))
    truth = swarm_b200.evaluate_batched(eng2, policy_t, faithful=False)
    assert 0.0 <= truth["aggregate"]["success_rate"] <= 1.0
    assert truth["per_episode"]["length"].tolist() == [r["length"] for r in ref]


FULL_SIZE = [
    # BASELINE.json configs at their FULL env counts (C2's 4096 envs is in CASES above)
    ("c3", {"num_drones": 16, "num_obstacles": 8}, 16384, 40, None),
    ("c4", {"num_drones": 32, "num_obstacles": 8}, 65536, 16, None),
    ("c4_dr", {"num_drones": 32, "num_obstacles": 8}, 65536, 12, "v1"),
    ("c4_dr_delay", {"num_drones": 32, "num_obstacles": 8}, 65536, 12, "v1+delay"),   # the yaml's whole actuation block
    ("c5_w20", {"num_drones": 128, "num_obstacles": 8}, 8192, 5, None),              # C5 as named: every env resets every step
    ("c5", {"num_drones": 128, "num_obstacles": 8, "world_size": 70.0}, 8192, 6, None),
    # round 2: BASELINE config 5 under domain_randomization_v1 (+ control delay) -- the wide kernel's DR instantiations
    ("c5_dr_delay", {"num_drones": 128, "num_obstacles": 8, "world_size": 70.0, "max_steps": 6}, 8192, 8, "v1+delay"),
    ("c5_w20_dr", {"num_drones": 128, "num_obstacles": 8}, 4096, 4, "v1"),
]


LONG_HORIZON = [
    # north_star: "over 1000 steps" -- every BASELINE swarm shape for 1000 steps against the C oracle
    ("c2", {"num_drones": 8, "num_obstacles": 4}, 256, 1000),
    ("c3_w20", {"num_drones": 16, "num_obstacles": 8}, 256, 1000),
    ("c4_w20", {"num_drones": 32, "num_obstacles": 8}, 256, 1000),
    ("c4_w44", {"num_drones": 32, "num_obstacles": 8, "world_size": 44.0}, 256, 1000),
    ("c5_w70", {"num_drones": 128, "num_obstacles": 8, "world_size": 70.0}, 256, 1000),
]


@pytest.mark.parametrize("name,cfg,E,T", LONG_HORIZON)
def test_cuda_matches_oracle_over_1000_steps(name, cfg, E, T):
    """1000 consecutive steps (auto-reset on, U(-1, 1) actions) of 256 env instances per BASELINE shape: every
    array bit for bit at every step, the obs rows of the valid agents included."""
    import os
    import swarm_oracle as so
    from parity_util import assert_biteq

    b = _backend(E, cfg)
    o = so.OracleSwarm(E, cfg)
    seeds = np.arange(5000, 5000 + E, dtype=np.uint64)
    for x in (b, o):
        x.seed(seeds)
        x.reset()
    rng = np.random.default_rng(321)
    N = o.N
    threads = len(os.sched_getaffinity(0))
    fields = ("positions", "velocities", "goal", "obstacles", "step_count", "reward", "dist", "terminated", "truncated",
              "reached", "collision", "obs_valid", "all_terminated", "all_truncated", "global_state", "active")
    for t in range(-1, T):
        if t >= 0:
            act = rng.uniform(-1.0, 1.0, size=(E, N, 3)).astype(np.float32)
            b.step(act, auto_reset=True)
            o.step(act, auto_reset=True, num_threads=threads)
        for fname in fields:
            assert_biteq(fname, getattr(b, fname), getattr(o, fname), t)
        valid = o.obs_valid.astype(bool)
        assert_biteq("obs", b.obs[valid], o.obs[valid], t)
    st = b.eng.stats()
    assert st["env_steps"] == E * T
    print(f"{name}: {E} envs x {N} drones x {T} steps bit-exact; episodes {st['episodes']}")


@pytest.mark.parametrize("name,cfg,E,T,dr", FULL_SIZE)
def test_cuda_matches_oracle_at_full_baseline_size(name, cfg, E, T, dr):
    """The whole BASELINE batch (tens of thousands of env instances) against the C oracle, every array
    bit for bit; the oracle needs a few seconds per config on the box's host threads."""
    import os
    import swarm_oracle as so
    from parity_util import assert_biteq

    dr_cfg = None
    if dr:
        from test_domain_randomization import DR_V1, DR_DELAY
        dr_cfg = DR_DELAY if dr.endswith("delay") else DR_V1
    kw = dict(domain_randomization=dr_cfg, dr_seed=2026) if dr_cfg else {}
    b = _backend(E, cfg, **kw)
    o = so.OracleSwarm(E, cfg, dr=dr_cfg, dr_seed=2026)
    seeds = np.arange(E, dtype=np.uint64)
    for x in (b, o):
        x.seed(seeds)
        x.reset()
    rng = np.random.default_rng(123)
    N = o.N
    threads = len(os.sched_getaffinity(0))
    for t in range(-1, T):
        if t >= 0:
            act = rng.uniform(-1.0, 1.0, size=(E, N, 3)).astype(np.float32)
            b.step(act, auto_reset=True)
            o.step(act, auto_reset=True, num_threads=threads)
        for fname in ("positions", "velocities", "goal", "obstacles", "step_count", "reward", "dist", "terminated",
                      "truncated", "reached", "collision", "obs_valid", "all_terminated", "all_truncated",
                      "global_state", "active"):
            assert_biteq(fname, getattr(b, fname), getattr(o, fname), t)
        valid = o.obs_valid.astype(bool)
        assert_biteq("obs", b.obs[valid], o.obs[valid], t)
    st = b.eng.stats()
    assert st["env_steps"] == E * T
    print(f"{name}: {E} envs x {N} drones x {T} steps bit-exact; episodes {st['episodes']}")
