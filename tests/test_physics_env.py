"""DronePhysicsEnv (reference src/swarm_marl/envs/drone_physics_env.py) as a point mass.

The reference integrates rigid bodies with PyBullet, a third-party dependency that is neither
vendored nor installed: PARITY UNPINNED.  What is checked: the CUDA path against the C restatement
(oracle/swarm_oracle.c, bit-exact), the env contract the reference's callers rely on, and the two
loose physical inequalities the reference's own manual scripts check (scripts/verify_physics.py:38-43:
z-drop > 0.5 m after 100 zero-action steps; scripts/verify_dashboard.py:73-78: 0 < z < 10).
"""
import numpy as np
import pytest

import parity_util as pu

FIELDS = ("positions", "velocities", "goal", "obstacles", "step_count", "reward", "dist", "terminated", "truncated",
          "reached", "collision", "obs_valid", "all_terminated", "all_truncated", "global_state", "active")


def test_oracle_zero_action_sinks_and_hover_holds():
    import swarm_oracle as so
    cfg = {"num_drones": 3, "num_obstacles": 0, "max_steps": 400, "world_size": 40.0}
    E = 64
    o = so.OracleSwarm(E, cfg, kind="physics")
    o.seed(np.arange(E, dtype=np.uint64))
    o.reset()
    assert np.all(o.positions[:, :, 2] >= 1.0)                      # :211-212
    assert np.all((o.goal[:, 2] >= 0.5) & (o.goal[:, 2] <= 2.0))    # :241-242
    c_lin = 1.0 - o.damp.astype(np.float64) ** 240
    assert np.all((c_lin > 0.399) & (c_lin < 0.601))                # 0.5 * U(0.8, 1.2) (:218-223)
    z0 = o.positions[:, :, 2].copy()
    high = z0 > 6.0
    for t in range(100):
        o.step(np.zeros((E, 3, 3), np.float32), auto_reset=False)
    drop = z0 - o.positions[:, :, 2]
    running = o.active.astype(bool)
    assert (high & running).sum() > 10
    assert np.all(drop[high & running] > 0.5)                        # verify_physics.py:38-43
    # an env whose lowest drone reached the ground plane ended with a collision
    ended = ~running.any(axis=1)
    assert ended.sum() > 10
    # hover: thrust 0.31 / max_accel on z cancels gravity minus g_comp
    o.reset()
    z1 = o.positions[:, :, 2].copy()
    act = np.zeros((E, 3, 3), np.float32)
    act[..., 2] = np.float32((9.81 - 9.5) / 2.0)
    for t in range(50):
        o.step(act, auto_reset=False)
    np.testing.assert_allclose(o.positions[:, :, 2], z1, atol=2e-3)


def test_oracle_contract_flags_and_rewards():
    import swarm_oracle as so
    cfg = {"num_drones": 4, "num_obstacles": 6, "max_steps": 30, "world_size": 12.0}
    E = 400
    o = so.OracleSwarm(E, cfg, kind="physics")
    o.seed(np.arange(50, 50 + E, dtype=np.uint64))
    o.reset()
    rng = np.random.default_rng(0)
    saw = dict(col=0, trunc=0)
    for t in range(40):
        was_active = o.active.astype(bool).copy()
        o.step(rng.uniform(-1, 1, size=(E, 4, 3)).astype(np.float32), auto_reset=False)
        live = was_active.any(axis=1)
        d = o.dist.astype(np.float64)
        want = -d * 0.1 - 10.0 * o.collision + 50.0 * ((o.reached == 1) & (o.collision == 0))
        np.testing.assert_array_equal(o.reward[live], want[live])            # :378-392
        done = (o.all_terminated | o.all_truncated).astype(bool)
        # one flag pair for every drone (:401-417)
        assert np.all(o.terminated[live] == o.all_terminated[live, None])
        assert np.all(o.truncated[live] == o.all_truncated[live, None])
        assert not np.any(o.all_terminated[live] & o.all_truncated[live])
        assert np.all(o.obs_valid[live] == 1)                                 # obs for every drone, always
        assert np.all(o.active[done] == 0)
        assert np.all(o.all_terminated[~live] == 1) and np.all(o.obs_valid[~live] == 0)
        saw["col"] += int(o.collision[live].any(axis=1).sum())
        saw["trunc"] += int(o.all_truncated[live].sum())
        speed = np.linalg.norm(o.obs[:, :, 3:6], axis=2)
        assert np.all(speed[live] <= 4.0 + 1e-5)                              # observed velocity clamp (:436-439)
    assert saw["col"] > 20 and saw["trunc"] > 5


GPU_CASES = [
    ({"num_drones": 3, "num_obstacles": 8}, 2000, 60),                                   # reference defaults
    ({"num_drones": 3, "num_obstacles": 4, "max_steps": 25, "world_size": 12.0}, 1500, 80),
    ({"num_drones": 8, "num_obstacles": 4, "max_steps": 40}, 600, 60),
    ({"num_drones": 5, "num_obstacles": 0, "max_steps": 30, "neighbor_k": 2, "sensed_obstacles": 3}, 333, 50),
    ({"num_drones": 32, "num_obstacles": 8, "world_size": 44.0, "max_steps": 20}, 128, 30),
    ({"num_drones": 1, "num_obstacles": 3, "max_steps": 20}, 500, 40),
    # more than 32 drones (round 2): the general large-N kernel
    ({"num_drones": 40, "num_obstacles": 4, "world_size": 60.0, "max_steps": 20}, 48, 45),
    ({"num_drones": 64, "num_obstacles": 8, "world_size": 80.0, "max_steps": 15, "neighbor_k": 4, "sensed_obstacles": 5}, 32, 35),
]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,E,T", GPU_CASES)
def test_cuda_physics_matches_oracle(cfg, E, T):
    import swarm_oracle as so
    from engine_backend import EngineBackend
    N = int(cfg["num_drones"])
    o = so.OracleSwarm(E, cfg, kind="physics")
    b = EngineBackend(E, cfg, kind="physics")
    seeds = np.arange(900, 900 + E, dtype=np.uint64)
    for x in (o, b):
        x.seed(seeds)
        x.reset()
    rng = np.random.default_rng(3)
    for t in range(-1, T):
        if t >= 0:
            if t % 4 == 3:   # goal seeking with gravity compensation: reaches goals
                d = o.goal[:, None, :] - o.positions
                d = d / np.maximum(np.linalg.norm(d, axis=2, keepdims=True), 1e-6)
                act = (d * 1.5).astype(np.float32)
                act[..., 2] += np.float32(0.155)
            else:
                act = rng.uniform(-1.6, 1.6, size=(E, N, 3)).astype(np.float32)   # (actions are not clipped, :336)
            o.step(act, auto_reset=True, num_threads=8)
            b.step(act, auto_reset=True)
        for name in FIELDS:
            pu.assert_biteq(name, getattr(b, name), getattr(o, name), t)
        pu.assert_biteq("damp", b.eng.damping.cpu().numpy(), o.damp, t)
        valid = o.obs_valid.astype(bool)
        pu.assert_biteq("obs", b.obs[valid], o.obs[valid], t)


DR_PHYS = {  # domain_randomization_v1.yaml's ranges on top of the physics env (engine semantics, DESIGN.md 9)
    "mass_scale": (0.85, 1.15), "max_accel_scale": (0.90, 1.10), "max_speed_scale": (0.90, 1.10),
    "dt_scale": (0.95, 1.05), "obstacle_radius_scale": (0.9, 1.1), "world_size_scale": (0.95, 1.05),
    "thrust_noise_std": 0.03, "position_noise_std": 0.02, "velocity_noise_std": 0.02,
    "obstacle_distance_noise_std": 0.03, "control_delay_steps": ((0, 1, 2), (0.7, 0.2, 0.1)),
}


def test_oracle_physics_neutral_randomisation_is_the_plain_path_and_constants_scale():
    import swarm_oracle as so
    cfg = {"num_drones": 4, "num_obstacles": 5, "max_steps": 20, "world_size": 12.0}
    E = 256
    neutral = {k: (1.0, 1.0) for k in DR_PHYS if k.endswith("_scale")}
    a, b = so.OracleSwarm(E, cfg, kind="physics"), so.OracleSwarm(E, cfg, kind="physics", dr=neutral, dr_seed=3)
    c = so.OracleSwarm(E, cfg, kind="physics", dr=DR_PHYS, dr_seed=3)
    for x in (a, b, c):
        x.seed(np.arange(E, dtype=np.uint64))
        x.reset()
    rng = np.random.default_rng(2)
    for t in range(50):
        act = rng.uniform(-1.5, 1.5, size=(E, 4, 3)).astype(np.float32)
        for x in (a, b, c):
            x.step(act, auto_reset=True)
        for name in FIELDS + ("obs",):
            pu.assert_biteq(name, getattr(b, name), getattr(a, name), t)
    p = c.dr_params
    assert p[:, 2].min() >= np.float32(0.95 / 240.0) and p[:, 2].max() <= np.float32(1.05 / 240.0)   # sub-step length
    assert p[:, 4].min() >= np.float32(0.15 + 0.8 * 0.9) and p[:, 4].max() <= np.float32(0.15 + 0.8 * 1.1)
    assert set(np.unique(p[:, 7]).astype(int)) <= {0, 1, 2} and len(np.unique(p[:, 7])) == 3
    assert not np.array_equal(c.positions, a.positions)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,E,T", [({"num_drones": 3, "num_obstacles": 8}, 1000, 60),
                                     ({"num_drones": 8, "num_obstacles": 4, "max_steps": 30}, 400, 70),
                                     ({"num_drones": 32, "num_obstacles": 8, "world_size": 44.0, "max_steps": 20}, 96, 30),
                                     ({"num_drones": 5, "num_obstacles": 6, "max_steps": 25, "neighbor_k": 2,
                                       "sensed_obstacles": 6}, 200, 50),
                                     ({"num_drones": 48, "num_obstacles": 6, "world_size": 70.0, "max_steps": 20}, 40, 45)])
def test_cuda_physics_with_domain_randomisation_matches_oracle(cfg, E, T):
    """DR on top of the physics env (round 2): per-episode max_accel / max_speed / sub-step length / obstacle radius /
    world, thrust + sensor noise, control delay -- CUDA and the C restatement agree bit for bit."""
    import swarm_oracle as so
    from engine_backend import EngineBackend
    N = int(cfg["num_drones"])
    o = so.OracleSwarm(E, cfg, kind="physics", dr=DR_PHYS, dr_seed=99, env_index_base=50)
    b = EngineBackend(E, cfg, kind="physics", domain_randomization=DR_PHYS, dr_seed=99, env_index_base=50)
    for x in (o, b):
        x.seed(np.arange(40, 40 + E, dtype=np.uint64))
        x.reset()
    rng = np.random.default_rng(6)
    for t in range(-1, T):
        if t >= 0:
            act = rng.uniform(-1.6, 1.6, size=(E, N, 3)).astype(np.float32)
            o.step(act, auto_reset=True, num_threads=8)
            b.step(act, auto_reset=True)
        for name in FIELDS + ("dr_params",):
            pu.assert_biteq(name, getattr(b, name), getattr(o, name), t)
        pu.assert_biteq("damp", b.eng.damping.cpu().numpy(), o.damp, t)
        valid = o.obs_valid.astype(bool)
        pu.assert_biteq("obs", b.obs[valid], o.obs[valid], t)


@pytest.mark.gpu
def test_cuda_physics_without_auto_reset_parks_the_env():
    import swarm_oracle as so
    from engine_backend import EngineBackend
    cfg = {"num_drones": 3, "num_obstacles": 6, "max_steps": 15, "world_size": 10.0}
    E = 256
    o, b = so.OracleSwarm(E, cfg, kind="physics"), EngineBackend(E, cfg, kind="physics")
    for x in (o, b):
        x.seed(np.arange(E, dtype=np.uint64))
        x.reset()
    rng = np.random.default_rng(8)
    for t in range(25):
        act = rng.uniform(-1, 1, size=(E, 3, 3)).astype(np.float32)
        o.step(act, auto_reset=False)
        b.step(act, auto_reset=False)
        for name in ("positions", "velocities", "step_count", "reward", "terminated", "truncated", "obs_valid",
                     "all_terminated", "all_truncated", "active", "collision", "reached"):
            pu.assert_biteq(name, getattr(b, name), getattr(o, name), t)
    assert not o.active.any()


@pytest.mark.gpu
def test_physics_facade_contract():
    """The dict contract of drone_physics_env.py:174-263, 279-419 on the façade class."""
    import swarm_b200
    env = swarm_b200.DronePhysicsEnv({"num_drones": 3, "num_obstacles": 4, "max_steps": 12})
    obs, infos = env.reset(seed=5)
    assert set(obs) == {"drone_0", "drone_1", "drone_2"} and all(o.shape == (37,) and o.dtype == np.float32 for o in obs.values())
    assert all(set(i) == {"distance_to_goal", "reached_goal", "collision"} for i in infos.values())
    z0 = env.positions[:, 2].copy()
    steps = 0
    while True:
        act = {a: np.zeros(3, np.float32) for a in env.agents}
        obs, rew, term, trunc, infos = env.step(act)
        steps += 1
        assert set(obs) == set(env.agent_ids) and set(rew) == set(env.agent_ids)
        assert all(isinstance(r, float) for r in rew.values())
        assert all({"global_state", "distance_to_goal", "reached_goal", "collision"} <= set(i) for i in infos.values())
        assert infos["drone_0"]["global_state"].shape == (21,)
        assert len({term[a] for a in env.agent_ids}) == 1 and len({trunc[a] for a in env.agent_ids}) == 1
        if term["__all__"] or trunc["__all__"]:
            break
        assert all(0.0 < p[2] < 10.5 for p in env.positions)       # verify_dashboard.py:73-78
    assert steps <= 12 and env.agents == []
    assert np.all(env.positions[:, 2] < z0)                        # zero action sinks (g_comp 9.5 < 9.81)
    obs2, infos2 = env.reset(seed=5)
    assert np.array_equal(obs2["drone_1"], env._engine.obs[0, 1].cpu().numpy())
    env.set_goal([1.0, 2.0, 1.5])
    assert np.allclose(env.goal, [1.0, 2.0, 1.5])
    env.close()
