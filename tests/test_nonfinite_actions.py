"""NaN and infinite actions: every kernel and the C oracle against numpy's semantics.

A policy that diverges emits NaN actions.  The reference handles them with plain numpy, and so must the engine:

  - np.clip maps +-inf to +-1 and lets NaN through (swarm and single-drone envs); the physics env does not clip,
    and an infinite velocity turns NaN at the next sub-step's speed clamp (inf / inf).
  - A NaN drone's velocity and position stay NaN: the speed clip, the wall clip and the physics clamps compare
    false with NaN and do not fire.
  - Every distance involving a NaN drone is NaN.  np.argsort sorts NaN after every number, so in the neighbour and
    obstacle blocks a NaN candidate ranks last and the slot it fills holds NaN in all four fields; zero padding
    appears only when there are fewer candidates than slots.
  - Pair, obstacle, ground and goal compares with NaN are false: a NaN drone never collides or reaches the goal,
    its env runs to the time limit and is truncated.  The formation mean of every active drone of the env takes
    the NaN drone in, so every active drone of that env gets a NaN reward.
  - The order among NaN candidates and the sign / payload bits of a NaN are not part of the contract (x86 and the
    GPU make different NaNs): comparisons here treat every NaN as equal and every other value bit for bit.

CPU half: the C oracle against a numpy restatement of the observation blocks and the flags, on built layouts.
GPU half: the engine against the oracle on the same kind of layouts, through every step kernel and launch mode,
with NaN envs in the same warps as clean envs and envs that end on the step, for max_steps + 2 steps so the NaN env
is truncated and re-drawn.
"""
import math
import os

import numpy as np
import pytest

import parity_util as pu
from test_selection_edges import _far_obstacles, _grid, drone_dist, kernels_run, obst_dist

F = np.float32
MAX_STEPS = 6
THR_PAIR = F(2 * 0.5)          # f32(2 collision_radius)
THR_OBST = F(0.5 + 0.8)        # f32(collision_radius + obstacle_radius)
PHYS_THR_PAIR = F(2 * 0.15)    # drone contact radius 0.15
PHYS_THR_OBST = F(0.8 + 0.15)
PHYS_LIFT = np.array([0.0, 0.0, 10.0], F)   # physics layouts sit above the ground (z >= 0.7)


def same(name, got, want, t=None):
    """Same shape, same NaN mask, and every element that is not NaN bit-identical."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (name, t, got.shape, want.shape)
    if got.dtype != want.dtype:
        got = got.astype(want.dtype)
    if want.dtype.kind == "f":
        gn, wn = np.isnan(got), np.isnan(want)
        if not np.array_equal(gn, wn):
            i = tuple(np.argwhere(gn != wn)[0])
            raise AssertionError(f"{name} NaN mask differs at step {t}, index {i}: got {got[i]!r} want {want[i]!r}")
        got, want = np.where(gn, 0, got).astype(want.dtype), np.where(wn, 0, want).astype(want.dtype)
    pu.assert_biteq(name, got, want, t)


# ---------------------------------------------------------------------------------------------- numpy restatement
def _block(rel, d, slots):
    """`slots` x (rx, ry, rz, d) of the nearest candidates, np.argsort order (NaN last), zero padded."""
    out = np.zeros((slots, 4), F)
    order = np.argsort(d, kind="stable")[:slots]
    out[:len(order), :3] = rel[order]
    out[:len(order), 3] = d[order]
    return out.ravel()


def restate_rows(kind, pos, vel, goal, obst, K=3, S=4, vmax=F(4.0)):
    """obs rows of every drone of one env as the reference builds them (drone_swarm_env.py:226-291,
    single_drone_env.py:128-159, drone_physics_env.py:436-439), randomisation off."""
    rows = []
    with np.errstate(all="ignore"):
        for i in range(len(pos)):
            v = vel[i]
            if kind == "physics":
                speed = drone_dist(v)[0]
                if speed > vmax:
                    v = (v / speed).astype(F) * vmax
            parts = [pos[i], v, goal - pos[i]]
            if kind != "single":
                rel = np.delete(pos, i, axis=0) - pos[i]
                parts.append(_block(rel, drone_dist(rel)[0], K))
            rel = obst - pos[i]
            parts.append(_block(rel, obst_dist(rel)[0], S))
            rows.append(np.concatenate(parts).astype(F))
    return np.stack(rows)


def restate_flags(kind, pos, goal, obst, active):
    """(reached, collision, reward is NaN) of every drone active in the step that produced this state."""
    N = len(pos)
    with np.errstate(all="ignore"):
        dist = drone_dist(goal - pos)[0].astype(np.float64)
        d_obst = obst_dist(obst[None, :, :] - pos[:, None, :])[0] if len(obst) else np.zeros((N, 0), F)
        d_pair = np.array([drone_dist(pos - pos[i])[0] for i in range(N)])
    nan_pos = np.isnan(pos).any(axis=1)
    if kind == "physics":
        reached = dist < 0.8
        others = ~np.eye(N, dtype=bool)
        col = (pos[:, 2] <= F(0.025)) | (d_obst <= PHYS_THR_OBST).any(axis=1) | ((d_pair <= PHYS_THR_PAIR) & others).any(axis=1)
        return reached, col, nan_pos
    reached = dist <= 0.8
    col = (d_obst <= THR_OBST).any(axis=1)
    if kind == "swarm":
        partner = active[None, :] & active[:, None] & ~np.eye(N, dtype=bool)
        col = col | ((d_pair <= THR_PAIR) & partner).any(axis=1)
        return reached & active, col & active, np.full(N, bool((nan_pos & active).any())) & active
    return reached, col, nan_pos


# ---------------------------------------------------------------------------------------------- layouts
def env_layout(kind, N, M, rng, role, nan_drones=(), parked=(), step_count=0):
    """One env: drones on the jittered grid of test_selection_edges (no pair, obstacle or goal contact), far
    obstacles, goal near the centre.  role "collide": two active drones exactly at the pair threshold, the rest
    parked, so the env ends on its first step."""
    pos = _grid(N, rng)
    obst = _far_obstacles(M, rng)
    goal = np.array([0.0, 0.0, 7.5], F)
    alive = np.ones(N, np.uint8)
    alive[list(parked)] = 0
    if role == "collide":
        alive[:] = 0
        alive[:2] = 1
        pos[0] = 0.0
        pos[1] = np.array([1, 0, 0], F) * THR_PAIR
    if kind == "physics":
        pos, obst, goal = pos + PHYS_LIFT, obst + PHYS_LIFT, goal + PHYS_LIFT
    return dict(pos=pos, alive=alive, goal=goal, obst=obst, step_count=step_count)


def stack(envs):
    b = {k: np.stack([np.asarray(e[k]) for e in envs]) for k in ("pos", "alive", "goal", "obst", "step_count")}
    b["step_count"] = b["step_count"].astype(np.int32)
    return b


def make_oracle(kind, N, M, b, K=3, S=4, dr=None, max_steps=MAX_STEPS):
    import swarm_oracle as so
    E = len(b["pos"])
    cfg = {"num_drones": N, "num_obstacles": M, "max_steps": max_steps, "world_size": 20.0, "neighbor_k": K,
           "sensed_obstacles": S}
    o = so.OracleSwarm(E, cfg, kind=kind, dr=dr, dr_seed=7)
    o.seed(np.arange(E, dtype=np.uint64))
    o.reset()
    o.positions[:] = b["pos"]
    o.velocities[:] = 0
    o.goal[:] = b["goal"]
    o.obstacles[:] = b["obst"]
    o.active[:] = b["alive"]
    o.step_count[:] = b["step_count"]
    o.observe()
    return o, cfg


def nonfinite_actions(T, E, N, rng, plan):
    """[T, E, N, 3] actions.  plan[e] = (role, drones): "nan" drones submit a NaN component (a different axis per
    drone), "inf" drones +-inf components, in steps 0-2 and zeros afterwards (so the next episode is clean);
    "still" envs submit zeros; "moving" envs small random actions."""
    acts = np.zeros((T, E, N, 3), F)
    for e, (role, drones) in enumerate(plan):
        if role == "moving":
            acts[:, e] = rng.uniform(-0.5, 0.5, (T, N, 3))
        for k, j in enumerate(drones):
            if role == "nan":
                acts[:3, e, j, k % 3] = np.nan
            elif role == "inf":
                acts[:3, e, j, k % 3] = np.inf if k % 2 == 0 else -np.inf
                acts[:3, e, j, (k + 1) % 3] = -np.inf
    return acts


# ---------------------------------------------------------------------------------------------- CPU half
@pytest.mark.parametrize("n", list(range(2, 128)))
def test_numpy_argsort_puts_nan_last(n):
    """The property the contract rests on, at every candidate count the envs produce (N - 1 <= 127, M): np.argsort
    (default and stable) places every NaN after every number, +inf included."""
    rng = np.random.default_rng(n)
    for trial in range(4):
        d = rng.uniform(0, 10, n).astype(F)
        d[rng.random(n) < 0.1] = np.inf
        nan_at = rng.choice(n, size=1 + trial * (n - 1) // 3, replace=False)
        d[nan_at] = np.nan
        for kind in ("quicksort", "stable"):
            order = np.argsort(d, kind=kind)
            k = n - len(nan_at)
            assert not np.isnan(d[order[:k]]).any() and np.isnan(d[order[k:]]).all(), (n, kind)
            assert np.array_equal(d[order[:k]], np.sort(d[~np.isnan(d)]))


CPU_CASES = [
    # id, kind, N, M, K, S, nan drones, parked drones, inf drones
    ("nan_lowest", "swarm", 8, 8, 3, 4, (0,), (), ()),
    ("nan_middle", "swarm", 8, 8, 3, 4, (3,), (), ()),
    ("nan_highest", "swarm", 8, 8, 3, 4, (7,), (), ()),
    ("two_nan", "swarm", 8, 8, 3, 4, (2, 5), (), ()),
    ("all_nan", "swarm", 8, 8, 3, 4, tuple(range(8)), (), ()),
    ("n4_k3", "swarm", 4, 8, 3, 4, (0,), (), ()),
    ("n6_k8_m3", "swarm", 6, 3, 8, 4, (2,), (), ()),
    ("beside_parked", "swarm", 8, 8, 3, 4, (4,), (3, 5), ()),
    ("n32_highest", "swarm", 32, 12, 3, 4, (31,), (), ()),
    ("n128_middle", "swarm", 128, 12, 3, 4, (64, 100), (), ()),
    ("inf_clipped", "swarm", 8, 8, 3, 4, (), (), (1, 6)),
    ("single", "single", 1, 8, 0, 4, (0,), (), ()),
    ("single_inf", "single", 1, 8, 0, 4, (), (), (0,)),
    ("physics_nan", "physics", 3, 8, 3, 4, (1,), (), ()),
    ("physics_inf", "physics", 3, 8, 3, 4, (), (), (0, 2)),
    ("physics_n40_nan", "physics", 40, 4, 3, 4, (0, 39), (), ()),
]


@pytest.mark.parametrize("case", CPU_CASES, ids=[c[0] for c in CPU_CASES])
def test_oracle_matches_numpy_on_nonfinite_actions(case):
    """The C oracle's observation rows, flags and reward NaN masks equal the numpy restatement at every step of
    envs with NaN / infinite actions (and clean envs beside them); the NaN env is truncated at max_steps and its
    next episode is clean."""
    name, kind, N, M, K, S, nan_d, parked, inf_d = case
    rng = np.random.default_rng(11)
    roles = [("nan", nan_d) if nan_d else ("inf", inf_d), ("moving", ()), ("still", ()), ("nan" if nan_d else "inf",
                                                                                       nan_d or inf_d)]
    envs = [env_layout(kind, N, M, rng, r, parked=parked if r == "nan" else ()) for r, _ in roles]
    b = stack(envs)
    T = MAX_STEPS + 2
    o, _ = make_oracle(kind, N, M, b, K=K, S=S)
    acts = nonfinite_actions(T, len(envs), N, rng, roles)
    nonfinite_envs = [e for e, (r, _) in enumerate(roles) if r == "nan" or (r == "inf" and kind == "physics")]
    nan_slots = 0   # neighbour / obstacle slots a NaN candidate filled: what the block check bites on
    for t in range(T):
        active = o.active.astype(bool).copy()
        o.step(acts[t], auto_reset=True)
        for e in range(len(envs)):
            ended = bool(o.all_terminated[e] or o.all_truncated[e])
            if not ended:   # (an ended env's state is the re-drawn one; its flags belong to the terminal state)
                reached, col, nan_r = restate_flags(kind, o.positions[e], o.goal[e], o.obstacles[e], active[e])
                same("reached", o.reached[e], reached.astype(np.uint8), t)
                same("collision", o.collision[e], col.astype(np.uint8), t)
                same("reward is NaN", np.isnan(o.reward[e]), nan_r, t)
            want = restate_rows(kind, o.positions[e], o.velocities[e], o.goal[e], o.obstacles[e], K, S)
            valid = o.obs_valid[e].astype(bool)
            same("obs", o.obs[e][valid], want[valid], t)
            nan_slots += int(np.isnan(o.obs[e][valid][:, 9::4]).sum())
            if e in nonfinite_envs and t < MAX_STEPS - 1:
                assert np.isnan(o.positions[e][list(nan_d or inf_d)]).any(axis=1).all(), (name, t, e)
                assert not ended, (name, t, e)                      # a NaN drone never collides or reaches
                assert np.isnan(o.reward[e][active[e]]).any()
            if e in nonfinite_envs and t == MAX_STEPS - 1:
                assert o.all_truncated[e] and not o.all_terminated[e], (name, e)
                same("truncated", o.truncated[e], active[e].astype(np.uint8), t)
            if e in nonfinite_envs and t >= MAX_STEPS:
                assert np.isfinite(o.positions[e]).all() and np.isfinite(o.reward[e]).all(), (name, t, e)
        if kind != "physics":
            inf_env = [e for e, (r, _) in enumerate(roles) if r == "inf"]
            for e in inf_env:
                assert np.isfinite(o.positions[e]).all(), (name, t, e)    # np.clip: +-inf -> +-1
    assert nan_slots > 0 or (kind != "physics" and not nan_d), name


# ---------------------------------------------------------------------------------------------- GPU half
KNOB_PREFIX = "SWARM_B200_"


@pytest.fixture(autouse=True)
def _clean_knobs(monkeypatch):
    """Clear inherited SWARM_B200_* knobs and pin N = 64 / 128 to the wide rotation kernel at every batch size."""
    for k in list(os.environ):
        if k.startswith(KNOB_PREFIX) and k != "SWARM_B200_LIB":
            monkeypatch.delenv(k)
    monkeypatch.setenv("SWARM_B200_ROTX_MIN_ENVS", "0")


def _dr(dr):
    if dr is None:
        return None
    from test_domain_randomization import DR_DELAY, DR_V1
    return {"v1": DR_V1, "delay": DR_DELAY}[dr]


def gpu_batch(kind, N, M, E=304, seed=5):
    """E envs, cycling through NaN envs (NaN drone at the lowest, a middle, the highest index, two of them, all of
    them, one beside parked drones), +-inf envs, and clean envs that keep running, end by truncation or end by a
    collision on the first step -- so at N = 8 / 16 one warp holds NaN envs and envs of the other kinds."""
    rng = np.random.default_rng(seed)
    nan_sets = [(0,), (N // 2,), (N - 1,), (1, N - 2), tuple(range(N)), (N // 2,)] if N > 1 else [(0,)]
    swarm = kind == "swarm"
    cycle = ["nan", "moving", "trunc", "nan", "collide" if swarm else "moving", "inf", "still", "nan"]
    envs, plan = [], []
    for e in range(E):
        role = cycle[e % len(cycle)]
        if role == "nan":
            drones = nan_sets[(e // len(cycle) * 3 + e % len(cycle)) % len(nan_sets)]
            parked = ()
            if swarm and N >= 4 and e % 3 == 0 and len(drones) == 1:
                parked = tuple({(drones[0] + 1) % N, (drones[0] + 2) % N})
            envs.append(env_layout(kind, N, M, rng, "nan", parked=parked))
            plan.append(("nan", drones + tuple(parked[:1])))     # (a parked drone's NaN action is never applied)
        elif role == "inf":
            envs.append(env_layout(kind, N, M, rng, "inf"))
            plan.append(("inf", (0, N - 1) if N > 1 else (0,)))
        else:
            envs.append(env_layout(kind, N, M, rng, role, step_count=MAX_STEPS - 1 if role == "trunc" else 0))
            plan.append(("moving" if role in ("moving", "trunc", "collide") else "still", ()))
    return stack(envs), plan


def applied_nan_count(o, submitted):
    """Active drones whose APPLIED command (after the control-delay ring, delay = dr_params[:, 7]) has a NaN."""
    t = o.step_count.astype(np.int64)
    d = o.dr_params[:, 7].astype(np.int64) if o._c.dr_enabled else np.zeros_like(t)
    H = o.act_hist.shape[1]
    applied = submitted.copy()
    for e in range(len(t)):
        if d[e] > 0:
            applied[e] = 0.0 if t[e] < d[e] else o.act_hist[e, (t[e] - d[e]) % H]
    return int((np.isnan(applied).any(axis=2) & o.active.astype(bool)).sum())


ORACLE_FIELDS = ("positions", "velocities", "goal", "obstacles", "step_count", "reward", "dist", "terminated",
                 "truncated", "reached", "collision", "obs_valid", "all_terminated", "all_truncated", "global_state",
                 "rng", "active", "obs", "dr_params", "act_hist")


def run_gpu(kind, N, M, K=3, dr=None, mode="step", E=304):
    """Engine and oracle from the same seeds and injected states, max_steps + 2 steps; every output compared after
    every step (step_many: after the last one).  Returns the step kernels that ran."""
    import torch
    import swarm_b200
    b, plan = gpu_batch(kind, N, M, E)
    dr_cfg = _dr(dr)
    T = MAX_STEPS + 2
    o, cfg = make_oracle(kind, N, M, b, K=K, dr=dr_cfg)
    acts = nonfinite_actions(T, E, N, np.random.default_rng(9), plan)
    want, nan_applied, episodes, timeouts = [], 0, 0, 0
    for t in range(T):
        nan_applied += applied_nan_count(o, acts[t])
        o.step(acts[t], auto_reset=True, num_threads=8)
        episodes += int((o.all_terminated | o.all_truncated).sum())
        timeouts += int((o.all_truncated & ~o.all_terminated).sum())
        want.append({k: getattr(o, k).copy() for k in ORACLE_FIELDS})
    assert nan_applied > 0 and any(np.isnan(w["reward"]).any() for w in want)

    eng = swarm_b200.SwarmEngine(E, cfg, kind=kind, device="cuda:0", reward64=True,
                                 **(dict(domain_randomization=dr_cfg, dr_seed=7) if dr_cfg else {}))
    eng.seed(np.arange(E, dtype=np.uint64))
    eng.reset()
    eng.set_state(b["pos"], np.zeros_like(b["pos"]), b["goal"], b["obst"], alive=b["alive"], step_count=b["step_count"])
    eng.reset_stats()
    a = torch.from_numpy(acts).cuda()
    got = lambda x: x.detach().cpu().numpy()  # noqa: E731

    def compare(t):
        w = want[t]
        for name in ORACLE_FIELDS[:15]:
            same(name, got(getattr(eng, name if name != "reward" else "reward64")), w[name], t)
        same("reward32", got(eng.reward), w["reward"].astype(F), t)
        same("rng", got(eng.rng), w["rng"].view(np.int64), t)
        same("alive", got(eng.alive).astype(np.uint8), w["active"], t)
        valid = w["obs_valid"].astype(bool)
        same("obs", got(eng.obs)[valid], w["obs"][valid], t)
        if dr_cfg:
            same("dr_params", got(eng.dr_params), w["dr_params"], t)
            if eng.act_hist is not None:
                same("act_hist", got(eng.act_hist), w["act_hist"], t)

    def go():
        if mode == "many":
            eng.step_many(a)
        else:
            for t in range(T):
                eng.step(a[t])
                compare(t)
    ran = kernels_run(go)
    compare(T - 1)
    # every NaN env was truncated and re-drawn: its new episode and running return are clean again
    assert np.isfinite(got(eng.positions)).all() and np.isfinite(got(eng.ep_return)).all()
    st = eng.stats()
    assert st["nan_actions"] == nan_applied, (st["nan_actions"], nan_applied)
    assert st["episodes"] == episodes and st["timeout"] == timeouts, (st, episodes, timeouts)
    # the return of a NaN episode is NaN, and so is the running return sum once such an episode has ended
    assert math.isnan(st["return_sum"]), st
    return ran


ROT = {8: "swarm_step_rot_kernel", 16: "swarm_step_rot_kernel", 32: "swarm_step_rot_kernel",
       64: "swarm_step_rotx_kernel", 128: "swarm_step_rotx_kernel"}
GENERAL = {"swarm_env_kernel", "swarm_env_kernel_small"}
GPU_SHAPES = [
    # id, kind, N, M, K, SWARM_B200_NO_ROT, kernel
    ("rot_n8", "swarm", 8, 4, 3, False, "rot"),
    ("rot_n16", "swarm", 16, 8, 3, False, "rot"),
    ("rot_n32", "swarm", 32, 12, 3, False, "rot"),
    ("wide_n64", "swarm", 64, 8, 3, False, "rot"),
    ("wide_n128", "swarm", 128, 12, 3, False, "rot"),
    ("general_n4", "swarm", 4, 8, 3, False, "general"),
    ("general_n6_k8", "swarm", 6, 3, 8, False, "general"),
    ("general_n12", "swarm", 12, 8, 3, False, "general"),
    ("general_n32_no_rot", "swarm", 32, 8, 3, True, "general"),
    ("general_large_n40", "swarm", 40, 8, 3, False, "general"),
    ("single_m8", "single", 1, 8, 0, False, "general"),
    ("physics_n3", "physics", 3, 8, 3, False, "general"),
    ("physics_n40", "physics", 40, 4, 3, False, "general"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["step", "many", "fused"])
@pytest.mark.parametrize("dr", [None, "v1", "delay"])
@pytest.mark.parametrize("shape", GPU_SHAPES, ids=[s[0] for s in GPU_SHAPES])
def test_kernels_match_oracle_on_nonfinite_actions(monkeypatch, shape, dr, mode):
    """NaN and +-inf actions through every step kernel: step() (step and auto-reset launches), step_many over all
    steps (the fused instantiation), or step() with SWARM_B200_FUSED_RESET=1; the same outputs as the oracle, NaN
    for NaN, every other value bit for bit, and the nan_actions / episodes / timeout statistics."""
    name, kind, N, M, K, no_rot, kernel = shape
    if no_rot:
        monkeypatch.setenv("SWARM_B200_NO_ROT", "1")
    if mode == "fused":
        monkeypatch.setenv("SWARM_B200_FUSED_RESET", "1")
    ran = run_gpu(kind, N, M, K=K, dr=dr, mode=mode)
    if kernel == "rot":
        assert ROT[N] in ran and not ran & GENERAL, ran
    else:
        assert ran and ran <= GENERAL, ran
