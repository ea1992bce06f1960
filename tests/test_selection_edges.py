"""Built states that reach the rotation-pass kernels' rarely taken selection branches, and the eligibility bounds.

The rotation kernels select neighbours on truncated packed keys: the distance bits with the low log2(N) bits replaced
by the drone index (obstacles: squared-distance or distance bits with the low 5 bits replaced by the obstacle index).
A few branches keep that exact, and random seeds reach them rarely:

  sort     two of the three smallest drone keys share a bucket: the picks are re-sorted by exact (distance, index)
  rescan   the 3rd and 4th drone keys share a bucket: exact neighbour rescan
  exact    a distance below 2^-14, or a zero / denormal square (NaN formation sum): the exact path
  obst     an obstacle key collision among the first five, equal roots of different squares, or a square below
           2^-101: the obstacle loop of the reference

Each layout here plants drones and obstacles on the axes around one drone (along an axis the distance is exactly
|x|, because sqrt(RN(x^2)) = |x|), so the distance bit patterns are chosen directly.  A zero-velocity, zero-action
step leaves the positions bit-identical, so the planted distances reach the selection code as built.

CPU half: predicates restating the key rules prove that every layout takes the branch it is built for, and the C
oracle's neighbour / obstacle blocks and flags are checked against a brute-force stable sort on (distance, index).
GPU half: the same layouts through every step kernel and launch mode, bit for bit against the oracle with no tie
tolerance, with torch.profiler proving which kernel ran.
"""
import os
import re

import numpy as np
import pytest

import parity_util as pu

F = np.float32
MAX_STEPS = 50
THR_PAIR = F(2 * 0.5)                 # f32(2 collision_radius)
THR_OBST = F(0.5 + 0.8)               # f32(collision_radius + obstacle_radius)
THR_GOAL = F(0.8) if float(F(0.8)) <= 0.8 else np.nextafter(F(0.8), F(0))   # largest f32 <= goal_radius
AXES = np.array([(1, 0, 0), (0, 1, 0), (0, 0, 1), (-1, 0, 0), (0, -1, 0), (0, 0, -1)], F)
EXACT_KEY = 0x38800000                # bits of 2^-14


def up(x, k=1):
    x = F(x)
    for _ in range(k):
        x = np.nextafter(x, F(np.inf))
    return x


def down(x, k=1):
    x = F(x)
    for _ in range(k):
        x = np.nextafter(x, F(-np.inf))
    return x


def u32(x):
    return int(np.asarray(x, F).view(np.uint32))


# ---------------------------------------------------------------------------------------------- distances and keys
def drone_dist(rel):
    """np.linalg.norm of a 3-vector as the reference computes it: float32 squares, float64 sum, float32 root."""
    sq = (rel * rel).astype(np.float64)
    s = ((sq[..., 0] + sq[..., 1]) + sq[..., 2]).astype(F)
    return np.sqrt(s), s


def obst_dist(rel):
    """np.linalg.norm(rel, axis=1): sequential float32 sum of squares, float32 root."""
    sq = rel * rel
    s = (sq[..., 0] + sq[..., 1]) + sq[..., 2]
    return np.sqrt(s), s


def drone_branches(pos, i):
    """The drone-selection branches drone i of an all-active env takes in the rotation kernels."""
    N = len(pos)
    IDX = N - 1
    js = np.array([j for j in range(N) if j != i])
    d, s = drone_dist(pos[js] - pos[i])
    keys = np.sort((d.view(np.uint32) & np.uint32(~IDX & 0xFFFFFFFF)) | js.astype(np.uint32)).astype(np.int64)
    k = list(keys[:4]) + [0xFFFFFFFF] * (4 - min(4, len(keys)))
    return {"sort": (k[0] ^ k[1]) <= IDX or (k[1] ^ k[2]) <= IDX,
            "rescan": (k[2] ^ k[3]) <= IDX,
            "exact": bool(s.min() < np.finfo(F).tiny) or k[0] < EXACT_KEY}


def obst_branch(obst, p, sqkey):
    """The obstacle fallback of the rotation kernels.  sqkey: keys on squared distances (swarm_step_rot.cu at M = 4 /
    8, swarm_step_rotx.cu at every M), then an exact tie among the first five roots is open too; otherwise keys on
    the distances (swarm_step_rot.cu's merge1_5 loop)."""
    M = len(obst)
    d, s = obst_dist(obst - p)
    base = s if sqkey else d
    keys = np.sort((base.view(np.uint32) & np.uint32(~31 & 0xFFFFFFFF)) | np.arange(M, dtype=np.uint32)).astype(np.int64)
    o = list(keys[:5]) + [0xFFFFFFFF] * (5 - min(5, M))
    bad = bool(s.min() < F(2.0 ** -101)) or any((o[q] ^ o[q + 1]) <= 31 for q in range(4))
    if sqkey:
        r = [d[int(x) & 31] if x != 0xFFFFFFFF else F(np.inf) for x in o]
        bad = bad or any(r[q] == r[q + 1] for q in range(4))
    return bad


# ---------------------------------------------------------------------------------------------- layout builder
def _grid(N, rng):
    """Drones not under test: a jittered grid (spacing >= 2.4, |coordinate| in [2.7, 9.3]), inside the smallest wall
    of DR_V1 (world 20 * 0.95 / 2); the planted cluster sits around the origin, more than 4.6 away from all of them."""
    c = np.array([-9.0, -6.0, -3.0, 3.0, 6.0, 9.0])
    g = np.array(np.meshgrid(c, c, c, indexing="ij")).reshape(3, -1).T
    g = g[rng.permutation(len(g))[:N]]
    return (g + rng.uniform(-0.3, 0.3, g.shape)).astype(F)


def _far_obstacles(M, rng):
    c = np.array([-7.5, -4.5, 4.5, 7.5])
    g = np.array(np.meshgrid(c, c, c, indexing="ij")).reshape(3, -1).T
    g = g[np.abs(g).max(axis=1) == 7.5]
    return (g[rng.permutation(len(g))[:M]] + rng.uniform(-0.2, 0.2, (M, 3))).astype(F)


def _partner_order(N, i, n, where):
    """n partner indices of drone i, reached by a forward round (fwd), a backward shuffle (bwd), the half round N / 2
    first (half), or, for N >= 64, the drones in the same lane as i first (lane)."""
    if where == "fwd":
        cand = [(i + 1 + k) % N for k in range(N)]
    elif where == "bwd":
        cand = [(i - 1 - k) % N for k in range(N)]
    elif where == "half":
        cand = [(i + N // 2) % N] + [(i + s * (1 + k)) % N for k in range(N) for s in (1, -1)]
    else:
        cand = [(i + 32 * (k + 1)) % N for k in range(N // 32)] + [(i + s * (1 + k)) % N for k in range(N) for s in (1, -1)]
    out = []
    for j in cand:
        if j != i and j not in out:
            out.append(j)
    return out[:n]


def _equal_root_pair():
    """Two obstacle offsets (x, y, 0) whose sequential float32 squares are adjacent floats in DIFFERENT key buckets
    (the first square's low 5 bits are all ones) but whose float32 roots are equal."""
    rng = np.random.default_rng(1)
    while True:
        x, y = rng.uniform(1.0, 1.4, 2).astype(F)
        s = x * x + y * y
        if u32(s) & 31 != 31 or np.sqrt(s) != np.sqrt(up(s)):
            continue
        for dx in range(8):
            for dy in range(8):
                x2, y2 = up(x, dx), up(y, dy)
                if x2 * x2 + y2 * y2 == up(s):
                    return np.array([x, y, 0], F), np.array([x2, y2, 0], F)


EQ_ROOT = _equal_root_pair()


def families(N, M):
    """Every planted layout for N drones and M obstacles: (family, name, spec).  spec keys:
      d: ascending distances of the planted partners, put on the axes around the drone under test (`axes`: the
         axis of each, default the first ones of AXES); rev: the nearest partner gets the HIGHEST index
      where: which rounds reach the partners (see _partner_order)
      obst / obst_rev: planted obstacle offsets in ascending distance / nearest gets the highest index
      goal: goal offset; parked: partner slots that are parked; want: branch -> expected value for the drone under test
    """
    wheres = ["fwd", "bwd", "half"] + (["lane"] if N >= 64 else [])
    out = []
    for w in wheres:
        out += [
            ("order", f"three_ulps_reversed_{w}", dict(d=[F(1.5), up(1.5), up(1.5, 2)], rev=True, where=w,
                                                       want={"sort": True, "rescan": False, "exact": False})),
            ("order", f"two_in_bucket_reversed_{w}", dict(d=[F(1.25), up(1.25), F(1.75)], rev=True, where=w,
                                                          want={"sort": True, "rescan": False, "exact": False})),
            ("set", f"third_fourth_reversed_{w}", dict(d=[F(1.2), F(1.35), F(1.5), up(1.5)], rev=True, where=w,
                                                       want={"sort": False, "rescan": True, "exact": False})),
            ("set", f"four_in_bucket_reversed_{w}", dict(d=[F(1.5), up(1.5), up(1.5, 2), up(1.5, 3)], rev=True, where=w,
                                                         want={"sort": True, "rescan": True, "exact": False})),
            ("tie", f"mirror_first_two_{w}", dict(d=[F(1.5), F(1.5), F(1.75)], axes=[0, 3, 1], where=w,
                                                 want={"sort": True, "rescan": False, "exact": False})),
            ("tie", f"mirror_reversed_{w}", dict(d=[F(1.25), F(1.5), F(1.5)], axes=[1, 0, 3], rev=True, where=w,
                                                 want={"sort": True, "rescan": False, "exact": False})),
            ("tie", f"third_fourth_{w}", dict(d=[F(1.2), F(1.35), F(1.6), F(1.6)], axes=[1, 2, 0, 3], where=w,
                                              want={"sort": False, "rescan": True, "exact": False})),
            ("tie", f"third_fourth_reversed_{w}", dict(d=[F(1.2), F(1.35), F(1.6), F(1.6), F(1.6)], axes=[1, 2, 0, 3, 5],
                                                       rev=True, where=w, want={"rescan": True, "exact": False})),
            ("tiny", f"coincident_{w}", dict(d=[F(0.0), F(1.5), F(1.75)], where=w, want={"exact": True})),
            ("tiny", f"below_2^-14_{w}", dict(d=[down(2.0 ** -14), F(1.5)], where=w, want={"exact": True})),
            ("tiny", f"at_2^-14_{w}", dict(d=[F(2.0 ** -14), F(1.5)], where=w, want={"exact": False})),
            ("tiny", f"above_2^-14_{w}", dict(d=[up(2.0 ** -14), F(1.5)], where=w, want={"exact": False})),
            ("tiny", f"denormal_square_{w}", dict(d=[F(2.0 ** -70), F(1.5)], where=w, want={"exact": True})),
            ("tiny", f"square_flushes_to_zero_{w}", dict(d=[F(2.0 ** -80), F(1.5)], where=w, want={"exact": True})),
        ]
    ax = AXES
    e0, e1 = EQ_ROOT
    out += [
        ("obstacles", "bucket_reversed", dict(obst=[ax[0] * F(1.5), ax[1] * up(1.5), ax[2] * up(1.5, 2)], obst_rev=True,
                                               want={"obst": True})),
        ("obstacles", "equal_roots_reversed", dict(obst=[e0, e1], obst_rev=True, want={"obst": True})),
        ("obstacles", "equal_roots", dict(obst=[e0, e1], want={"obst": True})),
        # equal roots of different squares at the 4th / 5th boundary: which obstacle is sensed at all is open
        ("obstacles", "equal_roots_at_last_slot_reversed", dict(obst=[ax[0] * F(1.4), ax[1] * F(1.45)] +
                                                                ([ax[4] * F(1.5)] if M >= 8 else []) + [e0, e1],
                                                                obst_rev=True, want={"obst": True})),
        ("obstacles", "tie_at_last_slot", dict(obst=[ax[0] * F(1.45), ax[1] * F(1.6)] +
                                               ([ax[4] * F(1.75)] if M >= 8 else []) + [ax[2] * F(1.9), ax[5] * F(1.9)],
                                               want={"obst": True})),
        ("obstacles", "tie_at_last_slot_reversed", dict(obst=[ax[0] * F(1.45), ax[1] * F(1.6)] +
                                                        ([ax[4] * F(1.75)] if M >= 8 else []) +
                                                        [ax[2] * F(1.9), ax[5] * F(1.9)], obst_rev=True, want={"obst": True})),
        ("obstacles", "on_the_drone", dict(obst=[np.zeros(3, F), ax[1] * F(1.6)], obst_rev=True, want={"obst": True})),
        ("obstacles", "clear", dict(obst=[ax[0] * F(1.45), ax[1] * F(1.6), ax[2] * F(1.75)], obst_rev=True,
                                    want={"obst": False})),
    ]
    for name, t in (("at", THR_PAIR), ("below", down(THR_PAIR)), ("above", up(THR_PAIR))):
        out.append(("threshold", f"pair_{name}", dict(d=[t, F(1.75)], where="half", want={"exact": False})))
        out.append(("threshold", f"obstacle_{name}", dict(obst=[ax[1] * (THR_OBST if name == "at" else
                                                                           down(THR_OBST) if name == "below" else up(THR_OBST))],
                                                          want={})))
        out.append(("threshold", f"goal_{name}", dict(goal=ax[2] * (THR_GOAL if name == "at" else
                                                                    down(THR_GOAL) if name == "below" else up(THR_GOAL)),
                                                      want={})))
        # three parked drones touching the drone under test, an active one exactly at / around the threshold behind
        out.append(("threshold", f"parked_then_active_{name}",
                    dict(d=[F(0.5), F(0.6), F(0.7), t], axes=[0, 1, 2, 3], parked=[0, 1, 2], where="fwd", want={})))
    return out


def build(N, M, fam, spec, i, rng, sqkey):
    """One env: (pos, alive, goal, obstacles, step_count) with spec planted around drone i at the origin."""
    pos = _grid(N, rng)
    obst = _far_obstacles(M, rng)
    goal = np.array([0.0, 0.0, 7.5], F) if fam != "threshold" else np.array([0.0, 0.0, -7.5], F)
    alive = np.ones(N, np.uint8)
    pos[i] = 0.0
    d = spec.get("d", [])
    js = _partner_order(N, i, len(d), spec.get("where", "fwd"))
    js = sorted(js, reverse=bool(spec.get("rev")))
    axes = spec.get("axes", list(range(len(d))))
    for q, (dist, j) in enumerate(zip(d, js)):
        pos[j] = AXES[axes[q]] * F(dist)
        if q in spec.get("parked", ()):
            alive[j] = 0
    po = spec.get("obst", [])
    ms = sorted(range(len(po)), reverse=bool(spec.get("obst_rev")))
    for v, m in zip(po, ms):
        obst[m] = v
    if "goal" in spec:
        goal = spec["goal"].astype(F)
    if "parked" not in spec and N & (N - 1) == 0:   # (packed keys: the rotation kernels' N, powers of two)
        br = drone_branches(pos, i)
        br["obst"] = obst_branch(obst, pos[i], sqkey)
        for k, v in spec["want"].items():
            assert br[k] == v, (N, M, fam, spec, i, k, br)
    return pos, alive, goal, obst, 0


def clean_env(N, M, rng, kind):
    """A filler env: nothing planted ("clean"), ending on this step by truncation ("trunc"), or two active drones
    exactly at the pair threshold and everyone else parked: both collide and the env ends ("collide")."""
    pos = _grid(N, rng)
    obst = _far_obstacles(M, rng)
    alive = np.ones(N, np.uint8)
    sc = MAX_STEPS - 1 if kind == "trunc" else 0
    if kind == "collide":
        alive[:] = 0
        alive[:2] = 1
        pos[0] = 0.0
        pos[1] = AXES[0] * THR_PAIR
    return pos, alive, np.array([0.0, 0.0, 7.5], F), obst, sc


def batch(N, M, sqkey, seed=0):
    """All layouts of `families` with the drone under test at varying indices, each followed by filler envs so that
    at N = 8 / 16 (several envs per warp) hazard envs sit beside clean envs and beside envs that end on the step."""
    rng = np.random.default_rng(seed)
    envs, meta = [], []
    focus_idx = [0, N - 1, N // 2 - 1, 1, N // 2 + 1, 5]
    fill = ["clean", "trunc", "clean", "collide"]
    for k, (fam, name, spec) in enumerate(families(N, M)):
        i = focus_idx[k % len(focus_idx)]
        envs.append(build(N, M, fam, spec, i, rng, sqkey))
        meta.append((fam, name, i))
        for _ in range(k % 3):
            kind = fill[len(envs) % 4]
            envs.append(clean_env(N, M, rng, kind))
            meta.append(("filler", kind, -1))
    pos, alive, goal, obst, sc = (np.stack([e[q] for e in envs]) for q in range(5))
    return dict(pos=pos, alive=alive, goal=goal, obst=obst, step_count=sc.astype(np.int32)), meta


def oracle_for(N, M, b, dr=None, seeds=None, world=20.0, spacing=2.5, steps=1, auto_reset=True, acts=None):
    import swarm_oracle as so
    E = len(b["pos"])
    cfg = {"num_drones": N, "num_obstacles": M, "max_steps": MAX_STEPS, "world_size": world, "desired_spacing": spacing}
    o = so.OracleSwarm(E, cfg, dr=dr, dr_seed=7)
    o.seed(np.arange(E, dtype=np.uint64) if seeds is None else seeds)
    o.reset()
    o.positions[:] = b["pos"]
    o.velocities[:] = 0
    o.goal[:] = b["goal"]
    o.obstacles[:] = b["obst"]
    o.active[:] = b["alive"]
    o.step_count[:] = b["step_count"]
    o.observe()
    for t in range(steps):
        o.step(np.zeros((E, N, 3), F) if acts is None else acts[t], auto_reset=auto_reset)
    return o, cfg


# ---------------------------------------------------------------------------------------------- CPU half
SHAPES = [(8, 4), (8, 12), (16, 8), (32, 12), (32, 4), (64, 8), (128, 12)]


def _sqkey(N, M):
    return N >= 64 or M in (4, 8)


@pytest.mark.parametrize("N,M", SHAPES)
def test_layouts_reach_their_branches(N, M):
    """Every planted layout takes the branch it is built for (asserted inside `build`), and across the batch each
    branch is reached by several drones under test."""
    b, meta = batch(N, M, _sqkey(N, M))
    seen = {"sort": 0, "rescan": 0, "exact": 0, "obst": 0}
    for e, (fam, name, i) in enumerate(meta):
        if i < 0 or not b["alive"][e].all():
            continue
        br = drone_branches(b["pos"][e], i)
        br["obst"] = obst_branch(b["obst"][e], b["pos"][e, i], _sqkey(N, M))
        for k in seen:
            seen[k] += int(br[k])
    assert min(seen.values()) >= 3, seen
    fams = {m[0] for m in meta}
    assert fams == {"order", "set", "tie", "tiny", "obstacles", "threshold", "filler"}


@pytest.mark.parametrize("N,M", SHAPES)
def test_oracle_blocks_are_the_stable_sort_of_every_layout(N, M):
    """The C oracle's neighbour and obstacle blocks are the k smallest (distance, index) pairs, lowest index first
    on ties, and its pair / obstacle / goal flags are the threshold compares, for every planted layout."""
    b, meta = batch(N, M, _sqkey(N, M))
    o, _ = oracle_for(N, M, b, steps=0)
    K, S = 3, 4
    for e, (fam, name, i) in enumerate(meta):
        if i < 0:
            continue
        pos, obst = b["pos"][e], b["obst"][e]
        for a in np.flatnonzero(o.obs_valid[e]):
            row = o.obs[e, a]
            js = np.array([j for j in range(N) if j != a])
            rel = pos[js] - pos[a]
            d, _ = drone_dist(rel)
            order = np.lexsort((js, d))[:K]
            want = np.concatenate([rel[order], d[order, None]], axis=1).ravel()
            assert np.array_equal(pu.bits(row[9:9 + 4 * K]), pu.bits(want)), (N, M, name, e, a)
            rel_o = obst - pos[a]
            do, _ = obst_dist(rel_o)
            order = np.lexsort((np.arange(M), do))[:S]
            want = np.concatenate([rel_o[order], do[order, None]], axis=1).ravel()
            assert np.array_equal(pu.bits(row[9 + 4 * K:]), pu.bits(want)), (N, M, name, e, a)
    o2, _ = oracle_for(N, M, b, steps=1, auto_reset=False)
    for e, (fam, name, i) in enumerate(meta):
        if i < 0:
            continue
        pos, alive = b["pos"][e], b["alive"][e].astype(bool)
        for a in np.flatnonzero(alive):
            js = np.array([j for j in range(N) if j != a and alive[j]])
            dmin = drone_dist(pos[js] - pos[a])[0].min() if len(js) else F(np.inf)
            omin = obst_dist(b["obst"][e] - pos[a])[0].min()
            assert o2.collision[e, a] == ((dmin <= THR_PAIR) or (omin <= THR_OBST)), (name, e, a)
            assert o2.reached[e, a] == (drone_dist(b["goal"][e] - pos[a])[0] <= THR_GOAL), (name, e, a)
        if fam == "threshold":   # the planted compare really sits on the threshold
            hit = {"at": 1, "below": 1, "above": 0}[name.rsplit("_", 1)[1]]
            flag = o2.reached if name.startswith("goal") else o2.collision
            assert flag[e, i] == hit, (name, e)
    assert np.array_equal(o2.positions, b["pos"])    # zero velocity, zero action: nothing moved


# ---------------------------------------------------------------------------------------------- GPU half
KERNEL_RE = re.compile(r"(swarm_step_rotx?_kernel|swarm_env_kernel(?:_small)?)\b")
KNOBS = ("SWARM_B200_NO_ROT", "SWARM_B200_FUSED_RESET", "SWARM_B200_ROTX_MIN_ENVS", "SWARM_B200_MULTI_STEP_MAX_GROUPS")


@pytest.fixture(autouse=True)
def _wide_kernel_everywhere(monkeypatch):
    """Clear inherited SWARM_B200_* knobs and pin N = 64 / 128 to the wide rotation kernel at every batch size."""
    for k in list(os.environ):
        if k.startswith("SWARM_B200_") and k != "SWARM_B200_LIB":
            monkeypatch.delenv(k)
    monkeypatch.setenv("SWARM_B200_ROTX_MIN_ENVS", "0")


def kernels_run(fn):
    """Names of the step kernels that ran on the device during fn() (torch.profiler, CUDA activity)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for ev in prof.events():
        m = KERNEL_RE.search(ev.name)
        if m:
            names.add(m.group(1))
    return names


def _dr(dr):
    if dr is None:
        return None
    from test_domain_randomization import DR_DELAY, DR_V1
    return {"v1": DR_V1, "delay": DR_DELAY}[dr]


def run_and_compare(N, M, b, *, dr=None, mode="step", world=20.0, spacing=2.5, acts=None):
    """Inject the batch into an engine and the oracle, step both (zero actions unless given), compare every output
    bit for bit and return the step kernels that ran."""
    import torch
    import swarm_b200
    E = len(b["pos"])
    steps = 3 if mode == "many" else (1 if acts is None else len(acts))
    dr_cfg = _dr(dr)
    o, cfg = oracle_for(N, M, b, dr=dr_cfg, world=world, spacing=spacing, steps=steps, acts=acts)
    eng = swarm_b200.SwarmEngine(E, cfg, device="cuda:0", reward64=True,
                                 **(dict(domain_randomization=dr_cfg, dr_seed=7) if dr_cfg else {}))
    eng.seed(np.arange(E, dtype=np.uint64))
    eng.reset()
    eng.set_state(b["pos"], np.zeros_like(b["pos"]), b["goal"], b["obst"], alive=b["alive"], step_count=b["step_count"])
    a = torch.zeros((steps, E, N, 3), device="cuda:0") if acts is None else torch.from_numpy(np.stack(acts)).cuda()

    def go():
        if mode == "many":
            eng.step_many(a)
        else:
            for t in range(steps):
                eng.step(a[t])
    ran = kernels_run(go)
    got = lambda t: t.detach().cpu().numpy()  # noqa: E731
    for name, want in (("positions", o.positions), ("velocities", o.velocities), ("goal", o.goal),
                       ("obstacles", o.obstacles), ("step_count", o.step_count), ("reward64", o.reward),
                       ("dist", o.dist), ("terminated", o.terminated), ("truncated", o.truncated),
                       ("reached", o.reached), ("collision", o.collision), ("obs_valid", o.obs_valid),
                       ("all_terminated", o.all_terminated), ("all_truncated", o.all_truncated),
                       ("global_state", o.global_state), ("rng", o.rng.view(np.int64))):
        pu.assert_biteq(name, got(getattr(eng, name)), want, mode)
    pu.assert_biteq("alive", got(eng.alive).astype(np.uint8), o.active, mode)
    valid = o.obs_valid.astype(bool)
    pu.assert_biteq("obs", got(eng.obs)[valid], o.obs[valid], mode)
    if dr_cfg:
        pu.assert_biteq("dr_params", got(eng.dr_params), o.dr_params, mode)
        if eng.act_hist is not None:
            pu.assert_biteq("act_hist", got(eng.act_hist), o.act_hist, mode)
    return ran


ROT = {8: "swarm_step_rot_kernel", 16: "swarm_step_rot_kernel", 32: "swarm_step_rot_kernel",
       64: "swarm_step_rotx_kernel", 128: "swarm_step_rotx_kernel"}
GENERAL = {"swarm_env_kernel", "swarm_env_kernel_small"}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["step", "many", "fused"])
@pytest.mark.parametrize("dr", [None, "v1", "delay"])
@pytest.mark.parametrize("N,M", SHAPES)
def test_rotation_kernels_match_oracle_on_built_states(monkeypatch, N, M, dr, mode):
    """Every layout through the rotation kernel (N <= 32) or the wide kernel (N = 64 / 128): one step() (step and
    auto-reset launches), step_many over three steps (the fused instantiation), or step() with the reset fused."""
    if mode == "fused":
        monkeypatch.setenv("SWARM_B200_FUSED_RESET", "1")
    b, _ = batch(N, M, _sqkey(N, M))
    ran = run_and_compare(N, M, b, dr=dr, mode=mode)
    assert ROT[N] in ran and not ran & GENERAL, ran


@pytest.mark.gpu
@pytest.mark.parametrize("dr", [None, "v1", "delay"])
@pytest.mark.parametrize("N,M,no_rot", [(12, 4, False), (40, 8, False), (8, 12, True), (32, 8, True)])
def test_general_kernels_match_oracle_on_built_states(monkeypatch, N, M, no_rot, dr):
    """The same layouts through the general kernels: N = 12 / 40, and N = 8 / 32 with SWARM_B200_NO_ROT=1."""
    if no_rot:
        monkeypatch.setenv("SWARM_B200_NO_ROT", "1")
    b, _ = batch(N, M, _sqkey(N, M))
    ran = run_and_compare(N, M, b, dr=dr)
    assert ran and ran <= GENERAL, ran


# ---------------------------------------------------------------------------------------------- eligibility bounds
def corner_batch(N, M, world, E=8, seed=3):
    """Drones split between opposite corners inside the smallest wall (world * 0.95 / 2), so pair distances and
    formation terms reach their largest values; goal and obstacles near the centre."""
    rng = np.random.default_rng(seed)
    c = world * 0.95 / 2 - 1.0
    pos = np.zeros((E, N, 3), F)
    for e in range(E):
        for j in range(N):
            s = np.array([1.0, 1.0, 1.0]) if j % 2 == 0 else np.array([-1.0, -1.0, -1.0])
            if e % 2:
                s[j % 3] = -s[j % 3]
            pos[e, j] = s * (c - 1.5 * (j // 2) * np.array([1.0, 0.0, 0.0]) - rng.uniform(0, 1, 3))
    obst = rng.uniform(-5, 5, (E, M, 3)).astype(F)
    goal = rng.uniform(-5, 5, (E, 3)).astype(F)
    return dict(pos=pos, alive=np.ones((E, N), np.uint8), goal=goal, obst=obst, step_count=np.zeros(E, np.int32))


BOUNDS = [
    # N, world, desired_spacing, dr, inside the rotation kernels' bounds
    (32, 1023.5, 1023.75, None, True),
    (128, 255.5, 511.5, None, True),
    (32, 975.0, 2.5, "v1", True),        # world-scale maximum 1.05: 1023.75
    (32, 1024.0, 2.5, None, False),
    (128, 256.0, 2.5, None, False),
    (32, 976.0, 2.5, "v1", False),
    (32, 20.0, 0.1, None, False),        # not a multiple of 2^-37
    (128, 70.0, 0.1, None, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("N,world,spacing,dr,inside", BOUNDS)
def test_eligibility_bounds(N, world, spacing, dr, inside):
    """Configs at the edge of rot_eligible / rotx_eligible match the oracle bit for bit, and run on the rotation
    kernels exactly when they are inside the bounds."""
    M = 8
    b = corner_batch(N, M, world)
    rng = np.random.default_rng(4)
    acts = [np.zeros((len(b["pos"]), N, 3), F)] + [rng.uniform(-1, 1, (len(b["pos"]), N, 3)).astype(F) for _ in range(2)]
    ran = run_and_compare(N, M, b, dr=dr, world=world, spacing=spacing, acts=acts)
    if inside:
        assert ROT[N] in ran and not ran & GENERAL, ran
    else:
        assert ran and ran <= GENERAL, ran
