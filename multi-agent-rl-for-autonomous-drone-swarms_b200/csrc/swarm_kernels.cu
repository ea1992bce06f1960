// swarm_kernels.cu -- sm_100a kernels of the batched drone-swarm env step.
//
// One fused launch performs, for every env instance of the batch, the whole of
//   DroneSwarmEnv.step   (reference src/swarm_marl/envs/drone_swarm_env.py:92-174)
//   SingleDroneEnv.step  (reference src/swarm_marl/envs/single_drone_env.py:73-111)
// integrate -> wall clip -> goal distance -> obstacle / pairwise distances (collision,
// formation, k-nearest features) -> reward -> done flags -> observation rows -> global_state,
// and, when an episode ends with auto_reset, env.reset() (drone_swarm_env.py:65-90) from the
// env's own numpy-compatible PCG64 stream.
//
// Mapping.  Envs are independent, so the unit of work is a WARP: one warp owns G = 32/N env
// instances (N <= 32; lane = env-local index * N + drone) or one env with ceil(N/32) drones per
// lane (N > 32).  A warp keeps its envs' positions / velocities / goal / obstacles in a private
// shared-memory slice (float4 tables: every pair-loop read is one LDS.128), needs no block
// barrier, and transposes its 32 x D observation rows through shared memory so the global
// writes are contiguous float4 streams.  All state traffic is float4 (coalesced 16 B).
//
// Arithmetic is bit-faithful to the reference's numpy expressions: explicit round-to-nearest
// float32 ops with no FMA contraction (the TU is compiled with -fmad=false as well), float64
// accumulation where np.linalg.norm goes through BLAS sdot (SURVEY.md 3.4 T1), float64 reward
// arithmetic with numpy's 8-lane pairwise summation order for np.mean (T4), lowest-index tie
// break for the k-nearest selections (T5), parked drones as neighbours but not colliders (T6).
#include "swarm_internal.h"
#include "swarm_device.cuh"

namespace swarm {


// ------------------------------------------------------------------------------------------
// per-drone scan: obstacle distances + pairwise distances
// ------------------------------------------------------------------------------------------
struct ScanOut {
    bool obst_hit, pair_hit;
    double form_sum;  // np.add.reduce(|d - d*|) in numpy's pairwise order
    int form_n;
};


// Eight consecutive "other drones" jp = jb .. jb+7 of drone i (jp skips i: j = jp + (jp >= i)).
// FORM 0: k-nearest only; 1: r[u] += |d - d*| (numpy pairwise lane u); 2: res += ... in order.
template <int KT, int NORM, bool FULL, int FORM>
__device__ __forceinline__ void pair_block8(const float4* __restrict__ tpos, int jb, int n_others, int i, float px,
                                            float py, float pz, float (&nd)[KT], int (&nj)[KT], double (&r)[8],
                                            double& res, double d_star) {
    float s[8];
    bool valid[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int jp = jb + u;
        valid[u] = FULL || jp < n_others;
        const int j = valid[u] ? jp + (jp >= i ? 1 : 0) : i;
        const float4 q = tpos[j];
        const float ss = sumsq1d<NORM>(__fsub_rn(q.x, px), __fsub_rn(q.y, py), __fsub_rn(q.z, pz));
        s[u] = valid[u] ? ss : 1.0f;
    }
    const float smin = fminf(fminf(fminf(s[0], s[1]), fminf(s[2], s[3])), fminf(fminf(s[4], s[5]), fminf(s[6], s[7])));
    float d[8];
    if (smin >= SQRT_FAST_MIN) {
#pragma unroll
        for (int u = 0; u < 8; ++u) d[u] = sqrt_rn_fast(s[u]);
    } else {  // coincident drones (d == 0) or denormal range: full IEEE path
#pragma unroll
        for (int u = 0; u < 8; ++u) d[u] = __fsqrt_rn(s[u]);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        topk_insert<KT>(valid[u] ? d[u] : TOPK_EMPTY, jb + u, nd, nj);
        if (FORM != 0) {
            const double err = fabs(__dsub_rn((double)d[u], d_star));
            if (FORM == 1) r[u] = __dadd_rn(r[u], err);
            else res = __dadd_rn(res, valid[u] ? err : 0.0);
        }
    }
}

template <int ST, bool FULL>
__device__ __forceinline__ void obst_block4(const float4* __restrict__ tobs, int mb, int M, float px, float py, float pz,
                                            float (&od)[ST], int (&om)[ST]) {
    float s[4];
    bool valid[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        valid[u] = FULL || mb + u < M;
        const float4 o = tobs[valid[u] ? mb + u : 0];
        const float ss = sumsq_axis(__fsub_rn(o.x, px), __fsub_rn(o.y, py), __fsub_rn(o.z, pz));
        s[u] = valid[u] ? ss : 1.0f;
    }
    const float smin = fminf(fminf(s[0], s[1]), fminf(s[2], s[3]));
    float d[4];
    if (smin >= SQRT_FAST_MIN) {
#pragma unroll
        for (int u = 0; u < 4; ++u) d[u] = sqrt_rn_fast(s[u]);
    } else {
#pragma unroll
        for (int u = 0; u < 4; ++u) d[u] = __fsqrt_rn(s[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) topk_insert<ST>(valid[u] ? d[u] : TOPK_EMPTY, mb + u, od, om);
}

// KT / ST: capacity of the k-nearest lists (>= K, S).  nj holds "other" indices jp (see above).
template <int KT, int ST, int NORM, int KIND, bool STEP>
__device__ __forceinline__ void scan_drone(const DevParams& P, const float4* __restrict__ tpos,
                                           const float4* __restrict__ tobs, int i, float px, float py, float pz,
                                           bool alive_i, int n_alive_env, float (&nd)[KT], int (&nj)[KT],
                                           float (&od)[ST], int (&om)[ST], ScanOut& out) {
    const int N = P.N, M = P.M;
#pragma unroll
    for (int q = 0; q < KT; ++q) { nd[q] = TOPK_EMPTY; nj[q] = -1; }
#pragma unroll
    for (int q = 0; q < ST; ++q) { od[q] = TOPK_EMPTY; om[q] = -1; }
    out.pair_hit = false;
    out.form_sum = 0.0;
    out.form_n = 0;

    // ---- obstacles: _nearest_obstacle_features (:273-291) + obstacle part of _collision_mask (:190-200)
    {
        int mb = 0;
        for (; mb + 4 <= M; mb += 4) obst_block4<ST, true>(tobs, mb, M, px, py, pz, od, om);
        if (mb < M) obst_block4<ST, false>(tobs, mb, M, px, py, pz, od, om);
    }
    out.obst_hit = od[0] <= P.thr_obst;  // nearest obstacle decides; TOPK_EMPTY (a NaN) when M == 0
    if (KIND == SWARM_KIND_SINGLE) return;

    // ---- drones: _nearest_neighbor_features (:245-271) over ALL j != i; pair part of
    //      _collision_mask (:202-207) and _formation_penalties (:210-224) over ACTIVE pairs
    const int n_others = N - 1;
    double r[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) r[u] = 0.0;
    double res = 0.0;

    if (!STEP) {
        int jb = 0;
        for (; jb + 8 <= n_others; jb += 8)
            pair_block8<KT, NORM, true, 0>(tpos, jb, n_others, i, px, py, pz, nd, nj, r, res, 0.0);
        if (jb < n_others) pair_block8<KT, NORM, false, 0>(tpos, jb, n_others, i, px, py, pz, nd, nj, r, res, 0.0);
        return;
    }

    if (alive_i && n_alive_env == N) {
        // fast path: every drone active -> the jp-th other drone is element jp of the mean's operand,
        // so numpy's pairwise-sum lane is static under 8x unrolling
        const double d_star = P.d_star;
        const int n8 = n_others >= 8 ? (n_others & ~7) : 0;
        for (int jb = 0; jb < n8; jb += 8)
            pair_block8<KT, NORM, true, 1>(tpos, jb, n_others, i, px, py, pz, nd, nj, r, res, d_star);
        if (n8 > 0) res = tree8(r);
        if (n8 < n_others) pair_block8<KT, NORM, false, 2>(tpos, n8, n_others, i, px, py, pz, nd, nj, r, res, d_star);
        out.pair_hit = nd[0] <= P.thr_pair;  // nearest drone decides (all drones active here)
        out.form_sum = res;
        out.form_n = n_others;
        return;
    }

    // general path: some drones are parked (or this one is) -> compact on the fly
    const int n_f = alive_i ? n_alive_env - 1 : 0;
    const int n8 = n_f >= 8 ? (n_f & ~7) : 0;
    bool tree_done = false;
    int cnt = 0;
    for (int jp = 0; jp < n_others; ++jp) {
        const int j = jp + (jp >= i ? 1 : 0);
        const float4 q = tpos[j];
        const float d = norm1d<NORM>(__fsub_rn(q.x, px), __fsub_rn(q.y, py), __fsub_rn(q.z, pz));
        topk_insert<KT>(d, jp, nd, nj);
        if (alive_i && q.w != 0.0f) {
            out.pair_hit |= d <= P.thr_pair;
            const double err = fabs(__dsub_rn((double)d, P.d_star));
            if (cnt < n8) {
                const int lane8 = cnt & 7;
#pragma unroll
                for (int u = 0; u < 8; ++u) r[u] = __dadd_rn(r[u], lane8 == u ? err : 0.0);
            } else {
                if (!tree_done && n8 > 0) res = tree8(r);
                tree_done = true;
                res = __dadd_rn(res, err);
            }
            ++cnt;
        }
    }
    if (!tree_done && n8 > 0) res = tree8(r);
    out.form_sum = res;
    out.form_n = n_f;
}

// observation row -> this lane's row of the staging tile:  _build_obs (:226-243)
template <int KT, int ST, bool EXACT, int KIND>
__device__ __forceinline__ void stage_obs_row(const DevParams& P, float* __restrict__ row,
                                              const float4* __restrict__ tpos, const float4* __restrict__ tobs, int i,
                                              float px, float py, float pz, float vx, float vy, float vz, float gx,
                                              float gy, float gz, const float (&nd)[KT], const int (&nj)[KT],
                                              const float (&od)[ST], const int (&om)[ST]) {
    const int K = EXACT ? KT : P.K, S = EXACT ? ST : P.S;
    row[0] = px; row[1] = py; row[2] = pz;
    row[3] = vx; row[4] = vy; row[5] = vz;
    row[6] = __fsub_rn(gx, px); row[7] = __fsub_rn(gy, py); row[8] = __fsub_rn(gz, pz);
    int off = 9;
    if (KIND != SWARM_KIND_SINGLE) {
#pragma unroll
        for (int q = 0; q < KT; ++q) {
            if (q < K) {
                float rx = 0.f, ry = 0.f, rz = 0.f, d = 0.f;
                if (nj[q] >= 0) {
                    const float4 t = tpos[nj[q] + (nj[q] >= i ? 1 : 0)];
                    rx = __fsub_rn(t.x, px); ry = __fsub_rn(t.y, py); rz = __fsub_rn(t.z, pz);
                    d = nd[q];
                }
                row[off + 4 * q + 0] = rx; row[off + 4 * q + 1] = ry;
                row[off + 4 * q + 2] = rz; row[off + 4 * q + 3] = d;
            }
        }
        off += 4 * K;
    }
#pragma unroll
    for (int q = 0; q < ST; ++q) {
        if (q < S) {
            float rx = 0.f, ry = 0.f, rz = 0.f, d = 0.f;
            if (om[q] >= 0) {
                const float4 t = tobs[om[q]];
                rx = __fsub_rn(t.x, px); ry = __fsub_rn(t.y, py); rz = __fsub_rn(t.z, pz);
                d = od[q];
            }
            row[off + 4 * q + 0] = rx; row[off + 4 * q + 1] = ry;
            row[off + 4 * q + 2] = rz; row[off + 4 * q + 3] = d;
        }
    }
}

// staged rows -> obs[base_agent .. base_agent + n_rows) as one contiguous stream
__device__ __forceinline__ void flush_stage(float* __restrict__ obs, int D, const float* __restrict__ stage,
                                            long long base_agent, int n_rows, int lane) {
    const int total = n_rows * D;
    float* dst = obs + base_agent * D;
    if (((base_agent & 3) == 0) && ((total & 3) == 0)) {  // D = 1 (mod 4): 16-byte aligned iff base % 4 == 0
        const float4* s4 = reinterpret_cast<const float4*>(stage);
        float4* d4 = reinterpret_cast<float4*>(dst);
        for (int idx = lane; idx < (total >> 2); idx += 32) __stcs(d4 + idx, s4[idx]);
    } else {
        for (int idx = lane; idx < total; idx += 32) __stcs(dst + idx, stage[idx]);
    }
}

// global_state row pieces of one drone: [pos.ravel | vel.ravel | goal] (:293-302)
__device__ __forceinline__ void write_gs_drone(float* __restrict__ row, int N, int i, float px, float py, float pz,
                                               float vx, float vy, float vz) {
    __stcs(row + 3 * i + 0, px); __stcs(row + 3 * i + 1, py); __stcs(row + 3 * i + 2, pz);
    __stcs(row + 3 * N + 3 * i + 0, vx); __stcs(row + 3 * N + 3 * i + 1, vy); __stcs(row + 3 * N + 3 * i + 2, vz);
}

// domain randomisation, sensor noise of one staged observation row (DESIGN.md 8): own position / velocity and the
// sensed obstacle distances get x + sigma z from the Philox block of (env, episode key, step_count of the observed
// state - 1, drone) -- the block the thrust noise of the step that produced the state was cut from
template <int KT, int ST, bool EXACT, int KIND>
__device__ __forceinline__ void add_sensor_noise(const DevParams& P, float* __restrict__ row, unsigned genv,
                                                 unsigned ekey, int sc_obs, int i, const int (&om)[ST]) {
    const int K = EXACT ? KT : P.K, S = EXACT ? ST : P.S;
    const uint4 rA = philox4x32_7(genv, ekey, (unsigned)(sc_obs - 1), (unsigned)i | (DR_STREAM_A << 16), P);
    uint4 rB = rA;
    if (S > 4) rB = philox4x32_7(genv, ekey, (unsigned)(sc_obs - 1), (unsigned)i | (DR_STREAM_B << 16), P);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        row[c] = __fmaf_rn(P.dr_std_pos, dr_normal(P.dr_qtable, dr_field(rA, 3 + c)), row[c]);
        row[3 + c] = __fmaf_rn(P.dr_std_vel, dr_normal(P.dr_qtable, dr_field(rA, 6 + c)), row[3 + c]);
    }
    const int off = 9 + (KIND != SWARM_KIND_SINGLE ? 4 * K : 0);
#pragma unroll
    for (int q = 0; q < ST; ++q)
        if (q < S && om[q] >= 0) {
            const unsigned f = q < 4 ? dr_field(rA, 9 + (q < 4 ? q : 0)) : dr_field(rB, q >= 4 ? q - 4 : 0);
            row[off + 4 * q + 3] = __fmaf_rn(P.dr_std_obst, dr_normal(P.dr_qtable, f), row[off + 4 * q + 3]);
        }
}

// ------------------------------------------------------------------------------------------
// the env kernel (step / reset / observe)
//   KT, ST  capacity of the k-nearest lists; EXACT: K == KT and S == ST (D is compile-time)
//   SMALLN  N <= 32: one drone per lane, drone state stays in registers between the phases
// ------------------------------------------------------------------------------------------
template <int KT, int ST, bool EXACT, int NORM, int KIND, bool SMALLN, bool DR>
__global__ void __launch_bounds__(kThreadsPerCta, kMinBlocksPerSm) swarm_env_kernel(const DevParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    unsigned char* wb = smem_raw + (size_t)warp * P.smem_per_warp;
    float4* tab_pos = reinterpret_cast<float4*>(wb);
    float4* tab_vel = tab_pos + P.n_tab;
    float4* tab_goal = tab_vel + P.n_tab;
    float4* tab_obst = tab_goal + P.G;
    float* stage = reinterpret_cast<float*>(tab_obst + P.G * P.m_pad);

    const int N = P.N, M = P.M, G = P.G;
    constexpr bool PHYS = KIND == SWARM_KIND_PHYSICS;   // DronePhysicsEnv as a point mass, above 32 drones (DESIGN.md 9)
    const int D = EXACT ? (KIND != SWARM_KIND_SINGLE ? 9 + 4 * KT + 4 * ST : 9 + 4 * ST) : P.D;
    const int nslots = SMALLN ? 1 : P.nslots;
    const int e_l = SMALLN ? lane / N : 0;  // env-local index of this lane
    const int i_base = SMALLN ? lane - e_l * N : lane;
    const unsigned env_lanes =
        SMALLN ? (e_l < G ? (N == 32 ? FULL_MASK : (((1u << N) - 1u) << (e_l * N))) : 0u) : FULL_MASK;

    // per-lane statistics (flushed once per warp at the end)
    unsigned st_eps = 0, st_succ = 0, st_col = 0, st_to = 0, st_len = 0, st_asteps = 0, st_esteps = 0, st_nan = 0;
    double st_ret = 0.0;

    asm volatile("griddepcontrol.wait;" ::: "memory");  // programmatic dependent launch: the previous launch is done
    // dynamic group queue (the first group of every warp is static): with only a few groups per warp a
    // static grid stride leaves most SMs idle during the last round
    const int warps_total = gridDim.x * kWarpsPerCta;
    int grp = blockIdx.x * kWarpsPerCta + warp;
    while (grp < P.n_groups) {
        int grp_next = 0;
        if (lane == 0) grp_next = (int)atomicAdd(P.work_counter, 1u);   // raw; + warps_total behind the shuffle
        const int env0 = P.env_begin + grp * G;
        const int n_env = min(G, P.env_begin + P.env_count - env0);
        const bool lane_env_ok = e_l < n_env;
        const int env = env0 + (lane_env_ok ? e_l : 0);
        const float4* tpos = tab_pos + e_l * N;  // this lane's env tables
        const float4* tobs = tab_obst + e_l * P.m_pad;
        float* gs_row = P.gs ? P.gs + (long long)env * P.R : nullptr;

        __syncwarp();  // previous group's shared-memory reads are done
        // ---- per-env tables: goal, obstacles
        if (lane < n_env) tab_goal[lane] = P.goal4[env0 + lane];
        for (int idx = lane; idx < n_env * M; idx += 32) {
            const int el = idx / M, m = idx - el * M;
            tab_obst[el * P.m_pad + m] = P.obst4[(long long)(env0 + el) * M + m];
        }
        float4 g4 = lane_env_ok ? P.goal4[env] : make_float4(0.f, 0.f, 0.f, 0.f);
        float gx = g4.x, gy = g4.y, gz = g4.z;
        const int sc = lane_env_ok ? P.step_count[env] : 0;
        // per-env dynamics constants: the config's, or this episode's randomised ones (DESIGN.md 8)
        float c_amax = P.amax, c_vmax = P.vmax, c_dt = P.dt, c_bound = P.bound, c_thr_obst = P.thr_obst;
        unsigned ekey = 0u;
        int ctrl_delay = 0;
        if (DR && lane_env_ok) {
            const float4 d0 = P.dr_params[(long long)env * 2 + 0], d1 = P.dr_params[(long long)env * 2 + 1];
            c_amax = d0.x; c_vmax = d0.y; c_dt = d0.z; c_bound = d0.w;
            c_thr_obst = d1.x; ekey = __float_as_uint(d1.y);
            ctrl_delay = (int)d1.w;
        }
        const unsigned genv = DR ? (unsigned)(P.env_index_base + env) : 0u;

        unsigned reset_envs = 0;  // bit el: env el of this group is (re)drawn in this launch

        if (P.mode == kModeStep) {
            // =========================== phase A: integrate (:98-118) ===========================
            int n_alive_env = 0;
            float4 p_reg = make_float4(0.f, 0.f, 0.f, 0.f), v_reg = p_reg;  // SMALLN: this lane's drone
            for (int slot = 0; slot < nslots; ++slot) {
                const int i = slot * 32 + i_base;
                const bool ok = lane_env_ok && i < N;
                bool alive = false;
                if (ok) {
                    const long long a = (long long)env * N + i;
                    float4 p = P.pos4[a];
                    float4 v = P.vel4[a];
                    alive = KIND == SWARM_KIND_SINGLE ? true : (p.w != 0.0f);
                    // prev distance (:98-101)
                    const float prev_d = norm1d<NORM>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));
                    if (alive) {
                        float ax = P.actions[a * 3 + 0], ay = P.actions[a * 3 + 1], az = P.actions[a * 3 + 2];
                        const bool clip_cmd = !PHYS;   // (the physics env neither clips nor casts the action, :336)
                        if (DR && P.dr_delay_hist > 0) delayed_command(P, env, N, i, sc, ctrl_delay, ax, ay, az);
                        if (clip_cmd) { ax = clipf(ax, -1.0f, 1.0f); ay = clipf(ay, -1.0f, 1.0f); az = clipf(az, -1.0f, 1.0f); }
                        if (!(ax == ax && ay == ay && az == az)) ++st_nan;   // NaN-action guard counter
                        if (DR) {
                            const uint4 r = philox4x32_7(genv, ekey, (unsigned)sc, (unsigned)i | (DR_STREAM_A << 16), P);
                            thrust_noise(P, [=](int f) { return dr_normal(P.dr_qtable, dr_field(r, f)); }, ax, ay, az);
                        }
                        if (PHYS) physics_substeps<NORM>(P, ax, ay, az, c_amax, c_vmax, DR ? c_dt : P.phys_h, p, v);
                        else point_mass_step<NORM>(P, ax, ay, az, c_amax, c_vmax, c_dt, p.x, p.y, p.z, v.x, v.y, v.z);
                    }
                    // wall clip for ALL drones (:113-117); velocity is not zeroed at the wall (the physics env has no walls)
                    if (!PHYS) {
                        p.x = clipf(p.x, -c_bound, c_bound);
                        p.y = clipf(p.y, -c_bound, c_bound);
                        p.z = clipf(p.z, -c_bound, c_bound);
                    }
                    p.w = alive ? 1.0f : 0.0f;
                    if (!PHYS) v.w = prev_d;   // (physics: .w keeps the drone's damping factor; its reward has no progress term)
                    tab_pos[e_l * N + i] = p;
                    if (SMALLN) { p_reg = p; v_reg = v; }
                    else tab_vel[e_l * N + i] = v;
                }
                n_alive_env += __popc(__ballot_sync(FULL_MASK, ok && alive) & env_lanes);
            }
            __syncwarp();

            // ================ phase B: distances, reward, obs rows (:120-162) ================
            unsigned m_alive = 0, m_done = 0;  // bit = slot
            float rew_sum = 0.0f;
            bool any_col = false;
            int n_cont = 0, n_open = 0;   // n_open (physics): active drones neither at the goal nor in contact
            for (int slot = 0; slot < nslots; ++slot) {
                const int i = slot * 32 + i_base;
                const bool ok = lane_env_ok && i < N;
                bool alive = false, reached = false, collided = false;
                float rew32 = 0.0f;
                if (ok) {
                    const float4 p = SMALLN ? p_reg : tpos[i];
                    const float4 v = SMALLN ? v_reg : tab_vel[e_l * N + i];
                    alive = p.w != 0.0f;
                    const float curr_d = norm1d<NORM>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));
                    float nd[KT]; int nj[KT]; float od[ST]; int om[ST];
                    ScanOut so;
                    scan_drone<KT, ST, NORM, KIND, true>(P, tpos, tobs, i, p.x, p.y, p.z, alive, n_alive_env, nd, nj,
                                                         od, om, so);
                    // physics env: reached = dist < goal_radius (strict, drone_physics_env.py:389); contact with the
                    // ground plane, an obstacle sphere or another drone (:368-372, point-mass radii set by the host)
                    reached = PHYS ? (alive && (double)curr_d < P.goal_radius_d)
                                   : (alive && curr_d <= P.thr_goal);   // :124-127 (double compare)
                    if (DR) so.obst_hit = od[0] <= c_thr_obst;         // this episode's obstacle radius
                    collided = alive && (so.obst_hit || so.pair_hit || (PHYS && p.z <= P.phys_ground_z));   // :128
                    double reward = 0.0;
                    if (PHYS) {
                        if (alive) {  // drone_physics_env.py:378-392
                            reward = __dmul_rn(-(double)curr_d, 0.1);
                            if (collided) reward = __dsub_rn(reward, 10.0);
                            else if (reached) reward = __dadd_rn(reward, 50.0);
                        }
                    } else if (alive) {
                        const double progress = __dmul_rn(__dsub_rn((double)v.w, (double)curr_d), P.k_p);  // :142
                        if (KIND == SWARM_KIND_SWARM) {
                            double pen = 0.0;  // :210-224
                            if (so.form_n > 0) pen = __dmul_rn(P.neg_k_f, __ddiv_rn(so.form_sum, (double)so.form_n));
                            reward = __dadd_rn(progress, pen);  // :143
                        } else {
                            reward = progress;
                        }
                        if (reached) reward = __dadd_rn(reward, P.r_goal);   // :144-145
                        if (collided) reward = __dadd_rn(reward, P.r_col);   // :146-147
                    }
                    rew32 = __double2float_rn(reward);
                    const long long a = (long long)env * N + i;
                    P.reward[a] = rew32;
                    if (P.reward64) P.reward64[a] = reward;
                    P.dist[a] = curr_d;
                    P.reached[a] = reached ? 1 : 0;
                    P.collision[a] = collided ? 1 : 0;
                    float ovx = v.x, ovy = v.y, ovz = v.z;
                    if (PHYS) {  // drone_physics_env.py:436-439: the observed velocity is clamped to max_speed
                        const float speed = norm1d<NORM>(v.x, v.y, v.z);
                        if (speed > c_vmax) {
                            ovx = __fmul_rn(__fdiv_rn(v.x, speed), c_vmax);
                            ovy = __fmul_rn(__fdiv_rn(v.y, speed), c_vmax);
                            ovz = __fmul_rn(__fdiv_rn(v.z, speed), c_vmax);
                        }
                    }
                    stage_obs_row<KT, ST, EXACT, KIND>(P, stage + lane * D, tpos, tobs, i, p.x, p.y, p.z, ovx, ovy,
                                                       ovz, gx, gy, gz, nd, nj, od, om);
                    if (DR) add_sensor_noise<KT, ST, EXACT, KIND>(P, stage + lane * D, genv, ekey, sc + 1, i, om);
                }
                __syncwarp();
                {
                    const int n_rows = SMALLN ? n_env * N : min(32, N - slot * 32);
                    const long long base = (long long)env0 * N + slot * 32;
                    flush_stage(P.obs, D, stage, base, n_rows, lane);
                }
                if (!SMALLN) __syncwarp();
                const bool done_agent = reached || collided;
                m_alive |= (alive ? 1u : 0u) << slot;
                m_done |= (done_agent ? 1u : 0u) << slot;
                any_col |= (__ballot_sync(FULL_MASK, collided) & env_lanes) != 0;
                n_cont += __popc(__ballot_sync(FULL_MASK, alive && !done_agent) & env_lanes);
                if (PHYS) n_open += __popc(__ballot_sync(FULL_MASK, alive && !collided && !reached) & env_lanes);
                // deterministic per-env reward sum (segmented tree over the env's lanes)
                float x = rew32;
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const float t = __shfl_down_sync(FULL_MASK, x, off);
                    if (SMALLN ? (i_base + off < N) : true) x = __fadd_rn(x, t);
                }
                rew_sum = __fadd_rn(rew_sum, x);  // meaningful on the env's first lane
            }

            // ====================== env-level flags (:137-138, :164-172) ======================
            const bool env_active = KIND == SWARM_KIND_SINGLE ? true : n_alive_env > 0;
            const int sc_new = env_active ? sc + 1 : sc;
            const bool time_limit = env_active && sc_new >= P.max_steps;
            bool all_term, all_trunc, ep_over;
            if (PHYS) {  // drone_physics_env.py:397-417: one flag pair for every drone
                const bool all_goals = n_open == 0;
                all_trunc = env_active && time_limit && !any_col && !all_goals;
                all_term = env_active ? (any_col || all_goals) : true;
                ep_over = env_active && (any_col || all_goals || time_limit);
                if (lane_env_ok && i_base == 0 && ep_over) {
                    st_eps++; st_succ += (all_goals && !any_col) ? 1 : 0; st_col += any_col ? 1 : 0; st_to += all_trunc ? 1 : 0;
                }
            } else if (KIND == SWARM_KIND_SWARM) {
                const bool all_reached = n_cont == 0 && !any_col && !time_limit;
                const bool episode_done = all_reached || any_col;
                all_term = env_active ? episode_done : true;  // :94-95 when no agent is left
                all_trunc = env_active ? (time_limit && !episode_done) : false;
                ep_over = env_active && (all_term || all_trunc);
                if (lane_env_ok && i_base == 0 && ep_over) {
                    st_eps++; st_succ += all_reached ? 1 : 0; st_col += any_col ? 1 : 0; st_to += all_trunc ? 1 : 0;
                }
            } else {
                all_term = (m_done & 1u) != 0;   // single env: terminated (:102)
                all_trunc = time_limit;          // truncated, not masked by terminated (:103)
                ep_over = all_term || all_trunc;
                if (lane_env_ok && ep_over) {
                    st_eps++; st_to += (all_trunc && !all_term) ? 1 : 0;
                }
            }
            const bool need_reset = P.auto_reset && (ep_over || !env_active);
            const bool cont_ok = !time_limit && !any_col;
            for (int slot = 0; slot < nslots; ++slot) {
                const int i = slot * 32 + i_base;
                if (!(lane_env_ok && i < N)) continue;
                const bool alive = (m_alive >> slot) & 1u, done_agent = (m_done >> slot) & 1u;
                const long long a = (long long)env * N + i;
                bool valid, alive_next;
                if (PHYS) {
                    P.terminated[a] = (alive && ep_over && !all_trunc) ? 1 : 0;
                    P.truncated[a] = (alive && ep_over && all_trunc) ? 1 : 0;
                    valid = alive;              // every drone is observed on every step
                    alive_next = alive && !ep_over;
                } else if (KIND == SWARM_KIND_SWARM) {
                    P.terminated[a] = (alive && done_agent) ? 1 : 0;                 // :150-151
                    P.truncated[a] = (alive && time_limit && !done_agent) ? 1 : 0;   // :152
                    valid = alive && !done_agent && cont_ok;                         // :154
                    alive_next = ep_over ? false : valid;                            // :169-172
                } else {
                    P.terminated[a] = all_term ? 1 : 0;
                    P.truncated[a] = all_trunc ? 1 : 0;
                    valid = true;
                    alive_next = true;
                }
                if (!need_reset) {  // (a reset env rewrites all of this in the observe pass)
                    P.obs_valid[a] = valid ? 1 : 0;
                    float4 p = SMALLN ? p_reg : tab_pos[e_l * N + i];
                    float4 v = SMALLN ? v_reg : tab_vel[e_l * N + i];
                    p.w = alive_next ? 1.0f : 0.0f;
                    if (!PHYS) v.w = 0.0f;   // (physics: the damping factor stays in .w)
                    P.pos4[a] = p;
                    P.vel4[a] = v;
                    if (gs_row) write_gs_drone(gs_row, N, i, p.x, p.y, p.z, v.x, v.y, v.z);
                }
            }
            if (lane_env_ok && i_base == 0) {
                st_esteps += env_active ? 1 : 0;
                st_asteps += n_alive_env;
                P.all_term[env] = all_term ? 1 : 0;
                P.all_trunc[env] = all_trunc ? 1 : 0;
                const float ret = __fadd_rn(P.ep_return[env], rew_sum);
                if (ep_over) { st_len += sc_new; st_ret += (double)ret; }
                if (P.episode_return) P.episode_return[env] = ep_over ? ret : 0.0f;
                if (P.episode_length) P.episode_length[env] = ep_over ? sc_new : 0;
                if (!need_reset) {
                    P.step_count[env] = sc_new;
                    P.ep_return[env] = ep_over ? 0.0f : ret;
                    if (gs_row) { __stcs(gs_row + 6 * N + 0, gx); __stcs(gs_row + 6 * N + 1, gy); __stcs(gs_row + 6 * N + 2, gz); }
                }
            }
            reset_envs = __ballot_sync(FULL_MASK, lane_env_ok && i_base == 0 && need_reset);
            if (SMALLN) {  // leader lane of env-local index el is el * N -> one bit per env
                unsigned packed = 0;
                for (int el = 0; el < n_env; ++el) packed |= ((reset_envs >> (el * N)) & 1u) << el;
                reset_envs = packed;
            } else {
                reset_envs = reset_envs & 1u;
            }
        } else {
            // ============ reset / observe: tables straight from the state buffers ============
            for (int slot = 0; slot < nslots; ++slot) {
                const int i = slot * 32 + i_base;
                if (lane_env_ok && i < N) {
                    const long long a = (long long)env * N + i;
                    tab_pos[e_l * N + i] = P.pos4[a];
                    tab_vel[e_l * N + i] = P.vel4[a];
                }
            }
            if (P.mode == kModeReset) {
                const bool want = lane < n_env && (P.env_mask == nullptr || P.env_mask[env0 + lane] != 0);
                reset_envs = __ballot_sync(FULL_MASK, want);
            }
        }
        __syncwarp();

        // ================================ reset (:65-80) ================================
        if (reset_envs) {
            for (int el = 0; el < n_env; ++el) {
                if (!((reset_envs >> el) & 1u)) continue;
                const int renv = env0 + el;
                const Pcg64State rng = load_rng(P, renv);
                double u_lo = P.rng_lo, u_range = P.rng_range;
                if (DR) {
                    const EpisodeDraw ep = draw_episode_constants(P, (unsigned)(P.env_index_base + renv), rng.sl);
                    u_lo = ep.u_lo(); u_range = ep.u_range();
                    float4 d0, d1;
                    episode_params(P, ep, d0, d1);
                    if (lane == 0) {
                        P.dr_params[(long long)renv * 2 + 0] = d0;
                        P.dr_params[(long long)renv * 2 + 1] = d1;
                    }
                    if (lane_env_ok && e_l == el) {
                        ekey = ep.key;
                        c_vmax = d0.y;   // (physics: the observed velocity is clamped to this episode's max_speed)
                    }
                }
                auto pos = [=](int j) { return reinterpret_cast<float*>(tab_pos + el * N + j); };
                auto goal = [=]() { return reinterpret_cast<float*>(tab_goal + el); };
                auto obst = [=](int m) { return reinterpret_cast<float*>(tab_obst + el * P.m_pad + m); };
                if (PHYS)
                    reset_env_physics_draws<1>(P, lane, N, M, rng, u_lo, u_range, pos,
                                               [=](int j) { return reinterpret_cast<float*>(tab_vel + el * N + j); }, goal, obst);
                else
                    reset_env_draws<1>(P, lane, N, rng, u_lo, u_range, pos, goal, obst);
                for (int k = lane; k < N; k += 32) {
                    reinterpret_cast<float*>(tab_pos + el * N + k)[3] = 1.0f;
                    float* tv = reinterpret_cast<float*>(tab_vel + el * N + k);
                    tv[0] = 0.f; tv[1] = 0.f; tv[2] = 0.f;
                    if (!PHYS) tv[3] = 0.f;  // (physics: .w holds this drone's new damping factor)
                }
                if (lane == 0) {
                    reset_env_finish(P, renv, rng);
                    reinterpret_cast<float*>(tab_goal + el)[3] = 0.0f;
                }
                for (int k = lane; k < M; k += 32) reinterpret_cast<float*>(tab_obst + el * P.m_pad + k)[3] = 0.0f;
            }
            __syncwarp();
            // new goal / obstacles back to the state buffers
            if (lane < n_env && ((reset_envs >> lane) & 1u)) P.goal4[env0 + lane] = tab_goal[lane];
            for (int idx = lane; idx < n_env * M; idx += 32) {
                const int el = idx / M, m = idx - el * M;
                if ((reset_envs >> el) & 1u) P.obst4[(long long)(env0 + el) * M + m] = tab_obst[el * P.m_pad + m];
            }
            if (lane_env_ok) { g4 = tab_goal[e_l]; gx = g4.x; gy = g4.y; gz = g4.z; }
        }

        // =========== observe pass: reset()'s obs / infos (:82-89), or swarm_observe ===========
        const unsigned observe_envs = P.mode == kModeObserve ? FULL_MASK : reset_envs;
        if (observe_envs) {
            const bool mine = lane_env_ok && ((observe_envs >> e_l) & 1u);
            const bool fresh = lane_env_ok && ((reset_envs >> e_l) & 1u);
            for (int slot = 0; slot < nslots; ++slot) {
                const int i = slot * 32 + i_base;
                const bool ok = mine && i < N;
                if (ok) {
                    const float4 p = tpos[i];
                    const float4 v = tab_vel[e_l * N + i];
                    float nd[KT]; int nj[KT]; float od[ST]; int om[ST];
                    ScanOut so;
                    scan_drone<KT, ST, NORM, KIND, false>(P, tpos, tobs, i, p.x, p.y, p.z, true, N, nd, nj, od, om, so);
                    const long long a = (long long)env * N + i;
                    P.dist[a] = norm1d<NORM>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));
                    // (the physics env observes every drone, always: drone_physics_env.py:421-462)
                    P.obs_valid[a] = KIND != SWARM_KIND_SWARM ? 1 : (p.w != 0.0f ? 1 : 0);
                    if (fresh) {
                        P.pos4[a] = p;
                        P.vel4[a] = make_float4(v.x, v.y, v.z, PHYS ? v.w : 0.0f);
                    }
                    if (P.mode != kModeStep) {
                        P.reward[a] = 0.0f;
                        if (P.reward64) P.reward64[a] = 0.0;
                        P.terminated[a] = 0; P.truncated[a] = 0; P.reached[a] = 0; P.collision[a] = 0;
                    }
                    if (gs_row) write_gs_drone(gs_row, N, i, p.x, p.y, p.z, v.x, v.y, v.z);
                    float ovx = v.x, ovy = v.y, ovz = v.z;
                    if (PHYS) {  // the observed velocity is clamped to max_speed (:436-439)
                        const float speed = norm1d<NORM>(v.x, v.y, v.z);
                        if (speed > c_vmax) {
                            ovx = __fmul_rn(__fdiv_rn(v.x, speed), c_vmax);
                            ovy = __fmul_rn(__fdiv_rn(v.y, speed), c_vmax);
                            ovz = __fmul_rn(__fdiv_rn(v.z, speed), c_vmax);
                        }
                    }
                    stage_obs_row<KT, ST, EXACT, KIND>(P, stage + lane * D, tpos, tobs, i, p.x, p.y, p.z, ovx, ovy, ovz,
                                                       gx, gy, gz, nd, nj, od, om);
                    // (a re-drawn env is observed at step_count 0, swarm_observe at the env's current step_count)
                    if (DR) add_sensor_noise<KT, ST, EXACT, KIND>(P, stage + lane * D, genv, ekey, fresh ? 0 : sc, i, om);
                }
                if (mine && i_base == 0 && slot == 0 && gs_row) {
                    __stcs(gs_row + 6 * N + 0, gx); __stcs(gs_row + 6 * N + 1, gy); __stcs(gs_row + 6 * N + 2, gz);
                }
                __syncwarp();
                // single-slot groups restage only the observed envs' rows; the other rows of the tile
                // still hold this step's rows, so the whole tile can be flushed again.  In reset mode
                // with a partial mask those other rows are stale -> flush per env there.
                if (SMALLN) {
                    if (P.mode == kModeStep || observe_envs == FULL_MASK ||
                        (reset_envs & ((1u << n_env) - 1u)) == ((1u << n_env) - 1u)) {
                        flush_stage(P.obs, D, stage, (long long)env0 * N, n_env * N, lane);
                    } else {
                        for (int el = 0; el < n_env; ++el)
                            if ((observe_envs >> el) & 1u)
                                flush_stage(P.obs, D, stage + el * N * D, (long long)(env0 + el) * N, N, lane);
                    }
                } else if (mine) {
                    flush_stage(P.obs, D, stage, (long long)env0 * N + slot * 32, min(32, N - slot * 32), lane);
                }
                if (!SMALLN) __syncwarp();
            }
            if (P.mode != kModeStep && lane < n_env && ((observe_envs >> lane) & 1u)) {
                P.all_term[env0 + lane] = 0;
                P.all_trunc[env0 + lane] = 0;
                if (P.episode_return) P.episode_return[env0 + lane] = 0.0f;
                if (P.episode_length) P.episode_length[env0 + lane] = 0;
            }
        }
        grp = warps_total + __shfl_sync(FULL_MASK, grp_next, 0);
    }
    // the last warp to leave re-arms the queue for the next launch
    if (lane == 0 && atomicAdd(P.work_counter + 1, 1u) == (unsigned)warps_total - 1u) {
        P.work_counter[0] = 0u;
        P.work_counter[1] = 0u;
    }

    // ---- statistics: one atomic per warp per counter
    if (P.stats && P.mode == kModeStep) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            st_eps += __shfl_xor_sync(FULL_MASK, st_eps, off);
            st_succ += __shfl_xor_sync(FULL_MASK, st_succ, off);
            st_col += __shfl_xor_sync(FULL_MASK, st_col, off);
            st_to += __shfl_xor_sync(FULL_MASK, st_to, off);
            st_len += __shfl_xor_sync(FULL_MASK, st_len, off);
            st_asteps += __shfl_xor_sync(FULL_MASK, st_asteps, off);
            st_esteps += __shfl_xor_sync(FULL_MASK, st_esteps, off);
            st_ret += __shfl_xor_sync(FULL_MASK, st_ret, off);
        }
        if (lane == 0) {
            if (st_eps) {
                atomicAdd(P.stats + SWARM_STAT_EPISODES, (unsigned long long)st_eps);
                atomicAdd(P.stats + SWARM_STAT_SUCCESS, (unsigned long long)st_succ);
                atomicAdd(P.stats + SWARM_STAT_COLLISION, (unsigned long long)st_col);
                atomicAdd(P.stats + SWARM_STAT_TIMEOUT, (unsigned long long)st_to);
                atomicAdd(P.stats + SWARM_STAT_LENGTH_SUM, (unsigned long long)st_len);
                atomicAdd(reinterpret_cast<double*>(P.stats + SWARM_STAT_RETURN_SUM), st_ret);
            }
            atomicAdd(P.stats + SWARM_STAT_AGENT_STEPS, (unsigned long long)st_asteps);
            atomicAdd(P.stats + SWARM_STAT_ENV_STEPS, (unsigned long long)st_esteps);
        }
        for (int off = 16; off >= 1; off >>= 1) st_nan += __shfl_xor_sync(FULL_MASK, st_nan, off);
        if (lane == 0 && st_nan) atomicAdd(P.stats + SWARM_STAT_NAN_ACTIONS, (unsigned long long)st_nan);
    }
}

// ------------------------------------------------------------------------------------------
// N <= 32 kernel.  One drone per lane; G = 32 / N env instances per warp.
//
// The O(N^2) pair work is split in two:
//   B1  every unordered pair (i, j) is evaluated ONCE (round r: lane i takes partner i + r, wrapping
//       inside its env) and the float32 distance is written into both drones' rows of a per-warp
//       distance matrix in shared memory, each row stored compacted (column c = j - (j > i));
//   B2  every lane scans its own row in ascending column order -- the reference's order for the
//       k-nearest selection (lowest index wins ties) and for np.mean's pairwise summation lanes.
// The matrix aliases the observation staging tile.  Step, auto-reset and observe share one copy
// of the scan code through a small warp-uniform state machine.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(unsigned saddr, const void* g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async4(unsigned saddr, const void* g) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

enum SmallMode : int { kSmallStep = 0, kSmallAux = 1 };  // aux = reset / auto-reset / observe launches


// The step kernel (MODE = kSmallStep) contains no reset / observe code and the aux kernel no
// reward / flag code: the instruction working set of each launch stays inside the SM's
// instruction cache (the fused single-kernel version measured 82 % icc hit rate).  With
// auto_reset the step launch writes a per-env reset mask and the host enqueues the aux kernel
// right behind it on the same stream.
// NT > 0: number of drones known at compile time (8 / 16 / 32 for the BASELINE shapes): every
// derived constant (G, row stride, block counts) folds and the matrix addressing becomes immediates.
__host__ __device__ constexpr int small_srow(int n) {
    int s = ((n - 1 + 7) & ~7) > 1 ? ((n - 1 + 7) & ~7) : 1;
    while ((s & 3) != 1) ++s;
    return s;
}

template <int KT, int ST, bool EXACT, int NORM, int KIND, int MODE, int NT, bool DR>
__global__ void __launch_bounds__(kThreadsPerCta, kMinBlocksPerSm) swarm_env_kernel_small(const DevParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // Per-warp slice: two "inboxes" (the next group's inputs land in one by cp.async while the current
    // group is processed out of the other) + the distance-matrix / obs-staging region.
    //   inbox: pos4[32] | vel4[32] | goal4[G] | obst4[G * m_pad] | actions[32 * 3] | step_count[G] | ep_return[G]
    unsigned char* wslice = smem_raw + (size_t)warp * P.smem_per_warp;
    float* region = reinterpret_cast<float*>(wslice + 2 * (size_t)P.inbox_bytes);  // distance matrix / obs staging tile
    const int N = NT ? NT : P.N, M = P.M, G = NT ? 32 / NT : P.G, srow = NT ? small_srow(NT) : P.srow;
    const int K = EXACT ? KT : P.K, S = EXACT ? ST : P.S;
    constexpr bool HAS_NEIGH = KIND != SWARM_KIND_SINGLE;  // swarm and physics envs observe neighbours
    constexpr bool PHYS = KIND == SWARM_KIND_PHYSICS;       // DronePhysicsEnv as a point mass (see oracle/swarm_oracle.c)
    const int D = EXACT ? (HAS_NEIGH ? 9 + 4 * KT + 4 * ST : 9 + 4 * ST) : P.D;
    const int goal_off = 64, obst_off = 64 + G, dr_off4 = 64 + G + G * P.m_pad;     // inbox offsets, float4 units
    const int act_off4 = dr_off4 + (DR ? 2 * G : 0);
    const int e_l = lane / N;
    const int i = lane - e_l * N;
    const int e_base = e_l * N;  // first lane of this lane's env
    const unsigned env_lanes = e_l < G ? (N == 32 ? FULL_MASK : (((1u << N) - 1u) << e_base)) : 0u;
    const int n_others = N - 1;
    const int n8 = n_others >= 8 ? (n_others & ~7) : 0;
    const int n_pad = (n_others + 7) & ~7;  // matrix rows are padded with +inf to whole blocks of 8
    const int half = N >> 1;
    // per-warp statistics live in shared memory (leader lanes update them; flushed once at the end)
    unsigned long long* wstats =
        reinterpret_cast<unsigned long long*>(smem_raw + (size_t)kWarpsPerCta * P.smem_per_warp) + warp * SWARM_STATS_WORDS;
    if (MODE == kSmallStep && lane < SWARM_STATS_WORDS) wstats[lane] = 0ull;

    asm volatile("griddepcontrol.wait;" ::: "memory");  // programmatic dependent launch: the previous launch is done
    const int warps_total = gridDim.x * kWarpsPerCta;
    const int gwarp = blockIdx.x * kWarpsPerCta + warp;
    // aux launches behind a step (auto-reset) walk the compacted list of groups that asked for a reset
    const bool listed = MODE == kSmallAux && P.mode == kModeAutoReset;
    // auto-reset hand-over: list (epoch & 1) is appended to by the step launch, list ((epoch - 1) & 1) is walked by
    // the aux launch behind it (swarm_internal.h)
    // (the step launch re-reads the epoch where it needs it -- a rare path -- instead of carrying list pointers in
    //  registers through the whole kernel: they cost the physics instantiation 48 bytes of spills and 13 %)
    const int* rlist = P.reset_list;
    int n_iter = P.n_groups;
    unsigned aux_epoch = 0u;
    if (listed) {
        aux_epoch = *reinterpret_cast<const volatile unsigned*>(P.reset_epoch);
        const unsigned lpar = (aux_epoch - 1u) & 1u;
        rlist = P.reset_list + lpar * P.reset_list_stride;
        n_iter = (int)*reinterpret_cast<const volatile unsigned*>(P.reset_count + lpar);
    }

    // cp.async prefetch of one group's inputs into an inbox (step kernel only)
    auto prefetch = [&](int grp, int buf) {
        const int env0 = P.env_begin + grp * G;
        const int n_env = min(G, P.env_begin + P.env_count - env0);
        const int n_ag = n_env * N;
        const long long a0 = (long long)env0 * N;
        unsigned char* ib = wslice + (size_t)buf * P.inbox_bytes;
        const unsigned sbase = (unsigned)__cvta_generic_to_shared(ib);
        if (lane < n_ag) {
            cp_async16(sbase + lane * 16, P.pos4 + a0 + lane);
            cp_async16(sbase + 512 + lane * 16, P.vel4 + a0 + lane);
        }
        if (lane < n_env) {
            cp_async16(sbase + goal_off * 16 + lane * 16, P.goal4 + env0 + lane);
            cp_async4(sbase + (act_off4 * 16 + 384) + lane * 4, P.step_count + env0 + lane);
            cp_async4(sbase + (act_off4 * 16 + 384 + 4 * G) + lane * 4, P.ep_return + env0 + lane);
        }
        for (int idx = lane; idx < n_env * M; idx += 32)
            cp_async16(sbase + obst_off * 16 + idx * 16, P.obst4 + (long long)env0 * M + idx);
        if (DR)
            for (int idx = lane; idx < 2 * n_env; idx += 32)
                cp_async16(sbase + dr_off4 * 16 + idx * 16, P.dr_params + (long long)env0 * 2 + idx);
        const float* act = P.actions + a0 * 3;
        // 16-byte copies need whole 16-byte chunks AND a 16-byte aligned base (a float32 view at a 4 / 8 / 12-byte
        // storage offset is a legal `actions` argument: it takes the 4-byte path)
        if ((((G * N) | n_ag) & 3) == 0 && (reinterpret_cast<unsigned long long>(P.actions) & 15ull) == 0) {
            if (lane * 4 < n_ag * 3) cp_async16(sbase + act_off4 * 16 + lane * 16, act + lane * 4);
        } else {
            for (int idx = lane; idx < n_ag * 3; idx += 32) cp_async4(sbase + act_off4 * 16 + idx * 4, act + idx);
        }
        cp_async_commit();
    };
    int buf = 0;
    if (MODE == kSmallStep && gwarp < n_iter) prefetch(gwarp, 0);

    // step launches: dynamic group queue (first group static, then an atomic counter drawn at the top of a
    // group and consumed after the integrator); aux launches keep the static stride
    // (short groups -- the single-drone env, tiny swarms -- are cheaper than the atomic: static stride there)
    const bool dyn_queue = MODE == kSmallStep && N >= 8;
    int it = gwarp;
    while (it < n_iter) {
        int it_next = it + warps_total;
        // (the raw counter value: an add placed here is scheduled right behind the atomic and waits out its round trip)
        if (dyn_queue && lane == 0) it_next = (int)atomicAdd(P.work_counter, 1u);
        const int env0 = listed ? rlist[it] : P.env_begin + it * G;
        const int n_env = min(G, P.env_begin + P.env_count - env0);
        const bool lane_ok = e_l < n_env;
        const int env = env0 + (lane_ok ? e_l : 0);
        const long long a0 = (long long)env0 * N;      // first agent of the group
        const long long a = a0 + (lane_ok ? lane : 0);  // this lane's agent
        const bool leader = lane_ok && i == 0;
        const unsigned ok_lanes = __ballot_sync(FULL_MASK, lane_ok);
        float4* tab_pos = reinterpret_cast<float4*>(wslice + (size_t)buf * P.inbox_bytes);
        float4* tab_vel = tab_pos + 32;
        float4* tab_goal = tab_pos + goal_off;
        float4* tab_obst = tab_pos + obst_off;
        const float4* tobs = tab_obst + e_l * P.m_pad;
        float* drow = region + lane * srow;  // this drone's row of the distance matrix

        unsigned reset_envs = 0;  // aux: bit el = env el is (re)drawn
        if (MODE == kSmallAux && P.mode != kModeObserve) {
            const bool want = lane < n_env && (P.env_mask == nullptr || P.env_mask[env0 + lane] != 0);
            reset_envs = __ballot_sync(FULL_MASK, want);
            if (reset_envs == 0) {  // nothing to reset in this group
                it = it_next;
                buf ^= 1;
                continue;
            }
        }

        float4 p = make_float4(0.f, 0.f, 0.f, 0.f), v = p, g4 = p;
        float ax = 0.f, ay = 0.f, az = 0.f, ep_ret = 0.f;
        int sc = 0;
        if (MODE == kSmallStep) {
            cp_async_wait_all();
            __syncwarp();  // this group's inbox is complete; the other inbox is free again
            if (lane_ok) {
                p = tab_pos[lane];
                v = tab_vel[lane];
                g4 = tab_goal[e_l];
                const float* act = reinterpret_cast<const float*>(tab_pos + act_off4);
                ax = act[lane * 3 + 0]; ay = act[lane * 3 + 1]; az = act[lane * 3 + 2];
                sc = reinterpret_cast<const int*>(act + 96)[e_l];
                ep_ret = (act + 96 + G)[e_l];
            }
            __syncwarp();  // everyone has read its inputs before positions are overwritten in place
        } else {
            __syncwarp();  // the previous group is done with the shared-memory slice
            if (lane_ok) {
                p = P.pos4[a];
                v = P.vel4[a];
                g4 = P.goal4[env];
            }
            for (int idx = lane; idx < n_env * M; idx += 32) tab_obst[idx] = P.obst4[(long long)env0 * M + idx];
        }
        float gx = g4.x, gy = g4.y, gz = g4.z;
        // per-env dynamics constants: the config's, or this episode's randomised ones
        float c_amax = P.amax, c_vmax = P.vmax, c_dt = P.dt, c_bound = P.bound, c_thr_obst = P.thr_obst;
        unsigned ekey = 0u;
        int ctrl_delay = 0;
        if (DR && lane_ok) {
            const float4* drp = MODE == kSmallStep ? tab_pos + dr_off4 + 2 * e_l : P.dr_params + (long long)env * 2;
            const float4 d0 = drp[0], d1 = drp[1];
            c_amax = d0.x; c_vmax = d0.y; c_dt = d0.z; c_bound = d0.w;
            c_thr_obst = d1.x; ekey = __float_as_uint(d1.y);
            ctrl_delay = (int)d1.w;
        }
        const unsigned genv = DR ? (unsigned)(P.env_index_base + env) : 0u;

        bool alive = KIND == SWARM_KIND_SINGLE ? lane_ok : (lane_ok && p.w != 0.0f);
        float prev_d = 0.f;
        bool nan_act = false;
        unsigned out_lanes = ok_lanes;  // lanes whose obs row is produced by this launch
        if (MODE == kSmallStep) {
            // =========================== phase A: integrate (:98-118) ===========================
            prev_d = norm1d<NORM>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));  // :98-101
            if (PHYS) {
                if (alive) {
                    // DR on top (DESIGN.md 9): the episode's sub-step length rides in c_dt; control delay and thrust
                    // noise act on the command, which is then held for the whole step (no clip: :336)
                    if (DR && P.dr_delay_hist > 0) delayed_command(P, env, N, i, sc, ctrl_delay, ax, ay, az);
                    if (DR) {
                        const uint4 r = philox4x32_7(genv, ekey, (unsigned)sc, (unsigned)i | (DR_STREAM_A << 16), P);
                        thrust_noise(P, [=](int f) { return dr_normal(P.dr_qtable, dr_field(r, f)); }, ax, ay, az);
                    }
                    physics_substeps<NORM>(P, ax, ay, az, c_amax, c_vmax, DR ? c_dt : P.phys_h, p, v);
                }
            } else if (alive) {
                if (DR && P.dr_delay_hist > 0) delayed_command(P, env, N, i, sc, ctrl_delay, ax, ay, az);
                ax = clipf(ax, -1.0f, 1.0f); ay = clipf(ay, -1.0f, 1.0f); az = clipf(az, -1.0f, 1.0f);
                nan_act = !(ax == ax && ay == ay && az == az);   // (np.clip lets NaN through; counted below)
                if (DR) {
                    const uint4 r = philox4x32_7(genv, ekey, (unsigned)sc, (unsigned)i | (DR_STREAM_A << 16), P);
                    thrust_noise(P, [=](int f) { return dr_normal(P.dr_qtable, dr_field(r, f)); }, ax, ay, az);
                }
                point_mass_step<NORM>(P, ax, ay, az, c_amax, c_vmax, c_dt, p.x, p.y, p.z, v.x, v.y, v.z);
            }
            if (PHYS) nan_act = alive && !(ax == ax && ay == ay && az == az);   // (the physics env does not clip)
            {   // NaN-action guard counter (rare: the vote is all a clean step pays)
                const unsigned nan_m = __ballot_sync(FULL_MASK, nan_act);
                if (nan_m != 0u && lane == 0) wstats[SWARM_STAT_NAN_ACTIONS] += (unsigned long long)__popc(nan_m);
            }
            // wall clip for ALL drones (:113-117); velocity is not zeroed at the wall (the physics env has no walls)
            if (!PHYS) {
                p.x = clipf(p.x, -c_bound, c_bound);
                p.y = clipf(p.y, -c_bound, c_bound);
                p.z = clipf(p.z, -c_bound, c_bound);
            }
        }
        if (MODE == kSmallStep) {  // next group's inputs -> the other inbox
            if (dyn_queue) it_next = warps_total + __shfl_sync(FULL_MASK, it_next, 0);
            if (it_next < n_iter) prefetch(it_next, buf ^ 1);
        }
        float damp = v.w;  // physics env: per-drone damping factor rides in vel4.w
        int sc_obs = MODE == kSmallStep ? sc + 1 : 0;  // step_count of the state the obs row describes (DR sensor stream)
        if (DR && MODE == kSmallAux && lane_ok) sc_obs = P.step_count[env];
        if (lane_ok) tab_pos[lane] = make_float4(p.x, p.y, p.z, alive ? 1.0f : 0.0f);
        tab_vel[lane] = make_float4(v.x, v.y, v.z, prev_d);  // parked here while the scans need the registers

        if (MODE == kSmallAux && reset_envs) {
            // ================================ reset (:65-80) ================================
            __syncwarp();
#pragma unroll 1
            for (int el = 0; el < n_env; ++el) {
                if (!((reset_envs >> el) & 1u)) continue;
                const int renv = env0 + el;
                const Pcg64State rng = load_rng(P, renv);
                double u_lo = P.rng_lo, u_range = P.rng_range;
                if (DR) {
                    const EpisodeDraw ep = draw_episode_constants(P, (unsigned)(P.env_index_base + renv), rng.sl);
                    u_lo = ep.u_lo(); u_range = ep.u_range();
                    float4 d0, d1;
                    episode_params(P, ep, d0, d1);
                    if (lane == 0) {
                        P.dr_params[(long long)renv * 2 + 0] = d0;
                        P.dr_params[(long long)renv * 2 + 1] = d1;
                    }
                    if (lane_ok && e_l == el) {
                        c_amax = d0.x; c_vmax = d0.y; c_dt = d0.z; c_bound = d0.w;
                        c_thr_obst = d1.x; ekey = ep.key;
                        sc_obs = 0;
                    }
                }
                auto pos = [=](int j) { return reinterpret_cast<float*>(tab_pos + el * N + j); };
                auto goal = [=]() { return reinterpret_cast<float*>(tab_goal + el); };
                auto obst = [=](int m) { return reinterpret_cast<float*>(tab_obst + el * P.m_pad + m); };
                if (PHYS)
                    reset_env_physics_draws<1>(P, lane, N, M, rng, u_lo, u_range, pos,
                                               [=](int j) { return reinterpret_cast<float*>(tab_vel + el * N + j); }, goal, obst);
                else
                    reset_env_draws<1>(P, lane, N, rng, u_lo, u_range, pos, goal, obst);
                if (lane < N) {
                    reinterpret_cast<float*>(tab_pos + el * N + lane)[3] = 1.0f;
                    float* tv = reinterpret_cast<float*>(tab_vel + el * N + lane);
                    tv[0] = 0.f; tv[1] = 0.f; tv[2] = 0.f;
                    if (!PHYS) tv[3] = 0.f;  // (physics: .w already holds this drone's damping factor)
                }
                if (lane == 0) {
                    reset_env_finish(P, renv, rng);
                    reinterpret_cast<float*>(tab_goal + el)[3] = 0.0f;
                }
                for (int k = lane; k < M; k += 32) reinterpret_cast<float*>(tab_obst + el * P.m_pad + k)[3] = 0.0f;
            }
            __syncwarp();
            const bool fresh = lane_ok && ((reset_envs >> e_l) & 1u);
            if (lane < n_env && ((reset_envs >> lane) & 1u)) P.goal4[env0 + lane] = tab_goal[lane];
            for (int idx = lane; idx < n_env * M; idx += 32)
                if ((reset_envs >> (idx / M)) & 1u) P.obst4[(long long)env0 * M + idx] = tab_obst[idx];
            if (fresh) {
                p = tab_pos[lane];
                g4 = tab_goal[e_l]; gx = g4.x; gy = g4.y; gz = g4.z;
                alive = true;
                P.pos4[a] = p;
                if (PHYS) damp = tab_vel[lane].w;
                P.vel4[a] = make_float4(0.f, 0.f, 0.f, PHYS ? damp : 0.f);
            }
            out_lanes = __ballot_sync(FULL_MASK, fresh);
        }
        const unsigned alive_mask = __ballot_sync(FULL_MASK, alive);
        const int n_alive_env = __popc(alive_mask & env_lanes);
        __syncwarp();  // position / obstacle tables complete

        // ========================= B1: symmetric distance matrix =========================
        if (HAS_NEIGH) {
            // Round r pairs drone i with j = i + r (wrapping inside the env).  Rounds 1 .. N/2 cover
            // every unordered pair; for even N the last round is visited from both ends, which only
            // stores the same value twice.  All addresses are (select of two lane constants) + r * stride.
            const int wrap_at = N - i;  // r >= wrap_at  <=>  i + r wraps
            const float4* tp_nw = tab_pos + lane;  // partner position, no wrap / wrap
            const float4* tp_w = tp_nw - N;
            float* own_nw = drow + (i - 1);        // own row, column j - 1 (j > i) / j (j < i)
            float* own_w = drow + (i - N);
            float* par_nw = drow + i;              // partner row j, column i (i < j) / i - 1 (i > j)
            float* par_w = drow - N * srow + (i - 1);
            int r0 = 1;
#pragma unroll 1
            for (; r0 + 3 <= half; r0 += 4) {
                float s[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int r = r0 + u;
                    const float4 q = (r >= wrap_at ? tp_w : tp_nw)[r];
                    s[u] = sumsq1d<NORM>(__fsub_rn(q.x, p.x), __fsub_rn(q.y, p.y), __fsub_rn(q.z, p.z));
                }
                const float smin = fminf(fminf(s[0], s[1]), fminf(s[2], s[3]));
                float d[4];
                if (smin >= SQRT_FAST_MIN) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) d[u] = sqrt_rn_fast(s[u]);
                } else {  // coincident drones (d == 0) or denormal range: full IEEE path
#pragma unroll
                    for (int u = 0; u < 4; ++u) d[u] = __fsqrt_rn(s[u]);
                }
                if (lane_ok) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int r = r0 + u;
                        const bool w = r >= wrap_at;
                        (w ? own_w : own_nw)[r] = d[u];
                        (w ? par_w : par_nw)[r * srow] = d[u];
                    }
                }
            }
#pragma unroll 1
            for (; r0 <= half; ++r0) {  // leftover rounds (N/2 not a multiple of 4)
                const bool w = r0 >= wrap_at;
                const float4 q = lane_ok ? (w ? tp_w : tp_nw)[r0] : p;
                const float dd = norm1d<NORM>(__fsub_rn(q.x, p.x), __fsub_rn(q.y, p.y), __fsub_rn(q.z, p.z));
                if (lane_ok) {
                    (w ? own_w : own_nw)[r0] = dd;
                    (w ? par_w : par_nw)[r0 * srow] = dd;
                }
            }
            // pad the row to a multiple of 8 columns with non-candidates so B2 runs whole blocks only
            if (lane_ok) {
#pragma unroll
                for (int u = 0; u < 7; ++u)
                    if (n_others + u < n_pad) drow[n_others + u] = TOPK_EMPTY;
            }
        }
        __syncwarp();

        // ================ B2: own row in ascending order: k-nearest (+ formation) ================
        float nd[KT]; int nj[KT];
#pragma unroll
        for (int q = 0; q < KT; ++q) { nd[q] = TOPK_EMPTY; nj[q] = -1; }
        bool pair_hit = false;
        double form_sum = 0.0;
        int form_n = 0;
        if (HAS_NEIGH && lane_ok) {
            if (MODE == kSmallAux) {
#pragma unroll 1
                for (int cb = 0; cb < n_pad; cb += 8) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) topk_insert<KT>(drow[cb + u], cb + u, nd, nj);
                }
            } else if (alive && n_alive_env == N) {
                // every drone active: column c is element c of np.mean's operand (:210-224).  numpy sums
                // columns [0, n8) in 8 lanes (tree-combined) and then adds columns [n8, N-1) in order; the
                // last block therefore runs on fresh lanes that are added sequentially afterwards.
                const double d_star = P.d_star;
                double r8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) r8[u] = 0.0;
                double res = 0.0;
#pragma unroll 1
                for (int cb = 0; cb < n_pad; cb += 8) {
                    if (cb == n8 && n8 > 0) {
                        res = tree8(r8);
#pragma unroll
                        for (int u = 0; u < 8; ++u) r8[u] = 0.0;
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const float d = drow[cb + u];  // TOPK_EMPTY in the padding columns: never selected
                        topk_insert<KT>(d, cb + u, nd, nj);
                        r8[u] = __dadd_rn(r8[u], fabs(__dsub_rn((double)d, d_star)));
                    }
                }
                if (n8 < n_others) {
#pragma unroll
                    for (int u = 0; u < 7; ++u) res = __dadd_rn(res, n8 + u < n_others ? r8[u] : 0.0);
                } else if (n8 > 0) {
                    res = tree8(r8);
                }
                pair_hit = nd[0] <= P.thr_pair;  // nearest drone decides (:202-207)
                form_sum = res;
                form_n = n_others;
            } else {
                // some drones are parked (or this one is): compact the active ones on the fly
                const unsigned em = (alive_mask & env_lanes) >> e_base;  // bit j: drone j of this env active
                const unsigned cm = (em & ((1u << i) - 1u)) | ((em >> (i + 1)) << i);  // bit c: column c active
                const int n_f = alive ? n_alive_env - 1 : 0;
                const int nf8 = n_f >= 8 ? (n_f & ~7) : 0;
                double r8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) r8[u] = 0.0;
                double res = 0.0;
                bool tree_done = false;
                int cnt = 0;
#pragma unroll 1
                for (int c = 0; c < n_others; ++c) {
                    const float d = drow[c];
                    topk_insert<KT>(d, c, nd, nj);
                    if (alive && ((cm >> c) & 1u)) {
                        pair_hit |= d <= P.thr_pair;
                        const double err = fabs(__dsub_rn((double)d, P.d_star));
                        if (cnt < nf8) {
                            const int lane8 = cnt & 7;
#pragma unroll
                            for (int u = 0; u < 8; ++u) r8[u] = __dadd_rn(r8[u], lane8 == u ? err : 0.0);
                        } else {
                            if (!tree_done && nf8 > 0) res = tree8(r8);
                            tree_done = true;
                            res = __dadd_rn(res, err);
                        }
                        ++cnt;
                    }
                }
                if (!tree_done && nf8 > 0) res = tree8(r8);
                form_sum = res;
                form_n = n_f;
            }
        }
        // ---- obstacles: _nearest_obstacle_features (:273-291) + obstacle part of _collision_mask
        float od[ST]; int om[ST];
#pragma unroll
        for (int q = 0; q < ST; ++q) { od[q] = TOPK_EMPTY; om[q] = -1; }
        {
            int mb = 0;
#pragma unroll 1
            for (; mb + 4 <= M; mb += 4) obst_block4<ST, true>(tobs, mb, M, p.x, p.y, p.z, od, om);
            if (mb < M) obst_block4<ST, false>(tobs, mb, M, p.x, p.y, p.z, od, om);
        }
        const float curr_d = norm1d<NORM>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));
        __syncwarp();  // every lane is done with the distance matrix: the region becomes the obs tile
        {
            const float4 t = tab_vel[lane];
            v = t; prev_d = t.w;
        }

        // ============================ obs row -> staging tile ============================
        if ((out_lanes >> lane) & 1u) {
            float* row = region + lane * D;
            // DR sensor noise of the observed state: blocks of counter (its step_count - 1), see swarm_device.cuh
            uint4 rA = make_uint4(0, 0, 0, 0), rB = rA;
            if (DR) {
                rA = philox4x32_7(genv, ekey, (unsigned)(sc_obs - 1), (unsigned)i | (DR_STREAM_A << 16), P);
                if (S > 4) rB = philox4x32_7(genv, ekey, (unsigned)(sc_obs - 1), (unsigned)i | (DR_STREAM_B << 16), P);
            }
            auto noisy = [&](float x, float sigma, unsigned idx) {
                return DR ? __fmaf_rn(sigma, dr_normal(P.dr_qtable, idx), x) : x;
            };
            auto obst_bits = [&](int q) { return q < 4 ? dr_field(rA, 9 + q) : dr_field(rB, q - 4); };
            row[0] = noisy(p.x, P.dr_std_pos, dr_field(rA, 3)); row[1] = noisy(p.y, P.dr_std_pos, dr_field(rA, 4));
            row[2] = noisy(p.z, P.dr_std_pos, dr_field(rA, 5));
            float ovx = v.x, ovy = v.y, ovz = v.z;
            if (PHYS) {  // drone_physics_env.py:436-439: the observed velocity is clamped to max_speed
                const float speed = norm1d<NORM>(v.x, v.y, v.z);
                if (speed > c_vmax) {
                    ovx = __fmul_rn(__fdiv_rn(v.x, speed), c_vmax);
                    ovy = __fmul_rn(__fdiv_rn(v.y, speed), c_vmax);
                    ovz = __fmul_rn(__fdiv_rn(v.z, speed), c_vmax);
                }
            }
            row[3] = noisy(ovx, P.dr_std_vel, dr_field(rA, 6)); row[4] = noisy(ovy, P.dr_std_vel, dr_field(rA, 7));
            row[5] = noisy(ovz, P.dr_std_vel, dr_field(rA, 8));
            row[6] = __fsub_rn(gx, p.x); row[7] = __fsub_rn(gy, p.y); row[8] = __fsub_rn(gz, p.z);
            int off = 9;
            const bool all_slots = (!HAS_NEIGH || n_others >= K) && M >= S;  // warp-uniform
            if (all_slots) {
                if (HAS_NEIGH) {
#pragma unroll
                    for (int q = 0; q < KT; ++q) {
                        if (q < K) {
                            const int c = nj[q];
                            const float4 t = (c >= i ? tab_pos + e_base + 1 : tab_pos + e_base)[c];
                            row[off + 4 * q + 0] = __fsub_rn(t.x, p.x);
                            row[off + 4 * q + 1] = __fsub_rn(t.y, p.y);
                            row[off + 4 * q + 2] = __fsub_rn(t.z, p.z);
                            row[off + 4 * q + 3] = nd[q];
                        }
                    }
                    off += 4 * K;
                }
#pragma unroll
                for (int q = 0; q < ST; ++q) {
                    if (q < S) {
                        const float4 t = tobs[om[q]];
                        row[off + 4 * q + 0] = __fsub_rn(t.x, p.x);
                        row[off + 4 * q + 1] = __fsub_rn(t.y, p.y);
                        row[off + 4 * q + 2] = __fsub_rn(t.z, p.z);
                        row[off + 4 * q + 3] = noisy(od[q], P.dr_std_obst, obst_bits(q));
                    }
                }
            } else {  // fewer candidates than slots: zero padding (:268-270, :288-290)
                if (HAS_NEIGH) {
#pragma unroll
                    for (int q = 0; q < KT; ++q) {
                        if (q < K) {
                            const int c = nj[q];
                            const bool has = c >= 0;
                            const float4 t = tab_pos[e_base + (has ? c + (c >= i ? 1 : 0) : i)];
                            row[off + 4 * q + 0] = has ? __fsub_rn(t.x, p.x) : 0.f;
                            row[off + 4 * q + 1] = has ? __fsub_rn(t.y, p.y) : 0.f;
                            row[off + 4 * q + 2] = has ? __fsub_rn(t.z, p.z) : 0.f;
                            row[off + 4 * q + 3] = has ? nd[q] : 0.f;
                        }
                    }
                    off += 4 * K;
                }
#pragma unroll
                for (int q = 0; q < ST; ++q) {
                    if (q < S) {
                        const int m = om[q];
                        const bool has = m >= 0;
                        const float4 t = tobs[has ? m : 0];
                        row[off + 4 * q + 0] = has ? __fsub_rn(t.x, p.x) : 0.f;
                        row[off + 4 * q + 1] = has ? __fsub_rn(t.y, p.y) : 0.f;
                        row[off + 4 * q + 2] = has ? __fsub_rn(t.z, p.z) : 0.f;
                        row[off + 4 * q + 3] = has ? noisy(od[q], P.dr_std_obst, obst_bits(q)) : 0.f;
                    }
                }
            }
        }
        __syncwarp();
        if (out_lanes == ok_lanes) {
            flush_stage(P.obs, D, region, a0, n_env * N, lane);  // whole tile, one contiguous stream
        } else {
#pragma unroll 1
            for (int el = 0; el < n_env; ++el)  // only the (re)observed envs' rows
                if ((out_lanes >> (el * N)) & 1u) flush_stage(P.obs, D, region + el * N * D, a0 + el * N, N, lane);
        }

        if (MODE == kSmallStep) {
            // ===================== rewards and flags (:120-172) =====================
            const bool obst_hit = od[0] <= c_thr_obst;
            // physics env: reached = dist < goal_radius (strict, drone_physics_env.py:389); contact with the
            // ground plane, an obstacle sphere or another drone (:368-372, point-mass radii set by the host)
            const bool reached = PHYS ? (alive && (double)curr_d < P.goal_radius_d)
                                      : (alive && curr_d <= P.thr_goal);  // :124-127 (double compare)
            const bool collided = alive && (obst_hit || pair_hit || (PHYS && p.z <= P.phys_ground_z));  // :128
            double reward = 0.0;
            if (PHYS) {
                if (alive) {  // drone_physics_env.py:378-392
                    reward = __dmul_rn(-(double)curr_d, 0.1);
                    if (collided) reward = __dsub_rn(reward, 10.0);
                    else if (reached) reward = __dadd_rn(reward, 50.0);
                }
            } else if (alive) {
                const double progress = __dmul_rn(__dsub_rn((double)prev_d, (double)curr_d), P.k_p);  // :142
                if (KIND == SWARM_KIND_SWARM) {
                    double pen = 0.0;  // :210-224
                    if (form_n > 0) {
                        const double mean = form_n == n_others ? mean_markstein(form_sum, P.n_others, P.inv_n_others)
                                                               : __ddiv_rn(form_sum, (double)form_n);
                        pen = __dmul_rn(P.neg_k_f, mean);
                    }
                    reward = __dadd_rn(progress, pen);  // :143
                } else {
                    reward = progress;
                }
                if (reached) reward = __dadd_rn(reward, P.r_goal);   // :144-145
                if (collided) reward = __dadd_rn(reward, P.r_col);   // :146-147
            }
            const float rew32 = __double2float_rn(reward);
            const bool done_agent = reached || collided;
            const bool any_col = (__ballot_sync(FULL_MASK, collided) & env_lanes) != 0;
            const int n_cont = __popc(__ballot_sync(FULL_MASK, alive && !done_agent) & env_lanes);
            // deterministic per-env reward sum (segmented tree over the env's lanes)
            float x = rew32;
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                const float t = __shfl_down_sync(FULL_MASK, x, off);
                if (i + off < N) x = __fadd_rn(x, t);
            }
            const bool env_active = KIND == SWARM_KIND_SINGLE ? true : n_alive_env > 0;
            const int sc_new = env_active ? sc + 1 : sc;
            const bool time_limit = env_active && sc_new >= P.max_steps;
            bool all_term, all_trunc, ep_over, all_reached = false;
            if (PHYS) {  // drone_physics_env.py:397-417: one flag pair for every drone
                const int n_open = __popc(__ballot_sync(FULL_MASK, alive && !collided && !reached) & env_lanes);
                all_reached = n_open == 0;
                const bool done = env_active && (any_col || all_reached || time_limit);
                all_trunc = env_active && time_limit && !any_col && !all_reached;
                all_term = env_active ? (any_col || all_reached) : true;
                ep_over = done;
                all_reached = all_reached && !any_col;
            } else if (KIND == SWARM_KIND_SWARM) {
                all_reached = n_cont == 0 && !any_col && !time_limit;
                const bool episode_done = all_reached || any_col;
                all_term = env_active ? episode_done : true;  // :94-95 when no agent is left
                all_trunc = env_active ? (time_limit && !episode_done) : false;
                ep_over = env_active && (all_term || all_trunc);
            } else {
                all_term = done_agent;   // single env: terminated (:102)
                all_trunc = time_limit;  // truncated, not masked by terminated (:103)
                ep_over = all_term || all_trunc;
            }
            const bool need_reset = P.auto_reset && (ep_over || !env_active);
            if (lane_ok) {
                bool valid, alive_next;
                if (PHYS) {
                    P.terminated[a] = (alive && ep_over && !all_trunc) ? 1 : 0;
                    P.truncated[a] = (alive && ep_over && all_trunc) ? 1 : 0;
                    valid = alive;              // every drone is observed on every step
                    alive_next = alive && !ep_over;
                } else if (KIND == SWARM_KIND_SWARM) {
                    P.terminated[a] = (alive && done_agent) ? 1 : 0;                 // :150-151
                    P.truncated[a] = (alive && time_limit && !done_agent) ? 1 : 0;   // :152
                    valid = alive && !done_agent && !time_limit && !any_col;         // :154
                    alive_next = ep_over ? false : valid;                            // :169-172
                } else {
                    P.terminated[a] = all_term ? 1 : 0;
                    P.truncated[a] = all_trunc ? 1 : 0;
                    valid = true;
                    alive_next = true;
                }
                P.reward[a] = rew32;
                if (P.reward64) P.reward64[a] = reward;
                P.reached[a] = reached ? 1 : 0;
                P.collision[a] = collided ? 1 : 0;
                if (!need_reset) {  // (a reset env gets these from the aux launch that follows)
                    P.dist[a] = curr_d;
                    P.obs_valid[a] = valid ? 1 : 0;
                    P.pos4[a] = make_float4(p.x, p.y, p.z, alive_next ? 1.0f : 0.0f);
                    P.vel4[a] = make_float4(v.x, v.y, v.z, PHYS ? damp : 0.0f);
                    if (P.gs) write_gs_drone(P.gs + (long long)env * P.R, N, i, p.x, p.y, p.z, v.x, v.y, v.z);
                }
            }
            if (leader) {
                P.all_term[env] = all_term ? 1 : 0;
                P.all_trunc[env] = all_trunc ? 1 : 0;
                if (P.reset_mask) P.reset_mask[env] = need_reset ? 1 : 0;
                const float ret = __fadd_rn(ep_ret, x);
                if (ep_over) {  // several env leaders per warp when G > 1: shared-memory atomics
                    atomicAdd(wstats + SWARM_STAT_EPISODES, 1ull);
                    atomicAdd(wstats + SWARM_STAT_LENGTH_SUM, (unsigned long long)sc_new);
                    atomicAdd(reinterpret_cast<double*>(wstats + SWARM_STAT_RETURN_SUM), (double)ret);
                    if (HAS_NEIGH) {
                        if (all_reached) atomicAdd(wstats + SWARM_STAT_SUCCESS, 1ull);
                        if (any_col) atomicAdd(wstats + SWARM_STAT_COLLISION, 1ull);
                        if (all_trunc) atomicAdd(wstats + SWARM_STAT_TIMEOUT, 1ull);
                    } else {  // single env (:92-103): the one drone's flags are the episode's
                        if (collided) atomicAdd(wstats + SWARM_STAT_COLLISION, 1ull);
                        else if (reached) atomicAdd(wstats + SWARM_STAT_SUCCESS, 1ull);
                        else if (all_trunc) atomicAdd(wstats + SWARM_STAT_TIMEOUT, 1ull);
                    }
                }
                if (P.episode_return) P.episode_return[env] = ep_over ? ret : 0.0f;
                if (P.episode_length) P.episode_length[env] = ep_over ? sc_new : 0;
                if (!need_reset) {
                    P.step_count[env] = sc_new;
                    P.ep_return[env] = ep_over ? 0.0f : ret;
                    if (P.gs) {
                        float* row = P.gs + (long long)env * P.R + 6 * N;
                        __stcs(row + 0, gx); __stcs(row + 1, gy); __stcs(row + 2, gz);
                    }
                }
            }
            if (P.auto_reset) {  // groups with an env to reset go on the list the aux launch walks
                const unsigned rl = __ballot_sync(FULL_MASK, leader && need_reset);
                if (rl != 0 && lane == 0) {
                    const unsigned lpar = *reinterpret_cast<const volatile unsigned*>(P.reset_epoch) & 1u;
                    P.reset_list[lpar * P.reset_list_stride + atomicAdd(P.reset_count + lpar, 1u)] = env0;
                }
            }
            {   // actions applied / envs stepped by this warp in this group
                const unsigned act_envs = __ballot_sync(FULL_MASK, leader && env_active);
                if (lane == 0) {
                    wstats[SWARM_STAT_AGENT_STEPS] += (unsigned long long)__popc(alive_mask);
                    wstats[SWARM_STAT_ENV_STEPS] += (unsigned long long)__popc(act_envs);
                }
            }
        } else {
            // =========== observe epilogue: reset()'s obs / infos (:82-89), or swarm_observe ===========
            if ((out_lanes >> lane) & 1u) {
                P.dist[a] = curr_d;
                P.obs_valid[a] = KIND == SWARM_KIND_SINGLE ? 1 : (alive ? 1 : 0);
                if (P.mode != kModeAutoReset) {  // an explicit reset / observe clears the step outputs
                    P.reward[a] = 0.0f;
                    if (P.reward64) P.reward64[a] = 0.0;
                    P.terminated[a] = 0; P.truncated[a] = 0; P.reached[a] = 0; P.collision[a] = 0;
                }
                if (P.gs) {
                    float* row = P.gs + (long long)env * P.R;
                    write_gs_drone(row, N, i, p.x, p.y, p.z, v.x, v.y, v.z);
                    if (i == 0) { __stcs(row + 6 * N + 0, gx); __stcs(row + 6 * N + 1, gy); __stcs(row + 6 * N + 2, gz); }
                }
                if (P.mode != kModeAutoReset && i == 0) {
                    P.all_term[env] = 0;
                    P.all_trunc[env] = 0;
                    if (P.episode_return) P.episode_return[env] = 0.0f;
                    if (P.episode_length) P.episode_length[env] = 0;
                }
            }
        }
        it = it_next;
        buf ^= 1;
    }
    if (dyn_queue || (MODE == kSmallStep && P.auto_reset)) {
        // the last warp to leave re-arms the queue for the next launch, hands the reset list over to the aux launch
        // and clears the other list for the next step
        if (lane == 0 && atomicAdd(P.work_counter + 1, 1u) == (unsigned)warps_total - 1u) {
            P.work_counter[0] = 0u;
            P.work_counter[1] = 0u;
            if (MODE == kSmallStep && P.auto_reset) {
                const unsigned epoch = *reinterpret_cast<const volatile unsigned*>(P.reset_epoch);
                P.reset_count[(epoch + 1u) & 1u] = 0u;
                *P.reset_epoch = epoch + 1u;
            }
        }
    }

    // ---- statistics: one global atomic per warp per counter
    if (MODE == kSmallStep) {
        __syncwarp();
        if (P.stats && lane < SWARM_STATS_WORDS) {
            const unsigned long long w = wstats[lane];
            if (lane == SWARM_STAT_RETURN_SUM) {
                const double dv = __longlong_as_double((long long)w);
                if (dv != 0.0) atomicAdd(reinterpret_cast<double*>(P.stats + lane), dv);
            } else if (w) {
                atomicAdd(P.stats + lane, w);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// np.random.default_rng(seed): SeedSequence(seed).generate_state(4, uint64) -> PCG64 seeding
// (numpy/random/bit_generator.pyx, _pcg64.pyx, src/pcg64/pcg64.h)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned ss_hashmix(unsigned value, unsigned& hc) {
    value ^= hc;
    hc *= 0x931e8875u;
    value *= hc;
    value ^= value >> 16;
    return value;
}
__device__ __forceinline__ unsigned ss_mix(unsigned x, unsigned y) {
    unsigned r = 0xca01f9ddu * x - 0x4973f715u * y;
    r ^= r >> 16;
    return r;
}

__global__ void swarm_seed_kernel(const DevParams P) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= P.E) return;
    if (P.env_mask && !P.env_mask[e]) return;
    const unsigned long long seed = P.seeds[e];
    const unsigned ent0 = (unsigned)(seed & 0xffffffffull), ent1 = (unsigned)(seed >> 32);
    const int n_ent = ent1 != 0 ? 2 : 1;
    unsigned pool[4];
    unsigned hc = 0x43b0d7e5u;
    pool[0] = ss_hashmix(ent0, hc);
    pool[1] = ss_hashmix(n_ent > 1 ? ent1 : 0u, hc);
    pool[2] = ss_hashmix(0u, hc);
    pool[3] = ss_hashmix(0u, hc);
#pragma unroll
    for (int s = 0; s < 4; ++s)
#pragma unroll
        for (int d = 0; d < 4; ++d)
            if (s != d) pool[d] = ss_mix(pool[d], ss_hashmix(pool[s], hc));
    unsigned w[8];
    hc = 0x8b51f9ddu;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        unsigned v = pool[k & 3];
        v ^= hc;
        hc *= 0x58f38dedu;
        v *= hc;
        v ^= v >> 16;
        w[k] = v;
    }
    const unsigned long long s_hi = (unsigned long long)w[0] | ((unsigned long long)w[1] << 32);
    const unsigned long long s_lo = (unsigned long long)w[2] | ((unsigned long long)w[3] << 32);
    const unsigned long long q_hi = (unsigned long long)w[4] | ((unsigned long long)w[5] << 32);
    const unsigned long long q_lo = (unsigned long long)w[6] | ((unsigned long long)w[7] << 32);
    // pcg_setseq_128_srandom_r: inc = (initseq << 1) | 1; state = 0; step; state += initstate; step
    const unsigned long long inc_hi = (q_hi << 1) | (q_lo >> 63), inc_lo = (q_lo << 1) | 1ull;
    const unsigned long long m_hi = 2549297995355413924ull, m_lo = 4865540595714422341ull;
    unsigned long long st_hi = inc_hi, st_lo = inc_lo;  // 0 * mult + inc
    st_lo += s_lo;
    st_hi += s_hi + (st_lo < s_lo ? 1ull : 0ull);
    unsigned long long ph, pl;
    mul128(st_hi, st_lo, m_hi, m_lo, ph, pl);
    st_lo = pl + inc_lo;
    st_hi = ph + inc_hi + (st_lo < pl ? 1ull : 0ull);
    P.rng[(long long)e * 4 + 0] = st_hi;
    P.rng[(long long)e * 4 + 1] = st_lo;
    P.rng[(long long)e * 4 + 2] = inc_hi;
    P.rng[(long long)e * 4 + 3] = inc_lo;
}

// ------------------------------------------------------------------------------------------
// host-side dispatch over the instantiated kernels
// ------------------------------------------------------------------------------------------
typedef void (*EnvKernel)(const DevParams);

template <int KT, int ST, bool EXACT, int KIND, int NT>
static EnvKernel pick_small(int norm_mode, bool step, bool dr) {
    if (dr)  // domain randomisation: norm_mode 0, runtime N
        return step ? swarm_env_kernel_small<KT, ST, EXACT, 0, KIND, kSmallStep, 0, true>
                    : swarm_env_kernel_small<KT, ST, EXACT, 0, KIND, kSmallAux, 0, true>;
    if (norm_mode == 0)
        return step ? swarm_env_kernel_small<KT, ST, EXACT, 0, KIND, kSmallStep, NT, false>
                    : swarm_env_kernel_small<KT, ST, EXACT, 0, KIND, kSmallAux, 0, false>;
    return step ? swarm_env_kernel_small<KT, ST, EXACT, 1, KIND, kSmallStep, 0, false>
                : swarm_env_kernel_small<KT, ST, EXACT, 1, KIND, kSmallAux, 0, false>;
}

template <int KT, int ST, bool EXACT, int KIND>
static EnvKernel pick_large(int norm_mode, bool dr) {
    if (dr) return swarm_env_kernel<KT, ST, EXACT, 0, KIND, false, true>;   // domain randomisation: norm_mode 0
    return norm_mode == 0 ? swarm_env_kernel<KT, ST, EXACT, 0, KIND, false, false>
                          : swarm_env_kernel<KT, ST, EXACT, 1, KIND, false, false>;
}

static EnvKernel resolve(const DevParams& p, int norm_mode, int env_kind) {
    const bool small_n = p.N <= 32;
    const bool step = p.mode == kModeStep;
    const bool dr = p.dr_enabled != 0;
    if (env_kind == SWARM_KIND_SWARM) {
        if (p.K == 3 && p.S == 4) {
            if (!small_n) return pick_large<3, 4, true, SWARM_KIND_SWARM>(norm_mode, dr);
            // (N = 32 measured faster on the runtime-N instantiation: 9.6e9 vs 9.1e9 agent-steps/s)
            if (p.N == 16) return pick_small<3, 4, true, SWARM_KIND_SWARM, 16>(norm_mode, step, dr);
            if (p.N == 8) return pick_small<3, 4, true, SWARM_KIND_SWARM, 8>(norm_mode, step, dr);
            return pick_small<3, 4, true, SWARM_KIND_SWARM, 0>(norm_mode, step, dr);
        }
        if (!small_n) return pick_large<SWARM_MAX_NEIGHBOR_K, SWARM_MAX_SENSED, false, SWARM_KIND_SWARM>(norm_mode, dr);
        return pick_small<SWARM_MAX_NEIGHBOR_K, SWARM_MAX_SENSED, false, SWARM_KIND_SWARM, 0>(norm_mode, step, dr);
    }
    if (env_kind == SWARM_KIND_PHYSICS) {  // point-mass DronePhysicsEnv
        if (p.K == 3 && p.S == 4) {
            if (!small_n) return pick_large<3, 4, true, SWARM_KIND_PHYSICS>(norm_mode, dr);
            return pick_small<3, 4, true, SWARM_KIND_PHYSICS, 0>(norm_mode, step, dr);
        }
        if (!small_n) return pick_large<SWARM_MAX_NEIGHBOR_K, SWARM_MAX_SENSED, false, SWARM_KIND_PHYSICS>(norm_mode, dr);
        return pick_small<SWARM_MAX_NEIGHBOR_K, SWARM_MAX_SENSED, false, SWARM_KIND_PHYSICS, 0>(norm_mode, step, dr);
    }
    if (p.S == 4) return pick_small<1, 4, true, SWARM_KIND_SINGLE, 1>(norm_mode, step, dr);
    return pick_small<1, SWARM_MAX_SENSED, false, SWARM_KIND_SINGLE, 0>(norm_mode, step, dr);
}

cudaError_t launch_env_kernel(const DevParams& p, int norm_mode, int env_kind, int grid, size_t smem_bytes,
                              cudaStream_t stream) {
    EnvKernel k = resolve(p, norm_mode, env_kind);
    cudaError_t err = ensure_dynamic_smem(reinterpret_cast<const void*>(k), smem_bytes);
    if (err != cudaSuccess) return err;
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)grid);
    lc.blockDim = dim3((unsigned)kThreadsPerCta);
    lc.dynamicSmemBytes = smem_bytes;
    lc.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    return cudaLaunchKernelEx(&lc, k, p);
}

cudaError_t env_kernel_occupancy(const DevParams& p, int norm_mode, int env_kind, size_t smem_bytes,
                                 int* blocks_per_sm) {
    EnvKernel k = resolve(p, norm_mode, env_kind);
    cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (err != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k, kThreadsPerCta, smem_bytes);
}

cudaError_t launch_seed_kernel(const DevParams& p, cudaStream_t stream) {
    const int threads = 128;
    swarm_seed_kernel<<<(p.E + threads - 1) / threads, threads, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace swarm
