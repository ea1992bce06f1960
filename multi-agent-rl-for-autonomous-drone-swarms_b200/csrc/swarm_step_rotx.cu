// swarm_step_rotx.cu -- rotation-pass step / auto-reset kernels for the dense swarms: N = 64 / 128 drones
// (BASELINE config 5), K = 3, S = 4, M a multiple of 4, norm_mode 0; DR = domain randomisation (DESIGN.md 8: per-episode
// dynamics constants, thrust / sensor noise, control delay -- same bits as the general kernels and the oracle).
// Reference: DroneSwarmEnv.step / reset, src/swarm_marl/envs/drone_swarm_env.py:92-174, 65-90.
//
// Same scheme as swarm_step_rot.cu (read its header first), with NS = N / 32 drones per lane:
// a warp owns ONE env, lane l holds drones s * 32 + l (slot s).  In round r = 1 .. 16 lane l meets lane
// l + r: it evaluates the NS x NS distances between its drones and that lane's once and hands each to the
// partner with one SHFL; round 0 covers the pairs inside a lane.  Keys carry log2(N) index bits; the 4
// smallest per drone are kept by the min/max merge network.  The rounds are a rolled loop (the body alone
// is ~10 KB of SASS) and the per-drone tail (neighbour picks, obstacles, observation row, reward) is ONE
// copy of code executed NS times over register arrays that are rotated between the passes, so the
// kernel stays inside the instruction cache.
#include <type_traits>

// float32 -> float64 by two integer ops instead of F2F (swarm_rot_common.cuh): with 6 conversions per pair the quarter-rate
// conversion unit is ~60 % busy at N = 128 and stalls the issue (MIO throttle 17 %); measured +3.5 % here, neutral at N <= 32
#define SWARM_ROT_INT_CVT 1
#include "swarm_rot_common.cuh"

namespace swarm {

// CTAs per SM (4 warps each): the step launch runs best with 3 (157 registers, no spills: +6 % at world 70 over
// 4 CTAs of 128 registers with ~20 spilled), the lighter reset launch with 4 (124 registers; +3 % at world 20)
#ifndef SWARM_ROTX_MINB_STEP
#define SWARM_ROTX_MINB_STEP 3
#endif
#ifndef SWARM_ROTX_MINB_RESET
#define SWARM_ROTX_MINB_RESET 4
#endif
// 0 (default): pos4 / vel4 / actions are prefetched by TMA into a per-warp inbox (14.8 KB of shared memory per
// warp at N = 128: 3 CTAs of 161 registers per SM);  1: they are read straight from global memory at the top
// of an item (9.2 KB, 4 CTAs of 128 registers) -- measured 6-8 % slower (spills, exposed load latency)
#ifndef SWARM_ROTX_DIRECT
#define SWARM_ROTX_DIRECT 0
#endif
// step launch: the rounds run on packed float32x2 instructions (FADD2 / FMUL2 / FFMA2, same roundings) like the N <= 32
// kernel -- (x, y) and (z, .) of a coordinate difference are one packed subtract + one packed multiply each, the square
// roots of two distances four packed operations; distances travel NEGATED (see neg_sqrt_rn_fast2).  The velocities and
// previous goal distances (16 values per lane at N = 128) wait in shared memory during the pass, which pays for the
// registers of the packed operands.
#ifndef SWARM_ROTX_PACKED
#define SWARM_ROTX_PACKED 1
#endif
constexpr int kXWarps = 4;  // warps per CTA

__host__ __device__ constexpr int rotx_envbox_bytes(int M, bool dr) { return 16 * (1 + M) + 16 + (dr ? 32 : 0); }
// per warp: mbarriers (16) | agent inbox pos4[N] vel4[N] actions[3N] | env inbox x 2 | position table
// (N float4; not doubled: the partner lane index is masked instead, which lets 4 CTAs = 16 warps fit an SM) |
// obs tile (one slot at a time)
__host__ __device__ constexpr int rotx_smem_per_warp(int N, int M, bool dr, bool step) {
    return 16 + (SWARM_ROTX_DIRECT ? 0 : 44 * N) + 2 * rotx_envbox_bytes(M, dr) + (N / 32) * 32 * 16 + kTileBytes;
}

namespace {

template <int NS, typename T>
__device__ __forceinline__ void rotate(T (&a)[NS]) {
    const T t = a[0];
#pragma unroll
    for (int s = 0; s + 1 < NS; ++s) a[s] = a[s + 1];
    a[NS - 1] = t;
}

}  // namespace

template <int NS, int MT, int MODE, bool DR>
__global__ void __launch_bounds__(kXWarps * 32, MODE == 0 ? SWARM_ROTX_MINB_STEP : SWARM_ROTX_MINB_RESET)
swarm_step_rotx_kernel(const DevParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int N = 32 * NS;
    constexpr unsigned IDX = N - 1;  // index bits of a neighbour key
    constexpr bool STEP = MODE == 0;
    const int warp = __shfl_sync(FULL_MASK, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const int M = MT ? MT : P.M;
    const int envbox_bytes = rotx_envbox_bytes(M, DR);
    constexpr int kAgentBox = SWARM_ROTX_DIRECT ? 0 : 44 * N;
    constexpr bool kPacked = SWARM_ROTX_PACKED && STEP;
    const int per_warp = 16 + kAgentBox + 2 * envbox_bytes + NS * 512 + kTileBytes;
    unsigned char* wslice = smem_raw + (size_t)warp * per_warp;
    const unsigned bar0 = smem_u32(wslice);
    const float4* in_pos = reinterpret_cast<const float4*>(wslice + 16);       // pos4[N] | vel4[N] | actions[3N]
    unsigned char* envbox0 = wslice + 16 + kAgentBox;
    float4* tab2 = reinterpret_cast<float4*>(wslice + 16 + kAgentBox + 2 * envbox_bytes);   // [NS][32]: drone j at tab2[j]; .w = drone index
    float* tile = reinterpret_cast<float*>(wslice + 16 + kAgentBox + 2 * envbox_bytes + NS * 512);
    unsigned long long* wstats =
        reinterpret_cast<unsigned long long*>(smem_raw + (size_t)kXWarps * per_warp) + warp * SWARM_STATS_WORDS;
    if (lane < SWARM_STATS_WORDS) wstats[lane] = 0ull;
    float* srow = tile + lane * kD;
    // kPacked: the obs tile is idle during the rotation pass -- velocities / previous goal distances wait there,
    // [4 * NS][32] floats, this lane's column (written once the previous item's tile has left, read back before the tail)
    float* const vstash = tile + lane;

    asm volatile("griddepcontrol.wait;" ::: "memory");  // programmatic dependent launch (see swarm_step_rot.cu)
    // auto-reset hand-over: list (epoch & 1) is appended to by the step launch, list ((epoch - 1) & 1) is walked by
    // the reset launch behind it (swarm_internal.h)
    const unsigned epoch = *reinterpret_cast<const volatile unsigned*>(P.reset_epoch);
    const unsigned lpar = STEP ? (epoch & 1u) : ((epoch - 1u) & 1u);
    unsigned* const rcount = P.reset_count + lpar;
    int* const rlist = P.reset_list + lpar * P.reset_list_stride;
    const int n_iter = STEP ? P.n_groups : (int)*reinterpret_cast<const volatile unsigned*>(rcount);
    unsigned* const queue = P.work_counter + (STEP ? 0 : 2);
    if (lane == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    // env inbox: goal4 | obst4[M] | step_count | ep_return | (DR) this episode's constants, 2 x float4
    const int obst_off = 16, sc_off = 16 * (1 + M), dr_off = 16 * (1 + M) + 16;
    auto issue = [&](int item, int buf) {
        if (!STEP) return;
        const int env0 = P.env_begin + item;
        if (lane == 0) {
            const unsigned bar = bar0 + 8 * buf;
            const unsigned dsta = bar0 + 16;
            const unsigned dst = smem_u32(envbox0 + (size_t)buf * envbox_bytes);
            const long long a0 = (long long)env0 * N;
            mbar_expect_tx(bar, (SWARM_ROTX_DIRECT ? 0u : (unsigned)N * 44u) + 16u + 16u * M + (DR ? 32u : 0u));
            if (!SWARM_ROTX_DIRECT) {
                bulk_g2s(dsta, P.pos4 + a0, N * 16u, bar);
                bulk_g2s(dsta + N * 16, P.vel4 + a0, N * 16u, bar);
                bulk_g2s(dsta + N * 32, P.actions + a0 * 3, N * 12u, bar);
            }
            bulk_g2s(dst, P.goal4 + env0, 16u, bar);
            bulk_g2s(dst + obst_off, P.obst4 + (long long)env0 * M, (unsigned)M * 16u, bar);
            if (DR) bulk_g2s(dst + dr_off, P.dr_params + (long long)env0 * 2, 32u, bar);
            cp_async4(dst + sc_off, P.step_count + env0);
            cp_async4(dst + sc_off + 4, P.ep_return + env0);
        }
        cp_async_commit();
    };
    const int warps_total = gridDim.x * kXWarps;
    int it = blockIdx.x * kXWarps + warp;
    if (it < n_iter) issue(it, 0);
    unsigned phase = 0;
    int buf = 0;

    while (it < n_iter) {
        // dynamic item queue in both launches (an item is >= 10k warp instructions and a warp sees only ~5 of them,
        // so a static stride would leave a fifth of the warps one item short)
        int it_next = 0;
        if (lane == 0) it_next = (int)atomicAdd(queue, 1u);   // raw: "+ warps_total" placed here would wait for the atomic
        const int env = STEP ? P.env_begin + it : rlist[it];
        const int a0 = env * N;
        unsigned char* ib = envbox0 + (size_t)buf * envbox_bytes;
        float4* tgoal = reinterpret_cast<float4*>(ib);
        float4* tobs = reinterpret_cast<float4*>(ib + obst_off);

        float px[NS], py[NS], pz[NS], vx[NS], vy[NS], vz[NS], prev_d[NS];
        bool alive[NS];
        float gx, gy, gz;
        int sc = 0;
        // per-env dynamics constants: the config's, or this episode's randomised ones
        float c_amax = P.amax, c_vmax = P.vmax, c_dt = P.dt, c_bound = P.bound, c_thr_obst = P.thr_obst;
        unsigned ekey = 0u;
        int ctrl_delay = 0;
        const unsigned genv = DR ? (unsigned)(P.env_index_base + env) : 0u;
        if (STEP) {
            float4 lp[NS], lv[NS];
            float la[NS][3];
            if (SWARM_ROTX_DIRECT) {  // coalesced loads, issued together before the inbox wait
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    lp[s] = P.pos4[a0 + s * 32 + lane];
                    lv[s] = P.vel4[a0 + s * 32 + lane];
                    const float* ga = P.actions + (long long)(a0 + s * 32 + lane) * 3;
                    la[s][0] = ga[0]; la[s][1] = ga[1]; la[s][2] = ga[2];
                }
            }
            cp_async_wait_all();
            mbar_wait(bar0 + 8 * buf, (phase >> buf) & 1u);
            phase ^= 1u << buf;
            __syncwarp();
            for (int idx = lane; idx < M; idx += 32) reinterpret_cast<unsigned*>(tobs)[idx * 4 + 3] = (unsigned)idx;
            const float4 g4 = tgoal[0];
            gx = g4.x; gy = g4.y; gz = g4.z;
            sc = reinterpret_cast<const int*>(ib + sc_off)[0];
            if (DR) {
                const float4* drp = reinterpret_cast<const float4*>(ib + dr_off);
                const float4 d0 = drp[0], d1 = drp[1];
                c_amax = d0.x; c_vmax = d0.y; c_dt = d0.z; c_bound = d0.w;
                c_thr_obst = d1.x; ekey = __float_as_uint(d1.y);
                ctrl_delay = (int)d1.w;
            }
            const float* act = reinterpret_cast<const float*>(in_pos + 2 * N);
            unsigned nan_n = 0u;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const float4 p = SWARM_ROTX_DIRECT ? lp[s] : in_pos[s * 32 + lane];
                float4 v = SWARM_ROTX_DIRECT ? lv[s] : in_pos[N + s * 32 + lane];
                float ax = SWARM_ROTX_DIRECT ? la[s][0] : act[(s * 32 + lane) * 3 + 0];
                float ay = SWARM_ROTX_DIRECT ? la[s][1] : act[(s * 32 + lane) * 3 + 1];
                float az = SWARM_ROTX_DIRECT ? la[s][2] : act[(s * 32 + lane) * 3 + 2];
                alive[s] = p.w != 0.0f;
                px[s] = p.x; py[s] = p.y; pz[s] = p.z;
                prev_d[s] = norm1d<0>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));  // :98-101
                if (alive[s]) {  // integrate (:103-111)
                    if (DR && P.dr_delay_hist > 0) delayed_command(P, env, N, s * 32 + lane, sc, ctrl_delay, ax, ay, az);
                    ax = clipf(ax, -1.0f, 1.0f); ay = clipf(ay, -1.0f, 1.0f); az = clipf(az, -1.0f, 1.0f);
                    nan_n += (ax == ax && ay == ay && az == az) ? 0u : 1u;   // (np.clip lets NaN through; counted)
                    if (DR) {
                        const uint4 r = philox4x32_7(genv, ekey, (unsigned)sc, (unsigned)(s * 32 + lane) | (DR_STREAM_A << 16), P);
                        thrust_noise(P, [=](int f) { return dr_normal(P.dr_qtable, dr_field(r, f)); }, ax, ay, az);
                    }
                    point_mass_step<0>(P, ax, ay, az, c_amax, c_vmax, c_dt, px[s], py[s], pz[s], v.x, v.y, v.z);
                }
                px[s] = clipf(px[s], -c_bound, c_bound);  // wall clip for ALL drones (:113-117)
                py[s] = clipf(py[s], -c_bound, c_bound);
                pz[s] = clipf(pz[s], -c_bound, c_bound);
                vx[s] = v.x; vy[s] = v.y; vz[s] = v.z;
            }
            // NaN-action guard counter (rare: the vote is all a clean step pays): drones, not components -- a lane
            // holds NS drones, so the lanes' counts are summed
            if (__any_sync(FULL_MASK, nan_n != 0u)) {
                const unsigned n = __reduce_add_sync(FULL_MASK, nan_n);
                if (lane == 0) wstats[SWARM_STAT_NAN_ACTIONS] += (unsigned long long)n;
            }
        } else {
            // ================================ reset (:65-80) ================================
            __syncwarp();
            const Pcg64State rng = load_rng(P, env);
            double u_lo = P.rng_lo, u_range = P.rng_range;
            if (DR) {
                const EpisodeDraw ep = draw_episode_constants(P, genv, rng.sl);
                u_lo = ep.u_lo(); u_range = ep.u_range();
                if (lane == 0) {
                    float4 d0, d1;
                    episode_params(P, ep, d0, d1);
                    P.dr_params[(long long)env * 2 + 0] = d0;
                    P.dr_params[(long long)env * 2 + 1] = d1;
                }
                ekey = ep.key;  // (the dynamics constants are not needed to observe)
            }
            // drone j lives at [slot j / 32][lane j % 32]
            reset_env_draws<4>(
                P, lane, N, rng, u_lo, u_range, [=](int j) { return reinterpret_cast<float*>(tab2 + j); },
                [=]() { return reinterpret_cast<float*>(tgoal); }, [=](int m) { return reinterpret_cast<float*>(tobs + m); });
            if (lane == 0) {
                reset_env_finish(P, env, rng);
                reinterpret_cast<float*>(tgoal)[3] = 0.0f;
            }
            for (int k = lane; k < M; k += 32) reinterpret_cast<unsigned*>(tobs + k)[3] = (unsigned)k;
            __syncwarp();
            if (lane == 0) P.goal4[env] = tgoal[0];
            for (int idx = lane; idx < M; idx += 32) {
                const float4 o = tobs[idx];
                P.obst4[(long long)env * M + idx] = make_float4(o.x, o.y, o.z, 0.0f);
            }
            const float4 g4 = tgoal[0];
            gx = g4.x; gy = g4.y; gz = g4.z;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const float4 p = tab2[s * 32 + lane];
                px[s] = p.x; py[s] = p.y; pz[s] = p.z;
                vx[s] = vy[s] = vz[s] = 0.0f;
                prev_d[s] = 0.0f;
                alive[s] = true;
            }
            __syncwarp();
        }

        // position table: tab2[j] is drone j (slot j / 32, lane j % 32); .w = drone index
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const float4 t = make_float4(px[s], py[s], pz[s], __int_as_float(s * 32 + lane));
            tab2[s * 32 + lane] = t;
        }
        bool all_alive_l = true;
        int n_alive_l = 0;
#pragma unroll
        for (int s = 0; s < NS; ++s) { all_alive_l = all_alive_l && alive[s]; n_alive_l += alive[s] ? 1 : 0; }
        const bool all_alive = __all_sync(FULL_MASK, all_alive_l);
        unsigned amask[NS];  // bit l of amask[s]: drone s * 32 + l is active
#pragma unroll
        for (int s = 0; s < NS; ++s) amask[s] = __ballot_sync(FULL_MASK, alive[s]);
        int n_alive_env = n_alive_l;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) n_alive_env += __shfl_xor_sync(FULL_MASK, n_alive_env, off);
        if (lane == 0) bulk_wait_read0();
        __syncwarp();
        it_next = warps_total + __shfl_sync(FULL_MASK, it_next, 0);
        if (STEP && it_next < n_iter) issue(it_next, buf ^ 1);
        if (kPacked) {   // not needed before the per-drone tail: out of the registers during the rotation pass
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                vstash[(4 * s + 0) * 32] = vx[s]; vstash[(4 * s + 1) * 32] = vy[s];
                vstash[(4 * s + 2) * 32] = vz[s]; vstash[(4 * s + 3) * 32] = prev_d[s];
            }
        }

        // ================= rotation pass =================
        // MASKED = some drone of the env is parked (it reached the goal earlier): neighbour keys still cover every
        // drone, but the formation sum runs over ACTIVE partners only -- each term is multiplied by the partner's
        // 0.0 / 1.0 flag (the float64 sum is order-free, DESIGN.md 4.1, so the masked pass gives the reference's
        // value too); collisions among active drones are read off the three picks in the tail
        unsigned k0[NS], k1[NS], k2[NS], k3[NS];
        double acc[NS];
#pragma unroll
        for (int s = 0; s < NS; ++s) { k0[s] = k1[s] = k2[s] = k3[s] = ~0u; acc[s] = 0.0; }
        bool bad = false;
        auto rotation_pass = [&](auto masked_tag) {
            constexpr bool MASKED = decltype(masked_tag)::value;
            const double d_star = P.d_star;
            constexpr unsigned KEYMASK = ~IDX & 0x7fffffffu;   // packed rounds: keys drop the sign of the negated distance
            f32x2 pxy[NS], pz0[NS];
#ifndef SWARM_ROTX_PACKED_RESET
#define SWARM_ROTX_PACKED_RESET 1
#endif
            constexpr bool kPackedReset = SWARM_ROTX_PACKED && SWARM_ROTX_PACKED_RESET && !STEP;   // packed differences / squares only
            if (kPacked || kPackedReset) {
#pragma unroll
                for (int s = 0; s < NS; ++s) { pxy[s] = pack2(px[s], py[s]); pz0[s] = pack2(pz[s], 0.0f); }
            }
            // round 0: the pairs inside a lane
#pragma unroll
            for (int s = 0; s < NS; ++s)
#pragma unroll
                for (int s2 = s + 1; s2 < NS; ++s2) {
                    // reset launch (no reward, so no formation sum and no exact distance per pair): the keys are built
                    // from a plain float32 sum of squares -- monotone in the distance up to 2 ulp, which the widened
                    // 3rd/4th-key check of the tail covers; the picks' distances are recomputed exactly there
                    const float sq = STEP ? sumsq1d_fast(__fsub_rn(px[s2], px[s]), __fsub_rn(py[s2], py[s]), __fsub_rn(pz[s2], pz[s]))
                                          : sumsq_axis(__fsub_rn(px[s2], px[s]), __fsub_rn(py[s2], py[s]), __fsub_rn(pz[s2], pz[s]));
                    const float d = STEP ? sqrt_rn_fast(sq) : sq;
                    const double t = STEP ? fabs(__dsub_rn(f64_of_pos_f32<(SWARM_ROT_CVT_FORM & 1) != 0>(d), d_star)) : 0.0;
                    merge1((__float_as_uint(d) & ~IDX) | (unsigned)(s2 * 32 + lane), k0[s], k1[s], k2[s], k3[s]);
                    merge1((__float_as_uint(d) & ~IDX) | (unsigned)(s * 32 + lane), k0[s2], k1[s2], k2[s2], k3[s2]);
                    if (STEP) {
                        acc[s] = __dadd_rn(acc[s], MASKED ? __dmul_rn(t, alive[s2] ? 1.0 : 0.0) : t);
                        acc[s2] = __dadd_rn(acc[s2], MASKED ? __dmul_rn(t, alive[s] ? 1.0 : 0.0) : t);
                    }
                }
            // one round: my NS drones against the NS drones of lane l + r; LAST = round 16, where lanes l and
            // l + 16 both evaluate their pairs and nothing is handed over
            auto round = [&](int r, auto last_tag) {
                constexpr bool LAST = decltype(last_tag)::value;
                const int lb = (lane - r) & 31;
                const float4* tq = tab2 + ((lane + r) & 31);
                unsigned kf[NS][NS], kb[NS][NS];
                double mf[NS], mb[NS];  // MASKED: 1.0 / 0.0 = partner (s2, lane + r) / (s, lane - r) is active
                if (MASKED) {
#pragma unroll
                    for (int u = 0; u < NS; ++u) {
                        mf[u] = ((amask[u] >> ((lane + r) & 31)) & 1u) ? 1.0 : 0.0;
                        mb[u] = ((amask[u] >> lb) & 1u) ? 1.0 : 0.0;
                    }
                }
#pragma unroll
                for (int s2 = 0; s2 < NS; ++s2) {
                    const float4 q = tq[s2 * 32];
                    if (kPacked) {
                        // NS distances to q: packed differences / squares, float64 accumulate (BLAS sdot), two packed
                        // square roots at a time; nd[] = MINUS the distance
                        float nd[NS];
#pragma unroll
                        for (int s = 0; s < NS; s += 2) {
                            float ax2, ay2, az2, bx2, by2, bz2;
                            sq_diff3(q, pxy[s], pz0[s], ax2, ay2, az2);
                            sq_diff3(q, pxy[s + 1], pz0[s + 1], bx2, by2, bz2);
                            unpack2(neg_sqrt_rn_fast2(neg_sumsq1d_of_squares(ax2, ay2, az2), neg_sumsq1d_of_squares(bx2, by2, bz2)),
                                    nd[s], nd[s + 1]);
                        }
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            kf[s][s2] = and_or<KEYMASK>(__float_as_uint(nd[s]), __float_as_uint(q.w));
                            const double t = fabs(__dadd_rn(f64_of_neg_f32(nd[s]), d_star));   // |(-d) + d*|
                            acc[s] = __dadd_rn(acc[s], MASKED ? __dmul_rn(t, mf[s2]) : t);
                            if (!LAST) {
                                const float db = __shfl_sync(FULL_MASK, nd[s], lb);  // -d(drone s of lane l - r, my drone s2)
                                kb[s][s2] = and_or<KEYMASK>(__float_as_uint(db), (unsigned)(s * 32 + lb));
                                const double tb = fabs(__dadd_rn(f64_of_neg_f32(db), d_star));
                                acc[s2] = __dadd_rn(acc[s2], MASKED ? __dmul_rn(tb, mb[s]) : tb);
                            }
                        }
                    }
#pragma unroll
                    for (int s = 0; s < (kPacked ? 0 : NS); ++s) {   // (scalar rounds: the reset launch, or SWARM_ROTX_PACKED = 0)
                        float sq;
                        if (kPackedReset) {   // sumsq_axis with packed differences / squares (same operations, same order)
                            float sx, sy, sz;
                            sq_diff3(q, pxy[s], pz0[s], sx, sy, sz);
                            sq = __fadd_rn(__fadd_rn(sx, sy), sz);
                        } else {
                            sq = STEP ? sumsq1d_fast(__fsub_rn(q.x, px[s]), __fsub_rn(q.y, py[s]), __fsub_rn(q.z, pz[s]))
                                      : sumsq_axis(__fsub_rn(q.x, px[s]), __fsub_rn(q.y, py[s]), __fsub_rn(q.z, pz[s]));
                        }
                        const float d = STEP ? sqrt_rn_fast(sq) : sq;  // (reset launch: key = squared distance, see round 0)
                        kf[s][s2] = and_or<~IDX>(__float_as_uint(d), __float_as_uint(q.w));
                        if (STEP) {
                            const double t = fabs(__dsub_rn(f64_of_pos_f32<(SWARM_ROT_CVT_FORM & 1) != 0>(d), d_star));
                            acc[s] = __dadd_rn(acc[s], MASKED ? __dmul_rn(t, mf[s2]) : t);
                        }
                        if (!LAST) {
                            const float db = __shfl_sync(FULL_MASK, d, lb);  // d(drone s of lane l - r, my drone s2)
                            kb[s][s2] = and_or<~IDX>(__float_as_uint(db), (unsigned)(s * 32 + lb));
                            if (STEP) {
                                const double tb = fabs(__dsub_rn(f64_of_pos_f32<(SWARM_ROT_CVT_FORM & 2) != 0>(db), d_star));
                                acc[s2] = __dadd_rn(acc[s2], MASKED ? __dmul_rn(tb, mb[s]) : tb);
                            }
                        }
                    }
                }
                // my drone s: forward keys kf[s][*]; my drone s2: backward keys kb[*][s2]
#pragma unroll
                for (int s = 0; s < NS; ++s)
#pragma unroll
                    for (int u = 0; u < NS; u += 2) {
                        merge2(kf[s][u], kf[s][u + 1], k0[s], k1[s], k2[s], k3[s]);
                        if (!LAST) merge2(kb[u][s], kb[u + 1][s], k0[s], k1[s], k2[s], k3[s]);
                    }
            };
#pragma unroll 1
            for (int r = 1; r < 16; ++r) round(r, std::false_type{});
            round(16, std::true_type{});
#pragma unroll
            for (int s = 0; s < NS; ++s)
                // (keys sharing a bucket are settled per drone in the tail: among keys 0-2 only the ORDER is open,
                //  a 3rd/4th-key collision triggers an exact neighbour rescan of that slot pass; only a distance
                //  below 2^-14 -- fast sqrt / exact-sum preconditions -- or a NaN position sends the whole item to the
                //  exact path.  The integer float32 -> float64 conversions of the rounds turn NaN into a finite value,
                //  so a NaN drone does not show up as a NaN formation sum here: its position is checked instead)
                bad = bad || (STEP && (!(acc[s] == acc[s]) || k0[s] < 0x38800000u ||
                                       !(px[s] == px[s] && py[s] == py[s] && pz[s] == pz[s])));
        };
        if (all_alive) rotation_pass(std::false_type{});
        else rotation_pass(std::true_type{});
        const bool exact = __any_sync(FULL_MASK, bad);
        if (kPacked) {
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                vx[s] = vstash[(4 * s + 0) * 32]; vy[s] = vstash[(4 * s + 1) * 32];
                vz[s] = vstash[(4 * s + 2) * 32]; prev_d[s] = vstash[(4 * s + 3) * 32];
            }
        }

        // ================= per-drone tail: one copy of code, NS passes over rotated register arrays =================
        double rew[NS];
        float cd[NS];
        unsigned fl[NS];  // bit 0 reached, bit 1 collided
        // step launch with auto-reset: the env is certain to be re-drawn (no active drone left, or the time limit is
        // reached on this step; collisions are added slot pass by slot pass) -- its obs rows are not stored
        bool doomed = STEP && P.auto_reset && (n_alive_env == 0 || sc + 1 >= P.max_steps);
#pragma unroll 1
        for (int s = 0; s < NS; ++s) {
            if (s > 0) {  // the previous slot's tile must have left shared memory before this pass scribbles on it
                if (lane == 0) bulk_wait_read0();
                __syncwarp();
            }
            const float p_x = px[0], p_y = py[0], p_z = pz[0];
            const int me = s * 32 + lane;
            float nd[3]; int nj[3];
            bool pair_hit = false;
            double form_sum = 0.0;
            int form_n = 0;
            if (!exact) {
                const unsigned kk[3] = {k0[0], k1[0], k2[0]};
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    nj[q] = (int)(kk[q] & IDX);
                    const float4 t = tab2[nj[q]];
                    nd[q] = norm1d<0>(__fsub_rn(t.x, p_x), __fsub_rn(t.y, p_y), __fsub_rn(t.z, p_z));
                }
                // exact (distance, index) order of the three picks -- the reference's argsort order
                auto cex3 = [&](int a, int b) {
                    const bool sw = nd[a] > nd[b] || (nd[a] == nd[b] && nj[a] > nj[b]);
                    const float td = sw ? nd[b] : nd[a], tD = sw ? nd[a] : nd[b];
                    const int tj = sw ? nj[b] : nj[a], tJ = sw ? nj[a] : nj[b];
                    nd[a] = td; nd[b] = tD; nj[a] = tj; nj[b] = tJ;
                };
                cex3(0, 1); cex3(1, 2); cex3(0, 1);
                // (reset launch: approximate squared-distance keys -> anything within one bucket of the 3rd key is open)
                constexpr int SH = NS == 4 ? 7 : 6;
                if (__any_sync(FULL_MASK, STEP ? (k2[0] ^ k3[0]) <= IDX : ((k3[0] >> SH) - (k2[0] >> SH)) <= 1u)) {
                    // some drone's 3rd and 4th key share a bucket: which candidates make its first three is open.
                    // Redo the neighbour selection of this slot pass exactly (ascending j, strict '<'); the
                    // formation sum is exact regardless.
#pragma unroll
                    for (int q = 0; q < 3; ++q) { nd[q] = TOPK_EMPTY; nj[q] = 0; }
#pragma unroll 1
                    for (int j = 0; j < N; ++j) {
                        if (j == me) continue;
                        const float4 q = tab2[j];
                        topk_insert<3>(norm1d<0>(__fsub_rn(q.x, p_x), __fsub_rn(q.y, p_y), __fsub_rn(q.z, p_z)), j, nd, nj);
                    }
                }
                form_sum = acc[0];
                if (all_alive) {
                    pair_hit = nd[0] <= P.thr_pair;
                    form_n = N - 1;
                } else {
                    // collisions count among ACTIVE drones only (:202-207): an active pick within the threshold
                    // settles it; three parked picks within the threshold leave it open -> scan the active drones
                    auto active = [&](int j) {
                        unsigned am = 0u;
#pragma unroll
                        for (int u = 0; u < NS; ++u) am = (j >> 5) == u ? amask[u] : am;
                        return ((am >> (j & 31)) & 1u) != 0u;
                    };
                    bool open = alive[0];
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const bool within = nd[q] <= P.thr_pair;
                        pair_hit = pair_hit || (within && active(nj[q]));
                        open = open && within;
                    }
                    open = open && !pair_hit;
                    if (__any_sync(FULL_MASK, open)) {
#pragma unroll 1
                        for (int j = 0; j < N; ++j) {
                            if (j == me || !active(j)) continue;
                            const float4 q = tab2[j];
                            pair_hit = pair_hit || norm1d<0>(__fsub_rn(q.x, p_x), __fsub_rn(q.y, p_y), __fsub_rn(q.z, p_z)) <= P.thr_pair;
                        }
                    }
                    pair_hit = pair_hit && alive[0];
                    form_n = alive[0] ? n_alive_env - 1 : 0;
                }
            } else {
                // exact path: the reference's loops as written (ascending j, strict '<', active pairs, numpy's
                // pairwise summation order)
#pragma unroll
                for (int q = 0; q < 3; ++q) { nd[q] = TOPK_EMPTY; nj[q] = 0; }
                const int n_f = alive[0] ? n_alive_env - 1 : 0;
                const int nf8 = n_f >= 8 ? (n_f & ~7) : 0;
                double r8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) r8[u] = 0.0;
                double res = 0.0;
                bool tree_done = false;
                int cnt = 0;
#pragma unroll 1
                for (int j = 0; j < N; ++j) {
                    if (j == me) continue;
                    unsigned am = 0u;
#pragma unroll
                    for (int u = 0; u < NS; ++u) am = (j >> 5) == u ? amask[u] : am;
                    const bool aj = (am >> (j & 31)) & 1u;
                    const float4 q = tab2[j];
                    const float d = norm1d<0>(__fsub_rn(q.x, p_x), __fsub_rn(q.y, p_y), __fsub_rn(q.z, p_z));
                    topk_insert<3>(d, j, nd, nj);
                    if (alive[0] && aj) {
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

            // ---- obstacles (:273-291, :190-200)
            float od[4]; int om[4];
            bool bad_o = false;
            {
                unsigned o0, o1, o2, o3, o4;
                if (MT == 8 || MT == 4) {
                    unsigned ok[MT ? MT : 1];
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
                        const float4 o = tobs[m];
                        const float sq = sumsq_axis(__fsub_rn(o.x, p_x), __fsub_rn(o.y, p_y), __fsub_rn(o.z, p_z));
                        srow[m] = sq;
                        ok[m] = and_or<~31u>(__float_as_uint(sq), __float_as_uint(o.w));
                    }
                    if (MT == 8) { sort8(reinterpret_cast<unsigned(&)[8]>(ok)); o4 = ok[MT == 8 ? 4 : 0]; }
                    else { sort4(reinterpret_cast<unsigned(&)[4]>(ok)); o4 = ~0u; }
                    o0 = ok[0]; o1 = ok[MT > 1 ? 1 : 0]; o2 = ok[MT > 2 ? 2 : 0]; o3 = ok[MT > 3 ? 3 : 0];
                } else {
                    o0 = o1 = o2 = o3 = o4 = ~0u;
#pragma unroll 1
                    for (int m = 0; m < M; ++m) {
                        const float4 o = tobs[m];
                        const float sq = sumsq_axis(__fsub_rn(o.x, p_x), __fsub_rn(o.y, p_y), __fsub_rn(o.z, p_z));
                        srow[m] = sq;
                        merge1_5(and_or<~31u>(__float_as_uint(sq), __float_as_uint(o.w)), o0, o1, o2, o3, o4);
                    }
                }
                bad_o = ((o0 ^ o1) <= 31u) || ((o1 ^ o2) <= 31u) || ((o2 ^ o3) <= 31u) || ((o3 ^ o4) <= 31u);
                const unsigned oo[4] = {o0, o1, o2, o3};
#pragma unroll
                for (int q = 0; q < 4; ++q) { om[q] = (int)(oo[q] & 31u); od[q] = srow[om[q]]; }
                bad_o = bad_o || !(od[0] >= SQRT_FAST_MIN);
#pragma unroll
                for (int q = 0; q < 4; ++q) od[q] = sqrt_rn_fast(od[q]);
                const float d4 = o4 != ~0u ? sqrt_rn_fast(srow[o4 & 31u]) : F32_INF;
                bad_o = bad_o || od[0] == od[1] || od[1] == od[2] || od[2] == od[3] || od[3] == d4;
            }
            if (__any_sync(FULL_MASK, bad_o)) {
#pragma unroll
                for (int q = 0; q < 4; ++q) { od[q] = TOPK_EMPTY; om[q] = 0; }
#pragma unroll 1
                for (int m = 0; m < M; ++m) {
                    const float4 o = tobs[m];
                    const float d = __fsqrt_rn(sumsq_axis(__fsub_rn(o.x, p_x), __fsub_rn(o.y, p_y), __fsub_rn(o.z, p_z)));
                    topk_insert<4>(d, m, od, om);
                }
            }
            const float curr_d = norm1d<0>(__fsub_rn(gx, p_x), __fsub_rn(gy, p_y), __fsub_rn(gz, p_z));

            // ---- per-drone reward pieces (:141-148); env-level flags need every slot: finished below
            double reward = 0.0;
            unsigned f = 0u;
            if (STEP) {
                const bool obst_hit = od[0] <= c_thr_obst;
                const bool reached = alive[0] && curr_d <= P.thr_goal;
                const bool collided = alive[0] && (obst_hit || pair_hit);
                if (alive[0]) {
                    const double progress = __dmul_rn(__dsub_rn((double)prev_d[0], (double)curr_d), P.k_p);
                    double pen = 0.0;
                    if (form_n > 0) {
                        const double mean = form_n == N - 1 ? mean_markstein(form_sum, P.n_others, P.inv_n_others)
                                                            : __ddiv_rn(form_sum, (double)form_n);
                        pen = __dmul_rn(P.neg_k_f, mean);
                    }
                    reward = __dadd_rn(progress, pen);
                    if (reached) reward = __dadd_rn(reward, P.r_goal);
                    if (collided) reward = __dadd_rn(reward, P.r_col);
                }
                f = (reached ? 1u : 0u) | (collided ? 2u : 0u);
            }
            // ---- obs row -> tile -> one TMA store per slot (:226-243)
            // (an env that is certain to be re-drawn by the auto-reset behind this launch -- time limit reached, or a
            //  collision seen in this or an earlier slot pass -- does not need this step's rows: the reset launch
            //  writes the new episode's.  At BASELINE's density 97 % of the envs end every step, and their rows were
            //  22 % of the launch's DRAM traffic.  An episode that ends because every drone reached the goal is only
            //  known after the last pass; its rows are written twice, as before.)
            if (STEP && P.auto_reset) doomed = doomed || __any_sync(FULL_MASK, (f & 2u) != 0u);
            if (!doomed) {
                const float4 t0 = tab2[nj[0]], t1 = tab2[nj[1]];
                const float4 t2 = tab2[nj[2]];
                const float4 b0 = tobs[om[0]], b1 = tobs[om[1]], b2 = tobs[om[2]], b3 = tobs[om[3]];
                // DR: sensor noise of the observed state -- the Philox block of counter (its step_count - 1), i.e. the
                // block this step's thrust noise was cut from (a reset observation: step_count 0, counter 0xFFFFFFFF)
                uint4 rA = make_uint4(0, 0, 0, 0);
                if (DR) rA = philox4x32_7(genv, ekey, STEP ? (unsigned)sc : 0xFFFFFFFFu, (unsigned)me | (DR_STREAM_A << 16), P);
                observe_row_k3s4<DR>(P, srow, p_x, p_y, p_z, vx[0], vy[0], vz[0], gx, gy, gz, t0, t1, t2, nd, b0, b1, b2, b3, od,
                                     [=](int f) { return dr_normal(P.dr_qtable, dr_field(rA, f)); });
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    bulk_s2g(P.obs + (long long)(a0 + s * 32) * kD, smem_u32(tile), (unsigned)kTileBytes);
                    bulk_commit();
                }
            }

            rew[0] = reward; cd[0] = curr_d; fl[0] = f;
            rotate<NS>(px); rotate<NS>(py); rotate<NS>(pz); rotate<NS>(vx); rotate<NS>(vy); rotate<NS>(vz);
            rotate<NS>(prev_d); rotate<NS>(alive); rotate<NS>(k0); rotate<NS>(k1); rotate<NS>(k2); rotate<NS>(k3); rotate<NS>(acc);
            rotate<NS>(rew); rotate<NS>(cd); rotate<NS>(fl);
        }

        // ================= env-level flags and outputs (:149-172) =================
        if (STEP) {
            bool col_l = false;
            int cont_l = 0;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                col_l = col_l || (fl[s] & 2u);
                cont_l += (alive[s] && fl[s] == 0u) ? 1 : 0;
            }
            const bool any_col = __any_sync(FULL_MASK, col_l);
            int n_cont = cont_l;
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) n_cont += __shfl_xor_sync(FULL_MASK, n_cont, off);
            const bool env_active = n_alive_env > 0;
            const int sc_new = env_active ? sc + 1 : sc;
            const bool time_limit = env_active && sc_new >= P.max_steps;
            const bool all_reached = n_cont == 0 && !any_col && !time_limit;
            const bool episode_done = all_reached || any_col;
            const bool all_term = env_active ? episode_done : true;
            const bool all_trunc = env_active ? (time_limit && !episode_done) : false;
            const bool ep_over = env_active && (all_term || all_trunc);
            const bool need_reset = P.auto_reset && (ep_over || !env_active);
            float x = 0.0f;  // per-env reward sum: slots in order inside a lane, then a tree over the lanes
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const int a = a0 + s * 32 + lane;
                const bool reached = fl[s] & 1u, collided = fl[s] & 2u, done_agent = fl[s] != 0u;
                const float rew32 = __double2float_rn(rew[s]);
                x = __fadd_rn(x, rew32);
                P.terminated[a] = (alive[s] && done_agent) ? 1 : 0;
                P.truncated[a] = (alive[s] && time_limit && !done_agent) ? 1 : 0;
                const bool valid = alive[s] && !done_agent && !time_limit && !any_col;
                const bool alive_next = ep_over ? false : valid;
                P.reward[a] = rew32;
                if (P.reward64) P.reward64[a] = rew[s];
                P.reached[a] = reached ? 1 : 0;
                P.collision[a] = collided ? 1 : 0;
                if (!need_reset) {
                    P.dist[a] = cd[s];
                    P.obs_valid[a] = valid ? 1 : 0;
                    P.pos4[a] = make_float4(px[s], py[s], pz[s], alive_next ? 1.0f : 0.0f);
                    P.vel4[a] = make_float4(vx[s], vy[s], vz[s], 0.0f);
                    if (P.gs) {
                        float* row = P.gs + (long long)env * P.R;
                        const int i = s * 32 + lane;
                        __stcs(row + 3 * i + 0, px[s]); __stcs(row + 3 * i + 1, py[s]); __stcs(row + 3 * i + 2, pz[s]);
                        __stcs(row + 3 * N + 3 * i + 0, vx[s]); __stcs(row + 3 * N + 3 * i + 1, vy[s]);
                        __stcs(row + 3 * N + 3 * i + 2, vz[s]);
                    }
                }
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) x = __fadd_rn(x, __shfl_down_sync(FULL_MASK, x, off));
            if (lane == 0) {
                P.all_term[env] = all_term ? 1 : 0;
                P.all_trunc[env] = all_trunc ? 1 : 0;
                if (P.reset_mask) P.reset_mask[env] = need_reset ? 1 : 0;
                const float ret = __fadd_rn(reinterpret_cast<const float*>(ib + sc_off)[1], x);
                if (ep_over) {
                    wstats[SWARM_STAT_EPISODES] += 1ull;
                    wstats[SWARM_STAT_LENGTH_SUM] += (unsigned long long)sc_new;
                    reinterpret_cast<double*>(wstats)[SWARM_STAT_RETURN_SUM] += (double)ret;
                    if (all_reached) wstats[SWARM_STAT_SUCCESS] += 1ull;
                    if (any_col) wstats[SWARM_STAT_COLLISION] += 1ull;
                    if (all_trunc) wstats[SWARM_STAT_TIMEOUT] += 1ull;
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
                wstats[SWARM_STAT_AGENT_STEPS] += (unsigned long long)n_alive_env;
                wstats[SWARM_STAT_ENV_STEPS] += env_active ? 1ull : 0ull;
                if (P.auto_reset && need_reset) rlist[atomicAdd(rcount, 1u)] = env;
            }
        } else {
            // reset()'s obs / infos (:82-89); reward / flags of the terminal step stay
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const int a = a0 + s * 32 + lane;
                P.dist[a] = cd[s];
                P.obs_valid[a] = 1;
                P.pos4[a] = make_float4(px[s], py[s], pz[s], 1.0f);
                P.vel4[a] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (P.gs) {
                    float* row = P.gs + (long long)env * P.R;
                    const int i = s * 32 + lane;
                    __stcs(row + 3 * i + 0, px[s]); __stcs(row + 3 * i + 1, py[s]); __stcs(row + 3 * i + 2, pz[s]);
                    __stcs(row + 3 * N + 3 * i + 0, 0.f); __stcs(row + 3 * N + 3 * i + 1, 0.f); __stcs(row + 3 * N + 3 * i + 2, 0.f);
                    if (i == 0) { __stcs(row + 6 * N + 0, gx); __stcs(row + 6 * N + 1, gy); __stcs(row + 6 * N + 2, gz); }
                }
            }
        }
        it = it_next;
        buf ^= 1;
    }
    // (only a step launch with its reset launch behind it -- which waits at its top -- may release its dependents
    //  before it has completed: see swarm_step_rot.cu)
    if (STEP && P.auto_reset) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (lane == 0 && atomicAdd(queue + 1, 1u) == (unsigned)warps_total - 1u) {  // last warp out re-arms the queue
        queue[0] = 0u;
        queue[1] = 0u;
        if (STEP && P.auto_reset) {  // hand the list over, clear the other one for the next step
            P.reset_count[(epoch + 1u) & 1u] = 0u;
            *P.reset_epoch = epoch + 1u;
        }
    }
    if (lane == 0) bulk_wait0();
    __syncwarp();
    if (STEP && P.stats && lane < SWARM_STATS_WORDS) {
        const unsigned long long w = wstats[lane];
        if (lane == SWARM_STAT_RETURN_SUM) {
            const double dv = __longlong_as_double((long long)w);
            if (dv != 0.0) atomicAdd(reinterpret_cast<double*>(P.stats + lane), dv);
        } else if (w) {
            atomicAdd(P.stats + lane, w);
        }
    }
}

// ------------------------------------------------------------------------------------------
typedef void (*RotxKernel)(const DevParams);

template <int NS, bool DR>
static RotxKernel pick_rotx_m(const DevParams& p) {
    const bool reset = p.mode == kModeAutoReset;
    if (p.M == 8) return reset ? swarm_step_rotx_kernel<NS, 8, 1, DR> : swarm_step_rotx_kernel<NS, 8, 0, DR>;
    if (p.M == 4) return reset ? swarm_step_rotx_kernel<NS, 4, 1, DR> : swarm_step_rotx_kernel<NS, 4, 0, DR>;
    return reset ? swarm_step_rotx_kernel<NS, 0, 1, DR> : swarm_step_rotx_kernel<NS, 0, 0, DR>;
}
static RotxKernel pick_rotx(const DevParams& p) {
    const bool dr = p.dr_enabled != 0;
    if (p.N == 128) return dr ? pick_rotx_m<4, true>(p) : pick_rotx_m<4, false>(p);
    if (p.N == 64) return dr ? pick_rotx_m<2, true>(p) : pick_rotx_m<2, false>(p);
    return nullptr;
}

size_t rotx_smem_bytes(const DevParams& p) {
    return (size_t)kXWarps * rotx_smem_per_warp(p.N, p.M, p.dr_enabled != 0, p.mode != kModeAutoReset) +
           (size_t)kXWarps * SWARM_STATS_WORDS * sizeof(unsigned long long);
}
int rotx_warps_per_cta() { return kXWarps; }

cudaError_t launch_rotx_kernel(const DevParams& p, int grid, cudaStream_t stream) {
    RotxKernel k = pick_rotx(p);
    if (!k) return cudaErrorInvalidValue;
    const size_t smem = rotx_smem_bytes(p);
    cudaError_t err = ensure_dynamic_smem(reinterpret_cast<const void*>(k), smem);
    if (err != cudaSuccess) return err;
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)grid);
    lc.blockDim = dim3((unsigned)(kXWarps * 32));
    lc.dynamicSmemBytes = smem;
    lc.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    return cudaLaunchKernelEx(&lc, k, p);
}

cudaError_t rotx_kernel_occupancy(const DevParams& p, int* blocks_per_sm) {
    RotxKernel k = pick_rotx(p);
    if (!k) return cudaErrorInvalidValue;
    const size_t smem = rotx_smem_bytes(p);
    cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k, kXWarps * 32, smem);
}

}  // namespace swarm
