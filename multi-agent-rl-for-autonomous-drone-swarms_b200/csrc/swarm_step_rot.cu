// swarm_step_rot.cu -- the step kernel of the BASELINE swarm shapes: DroneSwarmEnv.step
// (reference src/swarm_marl/envs/drone_swarm_env.py:92-174) for N in {8, 16, 32} drones, K = 3
// neighbours, S = 4 sensed obstacles, M a multiple of 4, norm_mode 0.  Every other shape runs on
// the general kernels of swarm_kernels.cu; the two produce bit-identical results (tests).
//
// Mapping: a warp owns 32 / N env instances, lane = env-local index * N + drone; no block barrier.
//
//   inputs    one lane issues TMA bulk copies (cp.async.bulk, SASS UBLKCP) of the next group's
//             pos4 / vel4 / actions / goal / obstacles into one of two per-warp inboxes, completion
//             on a per-warp mbarrier, while the current group is being processed.
//   pairs     "rotation" pass: in round r (1 .. N/2) lane i evaluates d(i, i+r) once and hands it to
//             lane i+r with one SHFL, so every unordered pair costs one distance evaluation and no
//             shared-memory matrix.  The 3 nearest neighbours are kept as packed keys
//             (distance bits with the low log2(N) bits replaced by the drone index) in a
//             branch-free min/max merge network (VIMNMX3); the 4th key is tracked so that any pair
//             of candidates that the truncation could have mis-ordered is DETECTED, and the warp
//             then redoes the scan on the exact path (same code shape as the reference loop).
//             Formation error sum |d - d*| (float64): every term is a multiple of 2^-37 and the sum
//             stays below 2^16, so float64 addition is exact and the order of np.mean's pairwise
//             summation does not matter (host checks d* and the world size, the kernel checks
//             d >= 2^-14; otherwise the exact path runs).
//   outputs   the 32 x 37 observation tile is staged in shared memory and leaves with ONE TMA bulk
//             store per group; state / flags are float4 / byte stores straight from registers.
#include <type_traits>
#include "swarm_rot_common.cuh"

// programmatic dependent launch of the step / reset kernels (hides the launch latency between them)
#ifndef SWARM_ROT_PDL
#define SWARM_ROT_PDL 1
#endif
// the step launch starts under the previous step's reset launch (see the kernel prologue)
#ifndef SWARM_ROT_OVERLAP
#define SWARM_ROT_OVERLAP 1
#endif
#ifndef SWARM_ROT_EARLY_TRIGGER
#define SWARM_ROT_EARLY_TRIGGER 1
#endif

namespace swarm {


// CTA shape (measured): N = 32 and N = 16 run best as 4 warps x 7 CTAs per SM (72 registers, 28 resident warps,
// 7 per scheduler; N = 16: +4 % over 8 x 3), N = 8 as 8 warps x 3 CTAs (80 registers; 4 x 7 is 5 % slower there).
// With domain randomisation every CTA carries the 2 KB quantile table, and seven copies of it do not fit beside
// 28 warp slices: the DR kernels run the same 28 warps as 4 CTAs of 7 (measured: 7 x 4 0.1620 ms per C4 step,
// 14 x 2 0.1625, 28 x 1 0.1710 -- warps of one CTA start in phase and then contend for the same pipes).
#ifndef SWARM_ROT_W32
#define SWARM_ROT_W32 4
#define SWARM_ROT_B32 7
#endif
// SWARM_ROT_DR_QTAB_GLOBAL = 1: the table is read from global memory (L1) instead, no per-CTA copy (measured slower:
// 0.1571 ms per C4 step as 7 x 4, 0.1557 as 4 x 7 -- which the missing copy makes possible -- against 0.1545)
#ifndef SWARM_ROT_DR_QTAB_GLOBAL
#define SWARM_ROT_DR_QTAB_GLOBAL 0
#endif
#ifndef SWARM_ROT_W32_DR
#define SWARM_ROT_W32_DR 7
#define SWARM_ROT_B32_DR 4
#endif
// N = 32 step launch: the per-env outputs (the __all__ flags, the reset mask, the episode outputs, step count, running
// return, the goal part of global_state: ten stores to seven different arrays) leave as TWO store instructions, lane k
// writing output k through a per-warp pointer table in shared memory, instead of ten stores with their own address
// arithmetic executed by one active lane (dropping that block altogether measured -1.9 % of the C4 step)
#ifndef SWARM_ROT_LANE_OUT
#define SWARM_ROT_LANE_OUT 1
#endif
constexpr int kLaneOutputs = 10;
constexpr int kLaneOutBytes = kLaneOutputs * (8 + 4 + 4);   // per warp: pointers | strides | staged values
__host__ __device__ constexpr int rot_warps(int n, bool dr) { return n >= 16 ? (dr ? SWARM_ROT_W32_DR : SWARM_ROT_W32) : 8; }
__host__ __device__ constexpr int rot_min_blocks(int n, bool dr) { return n >= 16 ? (dr ? SWARM_ROT_B32_DR : SWARM_ROT_B32) : 3; }

// smem per warp: mbarriers (16 B) | agent inbox: pos4[32] vel4[32] actions[96] (single buffer, refilled as
// soon as it has been read) | env inbox x 2: goal4[G] obst4[G*M] dr[2G] step_count[G] ep_return[G] |
// doubled position table (1 KB) | obs tile (4736 B)
__host__ __device__ constexpr int rot_envbox_bytes(int G, int M, bool dr) {
    return 16 * G * (1 + M) + (dr ? 32 * G : 0) + ((8 * G + 15) & ~15);
}
__host__ __device__ constexpr int rot_smem_per_warp(int G, int M, bool dr) {
    return 16 + 1408 + 2 * rot_envbox_bytes(G, M, dr) + 1024 + kTileBytes;
}

// MT: number of obstacles when known at compile time (4 / 8: sorting-network selection), 0 = P.M
// MODE: kRotStep = env.step() of every group (episode ends are put on the reset list);
//       kRotReset = env.reset() + first observation of the listed envs (the auto-reset launch that follows)
//       kRotFused = both in ONE launch: the warp that finds an episode over re-draws that env itself and runs the
//                   table / rotation / obstacle / tile code a second time (the SAME code, a runtime pass flag --
//                   a second copy would not fit the instruction cache) to produce the reset observation
enum RotMode : int { kRotStep = 0, kRotReset = 1, kRotFused = 2 };

// DRM: 0 = no domain randomisation, 1 = randomisation without a control delay, 2 = with the command ring (the ring code
// is kept out of the instantiation that does not need it: the DR kernels sit at the edge of the instruction cache,
// measured 0.1468 -> 0.1455 ms per C4 step)
template <int NT, int MT, int DRM, int MODE>
__global__ void __launch_bounds__(rot_warps(NT, DRM != 0) * 32, rot_min_blocks(NT, DRM != 0)) swarm_step_rot_kernel(const DevParams P) {
    constexpr bool DR = DRM != 0;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int N = NT, G = 32 / NT, HALF = NT / 2;
    constexpr unsigned IDX = NT - 1;  // index bits of a neighbour key
    constexpr int kRotWarps = rot_warps(NT, DR);
    constexpr bool kStepLike = MODE != kRotReset;   // items = env groups of the batch, inputs by TMA, dynamic queue
#ifndef SWARM_ROT_RAW_DRAW_MIN_N
#define SWARM_ROT_RAW_DRAW_MIN_N 16
#endif
    constexpr bool kRawDraw = NT >= SWARM_ROT_RAW_DRAW_MIN_N;   // queue draws keep the raw counter value until the shuffle
    constexpr bool kFused = MODE == kRotFused;
    // (the shuffle makes the warp index provably warp-uniform: addresses and branches that derive from
    //  it are then computed on the uniform datapath)
    const int warp = __shfl_sync(FULL_MASK, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const int M = MT ? MT : P.M;
    const int envbox_bytes = rot_envbox_bytes(G, M, DR);
    const int per_warp = 16 + 1408 + 2 * envbox_bytes + 1024 + kTileBytes;
    unsigned char* wslice = smem_raw + (size_t)warp * per_warp;
    const unsigned bar0 = smem_u32(wslice);
    const float4* in_pos = reinterpret_cast<const float4*>(wslice + 16);  // agent inbox
    unsigned char* envbox0 = wslice + 16 + 1408;
    float4* tab2 = reinterpret_cast<float4*>(wslice + 16 + 1408 + 2 * envbox_bytes);
    float* tile = reinterpret_cast<float*>(wslice + 16 + 1408 + 2 * envbox_bytes + 1024);
    unsigned long long* wstats =
        reinterpret_cast<unsigned long long*>(smem_raw + (size_t)kRotWarps * per_warp) + warp * SWARM_STATS_WORDS;
    if (lane < SWARM_STATS_WORDS) wstats[lane] = 0ull;
    // step launch: the groups with an env to reset are collected here and appended to the global list kLocalList
    // at a time (one atomic per flush instead of one per group)
    constexpr int kLocalList = 8;
    int* wlist = reinterpret_cast<int*>(smem_raw + (size_t)kRotWarps * per_warp +
                                        (size_t)kRotWarps * SWARM_STATS_WORDS * sizeof(unsigned long long)) + warp * kLocalList;
    int n_local = 0;
    const unsigned tid_y = threadIdx.y;   // zero (one-dimensional CTA), but not provably uniform: see atom_inc_lane
    auto flush_list = [&]() {
        __syncwarp();
        unsigned base = 0u;
        const unsigned par = *reinterpret_cast<const volatile unsigned*>(P.reset_epoch) & 1u;
        if (lane == 0) base = atom_add_lane(P.reset_count + par, (unsigned)n_local, tid_y);
        base = __shfl_sync(FULL_MASK, base, 0);
        if (lane < n_local) P.reset_list[par * P.reset_list_stride + base + lane] = wlist[lane];
        __syncwarp();
        n_local = 0;
    };
    // DR: the signed 512-entry normal quantile table lives in shared memory (13 lookups per agent-step)
    const float* qtab = SWARM_ROT_DR_QTAB_GLOBAL ? P.dr_qtable :
                        reinterpret_cast<const float*>(smem_raw + (size_t)kRotWarps * per_warp +
                                                       (size_t)kRotWarps * SWARM_STATS_WORDS * sizeof(unsigned long long) +
                                                       (size_t)kRotWarps * kLocalList * sizeof(int));
    // per-env outputs by lane (see SWARM_ROT_LANE_OUT): pointer / stride table of this warp, filled once
    // (the DR instantiations sit at the edge of the instruction cache: while they still carried the command-ring code they
    //  measured 1.3 % slower with it -- the plain ones 1.0 % faster; without that code, DRM = 1, 0.1455 -> 0.1433 ms)
#ifndef SWARM_ROT_LANE_OUT_DR
#define SWARM_ROT_LANE_OUT_DR 1
#endif
    constexpr bool kLaneOut = SWARM_ROT_LANE_OUT && MODE == kRotStep && NT == 32 && (DRM == 0 || (DRM == 1 && SWARM_ROT_LANE_OUT_DR));
    unsigned char* const lane_out = smem_raw + (size_t)kRotWarps * per_warp +
                                    (size_t)kRotWarps * SWARM_STATS_WORDS * sizeof(unsigned long long) +
                                    (size_t)kRotWarps * kLocalList * sizeof(int) +
                                    ((DR && !SWARM_ROT_DR_QTAB_GLOBAL) ? 2048 : 0) + (size_t)warp * kLaneOutBytes;
    unsigned long long* const optr = reinterpret_cast<unsigned long long*>(lane_out);
    unsigned* const ostride = reinterpret_cast<unsigned*>(lane_out + 8 * kLaneOutputs);
    unsigned* const ostage = reinterpret_cast<unsigned*>(lane_out + 12 * kLaneOutputs);
    if (kLaneOut && lane < kLaneOutputs) {
        const void* ptr = nullptr;
        unsigned stride = 4;
        switch (lane) {
            case 0: ptr = P.all_term; stride = 1; break;
            case 1: ptr = P.all_trunc; stride = 1; break;
            case 2: ptr = P.reset_mask; stride = 1; break;
            case 3: ptr = P.episode_return; break;
            case 4: ptr = P.episode_length; break;
            case 5: ptr = P.step_count; break;
            case 6: ptr = P.ep_return; break;
            default: ptr = P.gs ? P.gs + 6 * NT + (lane - 7) : nullptr; stride = 4u * (unsigned)P.R; break;
        }
        optr[lane] = reinterpret_cast<unsigned long long>(ptr);
        ostride[lane] = stride;
    }
    if (DR && !SWARM_ROT_DR_QTAB_GLOBAL) {
        float* qw = const_cast<float*>(qtab);
        for (int k = threadIdx.x; k < 512; k += kRotWarps * 32) qw[k] = P.dr_qtable[k];
        __syncthreads();
    }

    const int e_l = lane / N;
    const int i = lane - e_l * N;
    const int e_base = e_l * N;
    const unsigned env_lanes = N == 32 ? FULL_MASK : (((1u << N) - 1u) << e_base);
    float* srow = tile + lane * kD;  // this lane's tile row; before the obs is staged it stashes exact distances

    // Programmatic dependent launch: this grid may start while the previous launch of the stream is still running.
    //  * reset launch: waits for the step launch in front of it, reads its list, then lets the NEXT launch of the
    //    stream start at once (it only writes the listed envs);
    //  * step launch (kOverlap): does NOT wait at the top.  The launch in front of it is normally the previous
    //    step's reset launch, which touches only the envs flagged in reset_mask by that step: a warp waits for it
    //    the first time it is about to load a flagged group (issue()) and at the latest before it exits.  Every
    //    other group was last written by the previous STEP launch, which had completed before the reset launch
    //    released this one.  Anything else in front (a caller's kernel that never triggers early) has completed
    //    before this grid starts.
    constexpr bool kOverlap = SWARM_ROT_PDL && SWARM_ROT_OVERLAP && MODE == kRotStep;
    bool dep_waited = !kOverlap;
#if SWARM_ROT_PDL
    if (!kOverlap) asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
    // step: one item per env group; reset: one item per listed group
    // (reset launch: the first list entry is fetched together with the list length -- the entry is only used if
    //  it turns out to be inside the list -- so a warp's first item starts one memory round trip earlier)
#if SWARM_ROT_PDL && SWARM_ROT_EARLY_TRIGGER
    // step launch: let the reset launch behind it place its CTAs as slots come free during this launch's tail (they
    // sit in their griddepcontrol.wait until this launch has completed), instead of being launched only then
    // (only when that reset launch really follows: an early trigger releases whatever comes next in the stream, and a
    //  step launch of this kernel does not wait at its top)
    if (MODE == kRotStep && P.auto_reset) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
    int env0_pref = 0;
    const int* rlist = P.reset_list;
    int n_iter = P.n_groups;
    if (MODE == kRotReset) {
        const unsigned cur = (*reinterpret_cast<const volatile unsigned*>(P.reset_epoch) - 1u) & 1u;
        rlist = P.reset_list + cur * P.reset_list_stride;
        env0_pref = rlist[min((int)(blockIdx.x * kRotWarps + warp), P.n_groups - 1)];
        n_iter = (int)*reinterpret_cast<const volatile unsigned*>(P.reset_count + cur);
#if SWARM_ROT_PDL && SWARM_ROT_OVERLAP
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
    }
    const int env_end = P.env_begin + P.env_count;
    unsigned* const queue = P.work_counter + (kStepLike ? 0 : 2);

    if (lane == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    // env inbox: goal4[G] | obst4[G*M] | dr[2G] | step_count[G] | ep_return[G]
    const int goal_off = 0, obst_off = 16 * G, dr_off = 16 * G * (1 + M);
    const int sc_off = dr_off + (DR ? 32 * G : 0);
    // only_actions: the resident mode of the fused multi-step launch (one group per warp) -- the group's state is
    // already in this warp's inboxes, written back there by the previous step; only the next step's actions are fetched
    auto issue = [&](int grp, int buf, int t_step = 0, bool only_actions = false) {
        if (!kStepLike) return;
        const float* const actions = kFused ? P.actions + (long long)t_step * P.action_step_stride : P.actions;
        const int env0 = P.env_begin + grp * G;
        const int n_env = G == 1 ? 1 : min(G, env_end - env0);
        if (kFused && only_actions) {
            if (lane == 0) {
                const unsigned n_ag = (unsigned)(n_env * N);
                mbar_expect_tx(bar0 + 8 * buf, n_ag * 12u);
                bulk_g2s(bar0 + 16 + 1024, actions + (long long)env0 * N * 3, n_ag * 12u, bar0 + 8 * buf);
            }
            cp_async_commit();
            return;
        }
        if (kOverlap && !dep_waited) {   // (warp-uniform) a group the running reset launch may still be writing?
            const bool flagged = lane < n_env && P.reset_mask[env0 + lane] != 0;
            if (__any_sync(FULL_MASK, flagged)) {
                asm volatile("griddepcontrol.wait;" ::: "memory");
                dep_waited = true;
            }
        }
#if SWARM_ROT_TMA_LOADS
        if (lane == 0) {
            const unsigned n_ag = (unsigned)(n_env * N);
            const unsigned bar = bar0 + 8 * buf;
            const unsigned dsta = bar0 + 16;
            const unsigned dst = smem_u32(envbox0 + (size_t)buf * envbox_bytes);
            const long long a0 = (long long)env0 * N;
            mbar_expect_tx(bar, n_ag * 44u + (unsigned)n_env * (16u + 16u * M + (DR ? 32u : 0u)));
            bulk_g2s(dsta, P.pos4 + a0, n_ag * 16u, bar);
            bulk_g2s(dsta + 512, P.vel4 + a0, n_ag * 16u, bar);
            bulk_g2s(dsta + 1024, actions + a0 * 3, n_ag * 12u, bar);
            bulk_g2s(dst + goal_off, P.goal4 + env0, (unsigned)n_env * 16u, bar);
            bulk_g2s(dst + obst_off, P.obst4 + (long long)env0 * M, (unsigned)(n_env * M) * 16u, bar);
            if (DR) bulk_g2s(dst + dr_off, P.dr_params + (long long)env0 * 2, (unsigned)n_env * 32u, bar);
        }
#else
        {
            const int n_ag = n_env * N;
            const unsigned dsta = bar0 + 16;
            const unsigned dst = smem_u32(envbox0 + (size_t)buf * envbox_bytes);
            const long long a0 = (long long)env0 * N;
            if (G == 1 || lane < n_ag) {
                cp_async16(dsta + lane * 16, P.pos4 + a0 + lane);
                cp_async16(dsta + 512 + lane * 16, P.vel4 + a0 + lane);
            }
            if (lane * 4 < n_ag * 3) cp_async16(dsta + 1024 + lane * 16, actions + a0 * 3 + lane * 4);
            if (lane < n_env) cp_async16(dst + goal_off + lane * 16, P.goal4 + env0 + lane);
            for (int idx = lane; idx < n_env * M; idx += 32)
                cp_async16(dst + obst_off + idx * 16, P.obst4 + (long long)env0 * M + idx);
            if (DR && lane < 2 * n_env) cp_async16(dst + dr_off + lane * 16, P.dr_params + (long long)env0 * 2 + lane);
        }
#endif
        if (lane < n_env) {  // 4 bytes per env: too small for the bulk-copy engine
            const unsigned dst = smem_u32(envbox0 + (size_t)buf * envbox_bytes) + sc_off;
            cp_async4(dst + 4 * lane, P.step_count + env0 + lane);
            cp_async4(dst + 4 * (G + lane), P.ep_return + env0 + lane);
        }
        cp_async_commit();
    };
    // dynamic group queue: lane 0 draws the next group index while the current group is processed, so
    // every warp stays busy until the queue is empty (no static-stride tail)
    // (the first item of every warp is static, so the launch does not start with thousands of atomics on
    //  one address; the reset launch has ~1-2 items per warp and keeps a static stride throughout)
    const int warps_total = gridDim.x * kRotWarps;
    int it = blockIdx.x * kRotWarps + warp;
    // Fused launch: STATIC ownership -- this warp's groups are it, it + W, it + 2 W, ... -- and n_steps consecutive
    // steps in one launch (swarm_step_many on small batches): the items of a warp are (step 0: its groups in order),
    // (step 1: ...), ...  No warp ever touches another warp's envs, so the steps need no grid-wide barrier; a group's
    // state goes through global memory between steps (written by this warp's generic stores, read back by its bulk
    // copies: fence.proxy.async at the end of every item).
    const int ms_steps = kFused ? max(P.n_steps, 1) : 1;
    const int ms_own = (kFused && it < n_iter) ? (n_iter - it + warps_total - 1) / warps_total : 0;   // groups owned
    int ms_t = 0, ms_j = 0;          // current item: step ms_t, own group number ms_j
    // RESIDENT mode (one group per warp, several steps): the next item is the SAME group one step later, so its
    // state does not go through global memory and back -- the epilogue also writes pos / vel / step count / return
    // (and a reset its goal / obstacles / DR constants) into this warp's inboxes, the env inbox is not flipped, and
    // only the next step's actions are fetched, half an item ahead as usual.  (The global state is still written
    // every step: it is an output of the call.)
    const bool resident = kFused && ms_own == 1 && ms_steps > 1 && SWARM_ROT_TMA_LOADS;
    if (it < n_iter) issue(it, 0, 0);
    unsigned phase = 0;  // bit b: parity the next wait on mbarrier b uses

    int buf = 0;
    while (it < n_iter) {
        int it_next = 0;
        int ms_tn = ms_t, ms_jn = ms_j + 1;   // fused: the item after this one
        if (kFused) {
            if (ms_jn == ms_own) { ms_jn = 0; ++ms_tn; }
            it_next = ms_tn < ms_steps ? (int)(blockIdx.x * kRotWarps + warp) + ms_jn * warps_total : n_iter;
        } else if (kStepLike) {
            // (the RAW counter value: "+ warps_total" written here is scheduled right behind the atomic and waits out
            //  its round trip -- 4.6 % of the launch's stall samples in the ncu source view; it is added behind the
            //  shuffle that broadcasts the value, half an item later.  N = 8 keeps the add in place: its short items
            //  measured 4 % slower with the deferred add, N = 16 / 32 1.5 % / 1 % faster)
            if (lane == 0) it_next = (kRawDraw ? 0 : warps_total) + (int)atom_inc_lane(queue, tid_y);
        } else {
            it_next = it + warps_total;
        }
        const int env0 = kStepLike ? P.env_begin + it * G : env0_pref;
        if (MODE == kRotReset) env0_pref = rlist[min(it_next, P.n_groups - 1)];  // the next item's entry, early
        const int n_env = G == 1 ? 1 : min(G, env_end - env0);
        const bool lane_ok = G == 1 ? true : e_l < n_env;
        const int env = env0 + (lane_ok ? e_l : 0);
        const int a0 = env0 * N;                  // (num_envs * num_drones <= 2^30, checked at create)
        const int a = a0 + (lane_ok ? lane : 0);
        const bool leader = lane_ok && i == 0;
        const unsigned ok_lanes = __ballot_sync(FULL_MASK, lane_ok);
        unsigned char* ib = envbox0 + (size_t)buf * envbox_bytes;
        float4* tgoal = reinterpret_cast<float4*>(ib + goal_off);
        float4* tobs_all = reinterpret_cast<float4*>(ib + obst_off);
        const float4* tobs = tobs_all + e_l * M;

        float4 p = make_float4(0.f, 0.f, 0.f, 0.f), v = p;
        float gx = 0.f, gy = 0.f, gz = 0.f, prev_d = 0.f;
        int sc = 0;
        float c_amax = P.amax, c_vmax = P.vmax, c_dt = P.dt, c_bound = P.bound, c_thr_obst = P.thr_obst;
        unsigned ekey = 0u;
        int ctrl_delay = 0;
        const unsigned genv = DR ? (unsigned)(P.env_index_base + env) : 0u;
        bool alive = false;
        uint4 rA = make_uint4(0, 0, 0, 0);  // DR: this step's stream-A block (thrust + observation noise)
        unsigned reset_envs = 0u;  // reset launch: bit el = env el of the group is re-drawn
        if (MODE == kRotReset) {
            // one env per group: being on the list means it is re-drawn (no mask load in the dependency chain)
            if (G == 1) reset_envs = 1u;
            else reset_envs = __ballot_sync(FULL_MASK, lane < n_env && P.env_mask[env0 + lane] != 0);
        }

        // fused launch: pass 0 = env.step(); pass 1 (only when an episode of the group ended) = env.reset() + its
        // observation for those envs, through the same table / scan / tile code
        int pass = 0;
#pragma unroll 1
        for (;; ++pass) {
            // (the pass number is made opaque so that the compiler cannot specialise -- duplicate -- the scan / tile
            //  code for each pass: ONE copy must serve both or the loop leaves the 32 KB instruction cache)
            if (kFused) asm volatile("" : "+r"(pass));
            const bool step_now = MODE == kRotStep || (kFused && pass == 0);
            int step_flag = step_now ? 1 : 0;   // (re-read through an opaque copy after the input stage, see below)
            auto step_pass = [&]() { return MODE == kRotStep || (kFused && step_flag != 0); };
            if (step_now) {
                cp_async_wait_all();
#if SWARM_ROT_TMA_LOADS
                mbar_wait(bar0 + 8 * buf, (phase >> buf) & 1u);
                phase ^= 1u << buf;
#endif
                __syncwarp();  // the cp.async words of the other lanes
                // obstacle index -> .w of the inbox copy, so a key is one LOP3 (the table syncwarp below orders it)
                for (int idx = lane; idx < G * M; idx += 32)
                    reinterpret_cast<unsigned*>(tobs_all)[idx * 4 + 3] = (unsigned)(idx % M);
                float ax = 0.f, ay = 0.f, az = 0.f;
                bool nan_act = false;
                if (lane_ok) {
                    p = in_pos[lane];
                    v = in_pos[32 + lane];
                    const float4 g4 = tgoal[e_l];
                    gx = g4.x; gy = g4.y; gz = g4.z;
                    const float* act = reinterpret_cast<const float*>(in_pos + 64);
                    ax = act[lane * 3 + 0]; ay = act[lane * 3 + 1]; az = act[lane * 3 + 2];
                    sc = reinterpret_cast<const int*>(ib + sc_off)[e_l];
                    if (DR) {
                        const float4* drp = reinterpret_cast<const float4*>(ib + dr_off) + 2 * e_l;
                        const float4 d0 = drp[0], d1 = drp[1];
                        c_amax = d0.x; c_vmax = d0.y; c_dt = d0.z; c_bound = d0.w;
                        c_thr_obst = d1.x; ekey = __float_as_uint(d1.y);
                        ctrl_delay = (int)d1.w;
                    }
                }
                alive = lane_ok && p.w != 0.0f;

                // =========================== integrate (:98-118) ===========================
                prev_d = norm1d<0>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));  // :98-101
                if (alive) {
                    if (DRM == 2 && P.dr_delay_hist > 0) {
                        // control delay: apply the command submitted ctrl_delay steps ago (zero while the episode
                        // is younger), then file the one submitted now in ring slot step_count % H
                        const int H = P.dr_delay_hist;
                        float* ring = P.act_hist + ((long long)env * H * N + i) * 3;
                        const float sx = ax, sy = ay, sz = az;
                        const int slot_w = (int)((unsigned)sc % (unsigned)H);
                        if (ctrl_delay > 0) {
                            if (sc < ctrl_delay) {
                                ax = 0.f; ay = 0.f; az = 0.f;
                            } else {  // (sc - ctrl_delay) % H without a second division: ctrl_delay <= H
                                const int slot_r = slot_w - ctrl_delay + (slot_w < ctrl_delay ? H : 0);
                                const float* hp = ring + slot_r * (N * 3);
                                ax = hp[0]; ay = hp[1]; az = hp[2];
                            }
                        }
                        float* wp = ring + slot_w * (N * 3);
                        wp[0] = sx; wp[1] = sy; wp[2] = sz;
                    }
                    ax = clipf(ax, -1.0f, 1.0f); ay = clipf(ay, -1.0f, 1.0f); az = clipf(az, -1.0f, 1.0f);
                    nan_act = !(ax == ax && ay == ay && az == az);   // (np.clip lets NaN through; counted, see below)
                    if (DR) {  // thrust noise: a <- a * (1 + sigma z), one normal per axis
                        rA = philox4x32_7(genv, ekey, (unsigned)sc, (unsigned)i | (DR_STREAM_A << 16), P);
                        ax = __fmul_rn(ax, __fmaf_rn(P.dr_std_thrust, dr_normal_off(qtab, dr_field_off(rA, 0)), 1.0f));
                        ay = __fmul_rn(ay, __fmaf_rn(P.dr_std_thrust, dr_normal_off(qtab, dr_field_off(rA, 1)), 1.0f));
                        az = __fmul_rn(az, __fmaf_rn(P.dr_std_thrust, dr_normal_off(qtab, dr_field_off(rA, 2)), 1.0f));
                    }
                    v.x = __fadd_rn(v.x, __fmul_rn(__fmul_rn(ax, c_amax), c_dt));
                    v.y = __fadd_rn(v.y, __fmul_rn(__fmul_rn(ay, c_amax), c_dt));
                    v.z = __fadd_rn(v.z, __fmul_rn(__fmul_rn(az, c_amax), c_dt));
                    const float speed = norm1d<0>(v.x, v.y, v.z);  // _clip_speed (:179-183)
                    if (!(speed <= c_vmax || speed < P.eps_speed)) {
                        v.x = __fmul_rn(__fdiv_rn(v.x, speed), c_vmax);
                        v.y = __fmul_rn(__fdiv_rn(v.y, speed), c_vmax);
                        v.z = __fmul_rn(__fdiv_rn(v.z, speed), c_vmax);
                    }
                    p.x = __fadd_rn(p.x, __fmul_rn(v.x, c_dt));
                    p.y = __fadd_rn(p.y, __fmul_rn(v.y, c_dt));
                    p.z = __fadd_rn(p.z, __fmul_rn(v.z, c_dt));
                }
                {   // NaN-action guard counter (rare: the vote is all a clean step pays)
                    const unsigned nan_m = __ballot_sync(FULL_MASK, nan_act);
                    if (nan_m != 0u && lane == 0) wstats[SWARM_STAT_NAN_ACTIONS] += (unsigned long long)__popc(nan_m);
                }
                // wall clip for ALL drones (:113-117); velocity is not zeroed at the wall
                p.x = clipf(p.x, -c_bound, c_bound);
                p.y = clipf(p.y, -c_bound, c_bound);
                p.z = clipf(p.z, -c_bound, c_bound);
            } else {
                __syncwarp();  // every lane is done with the previous item's tables
                // ================================ reset (:65-80) ================================
                // draw order of env.reset(): positions (N,3) -> goal (3,) -> obstacles (M,3), each
                // rng.uniform(-W/2, W/2) in float64 then float32; 32 lanes draw in parallel by PCG64 jump-ahead
#pragma unroll 1
                for (int el = 0; el < n_env; ++el) {
                    if (!((reset_envs >> el) & 1u)) continue;
                    const int renv = env0 + el;
                    const unsigned long long sh = P.rng[(long long)renv * 4 + 0], sl = P.rng[(long long)renv * 4 + 1];
                    const unsigned long long ih = P.rng[(long long)renv * 4 + 2], il = P.rng[(long long)renv * 4 + 3];
                    double u_lo = P.rng_lo, u_range = P.rng_range;
                    if (DR) {
                        // this episode's constants: 6 uniforms + an episode key from one counter per (env, reset)
                        const unsigned ge = (unsigned)(P.env_index_base + renv);
                        const uint4 ra = philox4x32_10(ge, (unsigned)sl, (unsigned)(sl >> 32), DR_CTR_EPISODE, P);
                        const uint4 rb = philox4x32_10(ge, (unsigned)sl, (unsigned)(sl >> 32), DR_CTR_EPISODE + 1u, P);
                        const double inv24 = 1.0 / 16777216.0;
                        const double s_mass = __dadd_rn(P.dr_lo[0], __dmul_rn(P.dr_span[0], __dmul_rn((double)(ra.x >> 8), inv24)));
                        const double s_acc = __dadd_rn(P.dr_lo[1], __dmul_rn(P.dr_span[1], __dmul_rn((double)(ra.y >> 8), inv24)));
                        const double s_spd = __dadd_rn(P.dr_lo[2], __dmul_rn(P.dr_span[2], __dmul_rn((double)(ra.z >> 8), inv24)));
                        const double s_dt = __dadd_rn(P.dr_lo[3], __dmul_rn(P.dr_span[3], __dmul_rn((double)(ra.w >> 8), inv24)));
                        const double s_rad = __dadd_rn(P.dr_lo[4], __dmul_rn(P.dr_span[4], __dmul_rn((double)(rb.x >> 8), inv24)));
                        const double s_wld = __dadd_rn(P.dr_lo[5], __dmul_rn(P.dr_span[5], __dmul_rn((double)(rb.y >> 8), inv24)));
                        const double world = __dmul_rn(P.dr_world, s_wld);
                        const double half_w = __dmul_rn(world, 0.5);
                        u_lo = -half_w; u_range = __dsub_rn(half_w, -half_w);
                        if (lane == 0) {
                            float delay = 0.0f;  // this episode's control delay: 4th word of the second block
                            if (P.dr_delay_count > 0) {
                                const double uu = __dmul_rn((double)(rb.w >> 8), inv24);
                                int pick = P.dr_delay_count - 1;
#pragma unroll 1
                                for (int k = P.dr_delay_count - 1; k >= 0; --k)
                                    if (uu < P.dr_delay_cum[k]) pick = k;
                                delay = (float)P.dr_delay_values[pick];
                            }
                            const float4 d0 =
                                make_float4(__double2float_rn(__ddiv_rn(__dmul_rn(P.dr_max_accel, s_acc), s_mass)),
                                            __double2float_rn(__dmul_rn(P.dr_max_speed, s_spd)),
                                            __double2float_rn(__dmul_rn(P.dr_dt, s_dt)), __double2float_rn(half_w));
                            const float4 d1 =
                                make_float4(__double2float_rn(__dadd_rn(P.dr_r_c, __dmul_rn(P.dr_r_o, s_rad))),
                                            __uint_as_float(rb.z), __double2float_rn(world), delay);
                            P.dr_params[(long long)renv * 2 + 0] = d0;
                            P.dr_params[(long long)renv * 2 + 1] = d1;
                            if (kFused) {   // (resident mode reads them from here on the next step)
                                float4* drp = reinterpret_cast<float4*>(ib + dr_off) + 2 * el;
                                drp[0] = d0; drp[1] = d1;
                            }
                        }
                        if (e_l == el) ekey = rb.z;  // (the dynamics constants are not needed to observe)
                    }
#pragma unroll (kFused ? 1 : 4)
                    for (int k = lane; k < P.n_draws; k += 32) {
                        unsigned long long oh, ol;
                        pcg_jump(P.jump[k + 1], sh, sl, ih, il, oh, ol);
                        const float val = pcg_uniform_f32(oh, ol, u_lo, u_range);
                        if (k < 3 * N) {
                            reinterpret_cast<float*>(tab2 + 2 * el * N + k / 3)[k % 3] = val;
                        } else if (k < 3 * N + 3) {
                            reinterpret_cast<float*>(tgoal + el)[k - 3 * N] = val;
                        } else {
                            const int kk = k - 3 * N - 3;
                            reinterpret_cast<float*>(tobs_all + el * M + kk / 3)[kk % 3] = val;
                        }
                    }
                    if (lane == 0) {
                        unsigned long long oh, ol;
                        pcg_jump(P.jump[P.n_draws], sh, sl, ih, il, oh, ol);
                        P.rng[(long long)renv * 4 + 0] = oh;
                        P.rng[(long long)renv * 4 + 1] = ol;
                        P.step_count[renv] = 0;
                        P.ep_return[renv] = 0.0f;
                        reinterpret_cast<float*>(tgoal + el)[3] = 0.0f;
                    }
                    for (int k = lane; k < M; k += 32)  // obstacle index in .w (one-LOP3 keys, as in the step launch)
                        reinterpret_cast<unsigned*>(tobs_all + el * M + k)[3] = (unsigned)k;
                }
                __syncwarp();
                if (lane < n_env && ((reset_envs >> lane) & 1u)) P.goal4[env0 + lane] = tgoal[lane];
                for (int idx = lane; idx < n_env * M; idx += 32)
                    if ((reset_envs >> (idx / M)) & 1u) {
                        const float4 o = tobs_all[idx];
                        P.obst4[(long long)env0 * M + idx] = make_float4(o.x, o.y, o.z, 0.0f);
                    }
                const bool fresh = lane_ok && ((reset_envs >> e_l) & 1u);
                if (fresh) {
                    p = tab2[2 * e_base + i];
                    v = make_float4(0.f, 0.f, 0.f, 0.f);
                    const float4 g4 = tgoal[e_l];
                    gx = g4.x; gy = g4.y; gz = g4.z;
                    sc = -1;  // the observed state has step_count 0: its sensor noise is keyed by 0 - 1
                }
                alive = lane_ok;  // (only the re-drawn envs' results are used; every drone of theirs is active)
                __syncwarp();     // the drawn positions have been read before the table is rewritten
            }

            // (fused: the two input stages above rejoin here; without this the compiler threads the later tests of
            //  the pass flag back to them and emits the whole scan code twice)
            if (kFused) asm volatile("" : "+r"(step_flag));
            // doubled position table: entry [2N e_l + i + r] is drone (i + r) mod N for 0 <= r <= N; .w = drone index
            {
                const float4 t = make_float4(p.x, p.y, p.z, __int_as_float(i));
                tab2[2 * e_base + i] = t;
                tab2[2 * e_base + i + N] = t;
            }
            const unsigned alive_mask = __ballot_sync(FULL_MASK, alive);
            const int n_alive_env = __popc(alive_mask & env_lanes);
            if (lane == 0) bulk_wait_read0();  // the previous obs tile has left shared memory
            __syncwarp();
            // every lane has consumed the agent inbox (its values went through the integrator): refill it,
            // and the other env inbox, with the next group's inputs
            if (pass == 0) {
                if (!kFused) {
                    it_next = __shfl_sync(FULL_MASK, it_next, 0);
                    if (kStepLike && kRawDraw) it_next += warps_total;
                }
                // (fused, one group per warp: the next item is THIS group one step later -- its inputs are this
                //  item's outputs, so they are fetched at the end of the item instead)
                if (kStepLike && it_next < n_iter) {
                    if (resident) issue(it_next, buf, ms_tn, true);
                    else if (!(kFused && ms_own == 1)) issue(it_next, buf ^ 1, ms_tn);
                }
            }
            // velocity / previous goal distance wait in the tile row (slots 32-35) while the scans need the registers
            srow[32] = v.x; srow[33] = v.y; srow[34] = v.z; srow[35] = prev_d;

            float nd[3]; int nj[3];        // exact distances / drone indices of the 3 nearest neighbours
            float od[4]; int om[4];        // same for the 4 nearest obstacles
            bool pair_hit = false;
            double form_sum = 0.0;
            int form_n = 0;
            const float4* tp = tab2 + 2 * e_base + i;  // tp[r] = drone (i + r) mod N
            bool bad = false;
            // Groups with PARKED drones (they reached the goal earlier, the episode goes on) stay on the rotation pass
            // (round 2b, as in the wide kernel): neighbour keys cover every drone, each formation term is multiplied by
            // the partner's 0.0 / 1.0 activity flag (the float64 sum is exact, so the masked sum IS the reference's sum
            // over active pairs), collisions among ACTIVE drones are read off the three picks.  That instantiation of the
            // rounds is a rolled loop (it is the rarer one, and the hot loop must keep the instruction cache).  Under
            // goal-seeking actions 10 - 25 % of the groups hold a parked drone, and the serial exact path they used to
            // take (~2 000 instructions per item) made the whole launch 32 - 40 % slower (tools/parked_bench.py).
#ifndef SWARM_ROT_MASKED_PASS
#define SWARM_ROT_MASKED_PASS 1
#endif
            const bool masked = SWARM_ROT_MASKED_PASS && SWARM_ROT_PACKED && alive_mask != ok_lanes;   // (warp-uniform)
            if (alive_mask == ok_lanes || masked) {
                // ================= rotation pass: every drone of the group is active, or masked =================
                unsigned k0 = ~0u, k1 = ~0u, k2 = ~0u, k3 = ~0u;
                double acc_f = 0.0, acc_b = 0.0;
                float smin = F32_INF;
                const double d_star = P.d_star;
#ifndef SWARM_ROT_DR_UNROLL
#define SWARM_ROT_DR_UNROLL 5
#endif
#if SWARM_ROT_PACKED
                // Rounds in pairs (r, r + 1), the last pair holding the half round N/2: the coordinate differences /
                // squares of a round and the two square roots of a pair are packed float32x2 operations (same
                // roundings, half the issue slots).  Distances travel NEGATED through the pair (neg_sqrt_rn_fast2):
                // keys clear the sign in the LOP3 that packs them, the formation term is |(-d) + d*|, the stash holds
                // -d and the three picks take |.| when they are read back.
                const f32x2 p_xy = pack2(p.x, p.y), p_z0 = pack2(p.z, 0.0f);
                constexpr unsigned KEYMASK = ~IDX & 0x7fffffffu;
                const unsigned env_alive = alive_mask >> e_base;   // bit j: drone j of this lane's env is active
                // masked_tag: integral_constant<int, 0> = every drone active, 1 = masked, 2 = decided at run time (ONE copy
                // of the loop serves both: for instantiations whose loop is rolled anyway and which sit at the edge of the
                // instruction cache)
                auto full_round = [&](auto masked_tag, int r, const float4& q, float ndf) {
                    constexpr int MT_ = decltype(masked_tag)::value;
                    const bool MASKED = MT_ == 2 ? masked : (MT_ == 1);
                    const int src = lane + N - r;                                   // (i - r) mod N in the low bits
                    const float ndb = __shfl_sync(FULL_MASK, ndf, src, N);          // -d((i - r) mod N, i)
                    srow[r] = ndf;
                    srow[HALF + r] = ndb;
                    const unsigned kf = and_or<KEYMASK>(__float_as_uint(ndf), __float_as_uint(q.w));
                    const unsigned kb = merge_low<IDX | 0x80000000u>(__float_as_uint(ndb), (unsigned)src);
                    merge2(kf, kb, k0, k1, k2, k3);
                    if (kStepLike) {   // |d - d*| = |(-d) + d*|
                        double tf, tb;
                        if (SWARM_ROT_CVT_FORM & 1) tf = fabs(__dsub_rn(f64_of_pos_f32<true>(fabsf(ndf)), d_star));
                        else tf = fabs(__dadd_rn((double)ndf, d_star));
                        if (SWARM_ROT_CVT_FORM & 2) tb = fabs(__dsub_rn(f64_of_pos_f32<true>(fabsf(ndb)), d_star));
                        else tb = fabs(__dadd_rn((double)ndb, d_star));
                        if (MASKED) {   // only ACTIVE partners count (:210-224); q.w = the forward partner's index
                            tf = __dmul_rn(tf, ((env_alive >> (__float_as_uint(q.w) & IDX)) & 1u) ? 1.0 : 0.0);
                            tb = __dmul_rn(tb, ((env_alive >> ((unsigned)src & IDX)) & 1u) ? 1.0 : 0.0);
                        }
                        acc_f = __dadd_rn(acc_f, tf);
                        acc_b = __dadd_rn(acc_b, tb);
                    }
                };
                constexpr int kPairs = HALF / 2;
#ifndef SWARM_ROT_UNROLL_PAIRS
#define SWARM_ROT_UNROLL_PAIRS 8
#endif
#ifndef SWARM_ROT_UNROLL_PAIRS_DR
#define SWARM_ROT_UNROLL_PAIRS_DR 1   // (2 until the masked pass was added; re-measured: 1 0.1469 ms, 2 0.1485, 3 0.1484, 4 0.1559)
#endif
                // (the unroll factors are tuning knobs: the loop body must stay inside the instruction cache)
                // (the fused instantiation carries the reset code as well and misses the instruction cache -- 89 % hit rate,
                //  `no_instruction` 1.3 per issue at 8 192 envs: its pair loop stays rolled, measured 27.7 -> 25.7 us per step)
#ifndef SWARM_ROT_UNROLL_PAIRS_FUSED
#define SWARM_ROT_UNROLL_PAIRS_FUSED 1
#endif
                constexpr int kUnrollWant = kFused ? SWARM_ROT_UNROLL_PAIRS_FUSED : (DR ? SWARM_ROT_UNROLL_PAIRS_DR : SWARM_ROT_UNROLL_PAIRS);
                constexpr int kUnroll = kPairs > kUnrollWant ? kUnrollWant : kPairs;
                auto pair_rounds = [&](auto masked_tag) {
                    constexpr int MT_ = decltype(masked_tag)::value;
                    const bool MASKED = MT_ == 2 ? masked : (MT_ == 1);
                    constexpr int kUnrollHere = MT_ != 0 ? 1 : kUnroll;
#pragma unroll kUnrollHere
                    for (int u = 0; u < kPairs - 1; ++u) {
                        const int ra = 2 * u + 1, rb = 2 * u + 2;
                        const float4 qa = tp[ra], qb = tp[rb];
                        float ax2, ay2, az2, bx2, by2, bz2;
                        sq_diff3(qa, p_xy, p_z0, ax2, ay2, az2);
                        sq_diff3(qb, p_xy, p_z0, bx2, by2, bz2);
                        const float nsa = neg_sumsq1d_of_squares(ax2, ay2, az2), nsb = neg_sumsq1d_of_squares(bx2, by2, bz2);
                        float nda, ndb;
                        unpack2(neg_sqrt_rn_fast2(nsa, nsb), nda, ndb);
                        if (!kStepLike) smin = fminf(smin, fminf(-nsa, -nsb));  // reset(): only the range check of the sum
                        full_round(masked_tag, ra, qa, nda);
                        full_round(masked_tag, rb, qb, ndb);
                    }
                    {   // last pair: round N/2 - 1 and the half round N/2 (visited from both ends, each end keeps its copy)
                        const float4 qa = tp[HALF - 1], qb = tp[HALF];
                        float ax2, ay2, az2, bx2, by2, bz2;
                        sq_diff3(qa, p_xy, p_z0, ax2, ay2, az2);
                        sq_diff3(qb, p_xy, p_z0, bx2, by2, bz2);
                        const float nsa = neg_sumsq1d_of_squares(ax2, ay2, az2), nsb = neg_sumsq1d_of_squares(bx2, by2, bz2);
                        float nda, ndb;
                        unpack2(neg_sqrt_rn_fast2(nsa, nsb), nda, ndb);
                        if (!kStepLike) smin = fminf(smin, fminf(-nsa, -nsb));
                        full_round(masked_tag, HALF - 1, qa, nda);
                        srow[HALF] = ndb;
                        merge1(and_or<KEYMASK>(__float_as_uint(ndb), __float_as_uint(qb.w)), k0, k1, k2, k3);
                        if (kStepLike) {
                            double th = fabs(__dadd_rn((double)ndb, d_star));
                            if (MASKED) th = __dmul_rn(th, ((env_alive >> (__float_as_uint(qb.w) & IDX)) & 1u) ? 1.0 : 0.0);
                            acc_f = __dadd_rn(acc_f, th);
                        }
                    }
                };
#ifndef SWARM_ROT_MASKED_RUNTIME_DR
#define SWARM_ROT_MASKED_RUNTIME_DR 0
#endif
                if (SWARM_ROT_MASKED_RUNTIME_DR && DR && kUnroll == 1) pair_rounds(std::integral_constant<int, 2>{});
                else if (!masked) pair_rounds(std::integral_constant<int, 0>{});
                else pair_rounds(std::integral_constant<int, 1>{});
#else
                float4 qn = tp[1];
                // (the DR variant's loop + noise code sits at the edge of the instruction cache: its unroll
                //  factor is a tuning knob)
                constexpr int kUnroll = DR ? (HALF > SWARM_ROT_DR_UNROLL ? SWARM_ROT_DR_UNROLL : HALF) : HALF;
#pragma unroll kUnroll
                for (int r = 1; r < HALF; ++r) {
                    const float4 q = qn;
                    qn = tp[r + 1];
                    const float s = sumsq1d_fast(__fsub_rn(q.x, p.x), __fsub_rn(q.y, p.y), __fsub_rn(q.z, p.z));
                    const float d = sqrt_rn_fast(s);
                    const float db = __shfl_sync(FULL_MASK, d, lane - r, N);  // d((i - r) mod N, i)
                    srow[r] = d;
                    srow[HALF + r] = db;
                    const unsigned kf = and_or<~IDX>(__float_as_uint(d), __float_as_uint(q.w));
                    const unsigned kb = merge_low<IDX>(__float_as_uint(db), (unsigned)(lane - r));
                    merge2(kf, kb, k0, k1, k2, k3);
                    if (kStepLike) {
                        acc_f = __dadd_rn(acc_f, fabs(__dsub_rn(f64_of_pos_f32<(SWARM_ROT_CVT_FORM & 1) != 0>(d), d_star)));
                        acc_b = __dadd_rn(acc_b, fabs(__dsub_rn(f64_of_pos_f32<(SWARM_ROT_CVT_FORM & 2) != 0>(db), d_star)));
                    } else {
                        smin = fminf(smin, s);  // reset(): no reward, so no formation sum -- only its range check
                    }
                }
                {   // round N/2: the pair is visited from both ends, each end keeps its own copy
                    const float4 q = qn;
                    const float s = sumsq1d_fast(__fsub_rn(q.x, p.x), __fsub_rn(q.y, p.y), __fsub_rn(q.z, p.z));
                    const float d = sqrt_rn_fast(s);
                    srow[HALF] = d;
                    merge1(and_or<~IDX>(__float_as_uint(d), __float_as_uint(q.w)), k0, k1, k2, k3);
                    if (kStepLike) acc_f = __dadd_rn(acc_f, fabs(__dsub_rn(f64_of_pos_f32<(SWARM_ROT_CVT_FORM & 1) != 0>(d), d_star)));
                    else smin = fminf(smin, s);
                }
#endif
                form_sum = __dadd_rn(acc_f, acc_b);
                // s < 2^-28 (a distance below 2^-14: fast sqrt / exact-sum preconditions) shows up either as the
                // smallest key or, for s = 0 / denormal s (rsqrt -> inf -> NaN distance), as a NaN formation sum;
                // either sends the whole group to the exact path.  Candidates sharing a key bucket (truncation may
                // have mis-ordered them) are settled per drone: among keys 0-2 only the ORDER is open -> the
                // picks are sorted by their exact (distance, index) below; a 3rd/4th-key collision leaves the
                // SET open -> exact neighbour rescan
                // (the reset launch, which needs no formation sum, tracks the smallest squared distance instead)
                bad = !(form_sum == form_sum) || k0 < 0x38800000u /* 2^-14 */ || !(smin >= 0x1p-28f);
                const bool mine = lane_ok && (step_pass() || ((reset_envs >> e_l) & 1u));
                const unsigned kk[3] = {k0, k1, k2};
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    const int j = (int)(kk[q] & IDX);
                    const int t = (j - i) & (int)IDX;           // forward distance i -> j
                    nj[q] = j;
                    nd[q] = fabsf(srow[t <= HALF ? t : HALF + N - t]);  // backward round N - t was stashed at HALF + (N - t)
                                                                         // (|.|: the packed rounds stash -d)
                }
#ifndef SWARM_ROT_SORT_ALWAYS
#define SWARM_ROT_SORT_ALWAYS 0
#endif
                // keys in different buckets order their exact distances strictly (the truncation is monotone), so the
                // exact (distance, index) sort of the picks is only needed when two of the first three keys share a
                // bucket -- about one warp in a thousand (ncu source view: the sort was ~35 instructions per env-step)
                if (SWARM_ROT_SORT_ALWAYS || __any_sync(FULL_MASK, (k0 ^ k1) <= IDX || (k1 ^ k2) <= IDX)) {
                    auto cex3 = [&](int a, int b) {
                        const bool sw = nd[a] > nd[b] || (nd[a] == nd[b] && nj[a] > nj[b]);
                        const float td = sw ? nd[b] : nd[a], tD = sw ? nd[a] : nd[b];
                        const int tj = sw ? nj[b] : nj[a], tJ = sw ? nj[a] : nj[b];
                        nd[a] = td; nd[b] = tD; nj[a] = tj; nj[b] = tJ;
                    };
                    cex3(0, 1); cex3(1, 2); cex3(0, 1);
                }
                if (__any_sync(FULL_MASK, mine && (k2 ^ k3) <= IDX)) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) { nd[q] = TOPK_EMPTY; nj[q] = 0; }
                    const float4* te = tab2 + 2 * e_base;
#pragma unroll 1
                    for (int j = 0; j < N; ++j) {
                        if (j == i) continue;
                        const float4 q = te[j];
                        topk_insert<3>(norm1d<0>(__fsub_rn(q.x, p.x), __fsub_rn(q.y, p.y), __fsub_rn(q.z, p.z)), j, nd, nj);
                    }
                }
                if (!masked) {
                    pair_hit = nd[0] <= P.thr_pair;  // nearest drone decides (:202-207)
                    form_n = N - 1;
                } else {
                    // collisions count among ACTIVE drones only (:202-207): an active pick within the threshold settles
                    // it; three parked picks within the threshold leave it open -> scan the active drones
                    const unsigned env_alive = alive_mask >> e_base;
                    bool open = alive;
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const bool within = nd[q] <= P.thr_pair;
                        pair_hit = pair_hit || (within && ((env_alive >> nj[q]) & 1u));
                        open = open && within;
                    }
                    open = open && !pair_hit;
                    if (__any_sync(FULL_MASK, open)) {
                        const float4* te = tab2 + 2 * e_base;
#pragma unroll 1
                        for (int j = 0; j < N; ++j) {
                            if (j == i || !((env_alive >> j) & 1u)) continue;
                            const float4 q = te[j];
                            pair_hit = pair_hit || norm1d<0>(__fsub_rn(q.x, p.x), __fsub_rn(q.y, p.y), __fsub_rn(q.z, p.z)) <= P.thr_pair;
                        }
                    }
                    pair_hit = pair_hit && alive;
                    form_n = alive ? n_alive_env - 1 : 0;
                }

                // ---- obstacles: _nearest_obstacle_features (:273-291) + obstacle part of _collision_mask
                unsigned o0, o1, o2, o3, o4;
                float smin_o = F32_INF;
                if (MT == 8 || MT == 4) {
                    unsigned ok[MT ? MT : 1];
#pragma unroll
                    for (int m = 0; m < MT; m += 2) {
                        const float4 oa = tobs[m], ob = tobs[m + 1];
#if SWARM_ROT_PACKED
                        float oax, oay, oaz, obx, oby, obz;
                        sq_diff3(oa, p_xy, p_z0, oax, oay, oaz);
                        sq_diff3(ob, p_xy, p_z0, obx, oby, obz);
                        const float sa = __fadd_rn(__fadd_rn(oax, oay), oaz);   // np.linalg.norm(axis=): sequential f32
                        const float sb = __fadd_rn(__fadd_rn(obx, oby), obz);
#else
                        const float sa = sumsq_axis(__fsub_rn(oa.x, p.x), __fsub_rn(oa.y, p.y), __fsub_rn(oa.z, p.z));
                        const float sb = sumsq_axis(__fsub_rn(ob.x, p.x), __fsub_rn(ob.y, p.y), __fsub_rn(ob.z, p.z));
#endif
#if SWARM_ROT_OBST_SQKEY
                        // keys from the SQUARED distance (sqrt is monotone; squares that a truncated key cannot
                        // tell apart -- which includes every pair whose roots could coincide -- are flagged
                        // below): the sqrt is then taken for the 4 selected obstacles only
                        srow[m] = sa;
                        srow[m + 1] = sb;
                        ok[m] = and_or<~31u>(__float_as_uint(sa), __float_as_uint(oa.w));
                        ok[m + 1] = and_or<~31u>(__float_as_uint(sb), __float_as_uint(ob.w));
#else
                        smin_o = fminf(fminf(smin_o, sa), sb);
                        const float da = sqrt_rn_fast(sa), db = sqrt_rn_fast(sb);
                        srow[m] = da;
                        srow[m + 1] = db;
                        ok[m] = and_or<~31u>(__float_as_uint(da), __float_as_uint(oa.w));
                        ok[m + 1] = and_or<~31u>(__float_as_uint(db), __float_as_uint(ob.w));
#endif
                    }
                    if (MT == 8) {
                        sort8(reinterpret_cast<unsigned(&)[8]>(ok));
                        o4 = ok[MT == 8 ? 4 : 0];
                    } else {
                        sort4(reinterpret_cast<unsigned(&)[4]>(ok));
                        o4 = ~0u;
                    }
                    o0 = ok[0]; o1 = ok[MT > 1 ? 1 : 0]; o2 = ok[MT > 2 ? 2 : 0]; o3 = ok[MT > 3 ? 3 : 0];
                } else {
                    o0 = o1 = o2 = o3 = o4 = ~0u;
#pragma unroll 1
                    for (int mb = 0; mb < M; mb += 4) {
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float4 o = tobs[mb + u];
                            const float s = sumsq_axis(__fsub_rn(o.x, p.x), __fsub_rn(o.y, p.y), __fsub_rn(o.z, p.z));
                            smin_o = fminf(smin_o, s);
                            const float d = sqrt_rn_fast(s);
                            srow[mb + u] = d;
                            merge1_5(and_or<~31u>(__float_as_uint(d), __float_as_uint(o.w)), o0, o1, o2, o3, o4);
                        }
                    }
                }
                bool bad_o = !(smin_o >= SQRT_FAST_MIN) || ((o0 ^ o1) <= 31u) || ((o1 ^ o2) <= 31u) || ((o2 ^ o3) <= 31u) ||
                             ((o3 ^ o4) <= 31u);
                const unsigned oo[4] = {o0, o1, o2, o3};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    om[q] = (int)(oo[q] & 31u);
                    od[q] = srow[om[q]];
                }
#if SWARM_ROT_OBST_SQKEY
                if (MT == 8 || MT == 4) {
                    bad_o = bad_o || !(od[0] >= SQRT_FAST_MIN);   // od[] still holds squares here; od[0] is the smallest
#pragma unroll
                    for (int q = 0; q < 4; ++q) od[q] = sqrt_rn_fast(od[q]);
                    // different squares can round to the SAME distance (then the reference orders by index, the
                    // keys by square): any exact tie among the first five distances goes to the exact path
                    const float d4 = MT == 8 ? sqrt_rn_fast(srow[o4 & 31u]) : F32_INF;
                    bad_o = bad_o || od[0] == od[1] || od[1] == od[2] || od[2] == od[3] || od[3] == d4;
                }
#endif
                if (__any_sync(FULL_MASK, mine && bad_o)) {  // an undecided obstacle order: the reference's loop as written
#pragma unroll
                    for (int q = 0; q < 4; ++q) { od[q] = TOPK_EMPTY; om[q] = 0; }
#pragma unroll 1
                    for (int m = 0; m < M; ++m) {
                        const float4 o = tobs[m];
                        topk_insert<4>(__fsqrt_rn(sumsq_axis(__fsub_rn(o.x, p.x), __fsub_rn(o.y, p.y), __fsub_rn(o.z, p.z))), m, od, om);
                    }
                }
                bad = bad && mine;
            }
            if ((alive_mask != ok_lanes && !masked) || __any_sync(FULL_MASK, bad)) {
                // ============ exact path: parked drones, coincident drones, or a detected near-tie ============
                // the reference's loops as written: ascending j, strict '<' (lowest index wins ties),
                // collision / formation over ACTIVE pairs only, np.mean's pairwise summation order
#pragma unroll
                for (int q = 0; q < 3; ++q) { nd[q] = TOPK_EMPTY; nj[q] = 0; }
                pair_hit = false;
                const unsigned em = (alive_mask & env_lanes) >> e_base;  // bit j: drone j of this env active
                const int n_f = alive ? n_alive_env - 1 : 0;
                const int nf8 = n_f >= 8 ? (n_f & ~7) : 0;
                double r8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) r8[u] = 0.0;
                double res = 0.0;
                bool tree_done = false;
                int cnt = 0;
                const float4* te = tab2 + 2 * e_base;
#pragma unroll 1
                for (int j = 0; j < N; ++j) {
                    if (j == i) continue;
                    const float4 q = te[j];
                    const float d = norm1d<0>(__fsub_rn(q.x, p.x), __fsub_rn(q.y, p.y), __fsub_rn(q.z, p.z));
                    topk_insert<3>(d, j, nd, nj);
                    if (alive && ((em >> j) & 1u)) {
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
#pragma unroll
                for (int q = 0; q < 4; ++q) { od[q] = TOPK_EMPTY; om[q] = 0; }
#pragma unroll 1
                for (int m = 0; m < M; ++m) {
                    const float4 o = tobs[m];
                    const float d = __fsqrt_rn(sumsq_axis(__fsub_rn(o.x, p.x), __fsub_rn(o.y, p.y), __fsub_rn(o.z, p.z)));
                    topk_insert<4>(d, m, od, om);
                }
            }
            v.x = srow[32]; v.y = srow[33]; v.z = srow[34]; prev_d = srow[35];
            const float curr_d = norm1d<0>(__fsub_rn(gx, p.x), __fsub_rn(gy, p.y), __fsub_rn(gz, p.z));

            // ===================== rewards and flags (:120-172) =====================
            // (before the observation: an env whose episode ends here and is re-drawn by the auto-reset does not
            //  need this step's rows, so the tile / store below skip it)
            bool reached = false, collided = false, done_agent = false, any_col = false, time_limit = false;
            bool all_reached = false, all_term = false, all_trunc = false, ep_over = false, need_reset = false;
            bool env_active = false;
            double reward = 0.0;
            int sc_new = 0;
            unsigned redraw_envs = 0u;   // fused launch: bit el = env el of the group is re-drawn in pass 1
            if (step_pass()) {
                const bool obst_hit = od[0] <= c_thr_obst;
                reached = alive && curr_d <= P.thr_goal;    // :124-127 (double compare)
                collided = alive && (obst_hit || pair_hit);  // :128
                if (alive) {
                    const double progress = __dmul_rn(__dsub_rn((double)prev_d, (double)curr_d), P.k_p);  // :142
                    double pen = 0.0;  // :210-224
                    if (form_n > 0) {
                        const double mean = form_n == N - 1 ? mean_markstein(form_sum, P.n_others, P.inv_n_others)
                                                            : __ddiv_rn(form_sum, (double)form_n);
                        pen = __dmul_rn(P.neg_k_f, mean);
                    }
                    reward = __dadd_rn(progress, pen);                  // :143
                    if (reached) reward = __dadd_rn(reward, P.r_goal);  // :144-145
                    if (collided) reward = __dadd_rn(reward, P.r_col);  // :146-147
                }
                done_agent = reached || collided;
                any_col = (__ballot_sync(FULL_MASK, collided) & env_lanes) != 0;
                const int n_cont = __popc(__ballot_sync(FULL_MASK, alive && !done_agent) & env_lanes);
                env_active = n_alive_env > 0;
                sc_new = env_active ? sc + 1 : sc;
                time_limit = env_active && sc_new >= P.max_steps;
                all_reached = n_cont == 0 && !any_col && !time_limit;
                const bool episode_done = all_reached || any_col;
                all_term = env_active ? episode_done : true;  // :94-95 when no agent is left
                all_trunc = env_active ? (time_limit && !episode_done) : false;
                ep_over = env_active && (all_term || all_trunc);
                need_reset = P.auto_reset && (ep_over || !env_active);
                if (kFused) {
                    const unsigned nr = __ballot_sync(FULL_MASK, leader && need_reset);
                    if (G == 1) {
                        redraw_envs = nr & 1u;
                    } else {
#pragma unroll
                        for (int el = 0; el < G; ++el) redraw_envs |= ((nr >> (el * N)) & 1u) << el;
                    }
                }
            }

            // ============================ obs row -> staging tile (:226-243) ============================
            // rows this launch delivers: step = every env (fused: minus the ones about to be re-drawn),
            // reset = the re-drawn ones
            const unsigned out_envs = step_pass() ? (((1u << n_env) - 1u) & ~redraw_envs) : reset_envs;
            if (out_envs != 0u) {
                if (lane_ok && (!kFused || ((out_envs >> e_l) & 1u))) {
                    float* row = srow;
                    const float4 t0 = tab2[2 * e_base + nj[0]], t1 = tab2[2 * e_base + nj[1]], t2 = tab2[2 * e_base + nj[2]];
                    const float4 b0 = tobs[om[0]], b1 = tobs[om[1]], b2 = tobs[om[2]], b3 = tobs[om[3]];
                    if (DR) {  // sensor noise of the observed state (step_count sc + 1): the block of counter sc
                        if (!step_pass() || !alive)  // (an active drone drew this block for its thrust already)
                            rA = philox4x32_7(genv, ekey, (unsigned)sc, (unsigned)i | (DR_STREAM_A << 16), P);
                    }
                    auto noisy = [&](float x, float sigma, unsigned idx) {
                        return DR ? __fmaf_rn(sigma, dr_normal_off(qtab, idx), x) : x;
                    };
                    row[0] = noisy(p.x, P.dr_std_pos, dr_field_off(rA, 3)); row[1] = noisy(p.y, P.dr_std_pos, dr_field_off(rA, 4));
                    row[2] = noisy(p.z, P.dr_std_pos, dr_field_off(rA, 5));
                    row[3] = noisy(v.x, P.dr_std_vel, dr_field_off(rA, 6)); row[4] = noisy(v.y, P.dr_std_vel, dr_field_off(rA, 7));
                    row[5] = noisy(v.z, P.dr_std_vel, dr_field_off(rA, 8));
                    row[6] = __fsub_rn(gx, p.x); row[7] = __fsub_rn(gy, p.y); row[8] = __fsub_rn(gz, p.z);
                    row[9] = __fsub_rn(t0.x, p.x); row[10] = __fsub_rn(t0.y, p.y); row[11] = __fsub_rn(t0.z, p.z); row[12] = nd[0];
                    row[13] = __fsub_rn(t1.x, p.x); row[14] = __fsub_rn(t1.y, p.y); row[15] = __fsub_rn(t1.z, p.z); row[16] = nd[1];
                    row[17] = __fsub_rn(t2.x, p.x); row[18] = __fsub_rn(t2.y, p.y); row[19] = __fsub_rn(t2.z, p.z); row[20] = nd[2];
                    row[21] = __fsub_rn(b0.x, p.x); row[22] = __fsub_rn(b0.y, p.y); row[23] = __fsub_rn(b0.z, p.z);
                    row[24] = noisy(od[0], P.dr_std_obst, dr_field_off(rA, 9));
                    row[25] = __fsub_rn(b1.x, p.x); row[26] = __fsub_rn(b1.y, p.y); row[27] = __fsub_rn(b1.z, p.z);
                    row[28] = noisy(od[1], P.dr_std_obst, dr_field_off(rA, 10));
                    row[29] = __fsub_rn(b2.x, p.x); row[30] = __fsub_rn(b2.y, p.y); row[31] = __fsub_rn(b2.z, p.z);
                    row[32] = noisy(od[2], P.dr_std_obst, dr_field_off(rA, 11));
                    row[33] = __fsub_rn(b3.x, p.x); row[34] = __fsub_rn(b3.y, p.y); row[35] = __fsub_rn(b3.z, p.z);
                    row[36] = noisy(od[3], P.dr_std_obst, dr_field_off(rA, 12));
                }
                fence_async_smem();  // generic-proxy tile writes -> visible to the bulk-copy engine
                __syncwarp();
                if (lane == 0) {
                    if (out_envs == (1u << n_env) - 1u) {  // whole tile, one TMA store
                        bulk_s2g(P.obs + (long long)a0 * kD, smem_u32(tile), (unsigned)(n_env * N * kD * 4));
                    } else {
#pragma unroll 1
                        for (int el = 0; el < n_env; ++el)
                            if ((out_envs >> el) & 1u)
                                bulk_s2g(P.obs + (long long)(a0 + el * N) * kD, smem_u32(tile + el * N * kD),
                                         (unsigned)(N * kD * 4));
                    }
                    bulk_commit();
                }
            }

            if (step_pass()) {
                const float rew32 = __double2float_rn(reward);
                float x = rew32;  // deterministic per-env reward sum (segmented tree over the env's lanes)
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const float t = __shfl_down_sync(FULL_MASK, x, off);
                    if (off < N && i + off < N) x = __fadd_rn(x, t);
                }
                if (lane_ok) {
                    P.terminated[a] = (alive && done_agent) ? 1 : 0;                 // :150-151
                    P.truncated[a] = (alive && time_limit && !done_agent) ? 1 : 0;   // :152
                    const bool valid = alive && !done_agent && !time_limit && !any_col;  // :154
                    const bool alive_next = ep_over ? false : valid;                     // :169-172
                    P.reward[a] = rew32;
                    if (P.reward64) P.reward64[a] = reward;
                    P.reached[a] = reached ? 1 : 0;
                    P.collision[a] = collided ? 1 : 0;
                    if (!need_reset) {  // (a re-drawn env gets these from the reset pass / launch that follows)
                        P.dist[a] = curr_d;
                        P.obs_valid[a] = valid ? 1 : 0;
                        P.pos4[a] = make_float4(p.x, p.y, p.z, alive_next ? 1.0f : 0.0f);
                        P.vel4[a] = make_float4(v.x, v.y, v.z, 0.0f);
                        if (kFused && resident) {   // the next step reads its state from the inbox, not from global memory
                            float4* box = const_cast<float4*>(in_pos);
                            box[lane] = make_float4(p.x, p.y, p.z, alive_next ? 1.0f : 0.0f);
                            box[32 + lane] = make_float4(v.x, v.y, v.z, 0.0f);
                        }
                        if (P.gs) {
                            float* row = P.gs + (long long)env * P.R;
                            __stcs(row + 3 * i + 0, p.x); __stcs(row + 3 * i + 1, p.y); __stcs(row + 3 * i + 2, p.z);
                            __stcs(row + 3 * N + 3 * i + 0, v.x); __stcs(row + 3 * N + 3 * i + 1, v.y);
                            __stcs(row + 3 * N + 3 * i + 2, v.z);
                        }
                    }
                }
                if (kLaneOut) {
                    // (one env per warp: every value below is warp-uniform once the reward sum has been broadcast)
                    const float ret = __fadd_rn(reinterpret_cast<const float*>(ib + sc_off)[G + e_l], __shfl_sync(FULL_MASK, x, 0));
                    if (leader && ep_over) {
                        atomicAdd(wstats + SWARM_STAT_EPISODES, 1ull);
                        atomicAdd(wstats + SWARM_STAT_LENGTH_SUM, (unsigned long long)sc_new);
                        atomicAdd(reinterpret_cast<double*>(wstats + SWARM_STAT_RETURN_SUM), (double)ret);
                        if (all_reached) atomicAdd(wstats + SWARM_STAT_SUCCESS, 1ull);
                        if (any_col) atomicAdd(wstats + SWARM_STAT_COLLISION, 1ull);
                        if (all_trunc) atomicAdd(wstats + SWARM_STAT_TIMEOUT, 1ull);
                    }
                    ostage[0] = all_term ? 1u : 0u;
                    ostage[1] = all_trunc ? 1u : 0u;
                    ostage[2] = need_reset ? 1u : 0u;
                    ostage[3] = __float_as_uint(ep_over ? ret : 0.0f);
                    ostage[4] = (unsigned)(ep_over ? sc_new : 0);
                    ostage[5] = (unsigned)sc_new;
                    ostage[6] = __float_as_uint(ep_over ? 0.0f : ret);
                    ostage[7] = __float_as_uint(gx); ostage[8] = __float_as_uint(gy); ostage[9] = __float_as_uint(gz);
                    __syncwarp();
                    if (lane < kLaneOutputs) {
                        const unsigned long long base = optr[lane];
                        // outputs 5 .. 9 (state and global_state) belong to the reset launch when the env is re-drawn
                        if (base != 0ull && (lane < 5 || !need_reset)) {
                            unsigned char* dst = reinterpret_cast<unsigned char*>(base) + (unsigned long long)(unsigned)env * ostride[lane];
                            const unsigned val = ostage[lane];
                            if (lane < 3) *dst = (unsigned char)val;
                            else if (lane < 7) *reinterpret_cast<unsigned*>(dst) = val;
                            else __stcs(reinterpret_cast<unsigned*>(dst), val);
                        }
                    }
                } else if (leader) {
                    P.all_term[env] = all_term ? 1 : 0;
                    P.all_trunc[env] = all_trunc ? 1 : 0;
                    if (!kFused && P.reset_mask) P.reset_mask[env] = need_reset ? 1 : 0;
                    const float ret = __fadd_rn(reinterpret_cast<const float*>(ib + sc_off)[G + e_l], x);
                    if (ep_over) {  // several env leaders per warp when G > 1: shared-memory atomics
                        atomicAdd(wstats + SWARM_STAT_EPISODES, 1ull);
                        atomicAdd(wstats + SWARM_STAT_LENGTH_SUM, (unsigned long long)sc_new);
                        atomicAdd(reinterpret_cast<double*>(wstats + SWARM_STAT_RETURN_SUM), (double)ret);
                        if (all_reached) atomicAdd(wstats + SWARM_STAT_SUCCESS, 1ull);
                        if (any_col) atomicAdd(wstats + SWARM_STAT_COLLISION, 1ull);
                        if (all_trunc) atomicAdd(wstats + SWARM_STAT_TIMEOUT, 1ull);
                    }
                    if (P.episode_return) P.episode_return[env] = ep_over ? ret : 0.0f;
                    if (P.episode_length) P.episode_length[env] = ep_over ? sc_new : 0;
                    if (!need_reset) {
                        P.step_count[env] = sc_new;
                        P.ep_return[env] = ep_over ? 0.0f : ret;
                        if (kFused && resident) {
                            reinterpret_cast<int*>(ib + sc_off)[e_l] = sc_new;
                            reinterpret_cast<float*>(ib + sc_off)[G + e_l] = ep_over ? 0.0f : ret;
                        }
                        if (P.gs) {
                            float* row = P.gs + (long long)env * P.R + 6 * N;
                            __stcs(row + 0, gx); __stcs(row + 1, gy); __stcs(row + 2, gz);
                        }
                    }
                }
                {   // actions applied / envs stepped by this warp in this group
                    const unsigned act_envs = __ballot_sync(FULL_MASK, leader && env_active);
                    if (lane == 0) {
                        wstats[SWARM_STAT_AGENT_STEPS] += (unsigned long long)__popc(alive_mask);
                        wstats[SWARM_STAT_ENV_STEPS] += (unsigned long long)__popc(act_envs);
                    }
                }
                if (!kFused && P.auto_reset) {  // groups with an env to reset go on the list the reset launch walks
                    const unsigned rl = __ballot_sync(FULL_MASK, leader && need_reset);
                    if (rl != 0) {
                        if (lane == 0) wlist[n_local] = env0;
                        if (++n_local == kLocalList) flush_list();
                    }
                }
            } else {
                // =========== reset()'s obs / infos (:82-89) for the re-drawn envs; reward / flags stay ===========
                if (lane_ok && ((reset_envs >> e_l) & 1u)) {
                    P.dist[a] = curr_d;
                    P.obs_valid[a] = 1;
                    P.pos4[a] = make_float4(p.x, p.y, p.z, 1.0f);
                    P.vel4[a] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (kFused && resident) {   // (goal / obstacles / DR constants of the new episode are in the env inbox already)
                        float4* box = const_cast<float4*>(in_pos);
                        box[lane] = make_float4(p.x, p.y, p.z, 1.0f);
                        box[32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (i == 0) {
                            reinterpret_cast<int*>(ib + sc_off)[e_l] = 0;
                            reinterpret_cast<float*>(ib + sc_off)[G + e_l] = 0.0f;
                        }
                    }
                    if (P.gs) {
                        float* row = P.gs + (long long)env * P.R;
                        __stcs(row + 3 * i + 0, p.x); __stcs(row + 3 * i + 1, p.y); __stcs(row + 3 * i + 2, p.z);
                        __stcs(row + 3 * N + 3 * i + 0, 0.f); __stcs(row + 3 * N + 3 * i + 1, 0.f);
                        __stcs(row + 3 * N + 3 * i + 2, 0.f);
                        if (i == 0) { __stcs(row + 6 * N + 0, gx); __stcs(row + 6 * N + 1, gy); __stcs(row + 6 * N + 2, gz); }
                    }
                }
            }
            if (!kFused || pass != 0 || redraw_envs == 0u) break;
            reset_envs = redraw_envs;   // pass 1: env.reset() + observation of the envs whose episode just ended
        }
        if (kFused && ms_steps > 1) {
            // this item's state stores (generic proxy) must be visible to the bulk copies (async proxy) that read them
            // back one step later
            if (!resident) {
                asm volatile("fence.proxy.async.global;" ::: "memory");
                __syncwarp();
                if (ms_own == 1 && it_next < n_iter) issue(it_next, buf ^ 1, ms_tn);
            }
        }
        ms_t = ms_tn; ms_j = ms_jn;
        it = it_next;
        if (!resident) buf ^= 1;
    }
    if (MODE == kRotStep && n_local > 0) flush_list();
#if SWARM_ROT_PDL
    if (kOverlap && !dep_waited) asm volatile("griddepcontrol.wait;" ::: "memory");   // never exit without it
#endif
    // the last warp to leave re-arms the queue for the next launch
    // (no trigger here: a launch that has not triggered early releases its dependents when it has COMPLETED, with its
    //  stores flushed -- the step launch behind it relies on that, it does not wait at its top)
    if (kStepLike) {
        if (lane == 0 && atomicAdd(queue + 1, 1u) == (unsigned)warps_total - 1u) {
            queue[0] = 0u;
            queue[1] = 0u;
            if (MODE == kRotStep && P.auto_reset) {
                // every warp has flushed its list: hand it to the reset launch and clear the other list for the
                // next step (its reader -- the previous step's reset launch -- is done: see the wait below)
                const unsigned ep = *reinterpret_cast<const volatile unsigned*>(P.reset_epoch);
                P.reset_count[(ep + 1u) & 1u] = 0u;
                *P.reset_epoch = ep + 1u;
            }
        }
    }

    if (lane == 0) bulk_wait0();  // the last obs tile must have left shared memory before the CTA retires
    __syncwarp();
    if (kStepLike && P.stats && lane < SWARM_STATS_WORDS) {
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
// host side: eligibility and launch
// ------------------------------------------------------------------------------------------
typedef void (*RotKernel)(const DevParams);

template <int NT, int MODE>
static RotKernel pick_rot_m(const DevParams& p) {
    const int drm = p.dr_enabled == 0 ? 0 : (p.dr_delay_hist > 0 ? 2 : 1);
#define SWARM_PICK_DRM(MT_) \
    (drm == 0 ? swarm_step_rot_kernel<NT, MT_, 0, MODE> : drm == 1 ? swarm_step_rot_kernel<NT, MT_, 1, MODE> : swarm_step_rot_kernel<NT, MT_, 2, MODE>)
    if (p.M == 8) return SWARM_PICK_DRM(8);
    if (p.M == 4) return SWARM_PICK_DRM(4);
    return SWARM_PICK_DRM(0);
#undef SWARM_PICK_DRM
}

static RotKernel pick_rot(const DevParams& p) {
    const bool reset = p.mode == kModeAutoReset;
    const bool fused = p.mode == kModeStep && p.fused_reset != 0;
    switch (p.N) {
        case 8: return reset ? pick_rot_m<8, kRotReset>(p) : fused ? pick_rot_m<8, kRotFused>(p) : pick_rot_m<8, kRotStep>(p);
        case 16: return reset ? pick_rot_m<16, kRotReset>(p) : fused ? pick_rot_m<16, kRotFused>(p) : pick_rot_m<16, kRotStep>(p);
        case 32: return reset ? pick_rot_m<32, kRotReset>(p) : fused ? pick_rot_m<32, kRotFused>(p) : pick_rot_m<32, kRotStep>(p);
    }
    return nullptr;
}

size_t rot_smem_bytes(const DevParams& p) {
    return (size_t)rot_warps(p.N, p.dr_enabled != 0) * rot_smem_per_warp(32 / p.N, p.M, p.dr_enabled != 0) +
           (size_t)rot_warps(p.N, p.dr_enabled != 0) * (SWARM_STATS_WORDS * sizeof(unsigned long long) + 8 * sizeof(int)) +
           ((p.dr_enabled && !SWARM_ROT_DR_QTAB_GLOBAL) ? 2048 : 0) +
           ((p.dr_enabled && !SWARM_ROT_LANE_OUT_DR) ? 0 : (size_t)rot_warps(p.N, p.dr_enabled != 0) * kLaneOutBytes);
}

cudaError_t launch_rot_kernel(const DevParams& p, int grid, cudaStream_t stream) {
    RotKernel k = pick_rot(p);
    if (!k) return cudaErrorInvalidValue;
    const size_t smem = rot_smem_bytes(p);
    cudaError_t err = ensure_dynamic_smem(reinterpret_cast<const void*>(k), smem);
    if (err != cudaSuccess) return err;
#if SWARM_ROT_PDL
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)grid);
    lc.blockDim = dim3((unsigned)(rot_warps(p.N, p.dr_enabled != 0) * 32));
    lc.dynamicSmemBytes = smem;
    lc.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    return cudaLaunchKernelEx(&lc, k, p);
#else
    k<<<grid, rot_warps(p.N, p.dr_enabled != 0) * 32, smem, stream>>>(p);
    return cudaGetLastError();
#endif
}

cudaError_t rot_kernel_occupancy(const DevParams& p, int* blocks_per_sm) {
    RotKernel k = pick_rot(p);
    if (!k) return cudaErrorInvalidValue;
    const size_t smem = rot_smem_bytes(p);
    cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k, rot_warps(p.N, p.dr_enabled != 0) * 32, smem);
}

int rot_warps_per_cta(const DevParams& p) { return rot_warps(p.N, p.dr_enabled != 0); }

}  // namespace swarm
