/*
 * swarm_oracle.c -- CPU restatement of the reference's drone-swarm env step.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity ORACLE for the CUDA path:
 * a plain scalar C restatement of the algorithm in the reference repo
 *   nusRying/Multi-Agent-RL-for-Autonomous-Drone-Swarms
 *     src/swarm_marl/envs/common.py            (DroneEnvConfig)
 *     src/swarm_marl/envs/drone_swarm_env.py   (DroneSwarmEnv)
 *     src/swarm_marl/envs/single_drone_env.py  (SingleDroneEnv)
 * plus the numpy pieces those files lean on (np.random.default_rng = SeedSequence
 * + PCG64 XSL-RR 128/64, Generator.uniform, np.linalg.norm's two code paths,
 * np.mean's pairwise summation, NEP-50 weak-scalar comparisons).  Every function
 * cites the reference file:line it follows.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it; the product
 * package never does.
 *
 * PARITY PIN: tests/test_oracle_golden.py checks this file bit-for-bit against
 * the .npz fixtures under tests/golden/, which oracle/gen_golden.py produced by importing the
 * UNMODIFIED reference (numpy 2.3.5, OpenBLAS 0.3.30 x86-64) in the build
 * container; tests/test_oracle_vs_reference.py re-checks live, on seeds and configs that
 * are not among the fixtures, when /root/reference is present.
 * PARITY UNPINNED for two parts that have no runnable reference: the domain-randomisation
 * streams (configs/domain_randomization_v1.yaml is read by no reference code) and the
 * DronePhysicsEnv restatement (PyBullet is not vendored / installed).  Their semantics are
 * this repo's (DESIGN.md sections 8 and 9); here they only pin the CUDA path.
 *
 * Arithmetic rules restated here (SURVEY.md section 3.4, traps T1-T6):
 *  T1 norm1d  = np.linalg.norm(vec3)  -> sqrt(x.dot(x)) -> OpenBLAS sdot (x86-64
 *               kernel/x86_64/sdot.c tail loop: `double dot; dot += y[i]*x[i]` with
 *               the product rounded to f32 first) -> cast f32 -> sqrtf.
 *  T2 normAxis = np.linalg.norm(A, axis=k) -> sqrt(add.reduce(A*A)) = sequential f32.
 *  T3 thresholds: np.float32-vs-Python-float compares round the Python float to f32;
 *               Python-float-vs-Python-float compares (goal radius) stay in double.
 *  T4 rewards are Python floats (double); np.mean uses numpy's 8-lane pairwise sum.
 *  T5 argsort ties: this oracle breaks ties by lowest index (np.argsort's default
 *               introsort/simd-sort is not stable; ties are counted by the tests).
 *  T6 parked (goal-reached) drones: neighbours yes, colliders / formation no.
 *
 * Build: see oracle/Makefile  (gcc -O2 -ffp-contract=off -fno-fast-math).
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------- */
/* Config: mirror of DroneEnvConfig (envs/common.py:7-25) + num_drones        */
/* (drone_swarm_env.py:32) + oracle-only switches.                            */
/* ------------------------------------------------------------------------- */
#define ORACLE_MAX_DRONES 1024   /* scratch bound of this restatement */
#define ORACLE_MAX_OBSTACLES 256

typedef struct OracleConfig {
    double world_size, dt, max_speed, max_accel, collision_radius, goal_radius;
    double obstacle_radius, desired_spacing;
    double reward_progress_scale, reward_goal, reward_collision, reward_formation_scale;
    int32_t max_steps, num_obstacles, sensed_obstacles, neighbor_k;
    int32_t num_drones;
    int32_t env_kind;  /* 0 = SingleDroneEnv, 1 = DroneSwarmEnv, 2 = DronePhysicsEnv (point-mass restatement) */
    int32_t norm_mode; /* 0 = BLAS sdot (double accumulate), 1 = sequential f32 */
    int32_t reserved;
    /* domain randomisation: NOT reference behaviour (configs/domain_randomization_v1.yaml is read by no
     * reference code).  These semantics are the engine's (DESIGN.md section 8); this restatement only
     * pins the CUDA path to them.  dr_enabled == 0 -> everything below is ignored. */
    int32_t dr_enabled;
    int32_t dr_pad;
    uint64_t dr_seed;
    int64_t env_index_base;
    double dr_lo[6], dr_span[6]; /* mass, max_accel, max_speed, dt, obstacle_radius, world_size scales */
    double dr_std_thrust, dr_std_pos, dr_std_vel, dr_std_obst;
    /* control delay (yaml actuation.control_delay_steps): per episode a delay d is drawn from the discrete
     * distribution {values[k] with probability probs[k]}; the command applied at step t is the one
     * submitted at step t - d (zero while the episode is younger than d steps) */
    int32_t dr_delay_count;      /* 0 = no control delay */
    int32_t dr_delay_hist;       /* ring size of the command history = max(values), >= 1 when count > 0 */
    int32_t dr_delay_values[4];
    double dr_delay_cum[4];      /* cumulative probabilities */
} OracleConfig;

/* One batch of E environments, arrays laid out exactly like the reference's
 * numpy attributes with a leading env axis. */
typedef struct OracleBatch {
    int32_t num_envs;
    int32_t pad;
    float *positions;    /* [E][N][3]  DroneSwarmEnv.positions  (drone_swarm_env.py:59) */
    float *velocities;   /* [E][N][3]  .velocities (:60) */
    float *goal;         /* [E][3]     .goal (:61) */
    float *obstacles;    /* [E][M][3]  .obstacles (:62) */
    int32_t *step_count; /* [E]        .step_count (:63) */
    uint8_t *active;     /* [E][N]     membership of drone_i in .agents (:39,169-172) */
    uint64_t *rng;       /* [E][4]     PCG64 {state_hi, state_lo, inc_hi, inc_lo} */
    /* outputs of the last reset/step */
    float *obs;          /* [E][N][D]  D = 9 + 4K + 4S (swarm) or 9 + 4S (single) */
    double *reward;      /* [E][N]     Python-float rewards */
    float *dist;         /* [E][N]     info["distance_to_goal"] (f32-valued) */
    uint8_t *terminated; /* [E][N] */
    uint8_t *truncated;  /* [E][N] */
    uint8_t *reached;    /* [E][N]     info["reached_goal"] */
    uint8_t *collision;  /* [E][N]     info["collision"] */
    uint8_t *obs_valid;  /* [E][N]     1 where the reference would put agent i in the obs dict */
    uint8_t *all_terminated; /* [E]    terminated["__all__"] */
    uint8_t *all_truncated;  /* [E]    truncated["__all__"] */
    float *global_state; /* [E][6N+3]  info["global_state"] (drone_swarm_env.py:293-302) */
    float *dr_params;    /* [E][8]     DR only: {max_accel, max_speed, dt, bound, obst threshold, key, world, 0} */
    float *damp;         /* [E][N]     physics env only: per-drone velocity factor of one 1/240 s sub-step */
    float *act_hist;     /* [E][H][N][3] control delay only: ring of the last H submitted commands */
} OracleBatch;

/* ------------------------------------------------------------------------- */
/* numpy.random: SeedSequence + PCG64 + Generator.uniform                     */
/* (used by `np.random.default_rng(seed)` drone_swarm_env.py:35,66-67 and      */
/*  single_drone_env.py:31,55-57)                                              */
/* ------------------------------------------------------------------------- */
typedef unsigned __int128 u128;

#define SS_INIT_A 0x43b0d7e5u
#define SS_MULT_A 0x931e8875u
#define SS_INIT_B 0x8b51f9ddu
#define SS_MULT_B 0x58f38dedu
#define SS_MIX_L 0xca01f9ddu
#define SS_MIX_R 0x4973f715u
#define SS_XSHIFT 16
#define SS_POOL 4

static uint32_t ss_hashmix(uint32_t value, uint32_t *hash_const) {
    value ^= *hash_const;
    *hash_const *= SS_MULT_A;
    value *= *hash_const;
    value ^= value >> SS_XSHIFT;
    return value;
}

static uint32_t ss_mix(uint32_t x, uint32_t y) {
    uint32_t r = SS_MIX_L * x - SS_MIX_R * y;
    r ^= r >> SS_XSHIFT;
    return r;
}

/* numpy/random/bit_generator.pyx: SeedSequence.mix_entropy + generate_state(4, uint64)
 * followed by PCG64's pcg64_set_seed / pcg_setseq_128_srandom_r. */
void oracle_seed(uint64_t seed, uint64_t rng[4]) {
    uint32_t entropy[2];
    int n_ent = 1;
    entropy[0] = (uint32_t)(seed & 0xffffffffu);
    entropy[1] = (uint32_t)(seed >> 32);
    if (entropy[1] != 0) n_ent = 2;

    uint32_t pool[SS_POOL];
    uint32_t hc = SS_INIT_A;
    for (int i = 0; i < SS_POOL; ++i) pool[i] = ss_hashmix(i < n_ent ? entropy[i] : 0u, &hc);
    for (int s = 0; s < SS_POOL; ++s)
        for (int d = 0; d < SS_POOL; ++d)
            if (s != d) pool[d] = ss_mix(pool[d], ss_hashmix(pool[s], &hc));
    /* (entropy longer than the pool does not occur for 64-bit seeds) */

    uint32_t words[8];
    hc = SS_INIT_B;
    for (int i = 0; i < 8; ++i) {
        uint32_t v = pool[i % SS_POOL];
        v ^= hc;
        hc *= SS_MULT_B;
        v *= hc;
        v ^= v >> SS_XSHIFT;
        words[i] = v;
    }
    uint64_t w64[4];
    for (int i = 0; i < 4; ++i) w64[i] = (uint64_t)words[2 * i] | ((uint64_t)words[2 * i + 1] << 32);

    const u128 mult = ((u128)2549297995355413924ULL << 64) | (u128)4865540595714422341ULL;
    u128 initstate = ((u128)w64[0] << 64) | w64[1];
    u128 initseq = ((u128)w64[2] << 64) | w64[3];
    u128 inc = (initseq << 1) | 1u;
    u128 state = 0;
    state = state * mult + inc;
    state += initstate;
    state = state * mult + inc;
    rng[0] = (uint64_t)(state >> 64);
    rng[1] = (uint64_t)state;
    rng[2] = (uint64_t)(inc >> 64);
    rng[3] = (uint64_t)inc;
}

/* pcg64_next64: advance, then XSL-RR output of the new state. */
uint64_t oracle_pcg64_next(uint64_t rng[4]) {
    const u128 mult = ((u128)2549297995355413924ULL << 64) | (u128)4865540595714422341ULL;
    u128 state = ((u128)rng[0] << 64) | rng[1];
    u128 inc = ((u128)rng[2] << 64) | rng[3];
    state = state * mult + inc;
    rng[0] = (uint64_t)(state >> 64);
    rng[1] = (uint64_t)state;
    uint64_t hi = rng[0], lo = rng[1];
    uint64_t x = hi ^ lo;
    unsigned rot = (unsigned)(hi >> 58);
    return (x >> rot) | (x << ((-rot) & 63));
}

/* Generator.uniform(low, high) -> random_uniform: low + (high-low) * next_double,
 * next_double = (next_uint64 >> 11) * 2^-53; then `.astype(np.float32)`
 * (drone_swarm_env.py:72-80, single_drone_env.py:59-66). */
static float draw_uniform_f32(uint64_t rng[4], double lo, double range) {
    double u = (double)(oracle_pcg64_next(rng) >> 11) * (1.0 / 9007199254740992.0);
    volatile double scaled = range * u; /* no FMA contraction */
    double v = lo + scaled;
    return (float)v;
}

/* ------------------------------------------------------------------------- */
/* Domain randomisation streams (engine semantics, see OracleConfig)          */
/* ------------------------------------------------------------------------- */
/* Philox4x32 (Salmon et al., SC'11) with `rounds` rounds: 10 for the per-episode block (one per reset), 7 for the
 * per-step noise blocks (one per agent-step; 7 is the smallest round count the paper reports as Crush-resistant) */
static void philox4x32_r(uint32_t c[4], uint32_t k0, uint32_t k1, int rounds) {
    for (int r = 0; r < rounds; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
static void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) { philox4x32_r(c, k0, k1, 10); }
static void philox4x32_7(uint32_t c[4], uint32_t k0, uint32_t k1) { philox4x32_r(c, k0, k1, 7); }

static double inv_norm_cdf(double p) { /* Acklam's rational approximation */
    static const double a[] = {-3.969683028665376e+01, 2.209460984245205e+02, -2.759285104469687e+02,
                               1.383577518672690e+02, -3.066479806614716e+01, 2.506628277459239e+00};
    static const double b[] = {-5.447609879822406e+01, 1.615858368580409e+02, -1.556989798598866e+02,
                               6.680131188771972e+01, -1.328068155288572e+01};
    static const double c[] = {-7.784894002430293e-03, -3.223964580411365e-01, -2.400758277161838e+00,
                               -2.549732539343734e+00, 4.374664141464968e+00, 2.938163982698783e+00};
    static const double d[] = {7.784695709041462e-03, 3.224671290700398e-01, 2.445134137142996e+00,
                               3.754408661907416e+00};
    const double plow = 0.02425;
    if (p < plow) {
        double q = sqrt(-2.0 * log(p));
        return (((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) /
               ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1.0);
    }
    if (p > 1.0 - plow) {
        double q = sqrt(-2.0 * log(1.0 - p));
        return -(((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) /
               ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1.0);
    }
    double q = p - 0.5, r = q * q;
    return (((((a[0] * r + a[1]) * r + a[2]) * r + a[3]) * r + a[4]) * r + a[5]) * q /
           (((((b[0] * r + b[1]) * r + b[2]) * r + b[3]) * r + b[4]) * r + 1.0);
}

static float g_qtable[256];
static pthread_once_t g_qtable_once = PTHREAD_ONCE_INIT;
static void qtable_init(void) {
    for (int k = 0; k < 256; ++k) g_qtable[k] = (float)inv_norm_cdf(0.5 + ((double)k + 0.5) / 512.0);
}
static const float *qtable(void) {
    pthread_once(&g_qtable_once, qtable_init);
    return g_qtable;
}
void oracle_dr_quantile_table(float *out) { memcpy(out, qtable(), sizeof(float) * 256); }

/* per-env, per-episode view of the dynamics constants */
typedef struct DynConst {
    float amax, vmax, dt, bound, thr_obst;
    int dr;             /* randomisation on */
    uint32_t genv, ekey, k0, k1;
    float std_thrust, std_pos, std_vel, std_obst;
} DynConst;

/* 9-bit field f of a 128-bit Philox block (word 0 = bits 0-31) -> standard normal: sign = bit 8,
 * magnitude = half-normal quantile table[bits 0-7] */
static float dr_normal(const uint32_t r[4], int f) {
    int b = 9 * f, k = b >> 5, sh = b & 31;
    uint32_t v = r[k] >> sh;
    if (sh > 23) v |= r[k + 1] << (32 - sh);
    float q = qtable()[v & 0xFFu];
    return (v & 0x100u) ? -q : q;
}

/* ------------------------------------------------------------------------- */
/* np.linalg.norm restatements (T1, T2)                                       */
/* ------------------------------------------------------------------------- */
static float norm1d(const OracleConfig *c, float x, float y, float z) {
    /* np.linalg.norm(vec) with axis=None: sqrt(vec.dot(vec)) */
    volatile float px = x * x, py = y * y, pz = z * z;
    float s;
    if (c->norm_mode == 0) {
        volatile double acc = 0.0;
        acc = acc + (double)px;
        acc = acc + (double)py;
        acc = acc + (double)pz;
        s = (float)acc;
    } else {
        volatile float a = px + py;
        s = a + pz;
    }
    return sqrtf(s);
}

static float norm_axis(float x, float y, float z) {
    /* np.linalg.norm(A, axis=-1): sqrt(add.reduce(A*A, axis)) -- sequential f32 */
    volatile float px = x * x, py = y * y, pz = z * z;
    volatile float a = px + py;
    volatile float s = a + pz;
    return sqrtf(s);
}

/* np.add.reduce over a contiguous double vector: numpy's pairwise_sum
 * (numpy/_core/src/umath/loops_utils.h.src) -- what np.mean uses at
 * drone_swarm_env.py:222. */
static double np_pairwise_sum(const double *a, int n) {
    if (n < 8) {
        double r = -0.0;
        for (int i = 0; i < n; ++i) r += a[i];
        return r;
    } else if (n <= 128) {
        double r[8];
        int i;
        for (i = 0; i < 8; ++i) r[i] = a[i];
        for (i = 8; i < n - (n % 8); i += 8)
            for (int k = 0; k < 8; ++k) r[k] += a[i + k];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; ++i) res += a[i];
        return res;
    } else {
        int n2 = n / 2;
        n2 -= n2 % 8;
        return np_pairwise_sum(a, n2) + np_pairwise_sum(a + n2, n - n2);
    }
}

static int obs_dim(const OracleConfig *c) {
    /* drone_swarm_env.py:41-45 ; single_drone_env.py:33 */
    return c->env_kind != 0 ? 9 + 4 * c->neighbor_k + 4 * c->sensed_obstacles
                            : 9 + 4 * c->sensed_obstacles;
}

/* ------------------------------------------------------------------------- */
/* Observation pieces                                                         */
/* ------------------------------------------------------------------------- */

/* np.argsort's order of two distances: a ranks strictly after b.  NaN sorts after every number (+inf
 * included), so a NaN candidate is picked only when there are not enough numbers; NaNs tie with each other. */
static int ranks_after(float a, float b) {
    if (isnan(a)) return !isnan(b);
    return a > b;
}

/* _nearest_obstacle_features  drone_swarm_env.py:273-291 / single_drone_env.py:142-159 */
static void nearest_obstacle_features(const OracleConfig *c, const float *own, const float *obst,
                                      float *out) {
    int S = c->sensed_obstacles, M = c->num_obstacles;
    for (int k = 0; k < 4 * S; ++k) out[k] = 0.0f;
    if (M == 0 || S <= 0) return;
    float dist[ORACLE_MAX_OBSTACLES];
    int order[ORACLE_MAX_OBSTACLES];
    for (int m = 0; m < M; ++m) {
        float rx = obst[3 * m] - own[0], ry = obst[3 * m + 1] - own[1], rz = obst[3 * m + 2] - own[2];
        dist[m] = norm_axis(rx, ry, rz);
        order[m] = m;
    }
    /* stable insertion sort == argsort with lowest-index tie break, NaN last */
    for (int a = 1; a < M; ++a) {
        int key = order[a], b = a - 1;
        while (b >= 0 && ranks_after(dist[order[b]], dist[key])) { order[b + 1] = order[b]; --b; }
        order[b + 1] = key;
    }
    int k = S < M ? S : M;
    for (int q = 0; q < k; ++q) {
        int m = order[q];
        out[4 * q + 0] = obst[3 * m] - own[0];
        out[4 * q + 1] = obst[3 * m + 1] - own[1];
        out[4 * q + 2] = obst[3 * m + 2] - own[2];
        out[4 * q + 3] = dist[m];
    }
}

/* _nearest_neighbor_features  drone_swarm_env.py:245-271 (all drones j != i, parked included) */
static void nearest_neighbor_features(const OracleConfig *c, const float *pos, int index, float *out) {
    int K = c->neighbor_k, N = c->num_drones;
    for (int k = 0; k < 4 * K; ++k) out[k] = 0.0f;
    if (N <= 1 || K <= 0) return;
    int n = N - 1;
    float dist[ORACLE_MAX_DRONES];
    int who[ORACLE_MAX_DRONES], order[ORACLE_MAX_DRONES];
    const float *own = pos + 3 * index;
    int cnt = 0;
    for (int j = 0; j < N; ++j) {
        if (j == index) continue;
        float vx = pos[3 * j] - own[0], vy = pos[3 * j + 1] - own[1], vz = pos[3 * j + 2] - own[2];
        dist[cnt] = norm1d(c, vx, vy, vz);
        who[cnt] = j;
        order[cnt] = cnt;
        ++cnt;
    }
    for (int a = 1; a < n; ++a) {
        int key = order[a], b = a - 1;
        while (b >= 0 && ranks_after(dist[order[b]], dist[key])) { order[b + 1] = order[b]; --b; }
        order[b + 1] = key;
    }
    int k = K < n ? K : n;
    for (int q = 0; q < k; ++q) {
        int j = who[order[q]];
        out[4 * q + 0] = pos[3 * j] - own[0];
        out[4 * q + 1] = pos[3 * j + 1] - own[1];
        out[4 * q + 2] = pos[3 * j + 2] - own[2];
        out[4 * q + 3] = dist[order[q]];
    }
}

/* _build_obs  drone_swarm_env.py:226-243 / single_drone_env.py:128-140 */
static void build_obs(const OracleConfig *c, const DynConst *kc, int step_obs, const float *pos, const float *vel,
                      const float *goal, const float *obst, int index, float *out) {
    const float *p = pos + 3 * index, *v = vel + 3 * index;
    out[0] = p[0]; out[1] = p[1]; out[2] = p[2];
    out[3] = v[0]; out[4] = v[1]; out[5] = v[2];
    if (c->env_kind == 2) { /* drone_physics_env.py:436-439: the observed velocity is clamped to max_speed */
        float speed = norm1d(c, v[0], v[1], v[2]);
        float vmax = kc->vmax;   /* (DR: this episode's) */
        if (speed > vmax)
            for (int k = 0; k < 3; ++k) {
                volatile float q = v[k] / speed;
                out[3 + k] = q * vmax;
            }
    }
    out[6] = goal[0] - p[0]; out[7] = goal[1] - p[1]; out[8] = goal[2] - p[2];
    int off = 9;
    if (c->env_kind != 0) {
        nearest_neighbor_features(c, pos, index, out + off);
        off += 4 * c->neighbor_k;
    }
    nearest_obstacle_features(c, p, obst, out + off);
    if (kc->dr) {
        /* DR sensor noise of the observed state: Philox block of counter (genv, ekey, step_count - 1,
         * drone | stream << 16); stream A fields 3-5 position, 6-8 velocity, 9-12 sensed obstacle 0-3;
         * stream B field q - 4 = sensed obstacle q >= 4 */
        uint32_t ra[4] = {kc->genv, kc->ekey, (uint32_t)(step_obs - 1), (uint32_t)index};
        uint32_t rb[4] = {kc->genv, kc->ekey, (uint32_t)(step_obs - 1), (uint32_t)index | (1u << 16)};
        philox4x32_7(ra, kc->k0, kc->k1);
        philox4x32_7(rb, kc->k0, kc->k1);
        /* x + sigma z with ONE rounding (fused multiply-add) */
        for (int k = 0; k < 3; ++k) {
            out[k] = fmaf(kc->std_pos, dr_normal(ra, 3 + k), out[k]);
            out[3 + k] = fmaf(kc->std_vel, dr_normal(ra, 6 + k), out[3 + k]);
        }
        int filled = c->sensed_obstacles < c->num_obstacles ? c->sensed_obstacles : c->num_obstacles;
        for (int q = 0; q < filled; ++q)
            out[off + 4 * q + 3] = fmaf(kc->std_obst, q < 4 ? dr_normal(ra, 9 + q) : dr_normal(rb, q - 4),
                                        out[off + 4 * q + 3]);
    }
}

/* _distance_to_goal  drone_swarm_env.py:176-177 / single_drone_env.py:113-114 */
static float distance_to_goal(const OracleConfig *c, const float *goal, const float *p) {
    return norm1d(c, goal[0] - p[0], goal[1] - p[1], goal[2] - p[2]);
}

/* _global_state  drone_swarm_env.py:293-302 */
static void global_state(const OracleConfig *c, const float *pos, const float *vel, const float *goal,
                         float *out) {
    int N = c->num_drones;
    memcpy(out, pos, sizeof(float) * 3 * (size_t)N);
    memcpy(out + 3 * N, vel, sizeof(float) * 3 * (size_t)N);
    memcpy(out + 6 * N, goal, sizeof(float) * 3);
}

/* _clip_speed  drone_swarm_env.py:179-183 / single_drone_env.py:116-120 */
static void clip_speed(const OracleConfig *c, const DynConst *k, float *v) {
    float speed = norm1d(c, v[0], v[1], v[2]);
    float vmax = k->vmax; /* (float)max_speed: np.float32 <= python float -> f32 compare (NEP 50) */
    if (speed <= vmax || speed < (float)1e-8) return;
    for (int k = 0; k < 3; ++k) {
        volatile float q = v[k] / speed;
        v[k] = q * vmax;
    }
}

static float clipf(float x, float lo, float hi) {
    /* np.clip == minimum(maximum(x, lo), hi); NaN propagates */
    if (x < lo) return lo;
    if (x > hi) return hi;
    return x;
}

/* integrate block  drone_swarm_env.py:103-111 / single_drone_env.py:74-84
 * (DR: thrust noise a <- a * (1 + sigma z), stream (genv, ekey, step_count before the step, drone)) */
static void integrate(const OracleConfig *c, const DynConst *kc, int step_before, int drone, const float *action,
                      float *p, float *v) {
    float amax = kc->amax, dt = kc->dt;
    uint32_t ctr[4] = {kc->genv, kc->ekey, (uint32_t)step_before, (uint32_t)drone};
    if (kc->dr) philox4x32_7(ctr, kc->k0, kc->k1);
    for (int k = 0; k < 3; ++k) {
        float a = clipf(action[k], -1.0f, 1.0f);
        if (kc->dr) {
            volatile float one = fmaf(kc->std_thrust, dr_normal(ctr, k), 1.0f);   /* 1 + sigma z, one rounding */
            a = a * one;
        }
        volatile float accel = a * amax;
        volatile float dv = accel * dt;
        v[k] = v[k] + dv;
    }
    clip_speed(c, kc, v);
    for (int k = 0; k < 3; ++k) {
        volatile float dp = v[k] * dt;
        p[k] = p[k] + dp;
    }
}

/* ------------------------------------------------------------------------- */
/* Per-env views                                                              */
/* ------------------------------------------------------------------------- */
typedef struct EnvView {
    float *pos, *vel, *goal, *obst;
    int32_t *step_count;
    uint8_t *active;
    uint64_t *rng;
    float *obs, *dist, *gs;
    double *reward;
    uint8_t *terminated, *truncated, *reached, *collision, *obs_valid, *all_term, *all_trunc;
    float *dr;
    float *damp;
    float *act_hist;
    int env_index;
} EnvView;

static EnvView view(const OracleConfig *c, const OracleBatch *b, int e) {
    int N = c->num_drones, M = c->num_obstacles, D = obs_dim(c);
    EnvView v;
    v.pos = b->positions + (size_t)e * N * 3;
    v.vel = b->velocities + (size_t)e * N * 3;
    v.goal = b->goal + (size_t)e * 3;
    v.obst = b->obstacles + (size_t)e * M * 3;
    v.step_count = b->step_count + e;
    v.active = b->active + (size_t)e * N;
    v.rng = b->rng + (size_t)e * 4;
    v.obs = b->obs + (size_t)e * N * D;
    v.dist = b->dist + (size_t)e * N;
    v.gs = b->global_state ? b->global_state + (size_t)e * (6 * N + 3) : NULL;
    v.reward = b->reward + (size_t)e * N;
    v.terminated = b->terminated + (size_t)e * N;
    v.truncated = b->truncated + (size_t)e * N;
    v.reached = b->reached + (size_t)e * N;
    v.collision = b->collision + (size_t)e * N;
    v.obs_valid = b->obs_valid + (size_t)e * N;
    v.all_term = b->all_terminated + e;
    v.all_trunc = b->all_truncated + e;
    v.dr = b->dr_params ? b->dr_params + (size_t)e * 8 : NULL;
    v.damp = b->damp ? b->damp + (size_t)e * N : NULL;
    v.act_hist = (b->act_hist && c->dr_delay_hist > 0) ? b->act_hist + (size_t)e * c->dr_delay_hist * N * 3 : NULL;
    v.env_index = e;
    return v;
}

/* control delay: the command applied at step t (= step_count before the step) is the one submitted at
 * t - d; the ring slot t % H then takes the command submitted now.  out = 3 floats. */
static void delayed_command(const OracleConfig *c, const EnvView *v, int drone, const float *submitted, float *out) {
    int N = c->num_drones, H = c->dr_delay_hist;
    int d = (c->dr_enabled && v->dr && v->act_hist) ? (int)v->dr[7] : 0;
    int t = *v->step_count;
    if (d == 0) { out[0] = submitted[0]; out[1] = submitted[1]; out[2] = submitted[2]; }
    else if (t < d) { out[0] = out[1] = out[2] = 0.0f; }
    else {
        const float *h = v->act_hist + ((size_t)((t - d) % H) * N + drone) * 3;
        out[0] = h[0]; out[1] = h[1]; out[2] = h[2];
    }
    if (v->act_hist) {
        float *w = v->act_hist + ((size_t)(t % H) * N + drone) * 3;
        w[0] = submitted[0]; w[1] = submitted[1]; w[2] = submitted[2];
    }
}

/* the dynamics constants of one env: the config's, or (DR) this episode's */
static DynConst dyn_const(const OracleConfig *c, const EnvView *v) {
    DynConst k;
    memset(&k, 0, sizeof(k));
    k.amax = (float)c->max_accel;
    k.vmax = (float)c->max_speed;
    k.dt = (float)c->dt;
    k.bound = (float)(c->world_size / 2.0);
    k.thr_obst = (float)(c->collision_radius + c->obstacle_radius);
    if (c->dr_enabled && v->dr) {
        uint32_t key_bits;
        memcpy(&key_bits, v->dr + 5, 4);
        k.dr = 1;
        k.amax = v->dr[0]; k.vmax = v->dr[1]; k.dt = v->dr[2]; k.bound = v->dr[3]; k.thr_obst = v->dr[4];
        k.ekey = key_bits;
        k.genv = (uint32_t)(c->env_index_base + v->env_index);
        k.k0 = (uint32_t)(c->dr_seed & 0xffffffffu);
        k.k1 = (uint32_t)(c->dr_seed >> 32);
        k.std_thrust = (float)c->dr_std_thrust; k.std_pos = (float)c->dr_std_pos;
        k.std_vel = (float)c->dr_std_vel; k.std_obst = (float)c->dr_std_obst;
    }
    return k;
}

/* obs + info for every drone of one env (what reset() returns, and what the
 * batched contract reports after set_state):  drone_swarm_env.py:82-89. */
static void observe_env(const OracleConfig *c, EnvView *v) {
    int N = c->num_drones, D = obs_dim(c);
    DynConst kc = dyn_const(c, v);
    for (int i = 0; i < N; ++i) {
        build_obs(c, &kc, *v->step_count, v->pos, v->vel, v->goal, v->obst, i, v->obs + (size_t)i * D);
        v->dist[i] = distance_to_goal(c, v->goal, v->pos + 3 * i);
        v->obs_valid[i] = c->env_kind == 1 ? v->active[i] : 1;  /* the physics env observes every drone, always */
        v->reward[i] = 0.0;
        v->terminated[i] = v->truncated[i] = v->reached[i] = v->collision[i] = 0;
    }
    *v->all_term = 0;
    *v->all_trunc = 0;
    if (v->gs) global_state(c, v->pos, v->vel, v->goal, v->gs);
}

/* DR: this episode's constants from one Philox counter per (global env, PCG64 state_lo before the reset draws):
 * dr[0..7] = {max_accel s_acc / s_mass, max_speed s_spd, dt s_dt, world s_wld / 2, r_c + r_o s_rad, episode key,
 * world s_wld, control delay}.  base_dt / r_c: the kinematic envs pass cfg.dt / cfg.collision_radius, the physics env
 * its sub-step 1/240 s / the drone's contact radius.  Returns the half width of this episode's world. */
static double draw_episode_constants(const OracleConfig *c, EnvView *v, double base_dt, double r_c) {
    /* counter = (genv, PCG64 state_lo before the draws, 0xD5D5D5D5 [+1]) */
    uint32_t genv = (uint32_t)(c->env_index_base + v->env_index);
    uint32_t k0 = (uint32_t)(c->dr_seed & 0xffffffffu), k1 = (uint32_t)(c->dr_seed >> 32);
    uint64_t sl = v->rng[1];
    uint32_t ra[4] = {genv, (uint32_t)sl, (uint32_t)(sl >> 32), 0xD5D5D5D5u};
    uint32_t rb[4] = {genv, (uint32_t)sl, (uint32_t)(sl >> 32), 0xD5D5D5D5u + 1u};
    philox4x32_10(ra, k0, k1);
    philox4x32_10(rb, k0, k1);
    const double inv24 = 1.0 / 16777216.0;
    uint32_t u[6] = {ra[0], ra[1], ra[2], ra[3], rb[0], rb[1]};
    double sc[6];
    for (int k = 0; k < 6; ++k) {
        volatile double uu = (double)(u[k] >> 8) * inv24;
        volatile double sp = c->dr_span[k] * uu;
        sc[k] = c->dr_lo[k] + sp;
    }
    volatile double acc = c->max_accel * sc[1];
    volatile double spd = c->max_speed * sc[2];
    volatile double dtt = base_dt * sc[3];
    volatile double rad = c->obstacle_radius * sc[4];
    volatile double world = c->world_size * sc[5];
    volatile double half_w = world * 0.5;
    v->dr[0] = (float)(acc / sc[0]);
    v->dr[1] = (float)spd;
    v->dr[2] = (float)dtt;
    v->dr[3] = (float)half_w;
    v->dr[4] = (float)(r_c + rad);
    memcpy(v->dr + 5, &rb[2], 4);
    v->dr[6] = (float)world;
    v->dr[7] = 0.0f;
    if (c->dr_delay_count > 0) { /* this episode's control delay from the 4th word of the second block */
        double uu = (double)(rb[3] >> 8) * inv24;
        int pick = c->dr_delay_count - 1;
        for (int k = 0; k < c->dr_delay_count; ++k)
            if (uu < c->dr_delay_cum[k]) { pick = k; break; }
        v->dr[7] = (float)c->dr_delay_values[pick];
    }
    return half_w;
}

/* reset  drone_swarm_env.py:65-90 / single_drone_env.py:53-71.
 * Draw order: positions (N,3) -> goal (3,) -> obstacles (M,3). */
static void reset_env_physics(const OracleConfig *c, EnvView *v);
static void reset_env(const OracleConfig *c, EnvView *v) {
    int N = c->num_drones, M = c->num_obstacles;
    double bound = c->world_size / 2.0;
    if (c->env_kind == 2) { reset_env_physics(c, v); return; }
    if (c->dr_enabled && v->dr) bound = draw_episode_constants(c, v, c->dt, c->collision_radius);
    double lo = -bound, range = bound - (-bound);
    for (int i = 0; i < N; ++i) v->active[i] = 1;
    *v->step_count = 0;
    for (int k = 0; k < 3 * N; ++k) v->pos[k] = draw_uniform_f32(v->rng, lo, range);
    for (int k = 0; k < 3 * N; ++k) v->vel[k] = 0.0f;
    for (int k = 0; k < 3; ++k) v->goal[k] = draw_uniform_f32(v->rng, lo, range);
    for (int k = 0; k < 3 * M; ++k) v->obst[k] = draw_uniform_f32(v->rng, lo, range);
    observe_env(c, v);
}

/* _collision_mask  drone_swarm_env.py:185-208 (over active drones only) */
static void collision_mask(const OracleConfig *c, const DynConst *kc, const EnvView *v, uint8_t *collided) {
    int N = c->num_drones, M = c->num_obstacles;
    float thr_obst = kc->thr_obst; /* (float)(r_c + r_o): array <= py float */
    float thr_pair = (float)(2.0 * c->collision_radius);                /* np.float32 <= py float */
    for (int i = 0; i < N; ++i) collided[i] = 0;
    for (int i = 0; i < N; ++i) {
        if (!v->active[i]) continue;
        for (int m = 0; m < M; ++m) {
            float d = norm_axis(v->pos[3 * i] - v->obst[3 * m], v->pos[3 * i + 1] - v->obst[3 * m + 1],
                                v->pos[3 * i + 2] - v->obst[3 * m + 2]);
            if (d <= thr_obst) collided[i] = 1;
        }
    }
    for (int i = 0; i < N; ++i) {
        if (!v->active[i]) continue;
        for (int j = i + 1; j < N; ++j) {
            if (!v->active[j]) continue;
            float d = norm1d(c, v->pos[3 * i] - v->pos[3 * j], v->pos[3 * i + 1] - v->pos[3 * j + 1],
                             v->pos[3 * i + 2] - v->pos[3 * j + 2]);
            if (d <= thr_pair) { collided[i] = 1; collided[j] = 1; }
        }
    }
}

/* _formation_penalties  drone_swarm_env.py:210-224 */
static void formation_penalties(const OracleConfig *c, const EnvView *v, double *pen) {
    int N = c->num_drones, n_active = 0;
    for (int i = 0; i < N; ++i) { pen[i] = 0.0; n_active += v->active[i] ? 1 : 0; }
    if (n_active <= 1) return;
    double errs[ORACLE_MAX_DRONES];
    for (int i = 0; i < N; ++i) {
        if (!v->active[i]) continue;
        int n = 0;
        for (int j = 0; j < N; ++j) {
            if (j == i || !v->active[j]) continue;
            double d = (double)norm1d(c, v->pos[3 * i] - v->pos[3 * j], v->pos[3 * i + 1] - v->pos[3 * j + 1],
                                      v->pos[3 * i + 2] - v->pos[3 * j + 2]);
            errs[n++] = fabs(d - c->desired_spacing);
        }
        if (n > 0) {
            double spacing_error = np_pairwise_sum(errs, n) / (double)n;
            pen[i] = -c->reward_formation_scale * spacing_error;
        }
    }
}

/* DroneSwarmEnv.step  drone_swarm_env.py:92-174.  `action` is [N][3] f32 (a missing
 * dict key is a zero row, :104). */
static void step_swarm_env(const OracleConfig *c, EnvView *v, const float *action) {
    int N = c->num_drones, D = obs_dim(c);
    int n_active = 0;
    for (int i = 0; i < N; ++i) n_active += v->active[i] ? 1 : 0;
    for (int i = 0; i < N; ++i) {
        v->reward[i] = 0.0;
        v->terminated[i] = v->truncated[i] = v->reached[i] = v->collision[i] = v->obs_valid[i] = 0;
    }
    if (n_active == 0) { /* :94-95 */
        *v->all_term = 1;
        *v->all_trunc = 0;
        return;
    }
    double *prev = (double *)malloc(sizeof(double) * (size_t)N);
    double *curr = (double *)malloc(sizeof(double) * (size_t)N);
    double *pen = (double *)malloc(sizeof(double) * (size_t)N);
    uint8_t *collided = (uint8_t *)malloc((size_t)N);

    for (int i = 0; i < N; ++i) /* :98-101 */
        if (v->active[i]) prev[i] = (double)distance_to_goal(c, v->goal, v->pos + 3 * i);
    DynConst kc = dyn_const(c, v);
    for (int i = 0; i < N; ++i) /* :103-111 */
        if (v->active[i]) {
            float cmd[3];
            delayed_command(c, v, i, action + 3 * i, cmd);
            integrate(c, &kc, *v->step_count, i, cmd, v->pos + 3 * i, v->vel + 3 * i);
        }
    float bound = kc.bound; /* (float)(world_size / 2): :113-117, all drones */
    for (int k = 0; k < 3 * N; ++k) v->pos[k] = clipf(v->pos[k], -bound, bound);
    *v->step_count += 1; /* :118 */

    for (int i = 0; i < N; ++i) /* :120-127 */
        if (v->active[i]) {
            curr[i] = (double)distance_to_goal(c, v->goal, v->pos + 3 * i);
            v->reached[i] = curr[i] <= c->goal_radius; /* Python-float (double) compare, T3 */
        }
    collision_mask(c, &kc, v, collided);
    formation_penalties(c, v, pen);

    int any_collision = 0;
    for (int i = 0; i < N; ++i) if (v->active[i] && collided[i]) any_collision = 1; /* :137 */
    int time_limit = *v->step_count >= c->max_steps;                                 /* :138 */
    int n_next = 0;
    uint8_t *next_active = (uint8_t *)calloc((size_t)N, 1);

    for (int i = 0; i < N; ++i) { /* :141-162 */
        if (!v->active[i]) continue;
        double progress = (prev[i] - curr[i]) * c->reward_progress_scale;
        double reward = progress + pen[i];
        if (v->reached[i]) reward += c->reward_goal;
        if (collided[i]) reward += c->reward_collision;
        v->reward[i] = reward;
        int done_agent = v->reached[i] || collided[i];
        v->terminated[i] = (uint8_t)done_agent;
        v->truncated[i] = (uint8_t)(time_limit && !done_agent);
        v->collision[i] = collided[i];
        v->dist[i] = (float)curr[i];
        if (!done_agent && !time_limit && !any_collision) {
            build_obs(c, &kc, *v->step_count, v->pos, v->vel, v->goal, v->obst, i, v->obs + (size_t)i * D);
            v->obs_valid[i] = 1;
            next_active[i] = 1;
            ++n_next;
        }
    }
    int all_reached = n_next == 0 && !any_collision && !time_limit; /* :164 */
    int episode_done = all_reached || any_collision;
    *v->all_term = (uint8_t)episode_done;
    *v->all_trunc = (uint8_t)(time_limit && !episode_done);
    if (*v->all_term || *v->all_trunc) memset(v->active, 0, (size_t)N); /* :169-170 */
    else memcpy(v->active, next_active, (size_t)N);                     /* :171-172 */
    if (v->gs) global_state(c, v->pos, v->vel, v->goal, v->gs);

    free(prev); free(curr); free(pen); free(collided); free(next_active);
}

/* SingleDroneEnv.step  single_drone_env.py:73-111 */
static void step_single_env(const OracleConfig *c, EnvView *v, const float *action) {
    int M = c->num_obstacles;
    double prev = (double)distance_to_goal(c, v->goal, v->pos); /* :77 */
    DynConst kc = dyn_const(c, v);
    float cmd[3];
    delayed_command(c, v, 0, action, cmd);
    integrate(c, &kc, *v->step_count, 0, cmd, v->pos, v->vel); /* :74-75, 79-82 */
    float bound = kc.bound;
    for (int k = 0; k < 3; ++k) v->pos[k] = clipf(v->pos[k], -bound, bound); /* :83-87 */
    *v->step_count += 1;                                                       /* :89 */
    double curr = (double)distance_to_goal(c, v->goal, v->pos);               /* :91 */
    double reward = (prev - curr) * c->reward_progress_scale;                  /* :92 */
    int reached = curr <= c->goal_radius;                                      /* :93 */
    int collision = 0;                                                         /* :122-126 */
    float thr = kc.thr_obst; /* (float)(obstacle_radius + collision_radius) */
    for (int m = 0; m < M; ++m) {
        float d = norm_axis(v->obst[3 * m] - v->pos[0], v->obst[3 * m + 1] - v->pos[1],
                            v->obst[3 * m + 2] - v->pos[2]);
        if (d <= thr) collision = 1;
    }
    if (reached) reward += c->reward_goal;       /* :97-98 */
    if (collision) reward += c->reward_collision; /* :99-100 */
    v->reward[0] = reward;
    v->terminated[0] = (uint8_t)(reached || collision);               /* :102 */
    v->truncated[0] = (uint8_t)(*v->step_count >= c->max_steps);      /* :103 (not masked) */
    v->reached[0] = (uint8_t)reached;
    v->collision[0] = (uint8_t)collision;
    v->dist[0] = (float)curr;
    v->obs_valid[0] = 1;
    build_obs(c, &kc, *v->step_count, v->pos, v->vel, v->goal, v->obst, 0, v->obs); /* :105 */
    *v->all_term = v->terminated[0];
    *v->all_trunc = v->truncated[0];
    if (v->gs) global_state(c, v->pos, v->vel, v->goal, v->gs);
}

/* ------------------------------------------------------------------------- */
/* Batch entry points (ctypes)                                                */
/* ------------------------------------------------------------------------- */
int oracle_obs_dim(const OracleConfig *c) { return obs_dim(c); }

/* ------------------------------------------------------------------------- */
/* DronePhysicsEnv (drone_physics_env.py) as a POINT MASS.                     */
/* The reference integrates rigid bodies with PyBullet (pybullet>=3.2.5, not    */
/* vendored, not installed): PARITY UNPINNED.  What is restated here is the env */
/* contract and the force / drag / gravity / clamp model around the solver:     */
/*   per 1/240 s sub-step (:323-360, 24 per step at dt = 0.1):                  */
/*     speed clamp |v| <= max_speed (:353-358), force = action * max_accel * m  */
/*     + (0, 0, 9.5 m) (:336-343, action neither clipped nor cast), gravity     */
/*     -9.81 (:197), Bullet's integrateVelocities -> applyDamping               */
/*     (v *= (1 - c)^h) -> integrateTransforms order; the mass cancels.         */
/*   contacts (:368-372) end the episode, so the contact RESPONSE is never      */
/*   needed: ground z <= 0.025 (URDF box half height, assets/drone.urdf:12),    */
/*   obstacle |p - o| <= r_o + 0.15, drone pair |p_i - p_j| <= 0.30.            */
/* State is float32 (PyBullet's is double); distances use the swarm env's norms.*/
/* ------------------------------------------------------------------------- */
#define PHYS_SUBSTEP_HZ 240.0
#define PHYS_G_COMP 9.5
#define PHYS_GRAVITY 9.81
#define PHYS_HALF_HEIGHT 0.025f
#define PHYS_R_DRONE 0.15

/* (1 - c)^(1/240) with + - * / only, so the CUDA path reproduces it bit for bit:
 * ln x = 2 atanh((x - 1) / (x + 1)) (13 terms), exp by a 7-term Taylor series */
static double phys_damp_factor(double c_lin) {
    double x = 1.0 - c_lin;
    double t = (x - 1.0) / (x + 1.0), t2 = t * t;
    double term = t, acc = 0.0;
    for (int k = 0; k < 13; ++k) {
        volatile double q = term / (double)(2 * k + 1);
        acc = acc + q;
        volatile double nt = term * t2;
        term = nt;
    }
    volatile double lnx = 2.0 * acc;
    volatile double y = lnx / PHYS_SUBSTEP_HZ;
    double e = 1.0, pw = 1.0;
    for (int k = 1; k <= 7; ++k) {
        volatile double npw = pw * y;
        volatile double q = npw / (double)k;
        pw = q;
        e = e + pw;
    }
    return e;
}

static float draw_uniform_f64_to_f32_max(uint64_t rng[4], double lo, double range, double floor_) {
    double u = (double)(oracle_pcg64_next(rng) >> 11) * (1.0 / 9007199254740992.0);
    volatile double scaled = range * u;
    double v = lo + scaled;
    if (v < floor_) v = floor_;
    return (float)v;
}
static double draw_uniform_f64(uint64_t rng[4], double lo, double range) {
    double u = (double)(oracle_pcg64_next(rng) >> 11) * (1.0 / 9007199254740992.0);
    volatile double scaled = range * u;
    return lo + scaled;
}

/* reset  drone_physics_env.py:174-263.  Draw order per drone: position (3), mass noise, damping noise
 * (:207-223); then obstacles (3 each, z >= 0.5, :229-232); then goal (3) and goal z in [0.5, 2] (:240-242).
 * (The reference re-seeds from OS entropy when reset() gets no seed; here the env's stream continues.) */
static void reset_env_physics(const OracleConfig *c, EnvView *v) {
    int N = c->num_drones, M = c->num_obstacles;
    double bound = c->world_size / 2.0;
    /* DR on top (engine semantics, DESIGN.md 9): the sub-step length and the contact radius take the place of dt / r_c */
    if (c->dr_enabled && v->dr) bound = draw_episode_constants(c, v, 1.0 / PHYS_SUBSTEP_HZ, PHYS_R_DRONE);
    double lo = -bound, range = bound - (-bound);
    for (int i = 0; i < N; ++i) v->active[i] = 1;
    *v->step_count = 0;
    for (int i = 0; i < N; ++i) {
        v->pos[3 * i + 0] = draw_uniform_f32(v->rng, lo, range);
        v->pos[3 * i + 1] = draw_uniform_f32(v->rng, lo, range);
        v->pos[3 * i + 2] = draw_uniform_f64_to_f32_max(v->rng, lo, range, 1.0);  /* pos[2] = max(1.0, pos[2]) */
        (void)draw_uniform_f64(v->rng, 0.9, 1.1 - 0.9);                           /* mass noise: cancels for a point mass */
        double damp_noise = draw_uniform_f64(v->rng, 0.8, 1.2 - 0.8);
        volatile double c_lin = 0.5 * damp_noise;
        v->damp[i] = (float)phys_damp_factor(c_lin);
        v->vel[3 * i] = v->vel[3 * i + 1] = v->vel[3 * i + 2] = 0.0f;
    }
    for (int m = 0; m < M; ++m) {
        v->obst[3 * m + 0] = draw_uniform_f32(v->rng, lo, range);
        v->obst[3 * m + 1] = draw_uniform_f32(v->rng, lo, range);
        v->obst[3 * m + 2] = draw_uniform_f64_to_f32_max(v->rng, lo, range, 0.5);
    }
    v->goal[0] = draw_uniform_f32(v->rng, lo, range);
    v->goal[1] = draw_uniform_f32(v->rng, lo, range);
    (void)draw_uniform_f32(v->rng, lo, range);
    v->goal[2] = draw_uniform_f32(v->rng, 0.5, 2.0 - 0.5);
    observe_env(c, v);
}

/* step  drone_physics_env.py:279-419 */
static void step_physics_env(const OracleConfig *c, EnvView *v, const float *action) {
    int N = c->num_drones, M = c->num_obstacles, D = obs_dim(c);
    int n_active = 0;
    for (int i = 0; i < N; ++i) n_active += v->active[i];
    for (int i = 0; i < N; ++i) {
        v->reward[i] = 0.0;
        v->terminated[i] = v->truncated[i] = v->reached[i] = v->collision[i] = 0;
    }
    if (n_active == 0) { /* episode over and not reset: batched contract parks the env (swarm rule) */
        *v->all_term = 1;
        *v->all_trunc = 0;
        for (int i = 0; i < N; ++i) v->obs_valid[i] = 0;
        return;
    }
    const int substeps = (int)(c->dt * PHYS_SUBSTEP_HZ);                /* :323 */
    const DynConst kd = dyn_const(c, v);   /* DR: this episode's max_accel / max_speed / sub-step length / obstacle radius */
    const float h = kd.dr ? kd.dt : (float)(1.0 / PHYS_SUBSTEP_HZ);
    const float amax = kd.amax, vmax = kd.vmax;
    const float g_net = (float)(PHYS_G_COMP - PHYS_GRAVITY);            /* :343 minus :197 */
    for (int i = 0; i < N; ++i) {
        float *p = v->pos + 3 * i, *vel = v->vel + 3 * i;
        float a[3];
        delayed_command(c, v, i, action + 3 * i, a);                    /* DR control delay (identity without it) */
        if (kd.dr) {  /* thrust noise a (1 + sigma z): one normal per axis, held for the whole step; no clip (:336) */
            uint32_t ctr[4] = {kd.genv, kd.ekey, (uint32_t)*v->step_count, (uint32_t)i};
            philox4x32_7(ctr, kd.k0, kd.k1);
            for (int k = 0; k < 3; ++k) {
                volatile float one = fmaf(kd.std_thrust, dr_normal(ctr, k), 1.0f);
                a[k] = a[k] * one;
            }
        }
        const float f = v->damp[i];
        for (int s = 0; s < substeps; ++s) {
            float speed = norm1d(c, vel[0], vel[1], vel[2]);            /* :349-358 */
            if (speed > vmax)
                for (int k = 0; k < 3; ++k) {
                    volatile float q = vel[k] / speed;
                    vel[k] = q * vmax;
                }
            for (int k = 0; k < 3; ++k) {
                volatile float acc = a[k] * amax;                       /* :336 (mass cancels) */
                if (k == 2) { volatile float az = acc + g_net; acc = az; }
                volatile float dv = acc * h;
                volatile float vn = vel[k] + dv;
                vel[k] = vn * f;                                        /* linear damping */
            }
            for (int k = 0; k < 3; ++k) {
                volatile float dp = vel[k] * h;
                p[k] = p[k] + dp;
            }
        }
    }
    *v->step_count += 1;                                                /* :363 */
    const float thr_obst = kd.dr ? kd.thr_obst : (float)(c->obstacle_radius + PHYS_R_DRONE);
    const float thr_pair = (float)(2.0 * PHYS_R_DRONE);
    int any_collision = 0, all_goals = 1;
    for (int i = 0; i < N; ++i) {
        const float *p = v->pos + 3 * i;
        int hit = p[2] <= PHYS_HALF_HEIGHT;
        for (int m = 0; m < M; ++m) {
            float d = norm_axis(v->obst[3 * m] - p[0], v->obst[3 * m + 1] - p[1], v->obst[3 * m + 2] - p[2]);
            if (d <= thr_obst) hit = 1;
        }
        for (int j = 0; j < N; ++j) {
            if (j == i) continue;
            const float *q = v->pos + 3 * j;
            float d = norm1d(c, q[0] - p[0], q[1] - p[1], q[2] - p[2]);
            if (d <= thr_pair) hit = 1;
        }
        float dist = distance_to_goal(c, v->goal, p);
        double reward = -(double)dist * 0.1;                            /* :381 */
        int reached = (double)dist < c->goal_radius;                    /* :389, strict */
        if (hit) { reward -= 10.0; any_collision = 1; }                 /* :385-387 */
        else if (reached) reward += 50.0;                               /* :389-390 */
        else all_goals = 0;
        v->reward[i] = reward;
        v->collision[i] = (uint8_t)hit;
        v->reached[i] = (uint8_t)reached;                               /* infos reached_goal (:573) */
        v->dist[i] = dist;
        v->obs_valid[i] = 1;
    }
    int time_limit = *v->step_count >= c->max_steps;                    /* :397 */
    int done = any_collision || all_goals || time_limit;
    int trunc = time_limit && !any_collision && !all_goals;
    for (int i = 0; i < N; ++i) {                                       /* :401-417 */
        v->terminated[i] = (uint8_t)(done && !trunc);
        v->truncated[i] = (uint8_t)(done && trunc);
        if (done) v->active[i] = 0;
    }
    *v->all_term = (uint8_t)(any_collision || all_goals);
    *v->all_trunc = (uint8_t)trunc;
    DynConst kc = dyn_const(c, v);
    for (int i = 0; i < N; ++i)
        build_obs(c, &kc, *v->step_count, v->pos, v->vel, v->goal, v->obst, i, v->obs + (size_t)i * D);
    if (v->gs) global_state(c, v->pos, v->vel, v->goal, v->gs);
}

void oracle_seed_batch(const OracleBatch *b, const uint64_t *seeds) {
    for (int e = 0; e < b->num_envs; ++e) oracle_seed(seeds[e], b->rng + (size_t)e * 4);
}

void oracle_reset_batch(const OracleConfig *c, const OracleBatch *b, const uint8_t *mask) {
    for (int e = 0; e < b->num_envs; ++e) {
        if (mask && !mask[e]) continue;
        EnvView v = view(c, b, e);
        reset_env(c, &v);
    }
}

void oracle_observe_batch(const OracleConfig *c, const OracleBatch *b) {
    for (int e = 0; e < b->num_envs; ++e) {
        EnvView v = view(c, b, e);
        observe_env(c, &v);
    }
}

/* ep_done_out[e] (nullable) = 1 where the episode ended on this step; with
 * auto_reset the env is then reset (rng stream continues, like RLlib calling
 * env.reset() with no seed) and obs/dist/obs_valid/global_state hold the reset
 * observation while reward/flags keep the terminal step's values. */
static void step_range(const OracleConfig *c, const OracleBatch *b, const float *actions, int auto_reset,
                       int e0, int e1) {
    int N = c->num_drones;
    for (int e = e0; e < e1; ++e) {
        EnvView v = view(c, b, e);
        const float *act = actions + (size_t)e * N * 3;
        if (c->env_kind == 1) step_swarm_env(c, &v, act);
        else if (c->env_kind == 2) step_physics_env(c, &v, act);
        else step_single_env(c, &v, act);
        if (auto_reset && (*v.all_term || *v.all_trunc)) {
            /* keep terminal reward / flags, replace obs + info with the reset ones */
            double *rew = (double *)malloc(sizeof(double) * (size_t)N);
            uint8_t *fl = (uint8_t *)malloc((size_t)N * 4);
            memcpy(rew, v.reward, sizeof(double) * (size_t)N);
            memcpy(fl, v.terminated, (size_t)N);
            memcpy(fl + N, v.truncated, (size_t)N);
            memcpy(fl + 2 * N, v.reached, (size_t)N);
            memcpy(fl + 3 * N, v.collision, (size_t)N);
            uint8_t at = *v.all_term, atr = *v.all_trunc;
            reset_env(c, &v);
            memcpy(v.reward, rew, sizeof(double) * (size_t)N);
            memcpy(v.terminated, fl, (size_t)N);
            memcpy(v.truncated, fl + N, (size_t)N);
            memcpy(v.reached, fl + 2 * N, (size_t)N);
            memcpy(v.collision, fl + 3 * N, (size_t)N);
            *v.all_term = at;
            *v.all_trunc = atr;
            free(rew);
            free(fl);
        }
    }
}

typedef struct StepJob {
    const OracleConfig *c;
    const OracleBatch *b;
    const float *actions;
    int auto_reset, e0, e1;
} StepJob;

static void *step_worker(void *arg) {
    StepJob *j = (StepJob *)arg;
    step_range(j->c, j->b, j->actions, j->auto_reset, j->e0, j->e1);
    return NULL;
}

void oracle_step_batch(const OracleConfig *c, const OracleBatch *b, const float *actions, int auto_reset,
                       int num_threads) {
    int E = b->num_envs;
    if (num_threads <= 1 || E < 2 * num_threads) {
        step_range(c, b, actions, auto_reset, 0, E);
        return;
    }
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)num_threads);
    StepJob *jobs = (StepJob *)malloc(sizeof(StepJob) * (size_t)num_threads);
    for (int t = 0; t < num_threads; ++t) {
        jobs[t].c = c; jobs[t].b = b; jobs[t].actions = actions; jobs[t].auto_reset = auto_reset;
        jobs[t].e0 = (int)((int64_t)E * t / num_threads);
        jobs[t].e1 = (int)((int64_t)E * (t + 1) / num_threads);
        pthread_create(&th[t], NULL, step_worker, &jobs[t]);
    }
    for (int t = 0; t < num_threads; ++t) pthread_join(th[t], NULL);
    free(th);
    free(jobs);
}

#ifdef __cplusplus
}
#endif
