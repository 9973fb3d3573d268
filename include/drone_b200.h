/*
 * drone_b200.h -- C ABI of the B200-native batched delivery_drone simulator.
 *
 * Plain C, plain pointers and sizes, no torch types.  Every entry point is a pure
 * function over caller-owned DEVICE buffers: no global state, no allocation, no
 * host synchronisation (one documented exception: dd_policy_pack); work is enqueued
 * on the cudaStream_t passed in (as void*).
 * Return value: 0 = ok, < 0 = argument error (DD_E_*), > 0 = cudaError_t.
 * Safe to call concurrently on different streams / devices.  The device a call runs on is the one
 * that owns `stream` (a non-default stream) or, for the default stream, the one that owns the state
 * / first buffer argument: the entry points switch to it for the duration of the call and restore
 * the caller's current device, so an env on cuda:1 can be stepped while cuda:0 is current.
 *
 * The reference has no FFI: its "operator interface" for this path is the Python
 * class DroneGame (/root/reference/delivery_drone/game/game_engine.py).  Each entry
 * point below names the reference method(s) it replaces.
 */
#ifndef DRONE_B200_H
#define DRONE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DD_ABI_VERSION 6

/* ---- flag byte (per-step output and persistent state) ---------------------- */
#define DD_DONE        0x01u   /* game_engine.py:53  self.done            */
#define DD_LANDED      0x02u   /* drone.py:32        drone.landed         */
#define DD_CRASHED     0x04u   /* drone.py:31        drone.crashed        */
#define DD_TRUNCATED   0x08u   /* notebook-side time-out, Actor_Critic_PPO.ipynb c16:L89-93 */
#define DD_CAUSE_MASK  0x30u
#define DD_CAUSE_GROUND 0x10u  /* game_engine.py:193-197 */
#define DD_CAUSE_FUEL   0x20u  /* game_engine.py:200-204 */
#define DD_CAUSE_OOB    0x30u  /* game_engine.py:206-210 */

/* ---- action byte ------------------------------------------------------------ */
#define DD_ACT_MAIN   0x01u    /* action['main_thrust']  game_engine.py:115 */
#define DD_ACT_LEFT   0x02u    /* action['left_thrust']  game_engine.py:116 */
#define DD_ACT_RIGHT  0x04u    /* action['right_thrust'] game_engine.py:117 */
#define DD_ACT_SKIP   0x80u    /* env not stepped this call (per-game stepping of the socket API) */

/* ---- precision of the state / arithmetic ----------------------------------- */
#define DD_F32 0               /* throughput instantiation (north_star: fp32 within 1e-5) */
#define DD_F64 1               /* exact-parity instantiation (reference arithmetic is float64) */

/* ---- built-in action sources of dd_rollout ---------------------------------- */
#define DD_POLICY_TRACE    0   /* actions[t*n + i]                                         */
#define DD_POLICY_RANDOM   1   /* Philox bits, p = 0.5 per thruster (examples/random_agent.py:27-31) */
#define DD_POLICY_BANGBANG 2   /* main = vy > 1.5 (SURVEY.md 8c KAT6)                       */

#define DD_OBS_DIM      15     /* policy input, Actor_Critic_PPO.ipynb c10:L3-19           */
#define DD_STATS_SLOTS  64     /* contention-spreading copies of the stats block           */
#define DD_STATS_WORDS  8
#define DD_MAX_ENVS_PER_CALL 0x7fffff00   /* 32-bit env index inside one call; shard above that */
#define DD_RETURN_FIXED_SCALE 1048576.0   /* sum_return is accumulated as int64 in units of 2^-20 */

/* ---- DDEnvConfig.shaping -------------------------------------------------------- */
#define DD_SHAPING_PPO  0   /* calc_reward(state, prev_state): Actor_Critic_PPO.ipynb c7:L2-101 == Actor_Critic_Basic.ipynb */
#define DD_SHAPING_PG   1   /* calc_reward(state): Policy_Gradients.ipynb code cells 5-6 (stateless)                       */

/* ---- DDEnvConfig.launch_flags ------------------------------------------------- */
#define DD_LAUNCH_PDL        0x01   /* programmatic dependent launch: this kernel's CTAs may become
                                       resident while the previous kernel of the stream drains; the
                                       kernel itself waits (griddepcontrol.wait) before its first load */
#define DD_LAUNCH_BLOCK_128  0x10   /* dd_step CTA size (default 256) */
#define DD_LAUNCH_BLOCK_512  0x20

/* ---- DDEnvConfig.obs_format ---------------------------------------------------- */
/* Element format of the observation outputs (obs, final_obs, obs_tn) of dd_reset, dd_step, dd_step_plan and
 * dd_rollout / dd_rollout_shaped.  A 16-bit format writes uint16 bit patterns: every value is the one the same env
 * writes with DD_OBS_NATIVE, converted float -> 16 bit with round-to-nearest-even (what torch's .to(torch.float16) /
 * .to(torch.bfloat16) produce).  State, rewards, flags and statistics are unchanged.  DD_F32 state only (DD_F64 with a
 * 16-bit format: DD_E_DTYPE); an unknown value: DD_E_RANGE.  With obs_stride 16 the `steps` column is converted too,
 * so it is exact only up to 2048 (fp16) or 256 (bf16).
 * dd_policy_rollout and dd_gather_env ignore the field: their observations are always in the state precision. */
#define DD_OBS_NATIVE 0     /* the state precision (R) -- what a zero-initialised DDEnvConfig selects */
#define DD_OBS_F16    1     /* IEEE binary16 */
#define DD_OBS_BF16   2     /* bfloat16 */

/* error codes */
#define DD_E_NULL    (-1)
#define DD_E_RANGE   (-2)
#define DD_E_DTYPE   (-3)
#define DD_E_ALIGN   (-4)

/* All of config.py that the headless path reads (config.py:4-5,18-68).  Doubles;
 * the kernels derive their float / double constants from it on the host. */
typedef struct DDParams {
    double width, height;                 /* config.py:4-5   800, 600 */
    double gravity, drag, angular_drag;   /* config.py:18-20 0.3, 0.99, 0.95 */
    double drone_height;                  /* config.py:24    20 */
    double main_thrust, side_thrust;      /* config.py:25-26 0.6, 0.3 */
    double max_fuel, fuel_main, fuel_side;/* config.py:27-29 1000, 2, 1 */
    double platform_w, platform_h;        /* config.py:32-33 100, 20 */
    double land_speed, land_angle;        /* config.py:39-40 3.0, 20.0 */
    double oob_margin;                    /* config.py:45    50 */
    double ground_margin;                 /* game_engine.py:254 WINDOW_HEIGHT - 50 */
    double r_land, r_crash, r_fuel, r_oob, r_step;  /* config.py:54-58 */
    double shape_offset, shape_div;       /* game_engine.py:214 (500 - d) / 5000 */
    double start_x, start_y;              /* config.py:61-62 400, 100 */
    double plat_default_x, plat_default_y;/* game_engine.py:85 400, 500 */
    double spawn_x_min, spawn_x_count;    /* game_engine.py:66 randint(100, 701)  -> 100, 601 */
    double spawn_y_min, spawn_y_count;    /* game_engine.py:67 randint(50, 251)   -> 50, 201  */
    double plat_x_min, plat_x_count;      /* game_engine.py:74-77 randint(100, 700) -> 100, 600 */
    double plat_y_min, plat_y_count;      /* game_engine.py:78-81 randint(100, 550) -> 100, 450 */
    double vel_norm, angle_norm, angvel_norm;  /* game_engine.py:156-159 10, 180, 10 */
} DDParams;

/*
 * Environment state in HBM: structure of arrays, one entry per environment.
 * R = float (DD_F32) or double (DD_F64).
 *   pos_vel  : R[n][4] = x, y, vx, vy                  (drone.py:19-24)
 *   att_fuel : R[n][4] = angle, angular_velocity, fuel, ep_return (drone.py:27-30, game_engine.py:51)
 *   platform : R[n][2] = px, py                        (platform.py:19-20)
 *   steps    : int32[n]                                (game_engine.py:50)
 *   episode  : uint32[n] resets so far == Philox counter of the next spawn (game_engine.py:52)
 *   flags    : uint8[n] persistent DD_* flags (non-zero only when auto_reset == 0)
 * pos_vel / att_fuel must be 16-byte aligned, platform 8-byte (16 for DD_F64).
 */
typedef struct DDState {
    void *pos_vel;
    void *att_fuel;
    void *platform;
    int32_t *steps;
    uint32_t *episode;
    uint8_t *flags;
    int32_t dtype;           /* DD_F32 / DD_F64 */
    int32_t reserved;
    void *prev_dist;         /* R[n] or NULL: normalised distance_to_platform of the state observed before
                                the previous step, NaN = none (prev_state of Actor_Critic_PPO.ipynb
                                c16:L71-72,101-102).  Needed only when a shaped-reward output is requested.
                                Maintained by dd_rollout_shaped / dd_policy_rollout(shaped_tn) only: dd_step does
                                NOT advance it (it only writes NaN on an auto-reset), so a caller that interleaves
                                dd_step with the shaped rollouts must refill it with NaN first -- the shaped delta
                                then restarts as at an episode start (BatchedDroneEnv does this). */
} DDState;

/* Per-call knobs shared by reset / step / rollout. */
typedef struct DDEnvConfig {
    uint64_t seed;           /* Philox key */
    uint64_t env_id_base;    /* global id of env 0 of this shard: rank * n_local (SURVEY.md 8e) */
    int32_t max_steps;       /* <= 0: no truncation */
    int32_t auto_reset;      /* 0: freeze after done (game_engine.py:107-111); 1: same-step reset */
    int32_t randomize_drone; /* DroneGame(randomize_drone=...)    game_engine.py:14 */
    int32_t randomize_platform; /* DroneGame(randomize_platform=...) */
    int32_t launch_flags;    /* DD_LAUNCH_* bits; 0 = plain stream-ordered launch */
    int32_t shaping;         /* which notebook's client-side calc_reward the `shaped` outputs follow: DD_SHAPING_* */
    int32_t obs_format;      /* DD_OBS_*: element format of the observation outputs */
    int32_t reserved2;
} DDEnvConfig;

int  dd_abi_version(void);
void dd_default_params(DDParams *p);                 /* config.py defaults */
const char *dd_error_string(int code);

/* ---- per-environment physics parameter sets (domain randomisation, per-group curricula) ----------------------------
 * The _sets entry points below take a DDParamSets instead of one DDParams: a table of up to DD_MAX_PARAM_SETS derived
 * parameter sets and a per-env set index.
 *   Selection.  Env i steps, resets and observes exactly as the same env would under DDParams sets[min(index[i], count-1)]
 *     through the single-set entry point: spawn ranges and default spawn, max_fuel at reset, terminal rewards, shaping
 *     constants and observation normalisation.  An out-of-range index is clamped to count-1, never read out of bounds.
 *   Resampling (flags & DD_PARAM_SETS_RESAMPLE).  Each reset of env i -- masked resets of dd_reset_sets, same-step
 *     auto-resets of dd_step_sets / dd_rollout_sets -- draws s = mulhi32(r.a, count) with
 *     r = Philox4x32-10(counter = (env_id lo, env_id hi, episode, 3), key = seed), writes index[i] = s and spawns under
 *     set s.  `episode` is the counter the spawn itself uses (read before the increment); counter word 3 = 3 is a stream
 *     no other draw uses (spawns 0, random actions 1, dd_policy_rollout's Bernoulli uniforms 2).  The step that ends an
 *     episode runs under the old set (its reward, flags and final_obs row); the observation after the auto-reset is
 *     normalised by the new one.  Without the flag `index` is only read.
 *   Validation, before any CUDA call: NULL ps, or NULL table / index with n > 0: DD_E_NULL; count outside
 *     [1, DD_MAX_PARAM_SETS] or unknown flag bits: DD_E_RANGE; ps->dtype != s->dtype: DD_E_DTYPE; table not 16-byte
 *     aligned: DD_E_ALIGN; and every check of the single-set entry point, with the same codes.
 *   Plans.  dd_step_plan_sets keeps the table and index POINTERS: in-place edits of index[] or of the table contents
 *     reach the next dd_step_planned and captured graphs.  A different count or flags value needs a new plan.
 * dd_policy_rollout and dd_gather_env take no parameter sets. */
#define DD_MAX_PARAM_SETS      64
#define DD_PARAM_TABLE_BYTES   32768     /* fixed size: room for 64 sets of the float64 derived constants */
#define DD_PARAM_SETS_RESAMPLE 0x01

typedef struct DDParamSets {
    const void *table;       /* device, 16-byte aligned, DD_PARAM_TABLE_BYTES: the bytes dd_param_sets_build wrote */
    uint8_t *index;          /* device uint8[n]: the set env i runs under (written at resets under RESAMPLE) */
    int32_t count;           /* 1 .. DD_MAX_PARAM_SETS */
    int32_t dtype;           /* DD_F32 / DD_F64 the table was built for; must equal DDState.dtype */
    int32_t flags;           /* DD_PARAM_SETS_* */
    int32_t reserved;
} DDParamSets;

/* Pure host function, no CUDA call: derive `count` parameter sets (including the speed-threshold search) in `dtype` into
 * host_out (DD_PARAM_TABLE_BYTES; unused slots are zero), to be copied to the device table.  The layout is private. */
int dd_param_sets_build(const DDParams *sets, int32_t count, int32_t dtype, void *host_out);

/* DroneGame.reset (game_engine.py:59-93) for every env with mask[i] != 0 (mask == NULL: all).
 * obs (nullable): R[n][obs_stride] first observation of the new episode (uint16[n][obs_stride] under a 16-bit
 * c->obs_format, as for every obs / final_obs / obs_tn below). */
int dd_reset(const DDState *s, const DDParams *p, const DDEnvConfig *c, const uint8_t *mask,
             void *obs, int32_t obs_stride, int64_t n, void *stream);

/* DroneGame.step + get_state (+ reset when auto_reset) (game_engine.py:95-177).
 *   actions    uint8[n]  DD_ACT_* bits
 *   obs        R[n][obs_stride] or NULL (step-only)        game_engine.py:140-177
 *   reward     R[n] or NULL                                game_engine.py:179-216
 *   done_flags uint8[n] or NULL: flags of THIS step (non-zero iff the episode ended on it)
 *   final_obs  R[n][obs_stride] or NULL: terminal observation, written only for envs that ended
 *   stats      uint64[DD_STATS_SLOTS][DD_STATS_WORDS] or NULL: accumulated episode statistics */
int dd_step(const DDState *s, const DDParams *p, const DDEnvConfig *c, const uint8_t *actions,
            void *obs, int32_t obs_stride, void *reward, uint8_t *done_flags, void *final_obs,
            uint64_t *stats, int64_t n, void *stream);

/* ---- dd_step with the argument block built once -------------------------------------------------------
 * A gym loop calls dd_step with the same buffers every step; only `actions` (and the stream) change.
 * dd_step_plan validates the arguments once and stores the resolved launch (kernel, grid, argument block,
 * owning device) in caller-owned memory; dd_step_planned then costs one driver launch -- no validation,
 * no constant derivation, a 3-argument call for the binding.  Same kernel, same results as dd_step.
 * The plan goes stale when a buffer moves or DDEnvConfig changes (max_steps ...): plan again. */
#define DD_STEP_PLAN_BYTES 1024
typedef struct DDStepPlan { uint64_t opaque[DD_STEP_PLAN_BYTES / 8]; } DDStepPlan;
int dd_step_plan(const DDState *s, const DDParams *p, const DDEnvConfig *c,
                 void *obs, int32_t obs_stride, void *reward, uint8_t *done_flags, void *final_obs,
                 uint64_t *stats, int64_t n, DDStepPlan *plan);
int dd_step_planned(const DDStepPlan *plan, const uint8_t *actions, void *stream);

/* T steps in one launch, state held in registers (collect_episodes inner loop without a policy
 * network; Actor_Critic_PPO.ipynb c16:L42-108).  Optional [T][n] outputs.
 *   obs_tn[t] is the observation AFTER step t (after the same-step reset, if any) -- the `next_state` a
 *   gym loop gets back from step(), like dd_step's obs.  (dd_policy_rollout's obs_tn[t] is the observation
 *   BEFORE step t, the network input: the two differ by one step.)
 *   t0: DD_POLICY_RANDOM draws the action of call-local step t from Philox(seed, global env id, t0 + t), a pure
 *   function of its arguments.  The CALLER owns t0: consecutive rollouts of the same envs must pass a running
 *   offset (t0 += T), otherwise every rollout replays the same action noise.  BatchedDroneEnv keeps that counter. */
int dd_rollout(const DDState *s, const DDParams *p, const DDEnvConfig *c, int32_t policy,
               const uint8_t *actions_tn, uint32_t t0, int32_t T,
               void *reward_tn, uint8_t *done_tn, void *obs_tn, int32_t obs_stride,
               uint64_t *stats, int64_t n, void *stream);

/* dd_rollout + shaped_tn R[T][n]: the PPO notebook's client-side training reward
 * (calc_reward, Actor_Critic_PPO.ipynb c7:L2-101, and the -500 time-out of c16:L89-93) computed in the
 * same launch from the post-step state; needs s->prev_dist. */
int dd_rollout_shaped(const DDState *s, const DDParams *p, const DDEnvConfig *c, int32_t policy,
                      const uint8_t *actions_tn, uint32_t t0, int32_t T,
                      void *reward_tn, uint8_t *done_tn, void *obs_tn, int32_t obs_stride, void *shaped_tn,
                      uint64_t *stats, int64_t n, void *stream);

/* dd_reset / dd_step / dd_step_plan / dd_rollout_shaped with per-env parameter sets (DDParamSets above) in place of
 * DDParams.  A plan made by dd_step_plan_sets is launched by dd_step_planned.  dd_rollout_sets with shaped_tn NULL is
 * dd_rollout. */
int dd_reset_sets(const DDState *s, const DDParamSets *ps, const DDEnvConfig *c, const uint8_t *mask,
                  void *obs, int32_t obs_stride, int64_t n, void *stream);
int dd_step_sets(const DDState *s, const DDParamSets *ps, const DDEnvConfig *c, const uint8_t *actions,
                 void *obs, int32_t obs_stride, void *reward, uint8_t *done_flags, void *final_obs,
                 uint64_t *stats, int64_t n, void *stream);
int dd_step_plan_sets(const DDState *s, const DDParamSets *ps, const DDEnvConfig *c, void *obs, int32_t obs_stride,
                      void *reward, uint8_t *done_flags, void *final_obs, uint64_t *stats, int64_t n, DDStepPlan *plan);
int dd_rollout_sets(const DDState *s, const DDParamSets *ps, const DDEnvConfig *c, int32_t policy,
                    const uint8_t *actions_tn, uint32_t t0, int32_t T,
                    void *reward_tn, uint8_t *done_tn, void *obs_tn, int32_t obs_stride, void *shaped_tn,
                    uint64_t *stats, int64_t n, void *stream);

/* [T][n] synthetic random action trace (same bits DD_POLICY_RANDOM uses in-kernel). */
int dd_fill_random_actions(uint8_t *actions_tn, uint64_t seed, uint64_t env_id_base,
                           uint32_t t0, int32_t T, int64_t n, void *stream);

/* actions3[n][3] (any non-zero byte = pressed, game_engine.py:114-118) -> packed uint8[n]. */
int dd_pack_actions(const uint8_t *actions3, uint8_t *packed, int64_t n, void *stream);

/* Collapse the DD_STATS_SLOTS copies into out[DD_STATS_WORDS] (device):
 *   0 episodes, 1 landed, 2 crashed, 3 truncated, 4 sum_return (int64, 2^-20 units),
 *   5 sum_length (steps of the finished episodes), 6 env_steps = sum_length + the steps so far of
 *   the episodes still running (needs steps/flags of the n envs; NULL/NULL: finished only),
 *   7 reserved.  (Actor_Critic_PPO.ipynb c21:L94-95,L158-159,L169) */
int dd_stats_collapse(const uint64_t *stats, const int32_t *steps, const uint8_t *flags, int64_t n,
                      uint64_t *out, void *stream);

/* Everything the per-game surfaces (DroneGame.get_state / _get_info / .done .steps .episode, game_engine.py:140-177,
 * 281-298) read about env i, gathered into ONE record of DD_ENV_RECORD_DOUBLES doubles so that a per-game step of the
 * socket API costs one small copy instead of ten:  [0..15] obs row of env i (obs_stride 15: [15] = steps),
 * [16] reward and [17] flags of the last dd_step, [18] persistent flags, [19] steps, [20] episode,
 * [21..24] pos_vel, [25..28] att_fuel, [29..30] platform, [31] 0.   `out` may be device memory or pinned
 * (device-mapped) host memory; obs / reward / step_flags may be NULL (zeros).  `obs` is in the state precision (there
 * is no DDEnvConfig here: 16-bit observation rows cannot be read). */
#define DD_ENV_RECORD_DOUBLES 32
int dd_gather_env(const DDState *s, const void *obs, int32_t obs_stride, const void *reward,
                  const uint8_t *step_flags, int64_t i, int64_t n, double *out, void *stream);

/* n, sum x, sum x^2 of a float vector into out[3] (device doubles); ACCUMULATES into out.
 * (advantage normalisation moments, Actor_Critic_PPO.ipynb c21:L105) */
int dd_moments(const float *x, int64_t n, double *out, void *stream);

/* y = (x - mean) / (std + eps) with mean/std from moments[3] (unbiased std like torch.std). */
int dd_normalize(const float *x, float *y, const double *moments, double eps, int64_t n, void *stream);

/* compute_gae (Actor_Critic_PPO.ipynb c15:L49-53) for [T][n] rewards/dones and [T+1][n] values. */
int dd_gae(const float *rewards_tn, const float *values_t1n, const uint8_t *dones_tn, float *adv_tn,
           float *returns_tn, double gamma, double lambda, int32_t T, int64_t n, void *stream);
/* dd_gae that also ACCUMULATES the moments (n, sum, sum of squares) of the advantages it writes into moments[3]
 * (device doubles, nullable) in the same pass: dd_normalize can follow without dd_moments re-reading the buffer. */
int dd_gae_moments(const float *rewards_tn, const float *values_t1n, const uint8_t *dones_tn, float *adv_tn,
                   float *returns_tn, double *moments, double gamma, double lambda, int32_t T, int64_t n, void *stream);

/* compute_returns (Policy_Gradients.ipynb: G = r + gamma * G over reversed(rewards)) for [T][n] rewards; dones_tn
 * (nullable) marks the steps that ended an episode: G restarts behind them.  float64 accumulation like the
 * notebook's python floats, fp32 result. */
int dd_discounted_returns(const float *rewards_tn, const uint8_t *dones_tn, float *returns_tn, double gamma,
                          int32_t T, int64_t n, void *stream);

/* ---- K5: fused policy rollout (Actor_Critic_PPO.ipynb c11, c16) ---------------------------- */
/* fp32 parameters of DroneGamerBoi exactly as torch stores them: nn.Linear.weight is [out][in]
 * row-major; g / be are nn.LayerNorm weight / bias.  15-128-128-64-3. */
typedef struct DDPolicy {
    const float *w0, *b0, *g0, *be0;      /* network.0 (Linear 15->128), network.1 (LayerNorm 128) */
    const float *w1, *b1, *g1, *be1;      /* network.3 (Linear 128->128), network.4 */
    const float *w2, *b2, *g2, *be2;      /* network.6 (Linear 128->64), network.7 */
    const float *w3, *b3;                 /* network.9 (Linear 64->3) */
} DDPolicy;

#define DD_POLICY_BLOB_BYTES 67616        /* device workspace filled by dd_policy_pack */
#define DD_ACTION_THRESHOLD 0             /* action = probs > 0.5        (c18:L24-25) */
#define DD_ACTION_SAMPLE    1             /* action ~ Bernoulli(probs)   (c16:L61-63), Philox */

/* 16-bit format of the tensor-core operands (weight images and hidden activations; accumulation is fp32):
 *   DD_OPERANDS_FP16  10 mantissa bits: 8x lower rounding error than bf16 at the same MMA rate.  Needs the packed
 *                     network to fit the fp16 range, which dd_policy_pack verifies from the parameters alone
 *                     (|normalised activation| <= sqrt(N), so max |activation| <= sqrt(N) + max |beta / gamma|):
 *                     LayerNorm |gamma| in [2^-6, 2^6], |beta / gamma| <= 1024, weight-image maxima in [2^-8, 1024];
 *   DD_OPERANDS_BF16  8 exponent bits: any fp32 network (gamma = 0, huge beta / gamma ...);
 *   DD_OPERANDS_AUTO  fp16 when the check passes, else bf16 -- what dd_policy_pack / dd_value_pack use. */
#define DD_OPERANDS_AUTO 0
#define DD_OPERANDS_BF16 1
#define DD_OPERANDS_FP16 2

/* The per-column fp32 parameters the CUDA cores apply after each tensor-core layer.  HOST memory: the
 * launch passes them by value (kernel-argument constant bank), so every thread reads them as uniform
 * operands instead of replicating shared-memory loads.  Filled by dd_policy_pack.
 * With s = sign(gamma), g = |gamma| (floored at 1e-12): the accumulator of a layer is s (x - mean x), the activation
 * handed to the next layer is relu(s (x - mean x) rstd + beta / g), and g rides in the next layer's weight image
 * (relu(gamma n + beta) = g relu(s n + beta / g)); for the last hidden layer g is folded into w3. */
typedef struct DDPolicyConsts {
    float beta0[128];                     /* network.1: LayerNorm.bias / |LayerNorm.weight| */
    float beta1[128];                     /* network.4 */
    float beta2[64];                      /* network.7 */
    float w3[3][64];                      /* network.9.weight x |network.7.weight| (column-wise) */
    float b3[4];                          /* network.9.bias (+ pad) */
    int32_t operands;                     /* DD_OPERANDS_BF16 / DD_OPERANDS_FP16: what the blob's images are */
    int32_t reserved[3];
} DDPolicyConsts;

/* fp32 torch parameters (DEVICE pointers) -> `blob` (device, 16-byte aligned): 16-bit tensor-core operand
 * images with the LayerNorm centring, the sign of gamma, the previous layer's |gamma| and the biases folded in;
 * and `consts` (HOST).  This is the one entry point that synchronises `stream` (it copies 2 KB back to fill
 * `consts`); call it once per policy update.  dd_policy_pack == dd_policy_pack_ex(..., head 3, DD_OPERANDS_AUTO). */
int dd_policy_pack(const DDPolicy *p, void *blob, DDPolicyConsts *consts, void *stream);
int dd_policy_pack_ex(const DDPolicy *p, int32_t head, int32_t operands, void *blob, DDPolicyConsts *consts, void *stream);

/* probs[n][3] = policy(obs[n][15]) through the same tcgen05 path the rollout uses (parity hook).  Persistent
 * over the rows: any n up to DD_MAX_ENVS_PER_CALL, e.g. a whole [T*N][15] rollout buffer. */
int dd_policy_forward(const void *blob, const DDPolicyConsts *consts, const float *obs, float *probs, int64_t n,
                      void *stream);

/* The critic DroneTeacherBoi (Actor_Critic_PPO.ipynb: same trunk as the policy, Linear(64, 1) head, no sigmoid):
 * p->w3 is [1][64], p->b3 is [1].  values[n] = critic(obs[n][15]) -- what the training loop computes over the stored
 * states (`values = critic(states_tensor)` + the bootstrap value of the final state) before compute_gae. */
int dd_value_pack(const DDPolicy *p, void *blob, DDPolicyConsts *consts, void *stream);
int dd_value_forward(const void *blob, const DDPolicyConsts *consts, const float *obs, float *values, int64_t n,
                     void *stream);

/* `temperature` (DD_ACTION_SAMPLE, > 0): actions ~ Bernoulli(p^(1/tau) / (p^(1/tau) + (1-p)^(1/tau))) = Bernoulli(sigmoid(logit / tau)),
 * the evaluation sampling of evaluate_policy_simple (Actor_Critic_PPO.ipynb c18); 1 = the policy's own distribution
 * (collect_episodes_ppo).  probs / logp outputs always describe the untempered policy. */
/* T steps of {observe, policy, act, step} in one launch; DD_F32 state only; c->obs_format is ignored (obs_tn is fp32:
 * the critic's first layer reads these rows at full precision).  Optional [T][n] outputs:
 * actions (DD_ACT_* bits), logp (sum of the 3 Bernoulli log-probs), reward, done flags, obs [T][n][15],
 * probs [T][n][3], shaped (the notebook's training reward; needs s->prev_dist; c->shaping must be a DD_SHAPING_*
 * value, else DD_E_RANGE).
 *   obs_tn[t] is the observation BEFORE step t (what the policy saw; the `state` appended by
 *   collect_episodes_ppo, c16:L66-80) -- values for dd_gae come from these rows plus the observation after the
 *   last step as bootstrap row.
 *   t0: the Bernoulli uniforms of call-local step t are Philox(seed, global env id, t0 + t, stream 2); as for
 *   dd_rollout the caller owns t0 and must advance it by T between rollouts of the same envs. */
int dd_policy_rollout(const DDState *s, const DDParams *p, const DDEnvConfig *c, const void *blob,
                      const DDPolicyConsts *consts, int32_t mode, float temperature, uint32_t t0, int32_t T, uint8_t *actions_tn, float *logp_tn, float *reward_tn,
                      uint8_t *done_tn, float *obs_tn, float *probs_tn, float *shaped_tn, uint64_t *stats, int64_t n,
                      void *stream);

/* Launch shape of dd_policy_rollout (pure host function; what the launcher itself uses): the number of CTAs for n envs on
 * a device with `sms` SMs.  Slot g (0..3) of CTA b runs the tile of 128 envs number b + grid * g (if it exists).  Up to 3
 * tiles per SM the tiles are spread over the SMs, above that packed four to a CTA (per-SM throughput saturates with the
 * resident tiles; DESIGN.md 4b).  0 for n outside (0, DD_MAX_ENVS_PER_CALL]. */
int dd_policy_rollout_grid(int64_t n, int32_t sms);

#ifdef __cplusplus
}
#endif
#endif /* DRONE_B200_H */
