// drone_kernels.cu -- sm_100a kernels of the batched delivery_drone simulator + their C ABI.
//
//   K1 step_kernel     one DroneGame.step() (+ get_state, + same-step reset) per env per launch:
//                      one HBM round trip (SoA state in, state + reward + flags + obs out)
//   K2 reset_kernel    DroneGame.reset() for all / masked envs (Philox spawn)
//   K3 episode stats   warp ballot -> warp-aggregated REDs into one of DD_STATS_SLOTS copies, only
//                      in warps where an episode ended (fused into K1 and the rollout kernel)
//   rollout_kernel     T steps per launch with the env state in registers
//
// HBM-bound byte/float work: no tensor cores here.  What matters (ncu, profiles/):
//   * every load of a thread is issued before anything depends on one (one DRAM round trip),
//   * 16-byte coalesced loads and stores, 32-bit indexing, constants as immediates,
//   * ~100 issue slots per env-step so the SM never becomes the limiter,
//   * the observation tile staged through shared memory and written with one TMA bulk store
//     per CTA,
//   * programmatic dependent launch so the next step's CTAs are resident before this one drains.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include "drone_device.cuh"
#include "host_guard.h"

namespace dd {

// ---- observation tile: shared memory -> global ------------------------------------------------
// A CTA's tile is contiguous in global memory (BLOCK rows of obs_stride elements).  Full, 16-byte
// aligned tiles leave with ONE TMA bulk store (cp.async.bulk, SASS UBLKCP) issued by one thread;
// ragged tiles fall back to a coalesced copy loop.
template <typename R, int BLOCK>
__device__ __forceinline__ void obs_tile_store(const R* s_obs, R* g_tile, int rows, int stride) {
    const uint32_t bytes = (uint32_t)(rows * stride * sizeof(R));
    const bool bulk = (rows == BLOCK) && ((reinterpret_cast<uintptr_t>(g_tile) & 15u) == 0) && ((bytes & 15u) == 0);
    if (bulk) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // my smem writes -> async proxy
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(s_obs);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(g_tile), "r"(saddr), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem must outlive the read
        }
    } else {
        __syncthreads();
        const int total = rows * stride;
        for (int j = threadIdx.x; j < total; j += BLOCK) g_tile[j] = s_obs[j];
    }
}

// ---- observation element format (DDEnvConfig.obs_format) ---------------------------------------
// OF = DD_OBS_NATIVE: elements of type R, stored as the kernels always have.  OF = DD_OBS_F16 / DD_OBS_BF16 (float
// state only): uint16 bit patterns, converted in pairs by write_obs16; the KArgs / RArgs pointers (obs, final_obs,
// obs_tn) then hold uint16 buffers and are cast here.
template <typename R, int OF> struct ObsElem { using type = uint16_t; };
template <typename R> struct ObsElem<R, DD_OBS_NATIVE> { using type = R; };
template <typename R, int OF> using obs_elem_t = typename ObsElem<R, OF>::type;

template <int OF, typename R>
__device__ __forceinline__ obs_elem_t<R, OF>* obs_ptr(R* p) { return reinterpret_cast<obs_elem_t<R, OF>*>(p); }

// =================================================================================================
// K1: one step per env per launch.
// =================================================================================================
// SETS: per-env parameter sets (KArgsPS): env i's constants are set min(index[i], count - 1) of the table, read through
// L1 after the index byte arrives; under ps_resample each auto-reset draws a new set (param_set_draw) before it spawns.
template <typename R, bool AUTO, bool OBS, bool DEF, int BLOCK, int OF, bool SETS>
__global__ void __launch_bounds__(BLOCK) step_kernel(const __grid_constant__ KArgsOf<R, SETS> a)
{
    using O = obs_elem_t<R, OF>;
    __shared__ __align__(128) O s_obs[OBS ? BLOCK * kMaxObsStride : 1];
    Consts<R> k;
    if constexpr (!SETS) k = consts_of<R, DEF>(a);

    const uint32_t tile0 = blockIdx.x * BLOCK;
    const uint32_t i = tile0 + threadIdx.x;
    const bool live = i < a.n;

    pdl_wait();                                            // state / actions may come from the previous launch
    uint32_t f_stat = 0; R ret_stat = 0; int32_t len_stat = 0;
    if (live) {
        // ---- every load of this thread, back to back ----
        Env<R> e;
        uint32_t act = a.actions[i];
        load_env(a, i, e);
        uint32_t pflags = AUTO ? 0u : (uint32_t)a.flags[i];   // persistent flags are always 0 under auto-reset
        uint32_t set = 0;
        if constexpr (SETS) set = a.ps_index[i];
        pin(act); pin(pflags);
        if constexpr (SETS) { pin(set); k = param_set<R>(a.ps_table, param_set_clamp(set, a.ps_count)); }
        pdl_launch_dependents();

        uint32_t oflags = pflags;                              // what this step reports
        R reward = (R)0, speed = (R)0, dist = (R)0;
        const bool stepped = !(act & DD_ACT_SKIP) && !(pflags & DD_DONE);

        if (stepped) {
            uint32_t f = step_core<R, OBS>(e, act, k, reward, speed, dist);
            if (!f && a.max_steps > 0 && e.steps >= a.max_steps) f = DD_DONE | DD_TRUNCATED;
            oflags = f;
            if (f) {                                           // rare: ~1 % of env-steps
                f_stat = f; ret_stat = e.ret; len_stat = e.steps;
                if (a.final_obs) {                             // terminal observation (scattered rows)
                    O* fo = obs_ptr<OF>(a.final_obs) + (size_t)i * a.obs_stride;
                    if (!OBS) speed = Arith<R>::sqrt_(Arith<R>::fma_(e.vx, e.vx, Arith<R>::mul(e.vy, e.vy)));
                    if constexpr (OF == DD_OBS_NATIVE) write_obs(e, f, speed, dist, k, [&](int j, R v) { fo[j] = v; });
                    else write_obs16<OF>(e, f, speed, dist, k, false, 0.0f, [&](int j, O v) { fo[j] = v; });
                }
                if (AUTO) {                                    // same-step reset
                    const uint32_t ep = a.episode[i];
                    if constexpr (SETS) {
                        if (a.ps_resample) {                   // the new episode's set; final_obs above is the old one's
                            set = param_set_draw(a.seed, a.env_id_base + (uint64_t)i, ep, a.ps_count);
                            a.ps_index[i] = (uint8_t)set;
                            k = param_set<R>(a.ps_table, set);
                        }
                    }
                    spawn(e, k, a.seed, a.env_id_base + (uint64_t)i, ep, a.rand_drone != 0, a.rand_platform != 0);
                    a.episode[i] = ep + 1;
                    store2(a.platform, i, e.px, e.py);
                    if (a.prev_dist) a.prev_dist[i] = nan_of<R>();
                    f = 0;
                    if (OBS) speed_dist(e, speed, dist);
                }
            }
            pflags = f;
            store_env(a, i, e);
            if (!AUTO) a.flags[i] = (uint8_t)pflags;
        } else if (OBS) {
            speed_dist(e, speed, dist);                        // frozen / skipped env: obs of the state as is
        }

        if (a.reward) a.reward[i] = reward;
        if (a.done_flags) a.done_flags[i] = (uint8_t)oflags;
        if (OBS) {
            O* row = s_obs + threadIdx.x * a.obs_stride;
            if constexpr (OF == DD_OBS_NATIVE) {
                write_obs(e, pflags, speed, dist, k, [&](int j, R v) { row[j] = v; });
                if (a.obs_stride > DD_OBS_DIM) row[DD_OBS_DIM] = (R)e.steps;     // 16th key: 'steps'
            } else {
                write_obs16<OF>(e, pflags, speed, dist, k, a.obs_stride > DD_OBS_DIM, (float)e.steps,
                                [&](int j, O v) { row[j] = v; });
            }
        }
    } else {
        pdl_launch_dependents();
    }

    if (a.stats) stats_warp_commit(a.stats, f_stat, ret_stat, len_stat);
    if (OBS) {
        const uint32_t rem = a.n - tile0;
        const int rows = rem < (uint32_t)BLOCK ? (int)rem : BLOCK;
        obs_tile_store<O, BLOCK>(s_obs, obs_ptr<OF>(a.obs) + (size_t)tile0 * a.obs_stride, rows, a.obs_stride);
    }
}

// =================================================================================================
// K2: reset.
// =================================================================================================
constexpr int kBlock = 256;

// The constants env i resets under: the launch's (SETS = false) or its set, drawn anew under ps_resample.
template <typename R, bool SETS>
__device__ __forceinline__ Consts<R> reset_consts(const KArgsOf<R, SETS>& a, uint32_t i, uint32_t ep)
{
    if constexpr (SETS) {
        uint32_t s;
        if (a.ps_resample) {
            s = param_set_draw(a.seed, a.env_id_base + (uint64_t)i, ep, a.ps_count);
            a.ps_index[i] = (uint8_t)s;
        } else {
            s = param_set_clamp(a.ps_index[i], a.ps_count);
        }
        return param_set<R>(a.ps_table, s);
    } else {
        return a.k;
    }
}

template <typename R, int OF, bool SETS>
__global__ void __launch_bounds__(kBlock) reset_kernel(const __grid_constant__ KArgsOf<R, SETS> a, const uint8_t* mask)
{
    const uint32_t i = blockIdx.x * kBlock + threadIdx.x;
    pdl_wait();
    if (i >= a.n) return;
    if (mask && !mask[i]) return;
    Env<R> e;
    const uint32_t ep = a.episode[i];
    const Consts<R> k = reset_consts<R, SETS>(a, i, ep);
    spawn(e, k, a.seed, a.env_id_base + (uint64_t)i, ep, a.rand_drone != 0, a.rand_platform != 0);
    a.episode[i] = ep + 1;                                     // game_engine.py:91
    store_env(a, i, e);
    store2(a.platform, i, e.px, e.py);
    a.flags[i] = 0;
    if (a.prev_dist) a.prev_dist[i] = nan_of<R>();              // prev_state = None (c16:L38)
    if (a.obs) {
        R speed, dist;
        speed_dist(e, speed, dist);
        obs_elem_t<R, OF>* row = obs_ptr<OF>(a.obs) + (size_t)i * a.obs_stride;
        if constexpr (OF == DD_OBS_NATIVE) {
            write_obs(e, 0u, speed, dist, k, [&](int j, R v) { row[j] = v; });
            if (a.obs_stride > DD_OBS_DIM) row[DD_OBS_DIM] = (R)0;
        } else {
            write_obs16<OF>(e, 0u, speed, dist, k, a.obs_stride > DD_OBS_DIM, 0.0f, [&](int j, uint16_t v) { row[j] = v; });
        }
    }
}

// =================================================================================================
// Rollout: T steps per launch, env state in registers, one state round trip per launch.
// =================================================================================================
template <typename R, typename KA = KArgs<R>>
struct RArgs {
    KA a;
    const uint8_t* actions_tn;
    R* reward_tn;
    uint8_t* done_tn;
    R* obs_tn;
    R* shaped_tn;
    uint32_t t0;
    int32_t T, policy, auto_reset;
};

// POLICY (the action source) is a template parameter and every launch-constant switch is read once before the
// loop: the kernel is bound by issue slots (no memory traffic to hide behind), so each instruction of the
// per-step path is throughput.
// OUTS = false: no per-step [T][n] outputs (reward / done / shaped) -- the pure statistics rollout of the curriculum
// sweep and the throughput bench -- compiles their address arithmetic and predicated stores away.
// SETS: as in step_kernel; the env's constants stay in registers over the T steps and are reloaded when a resampling
// auto-reset draws a new set (index[i] is written back once, at the end).
template <typename R, bool OBS, bool DEF, int POLICY, bool OUTS, int OF, bool SETS>
__global__ void __launch_bounds__(kBlock) rollout_kernel(const __grid_constant__ RArgs<R, KArgsOf<R, SETS>> ra)
{
    using O = obs_elem_t<R, OF>;
    __shared__ __align__(128) O s_obs[OBS ? kBlock * kMaxObsStride : 1];
    const auto& a = ra.a;
    Consts<R> k;
    if constexpr (!SETS) k = consts_of<R, DEF>(a);
    const uint32_t tile0 = blockIdx.x * kBlock;
    const uint32_t i = tile0 + threadIdx.x;
    const bool live = i < a.n;
    const uint32_t rem = a.n - tile0;
    const int rows = rem < (uint32_t)kBlock ? (int)rem : kBlock;

    pdl_wait();
    Env<R> e = {};
    uint32_t pflags = 0, ep = 0, set = 0;
    bool platform_dirty = false, set_dirty = false;
    if (live) {
        load_env(a, i, e);
        pflags = a.flags[i];
        ep = a.episode[i];
        if constexpr (SETS) set = param_set_clamp(a.ps_index[i], a.ps_count);
    }
    if constexpr (SETS) k = param_set<R>(a.ps_table, set);
    pdl_launch_dependents();
    const uint64_t gid = a.env_id_base + (uint64_t)i;
    // DD_POLICY_RANDOM: the 96 action bits of the current block of 32 steps (action_block) as a shift register --
    // the step's action is its low 3 bits (== action_from_block), then it moves on by 3 bits
    uint32_t rb0 = 0, rb1 = 0, rb2 = 0, tt = ra.t0;
    if (POLICY == DD_POLICY_RANDOM) {
        const U4 b = action_block(a.seed, gid, tt);
        rb0 = b.a; rb1 = b.b; rb2 = b.c;
        for (uint32_t j = 0; j < (tt & 31u); ++j) {          // a rollout may start inside a block
            rb0 = __funnelshift_r(rb0, rb1, 3); rb1 = __funnelshift_r(rb1, rb2, 3); rb2 >>= 3;
        }
    }
    const bool out_rew = OUTS && ra.reward_tn != nullptr, out_done = OUTS && ra.done_tn != nullptr,
               do_stats = a.stats != nullptr, auto_reset = ra.auto_reset != 0;
    const int32_t max_steps = a.max_steps;
    // N2 (shaped training reward): normalised distance of the current state and of the one before it
    const bool shaping = OUTS && ra.shaped_tn != nullptr;
    R dprev = nan_of<R>(), dcur = (R)0;
    if (live && shaping) {
        R s_, d_;
        speed_dist(e, s_, d_);
        dcur = Arith<R>::div(d_, k.width, k.inv_width);
        dprev = a.prev_dist[i];
    }

    StatsAcc st;                                             // per-thread statistics, one commit per warp and launch
    auto one_step = [&](const int32_t t) {
        uint32_t oflags = pflags;
        R reward = (R)0, speed = (R)0, dist = (R)0, shaped = (R)0;
        if (live) {
            const size_t o = (size_t)t * a.n + i;
            uint32_t act;
            if (POLICY == DD_POLICY_TRACE) {
                act = ra.actions_tn[o];
            } else if (POLICY == DD_POLICY_RANDOM) {
                act = rb0 & 7u;
                rb0 = __funnelshift_r(rb0, rb1, 3); rb1 = __funnelshift_r(rb1, rb2, 3); rb2 >>= 3;
            } else {
                act = (e.vy > (R)1.5) ? DD_ACT_MAIN : 0u;
            }
            if (!(act & DD_ACT_SKIP) && !(pflags & DD_DONE)) {
                uint32_t f = step_core<R, OBS>(e, act, k, reward, speed, dist);
                if (!f && max_steps > 0 && e.steps >= max_steps) f = DD_DONE | DD_TRUNCATED;
                oflags = f;
                if (shaping) {
                    const R sp = OBS ? speed : Arith<R>::sqrt_(Arith<R>::fma_(e.vx, e.vx, Arith<R>::mul(e.vy, e.vy)));
                    shaped = shaped_reward(a.shaping, e, f, sp, dist, dprev, max_steps > 0 && e.steps >= max_steps, k);
                    dprev = dcur;
                    dcur = Arith<R>::div(dist, k.width, k.inv_width);
                }
                if (f) {
                    if (do_stats) st.add(f, e.ret, e.steps);          // per-thread totals, committed once after the loop
                    if (auto_reset) {
                        if constexpr (SETS) {
                            if (a.ps_resample) {
                                set = param_set_draw(a.seed, gid, ep, a.ps_count);
                                set_dirty = true;
                                k = param_set<R>(a.ps_table, set);
                            }
                        }
                        spawn(e, k, a.seed, gid, ep, a.rand_drone != 0, a.rand_platform != 0);
                        ep += 1;
                        platform_dirty = true;
                        f = 0;
                        if (OBS || shaping) speed_dist(e, speed, dist);
                        if (shaping) { dprev = nan_of<R>(); dcur = Arith<R>::div(dist, k.width, k.inv_width); }
                    }
                }
                pflags = f;
            } else if (OBS) {
                speed_dist(e, speed, dist);
            }
            if (shaping) ra.shaped_tn[o] = shaped;
            if (out_rew) ra.reward_tn[o] = reward;
            if (out_done) ra.done_tn[o] = (uint8_t)oflags;
            if (OBS) {
                O* row = s_obs + threadIdx.x * a.obs_stride;
                if constexpr (OF == DD_OBS_NATIVE) {
                    write_obs(e, pflags, speed, dist, k, [&](int j, R v) { row[j] = v; });
                    if (a.obs_stride > DD_OBS_DIM) row[DD_OBS_DIM] = (R)e.steps;
                } else {
                    write_obs16<OF>(e, pflags, speed, dist, k, a.obs_stride > DD_OBS_DIM, (float)e.steps,
                                    [&](int j, O v) { row[j] = v; });
                }
            }
        }
        if (OBS) {
            obs_tile_store<O, kBlock>(s_obs, obs_ptr<OF>(ra.obs_tn) + ((size_t)t * a.n + tile0) * a.obs_stride, rows, a.obs_stride);
            __syncthreads();                                   // tile is reused next step
        }
    };
    if constexpr (POLICY == DD_POLICY_RANDOM) {
        // the steps are walked block by block (32 steps = one action_block): the refill of the shift register sits between
        // the blocks instead of behind a test in every step
        for (int32_t t = 0; t < ra.T;) {
            if (t > 0) {                                     // (tt & 31) == 0 here: the next block
                const U4 b = action_block(a.seed, gid, tt);
                rb0 = b.a; rb1 = b.b; rb2 = b.c;
            }
            const int32_t left = 32 - (int32_t)(tt & 31u);
            const int32_t t_end = ra.T - t < left ? ra.T : t + left;
            tt += (uint32_t)(t_end - t);
            for (; t < t_end; ++t) one_step(t);
        }
    } else {
        for (int32_t t = 0; t < ra.T; ++t) one_step(t);
    }

    if (do_stats) st.commit(a.stats);
    if (live) {
        store_env(a, i, e);
        a.flags[i] = (uint8_t)pflags;
        a.episode[i] = ep;
        if (platform_dirty) store2(a.platform, i, e.px, e.py);
        if (shaping) a.prev_dist[i] = dprev;
        if constexpr (SETS) { if (set_dirty) a.ps_index[i] = (uint8_t)set; }
    }
}

// ---- small utility kernels ----------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) fill_random_actions_kernel(uint8_t* out, uint64_t seed, uint64_t env_id_base,
                                                                      uint32_t t0, int32_t T, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    U4 blk = {0, 0, 0, 0};
    uint32_t blk_id = 0xffffffffu;
    for (int32_t t = 0; t < T; ++t) {
        const uint32_t tt = t0 + (uint32_t)t;
        if ((tt >> 5) != blk_id) { blk = action_block(seed, env_id_base + (uint64_t)i, tt); blk_id = tt >> 5; }
        out[(int64_t)t * n + i] = (uint8_t)action_from_block(blk, tt);
    }
}

__global__ void __launch_bounds__(kBlock) pack_actions_kernel(const uint8_t* a3, uint8_t* packed, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const uint8_t m = a3[3 * i], l = a3[3 * i + 1], r = a3[3 * i + 2];
    packed[i] = (uint8_t)((m ? DD_ACT_MAIN : 0u) | (l ? DD_ACT_LEFT : 0u) | (r ? DD_ACT_RIGHT : 0u));
}

// one env's observation row, last step outputs and raw state as doubles (compat layer: one copy per per-game step)
template <typename R>
__global__ void gather_env_kernel(const R* pos_vel, const R* att_fuel, const R* platform, const int32_t* steps,
                                  const uint32_t* episode, const uint8_t* flags, const R* obs, int obs_stride,
                                  const R* reward, const uint8_t* step_flags, int64_t i, double* out)
{
    const int j = threadIdx.x;
    if (j >= DD_ENV_RECORD_DOUBLES) return;
    double v = 0.0;
    if (j < 16) v = obs ? (j < obs_stride ? (double)obs[i * obs_stride + j] : (double)steps[i]) : 0.0;
    else if (j == 16) v = reward ? (double)reward[i] : 0.0;
    else if (j == 17) v = step_flags ? (double)step_flags[i] : 0.0;
    else if (j == 18) v = (double)flags[i];
    else if (j == 19) v = (double)steps[i];
    else if (j == 20) v = (double)episode[i];
    else if (j < 25) v = (double)pos_vel[4 * i + (j - 21)];
    else if (j < 29) v = (double)att_fuel[4 * i + (j - 25)];
    else if (j < 31) v = (double)platform[2 * i + (j - 29)];
    out[j] = v;
}

// out[0..5] = column sums of the slot copies; out[6] = out[5] (+ live steps, added by the next kernel)
__global__ void stats_collapse_kernel(const unsigned long long* stats, unsigned long long* out)
{
    const int w = threadIdx.x;
    if (w >= DD_STATS_WORDS) return;
    unsigned long long t = 0;
    const int col = (w == 6) ? 5 : w;
    for (int s = 0; s < DD_STATS_SLOTS; ++s) t += stats[s * DD_STATS_WORDS + col];
    out[w] = (w == 7) ? 0ull : t;
}

// out[6] += sum of steps[i] over episodes still running
__global__ void __launch_bounds__(kBlock) live_steps_kernel(const int32_t* steps, const uint8_t* flags, int64_t n,
                                                             unsigned long long* out)
{
    unsigned long long t = 0;
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock)
        if (!(flags[i] & DD_DONE)) t += (unsigned long long)steps[i];
    t = (unsigned long long)warp_sum((long long)t);
    if ((threadIdx.x & 31) == 0 && t) atomicAdd(out + 6, t);
}

// =================================================================================================
// host side of the ABI
// =================================================================================================
static inline int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

static bool params_are_default(const DDParams& p)
{
    const DDParams d = kDefaultParams;
    if (memcmp(&p, &d, sizeof d) != 0) return false;
    // the compile-time constants assume sqrt thresholds that the search confirms
    return speed2_threshold<float>((float)p.land_speed) == (float)p.land_speed * (float)p.land_speed &&
           speed2_threshold<double>(p.land_speed) == p.land_speed * p.land_speed;
}

// Everything of the argument block but the constants.
template <typename R>
static int fill_state(KArgs<R>& a, const DDState* s, const DDEnvConfig* c, int64_t n)
{
    if (!s || !c) return DD_E_NULL;
    if (n < 0 || n > (int64_t)0x7fffff00) return DD_E_RANGE;          // 32-bit env index inside one call
    if (n > 0 && (!s->pos_vel || !s->att_fuel || !s->platform || !s->steps || !s->episode || !s->flags)) return DD_E_NULL;
    if ((reinterpret_cast<uintptr_t>(s->pos_vel) | reinterpret_cast<uintptr_t>(s->att_fuel)) & 15u) return DD_E_ALIGN;
    if (reinterpret_cast<uintptr_t>(s->platform) & (2 * sizeof(R) - 1)) return DD_E_ALIGN;
    a = KArgs<R>{};
    a.pos_vel = (R*)s->pos_vel; a.att_fuel = (R*)s->att_fuel; a.platform = (R*)s->platform;
    a.prev_dist = (R*)s->prev_dist;
    a.steps = s->steps; a.episode = s->episode; a.flags = s->flags;
    a.n = (uint32_t)n; a.seed = c->seed; a.env_id_base = c->env_id_base;
    a.max_steps = c->max_steps; a.obs_stride = DD_OBS_DIM; a.shaping = c->shaping;
    a.rand_drone = c->randomize_drone; a.rand_platform = c->randomize_platform;
    return 0;
}

template <typename R>
static int fill_args(KArgs<R>& a, const DDState* s, const DDParams* p, const DDEnvConfig* c, int64_t n)
{
    if (!p) return DD_E_NULL;
    if (int rc = fill_state(a, s, c, n)) return rc;
    a.k = make_consts<R>(*p);
    return 0;
}

// The DDParamSets checks of include/drone_b200.h, then the argument block of the per-env kernels.
template <typename R>
static int fill_args(KArgsPS<R>& a, const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, int64_t n)
{
    if (!ps) return DD_E_NULL;
    if (int rc = fill_state(a, s, c, n)) return rc;
    if (n > 0 && (!ps->table || !ps->index)) return DD_E_NULL;
    if (ps->count < 1 || ps->count > DD_MAX_PARAM_SETS || (ps->flags & ~DD_PARAM_SETS_RESAMPLE)) return DD_E_RANGE;
    if (ps->dtype != s->dtype) return DD_E_DTYPE;
    if (reinterpret_cast<uintptr_t>(ps->table) & 15u) return DD_E_ALIGN;
    a.ps_table = ps->table; a.ps_index = ps->index;
    a.ps_count = (uint32_t)ps->count; a.ps_resample = (ps->flags & DD_PARAM_SETS_RESAMPLE) ? 1 : 0;
    return 0;
}

// Kernel mode of a call: single-set calls use the immediates when the parameters are config.py's; per-env sets never.
static bool params_are_default(const DDParamSets&) { return false; }

static inline int check_stride(int32_t stride) {
    return (stride == DD_OBS_DIM || stride == kMaxObsStride) ? 0 : DD_E_RANGE;
}

// DDEnvConfig.obs_format, checked before any CUDA call: DD_E_RANGE for an unknown value, DD_E_DTYPE for a 16-bit format
// with float64 state (the exact-parity instantiation writes its own precision only).  NULL structs are left to the
// callee's checks.
static int check_obs_format(const DDState* s, const DDEnvConfig* c)
{
    if (!s || !c) return 0;
    if (c->obs_format < DD_OBS_NATIVE || c->obs_format > DD_OBS_BF16) return DD_E_RANGE;
    if (c->obs_format != DD_OBS_NATIVE && s->dtype != DD_F32) return DD_E_DTYPE;
    return 0;
}

template <typename R, bool SETS, typename P>
static int reset_impl(const DDState* s, const P* p, const DDEnvConfig* c, const uint8_t* mask,
                      void* obs, int32_t obs_stride, int64_t n, cudaStream_t st)
{
    KArgsOf<R, SETS> a;
    if (int rc = fill_args(a, s, p, c, n)) return rc;
    if (obs) { if (int rc = check_stride(obs_stride)) return rc; a.obs_stride = obs_stride; }
    a.obs = (R*)obs;
    if (n == 0) return 0;
    DeviceGuard g(st, s->pos_vel);
    if (g.err != cudaSuccess) return (int)g.err;
    const bool pdl = (c->launch_flags & DD_LAUNCH_PDL) != 0;
    if constexpr (sizeof(R) == 4) {                        // 16-bit observations: float state only
        if (c->obs_format == DD_OBS_F16) return launch(reset_kernel<R, DD_OBS_F16, SETS>, grid_for(n, kBlock), kBlock, st, pdl, a, mask);
        if (c->obs_format == DD_OBS_BF16) return launch(reset_kernel<R, DD_OBS_BF16, SETS>, grid_for(n, kBlock), kBlock, st, pdl, a, mask);
    }
    return launch(reset_kernel<R, DD_OBS_NATIVE, SETS>, grid_for(n, kBlock), kBlock, st, pdl, a, mask);
}

// The resolved launch of one dd_step call: what dd_step_plan stores in the caller's DDStepPlan.
template <typename R, bool SETS = false>
struct StepPlanT {
    uint32_t magic;
    int32_t dtype, device, grid, block, pdl;
    void (*kern)(KArgsOf<R, SETS>);
    KArgsOf<R, SETS> a;                                    // everything but `actions`
};
constexpr uint32_t kPlanMagic = 0x44445034u;               // "DDP4"
constexpr uint32_t kPlanMagicSets = 0x44445334u;           // "DDS4": a plan of dd_step_plan_sets
static_assert(sizeof(StepPlanT<double, true>) <= DD_STEP_PLAN_BYTES && sizeof(StepPlanT<float, true>) <= DD_STEP_PLAN_BYTES,
              "DD_STEP_PLAN_BYTES too small for the argument block");

template <typename R, bool AUTO, bool OBS, bool DEF, int OF, bool SETS>
static void (*step_kernel_of(int block))(KArgsOf<R, SETS>)
{
    if constexpr (sizeof(R) == 4) {                        // CTA-size variants: float only (tuning knob)
        if (block == 128) return step_kernel<R, AUTO, OBS, DEF, 128, OF, SETS>;
        if (block == 512) return step_kernel<R, AUTO, OBS, DEF, 512, OF, SETS>;
    }
    return step_kernel<R, AUTO, OBS, DEF, 256, OF, SETS>;
}

template <typename R, int OF, bool SETS>
static void (*step_kernel_sel(bool au, bool ob, bool def, int block))(KArgsOf<R, SETS>)
{
#define DD_STEP(AU, OB, DF) step_kernel_of<R, AU, OB, DF, OF, SETS>(block)
    if (!SETS && def)                                      // per-env sets: DEF = false only
        return au ? (ob ? DD_STEP(true, true, !SETS) : DD_STEP(true, false, !SETS))
                  : (ob ? DD_STEP(false, true, !SETS) : DD_STEP(false, false, !SETS));
    return au ? (ob ? DD_STEP(true, true, false) : DD_STEP(true, false, false))
              : (ob ? DD_STEP(false, true, false) : DD_STEP(false, false, false));
#undef DD_STEP
}

// Validate a dd_step call and resolve it to (kernel, grid, block, argument block).
template <typename R, bool SETS, typename P>
static int step_resolve(StepPlanT<R, SETS>& pl, const DDState* s, const P* p, const DDEnvConfig* c,
                        void* obs, int32_t obs_stride, void* reward, uint8_t* done_flags, void* final_obs,
                        uint64_t* stats, int64_t n)
{
    KArgsOf<R, SETS>& a = pl.a;
    if (int rc = fill_args(a, s, p, c, n)) return rc;
    if (obs || final_obs) { if (int rc = check_stride(obs_stride)) return rc; a.obs_stride = obs_stride; }
    a.obs = (R*)obs; a.reward = (R*)reward; a.final_obs = (R*)final_obs;
    a.done_flags = done_flags; a.stats = (unsigned long long*)stats;
    const bool au = c->auto_reset != 0, ob = obs != nullptr, def = params_are_default(*p);
    const int bsel = (c->launch_flags >> 4) & 3;
    int block = bsel == 1 ? 128 : (bsel == 2 ? 512 : 256);
    if (sizeof(R) != 4) block = 256;
    pl.magic = SETS ? kPlanMagicSets : kPlanMagic; pl.dtype = sizeof(R) == 4 ? DD_F32 : DD_F64; pl.device = -1;
    pl.block = block; pl.grid = grid_for(n, block); pl.pdl = (c->launch_flags & DD_LAUNCH_PDL) ? 1 : 0;
    pl.kern = step_kernel_sel<R, DD_OBS_NATIVE, SETS>(au, ob, def, block);
    if constexpr (sizeof(R) == 4) {                        // 16-bit observations: float state only
        if (c->obs_format == DD_OBS_F16) pl.kern = step_kernel_sel<R, DD_OBS_F16, SETS>(au, ob, def, block);
        if (c->obs_format == DD_OBS_BF16) pl.kern = step_kernel_sel<R, DD_OBS_BF16, SETS>(au, ob, def, block);
    }
    return 0;
}

template <typename R, bool SETS, typename P>
static int step_impl(const DDState* s, const P* p, const DDEnvConfig* c, const uint8_t* actions,
                     void* obs, int32_t obs_stride, void* reward, uint8_t* done_flags, void* final_obs,
                     uint64_t* stats, int64_t n, cudaStream_t st)
{
    StepPlanT<R, SETS> pl;
    if (int rc = step_resolve(pl, s, p, c, obs, obs_stride, reward, done_flags, final_obs, stats, n)) return rc;
    if (!actions && n > 0) return DD_E_NULL;
    if (n == 0) return 0;
    DeviceGuard g(st, s->pos_vel);
    if (g.err != cudaSuccess) return (int)g.err;
    pl.a.actions = actions;
    return launch(pl.kern, pl.grid, pl.block, st, pl.pdl != 0, pl.a);
}

template <typename R, bool SETS>
static int step_planned(const StepPlanT<R, SETS>& pl, const uint8_t* actions, cudaStream_t st)
{
    if (pl.a.n == 0) return 0;
    if (!actions) return DD_E_NULL;
    DeviceGuard g(pl.device);
    if (g.err != cudaSuccess) return (int)g.err;
    KArgsOf<R, SETS> a = pl.a;
    a.actions = actions;
    return launch(pl.kern, pl.grid, pl.block, st, pl.pdl != 0, a);
}

template <typename R, bool SETS, typename P>
static int rollout_impl(const DDState* s, const P* p, const DDEnvConfig* c, int32_t policy,
                        const uint8_t* actions_tn, uint32_t t0, int32_t T, void* reward_tn, uint8_t* done_tn,
                        void* obs_tn, int32_t obs_stride, void* shaped_tn, uint64_t* stats, int64_t n, cudaStream_t st)
{
    RArgs<R, KArgsOf<R, SETS>> ra{};
    if (int rc = fill_args(ra.a, s, p, c, n)) return rc;
    if (policy < DD_POLICY_TRACE || policy > DD_POLICY_BANGBANG) return DD_E_RANGE;
    if (policy == DD_POLICY_TRACE && !actions_tn && n > 0 && T > 0) return DD_E_NULL;
    if (T < 0) return DD_E_RANGE;
    if (obs_tn) { if (int rc = check_stride(obs_stride)) return rc; ra.a.obs_stride = obs_stride; }
    ra.a.stats = (unsigned long long*)stats;
    if (shaped_tn && !s->prev_dist && n > 0) return DD_E_NULL;
    if (shaped_tn && c->shaping != DD_SHAPING_PPO && c->shaping != DD_SHAPING_PG) return DD_E_RANGE;
    ra.actions_tn = actions_tn; ra.reward_tn = (R*)reward_tn; ra.done_tn = done_tn; ra.obs_tn = (R*)obs_tn;
    ra.shaped_tn = (R*)shaped_tn;
    ra.t0 = t0; ra.T = T; ra.policy = policy; ra.auto_reset = c->auto_reset;
    if (n == 0 || T == 0) return 0;
    DeviceGuard guard(st, s->pos_vel);
    if (guard.err != cudaSuccess) return (int)guard.err;
    const bool pdl = (c->launch_flags & DD_LAUNCH_PDL) != 0, def = params_are_default(*p);
    const int g = grid_for(n, kBlock);
    const bool outs = reward_tn || done_tn || shaped_tn;
#define DD_ROLL2(OBS_, DEF_, OUTS_, OF_)                                                                                          \
    (policy == DD_POLICY_TRACE    ? launch(rollout_kernel<R, OBS_, DEF_, DD_POLICY_TRACE, OUTS_, OF_, SETS>, g, kBlock, st, pdl, ra)  \
     : policy == DD_POLICY_RANDOM ? launch(rollout_kernel<R, OBS_, DEF_, DD_POLICY_RANDOM, OUTS_, OF_, SETS>, g, kBlock, st, pdl, ra) \
                                  : launch(rollout_kernel<R, OBS_, DEF_, DD_POLICY_BANGBANG, OUTS_, OF_, SETS>, g, kBlock, st, pdl, ra))
#define DD_ROLL(OBS_, DEF_, OF_) (outs ? DD_ROLL2(OBS_, DEF_, true, OF_) : DD_ROLL2(OBS_, DEF_, false, OF_))
    // per-env sets: DEF = false only (DEF = !SETS below instantiates nothing new for them)
    if constexpr (sizeof(R) == 4) {                        // 16-bit obs_tn: float state only
        if (obs_tn && c->obs_format == DD_OBS_F16) return def ? DD_ROLL(true, !SETS, DD_OBS_F16) : DD_ROLL(true, false, DD_OBS_F16);
        if (obs_tn && c->obs_format == DD_OBS_BF16) return def ? DD_ROLL(true, !SETS, DD_OBS_BF16) : DD_ROLL(true, false, DD_OBS_BF16);
    }
    if (def) return obs_tn ? DD_ROLL(true, !SETS, DD_OBS_NATIVE) : DD_ROLL(false, !SETS, DD_OBS_NATIVE);
    return obs_tn ? DD_ROLL(true, false, DD_OBS_NATIVE) : DD_ROLL(false, false, DD_OBS_NATIVE);
#undef DD_ROLL
#undef DD_ROLL2
}

}  // namespace dd

extern "C" {

int dd_abi_version(void) { return DD_ABI_VERSION; }

void dd_default_params(DDParams* p)
{
    if (!p) return;
    *p = dd::kDefaultParams;
}

const char* dd_error_string(int code)
{
    switch (code) {
        case 0: return "ok";
        case DD_E_NULL: return "null pointer argument";
        case DD_E_RANGE: return "argument out of range";
        case DD_E_DTYPE: return "unknown dtype";
        case DD_E_ALIGN: return "buffer not sufficiently aligned";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int dd_reset(const DDState* s, const DDParams* p, const DDEnvConfig* c, const uint8_t* mask,
             void* obs, int32_t obs_stride, int64_t n, void* stream)
{
    if (!s) return DD_E_NULL;
    if (int rc = dd::check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32) return dd::reset_impl<float, false>(s, p, c, mask, obs, obs_stride, n, (cudaStream_t)stream);
    if (s->dtype == DD_F64) return dd::reset_impl<double, false>(s, p, c, mask, obs, obs_stride, n, (cudaStream_t)stream);
    return DD_E_DTYPE;
}

int dd_step(const DDState* s, const DDParams* p, const DDEnvConfig* c, const uint8_t* actions,
            void* obs, int32_t obs_stride, void* reward, uint8_t* done_flags, void* final_obs,
            uint64_t* stats, int64_t n, void* stream)
{
    if (!s) return DD_E_NULL;
    if (int rc = dd::check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32)
        return dd::step_impl<float, false>(s, p, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n, (cudaStream_t)stream);
    if (s->dtype == DD_F64)
        return dd::step_impl<double, false>(s, p, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n, (cudaStream_t)stream);
    return DD_E_DTYPE;
}

}  // extern "C"

namespace dd {
template <bool SETS, typename P>
static int step_plan_impl(const DDState* s, const P* p, const DDEnvConfig* c, void* obs, int32_t obs_stride,
                          void* reward, uint8_t* done_flags, void* final_obs, uint64_t* stats, int64_t n, DDStepPlan* plan)
{
    if (!s || !plan) return DD_E_NULL;
    if (s->dtype != DD_F32 && s->dtype != DD_F64) return DD_E_DTYPE;
    if (int rc = dd::check_obs_format(s, c)) { memset(plan, 0, sizeof *plan); return rc; }
    memset(plan, 0, sizeof *plan);
    int rc, *device;
    if (s->dtype == DD_F32) {
        auto* pl = reinterpret_cast<dd::StepPlanT<float, SETS>*>(plan);
        rc = dd::step_resolve(*pl, s, p, c, obs, obs_stride, reward, done_flags, final_obs, stats, n);
        device = &pl->device;
    } else {
        auto* pl = reinterpret_cast<dd::StepPlanT<double, SETS>*>(plan);
        rc = dd::step_resolve(*pl, s, p, c, obs, obs_stride, reward, done_flags, final_obs, stats, n);
        device = &pl->device;
    }
    if (rc) { memset(plan, 0, sizeof *plan); return rc; }
    // the state buffers name the device the planned launches run on
    const cudaError_t e = dd::owning_device(nullptr, n > 0 ? s->pos_vel : nullptr, device);
    if (e != cudaSuccess) { memset(plan, 0, sizeof *plan); return (int)e; }
    return 0;
}
}  // namespace dd

extern "C" {

int dd_step_plan(const DDState* s, const DDParams* p, const DDEnvConfig* c, void* obs, int32_t obs_stride,
                 void* reward, uint8_t* done_flags, void* final_obs, uint64_t* stats, int64_t n, DDStepPlan* plan)
{
    return dd::step_plan_impl<false>(s, p, c, obs, obs_stride, reward, done_flags, final_obs, stats, n, plan);
}

int dd_step_plan_sets(const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, void* obs, int32_t obs_stride,
                      void* reward, uint8_t* done_flags, void* final_obs, uint64_t* stats, int64_t n, DDStepPlan* plan)
{
    return dd::step_plan_impl<true>(s, ps, c, obs, obs_stride, reward, done_flags, final_obs, stats, n, plan);
}

int dd_param_sets_build(const DDParams* sets, int32_t count, int32_t dtype, void* host_out)
{
    return dd::param_sets_build_checked(sets, count, dtype, host_out);
}

int dd_reset_sets(const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, const uint8_t* mask,
                  void* obs, int32_t obs_stride, int64_t n, void* stream)
{
    if (!s) return DD_E_NULL;
    if (int rc = dd::check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32) return dd::reset_impl<float, true>(s, ps, c, mask, obs, obs_stride, n, (cudaStream_t)stream);
    if (s->dtype == DD_F64) return dd::reset_impl<double, true>(s, ps, c, mask, obs, obs_stride, n, (cudaStream_t)stream);
    return DD_E_DTYPE;
}

int dd_step_sets(const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, const uint8_t* actions,
                 void* obs, int32_t obs_stride, void* reward, uint8_t* done_flags, void* final_obs,
                 uint64_t* stats, int64_t n, void* stream)
{
    if (!s) return DD_E_NULL;
    if (int rc = dd::check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32)
        return dd::step_impl<float, true>(s, ps, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n, (cudaStream_t)stream);
    if (s->dtype == DD_F64)
        return dd::step_impl<double, true>(s, ps, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n, (cudaStream_t)stream);
    return DD_E_DTYPE;
}

int dd_rollout_sets(const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, int32_t policy,
                    const uint8_t* actions_tn, uint32_t t0, int32_t T, void* reward_tn, uint8_t* done_tn,
                    void* obs_tn, int32_t obs_stride, void* shaped_tn, uint64_t* stats, int64_t n, void* stream)
{
    if (!s) return DD_E_NULL;
    if (int rc = dd::check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32)
        return dd::rollout_impl<float, true>(s, ps, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n, (cudaStream_t)stream);
    if (s->dtype == DD_F64)
        return dd::rollout_impl<double, true>(s, ps, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n, (cudaStream_t)stream);
    return DD_E_DTYPE;
}

int dd_step_planned(const DDStepPlan* plan, const uint8_t* actions, void* stream)
{
    if (!plan) return DD_E_NULL;
    const auto* hdr = reinterpret_cast<const dd::StepPlanT<float>*>(plan);
    if (hdr->magic == dd::kPlanMagicSets) {                           // dd_step_plan_sets
        if (hdr->dtype == DD_F32) return dd::step_planned(*reinterpret_cast<const dd::StepPlanT<float, true>*>(plan), actions, (cudaStream_t)stream);
        if (hdr->dtype == DD_F64) return dd::step_planned(*reinterpret_cast<const dd::StepPlanT<double, true>*>(plan), actions, (cudaStream_t)stream);
        return DD_E_DTYPE;
    }
    if (hdr->magic != dd::kPlanMagic) return DD_E_RANGE;             // not (or no longer) a plan
    if (hdr->dtype == DD_F32) return dd::step_planned(*hdr, actions, (cudaStream_t)stream);
    if (hdr->dtype == DD_F64) return dd::step_planned(*reinterpret_cast<const dd::StepPlanT<double>*>(plan), actions, (cudaStream_t)stream);
    return DD_E_DTYPE;
}

int dd_rollout_shaped(const DDState* s, const DDParams* p, const DDEnvConfig* c, int32_t policy,
                      const uint8_t* actions_tn, uint32_t t0, int32_t T, void* reward_tn, uint8_t* done_tn,
                      void* obs_tn, int32_t obs_stride, void* shaped_tn, uint64_t* stats, int64_t n, void* stream)
{
    if (!s) return DD_E_NULL;
    if (int rc = dd::check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32)
        return dd::rollout_impl<float, false>(s, p, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n, (cudaStream_t)stream);
    if (s->dtype == DD_F64)
        return dd::rollout_impl<double, false>(s, p, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n, (cudaStream_t)stream);
    return DD_E_DTYPE;
}

int dd_rollout(const DDState* s, const DDParams* p, const DDEnvConfig* c, int32_t policy,
               const uint8_t* actions_tn, uint32_t t0, int32_t T, void* reward_tn, uint8_t* done_tn,
               void* obs_tn, int32_t obs_stride, uint64_t* stats, int64_t n, void* stream)
{
    return dd_rollout_shaped(s, p, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, nullptr, stats, n, stream);
}

int dd_fill_random_actions(uint8_t* actions_tn, uint64_t seed, uint64_t env_id_base, uint32_t t0, int32_t T,
                           int64_t n, void* stream)
{
    if (!actions_tn) return DD_E_NULL;
    if (n < 0 || T < 0) return DD_E_RANGE;
    if (n == 0 || T == 0) return 0;
    dd::DeviceGuard g((cudaStream_t)stream, actions_tn);
    if (g.err != cudaSuccess) return (int)g.err;
    dd::fill_random_actions_kernel<<<dd::grid_for(n, dd::kBlock), dd::kBlock, 0, (cudaStream_t)stream>>>(actions_tn, seed, env_id_base, t0, T, n);
    return (int)cudaGetLastError();
}

int dd_gather_env(const DDState* s, const void* obs, int32_t obs_stride, const void* reward,
                  const uint8_t* step_flags, int64_t i, int64_t n, double* out, void* stream)
{
    if (!s || !out) return DD_E_NULL;
    if (!s->pos_vel || !s->att_fuel || !s->platform || !s->steps || !s->episode || !s->flags) return DD_E_NULL;
    if (i < 0 || i >= n) return DD_E_RANGE;
    if (obs && obs_stride != 15 && obs_stride != 16) return DD_E_RANGE;
    if (s->dtype != DD_F32 && s->dtype != DD_F64) return DD_E_DTYPE;
    dd::DeviceGuard g((cudaStream_t)stream, s->pos_vel);
    if (g.err != cudaSuccess) return (int)g.err;
    if (s->dtype == DD_F32)
        dd::gather_env_kernel<float><<<1, 32, 0, (cudaStream_t)stream>>>(
            (const float*)s->pos_vel, (const float*)s->att_fuel, (const float*)s->platform, s->steps, s->episode, s->flags,
            (const float*)obs, obs_stride, (const float*)reward, step_flags, i, out);
    else if (s->dtype == DD_F64)
        dd::gather_env_kernel<double><<<1, 32, 0, (cudaStream_t)stream>>>(
            (const double*)s->pos_vel, (const double*)s->att_fuel, (const double*)s->platform, s->steps, s->episode, s->flags,
            (const double*)obs, obs_stride, (const double*)reward, step_flags, i, out);
    else return DD_E_DTYPE;
    return (int)cudaGetLastError();
}

int dd_pack_actions(const uint8_t* actions3, uint8_t* packed, int64_t n, void* stream)
{
    if (!actions3 || !packed) return DD_E_NULL;
    if (n < 0) return DD_E_RANGE;
    if (n == 0) return 0;
    dd::DeviceGuard g((cudaStream_t)stream, packed);
    if (g.err != cudaSuccess) return (int)g.err;
    dd::pack_actions_kernel<<<dd::grid_for(n, dd::kBlock), dd::kBlock, 0, (cudaStream_t)stream>>>(actions3, packed, n);
    return (int)cudaGetLastError();
}

int dd_stats_collapse(const uint64_t* stats, const int32_t* steps, const uint8_t* flags, int64_t n,
                      uint64_t* out, void* stream)
{
    if (!stats || !out) return DD_E_NULL;
    if (n < 0) return DD_E_RANGE;
    if (n > 0 && ((steps == nullptr) != (flags == nullptr))) return DD_E_NULL;
    dd::DeviceGuard g((cudaStream_t)stream, stats);
    if (g.err != cudaSuccess) return (int)g.err;
    dd::stats_collapse_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const unsigned long long*)stats, (unsigned long long*)out);
    if (steps && n > 0) {
        int g = dd::grid_for(n, dd::kBlock * 8);
        if (g > 148 * 8) g = 148 * 8;
        dd::live_steps_kernel<<<g, dd::kBlock, 0, (cudaStream_t)stream>>>(steps, flags, n, (unsigned long long*)out);
    }
    return (int)cudaGetLastError();
}

}  // extern "C"
