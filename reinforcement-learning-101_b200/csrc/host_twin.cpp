// host_twin.cpp -- host instantiation of the per-environment code of the kernels (include/drone_b200_host.h).
//
// TEST INFRASTRUCTURE.  Compiled by g++ (-O2 -ffp-contract=off, no -ffast-math, no -mfma) into its own library
// libdrone_b200_host.so; the product never loads it.  Everything numeric comes from drone_core.cuh -- the same
// step_core / write_obs / spawn / shaped_reward / Philox source that step_kernel, rollout_kernel and the fused
// policy kernel inline; only the orchestration around it (which env resets, what is stored where) is restated
// here, following step_kernel / rollout_kernel of drone_kernels.cu statement by statement.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include "drone_core.cuh"
#include "../../include/drone_b200_host.h"

namespace {

using namespace dd;

template <typename R>
struct HostState {
    R *pos_vel, *att_fuel, *platform, *prev_dist;
    int32_t* steps;
    uint32_t* episode;
    uint8_t* flags;
};

template <typename R>
int bind(HostState<R>& h, const DDState* s, const DDEnvConfig* c, int64_t n)
{
    if (!s || !c) return DD_E_NULL;
    if (n < 0 || n > (int64_t)DD_MAX_ENVS_PER_CALL) return DD_E_RANGE;
    if (n > 0 && (!s->pos_vel || !s->att_fuel || !s->platform || !s->steps || !s->episode || !s->flags)) return DD_E_NULL;
    h.pos_vel = (R*)s->pos_vel; h.att_fuel = (R*)s->att_fuel; h.platform = (R*)s->platform; h.prev_dist = (R*)s->prev_dist;
    h.steps = s->steps; h.episode = s->episode; h.flags = s->flags;
    return 0;
}

template <typename R>
void load_env(const HostState<R>& h, int64_t i, Env<R>& e)
{
    e.x = h.pos_vel[4 * i]; e.y = h.pos_vel[4 * i + 1]; e.vx = h.pos_vel[4 * i + 2]; e.vy = h.pos_vel[4 * i + 3];
    e.angle = h.att_fuel[4 * i]; e.angvel = h.att_fuel[4 * i + 1]; e.fuel = h.att_fuel[4 * i + 2]; e.ret = h.att_fuel[4 * i + 3];
    e.px = h.platform[2 * i]; e.py = h.platform[2 * i + 1];
    e.steps = h.steps[i];
}

template <typename R>
void store_env(const HostState<R>& h, int64_t i, const Env<R>& e)
{
    h.pos_vel[4 * i] = e.x; h.pos_vel[4 * i + 1] = e.y; h.pos_vel[4 * i + 2] = e.vx; h.pos_vel[4 * i + 3] = e.vy;
    h.att_fuel[4 * i] = e.angle; h.att_fuel[4 * i + 1] = e.angvel; h.att_fuel[4 * i + 2] = e.fuel; h.att_fuel[4 * i + 3] = e.ret;
    h.steps[i] = e.steps;
}

template <typename R> long long return_fx(R ret) { return std::llrint((double)ret * DD_RETURN_FIXED_SCALE); }

template <typename R>
void stats_commit(uint64_t* st, uint32_t f, R ret, int32_t steps)
{
    if (!st || !f) return;
    st[0] += 1;
    if (f & DD_LANDED) st[1] += 1;
    if (f & DD_CRASHED) st[2] += 1;
    if (f & DD_TRUNCATED) st[3] += 1;
    st[4] += (uint64_t)return_fx(ret);
    st[5] += (uint64_t)steps;
}

// Where env i's constants come from: the call's DDParams, or its entry of a DDParamSets table (the _sets twins).
template <typename R>
struct ConstSource {
    Consts<R> k0{};
    const DDParamSets* ps = nullptr;
    int init(const DDState* s, const DDParams* p, const DDParamSets* sets, int64_t n)     // fill_args of drone_kernels.cu
    {
        if (!sets) { if (!p) return DD_E_NULL; k0 = make_consts<R>(*p); return 0; }
        if (n > 0 && (!sets->table || !sets->index)) return DD_E_NULL;
        if (sets->count < 1 || sets->count > DD_MAX_PARAM_SETS || (sets->flags & ~DD_PARAM_SETS_RESAMPLE)) return DD_E_RANGE;
        if (sets->dtype != s->dtype) return DD_E_DTYPE;
        if (reinterpret_cast<uintptr_t>(sets->table) & 15u) return DD_E_ALIGN;
        ps = sets;
        return 0;
    }
    Consts<R> of(int64_t i) const
    {
        return ps ? param_set<R>(ps->table, param_set_clamp(ps->index[i], (uint32_t)ps->count)) : k0;
    }
    // the constants of env i's reset number `ep`: under DD_PARAM_SETS_RESAMPLE a new set, recorded in index[i]
    Consts<R> at_reset(int64_t i, const Consts<R>& cur, uint64_t seed, uint64_t gid, uint32_t ep) const
    {
        if (!ps || !(ps->flags & DD_PARAM_SETS_RESAMPLE)) return cur;
        const uint32_t s = param_set_draw(seed, gid, ep, (uint32_t)ps->count);
        ps->index[i] = (uint8_t)s;
        return param_set<R>(ps->table, s);
    }
};

inline int check_stride(int32_t stride) { return (stride == DD_OBS_DIM || stride == 16) ? 0 : DD_E_RANGE; }

// check_obs_format of drone_kernels.cu
inline int check_obs_format(const DDState* s, const DDEnvConfig* c)
{
    if (!s || !c) return 0;
    if (c->obs_format < DD_OBS_NATIVE || c->obs_format > DD_OBS_BF16) return DD_E_RANGE;
    if (c->obs_format != DD_OBS_NATIVE && s->dtype != DD_F32) return DD_E_DTYPE;
    return 0;
}

// Row r of an observation buffer in format `fmt` (DD_OBS_*; 16-bit formats: float state only): write_obs, or
// write_obs16 as the kernels' 16-bit instantiations call it.  steps_col: column 15 = `steps`.
template <typename R>
void obs_row(void* base, int64_t r, int32_t stride, int32_t fmt, const Env<R>& e, uint32_t flags, R speed, R dist,
             const Consts<R>& k, bool steps_col, R steps)
{
    if constexpr (sizeof(R) == 4) {
        if (fmt != DD_OBS_NATIVE) {
            uint16_t* row = (uint16_t*)base + r * stride;
            auto put = [&](int j, uint16_t v) { row[j] = v; };
            if (fmt == DD_OBS_F16) write_obs16<DD_OBS_F16>(e, flags, speed, dist, k, steps_col, steps, put);
            else write_obs16<DD_OBS_BF16>(e, flags, speed, dist, k, steps_col, steps, put);
            return;
        }
    }
    R* row = (R*)base + r * stride;
    write_obs(e, flags, speed, dist, k, [&](int j, R v) { row[j] = v; });
    if (steps_col) row[DD_OBS_DIM] = steps;
}

template <typename R>
int reset_host(const DDState* s, const DDParams* p, const DDParamSets* ps, const DDEnvConfig* c, const uint8_t* mask,
               void* obs_, int32_t stride, int64_t n)
{
    HostState<R> h;
    if (int rc = bind(h, s, c, n)) return rc;
    ConstSource<R> src;
    if (int rc = src.init(s, p, ps, n)) return rc;
    if (obs_) if (int rc = check_stride(stride)) return rc;
    void* obs = obs_;
    for (int64_t i = 0; i < n; ++i) {                                  // reset_kernel
        if (mask && !mask[i]) continue;
        Env<R> e;
        const uint32_t ep = h.episode[i];
        const Consts<R> k = src.at_reset(i, src.of(i), c->seed, c->env_id_base + (uint64_t)i, ep);
        spawn(e, k, c->seed, c->env_id_base + (uint64_t)i, ep, c->randomize_drone != 0, c->randomize_platform != 0);
        h.episode[i] = ep + 1;
        store_env(h, i, e);
        h.platform[2 * i] = e.px; h.platform[2 * i + 1] = e.py;
        h.flags[i] = 0;
        if (h.prev_dist) h.prev_dist[i] = std::numeric_limits<R>::quiet_NaN();
        if (obs) {
            R speed, dist;
            speed_dist(e, speed, dist);
            obs_row(obs, i, stride, c->obs_format, e, 0u, speed, dist, k, stride > DD_OBS_DIM, (R)0);
        }
    }
    return 0;
}

template <typename R>
int step_host(const DDState* s, const DDParams* p, const DDParamSets* ps, const DDEnvConfig* c, const uint8_t* actions,
              void* obs_, int32_t stride, void* reward_, uint8_t* done_flags, void* final_obs_, uint64_t* stats, int64_t n)
{
    HostState<R> h;
    if (int rc = bind(h, s, c, n)) return rc;
    ConstSource<R> src;
    if (int rc = src.init(s, p, ps, n)) return rc;
    if (!actions && n > 0) return DD_E_NULL;
    if (obs_ || final_obs_) if (int rc = check_stride(stride)) return rc;
    void *obs = obs_, *final_obs = final_obs_;
    R* reward_out = (R*)reward_;
    const bool AUTO = c->auto_reset != 0, OBS = obs != nullptr;
    for (int64_t i = 0; i < n; ++i) {                                  // step_kernel, one "thread" at a time
        Env<R> e;
        const uint32_t act = actions[i];
        load_env(h, i, e);
        Consts<R> k = src.of(i);
        uint32_t pflags = AUTO ? 0u : (uint32_t)h.flags[i];
        uint32_t oflags = pflags;
        R reward = (R)0, speed = (R)0, dist = (R)0;
        const bool stepped = !(act & DD_ACT_SKIP) && !(pflags & DD_DONE);
        if (stepped) {
            uint32_t f = step_core<R, true>(e, act, k, reward, speed, dist);
            if (!f && c->max_steps > 0 && e.steps >= c->max_steps) f = DD_DONE | DD_TRUNCATED;
            oflags = f;
            if (f) {
                stats_commit(stats, f, e.ret, e.steps);
                if (final_obs) obs_row(final_obs, i, stride, c->obs_format, e, f, speed, dist, k, false, (R)0);
                if (AUTO) {
                    const uint32_t ep = h.episode[i];
                    k = src.at_reset(i, k, c->seed, c->env_id_base + (uint64_t)i, ep);
                    spawn(e, k, c->seed, c->env_id_base + (uint64_t)i, ep, c->randomize_drone != 0, c->randomize_platform != 0);
                    h.episode[i] = ep + 1;
                    h.platform[2 * i] = e.px; h.platform[2 * i + 1] = e.py;
                    if (h.prev_dist) h.prev_dist[i] = std::numeric_limits<R>::quiet_NaN();
                    f = 0;
                    if (OBS) speed_dist(e, speed, dist);
                }
            }
            pflags = f;
            store_env(h, i, e);
            if (!AUTO) h.flags[i] = (uint8_t)pflags;
        } else if (OBS) {
            speed_dist(e, speed, dist);
        }
        if (reward_out) reward_out[i] = reward;
        if (done_flags) done_flags[i] = (uint8_t)oflags;
        if (OBS) obs_row(obs, i, stride, c->obs_format, e, pflags, speed, dist, k, stride > DD_OBS_DIM, (R)e.steps);
    }
    return 0;
}

template <typename R>
int rollout_host(const DDState* s, const DDParams* p, const DDParamSets* ps, const DDEnvConfig* c, int32_t policy,
                 const uint8_t* actions_tn, uint32_t t0, int32_t T, void* reward_tn_, uint8_t* done_tn, void* obs_tn_,
                 int32_t stride, void* shaped_tn_, uint64_t* stats, int64_t n)
{
    HostState<R> h;
    if (int rc = bind(h, s, c, n)) return rc;
    ConstSource<R> src;
    if (int rc = src.init(s, p, ps, n)) return rc;
    if (policy < DD_POLICY_TRACE || policy > DD_POLICY_BANGBANG) return DD_E_RANGE;
    if (policy == DD_POLICY_TRACE && !actions_tn && n > 0 && T > 0) return DD_E_NULL;
    if (T < 0) return DD_E_RANGE;
    if (obs_tn_) if (int rc = check_stride(stride)) return rc;
    if (shaped_tn_ && !s->prev_dist && n > 0) return DD_E_NULL;
    if (shaped_tn_ && c->shaping != DD_SHAPING_PPO && c->shaping != DD_SHAPING_PG) return DD_E_RANGE;
    R *reward_tn = (R*)reward_tn_, *shaped_tn = (R*)shaped_tn_;
    void* obs_tn = obs_tn_;
    const bool OBS = obs_tn != nullptr, shaping = shaped_tn != nullptr, auto_reset = c->auto_reset != 0;
    const int32_t max_steps = c->max_steps;
    const R nan = std::numeric_limits<R>::quiet_NaN();
    for (int64_t i = 0; i < n; ++i) {                                  // rollout_kernel, one "thread" at a time
        Env<R> e;
        load_env(h, i, e);
        Consts<R> k = src.of(i);
        uint32_t pflags = h.flags[i], ep = h.episode[i];
        bool platform_dirty = false;
        const uint64_t gid = c->env_id_base + (uint64_t)i;
        R dprev = nan, dcur = (R)0;
        if (shaping) {
            R s_, d_;
            speed_dist(e, s_, d_);
            dcur = Arith<R>::div(d_, k.width, k.inv_width);
            dprev = h.prev_dist[i];
        }
        for (int32_t t = 0; t < T; ++t) {
            const int64_t o = (int64_t)t * n + i;
            uint32_t oflags = pflags;
            R reward = (R)0, speed = (R)0, dist = (R)0, shaped = (R)0;
            uint32_t act;
            if (policy == DD_POLICY_TRACE) act = actions_tn[o];
            else if (policy == DD_POLICY_RANDOM) act = action_from_block(action_block(c->seed, gid, t0 + (uint32_t)t), t0 + (uint32_t)t);
            else act = (e.vy > (R)1.5) ? DD_ACT_MAIN : 0u;
            if (!(act & DD_ACT_SKIP) && !(pflags & DD_DONE)) {
                uint32_t f = step_core<R, true>(e, act, k, reward, speed, dist);
                if (!f && max_steps > 0 && e.steps >= max_steps) f = DD_DONE | DD_TRUNCATED;
                oflags = f;
                if (shaping) {
                    shaped = shaped_reward(c->shaping, e, f, speed, dist, dprev, max_steps > 0 && e.steps >= max_steps, k);
                    dprev = dcur;
                    dcur = Arith<R>::div(dist, k.width, k.inv_width);
                }
                if (f) {
                    stats_commit(stats, f, e.ret, e.steps);
                    if (auto_reset) {
                        k = src.at_reset(i, k, c->seed, gid, ep);
                        spawn(e, k, c->seed, gid, ep, c->randomize_drone != 0, c->randomize_platform != 0);
                        ep += 1;
                        platform_dirty = true;
                        f = 0;
                        speed_dist(e, speed, dist);
                        if (shaping) { dprev = nan; dcur = Arith<R>::div(dist, k.width, k.inv_width); }
                    }
                }
                pflags = f;
            } else if (OBS) {
                speed_dist(e, speed, dist);
            }
            if (shaping) shaped_tn[o] = shaped;
            if (reward_tn) reward_tn[o] = reward;
            if (done_tn) done_tn[o] = (uint8_t)oflags;
            if (OBS) obs_row(obs_tn, o, stride, c->obs_format, e, pflags, speed, dist, k, stride > DD_OBS_DIM, (R)e.steps);
        }
        store_env(h, i, e);
        h.flags[i] = (uint8_t)pflags;
        h.episode[i] = ep;
        if (platform_dirty) { h.platform[2 * i] = e.px; h.platform[2 * i + 1] = e.py; }
        if (shaping) h.prev_dist[i] = dprev;
    }
    return 0;
}

}  // namespace

extern "C" {

int dd_host_abi_version(void) { return DD_ABI_VERSION; }

int dd_reset_host(const DDState* s, const DDParams* p, const DDEnvConfig* c, const uint8_t* mask, void* obs, int32_t obs_stride, int64_t n)
{
    if (!s) return DD_E_NULL;
    if (int rc = check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32) return reset_host<float>(s, p, nullptr, c, mask, obs, obs_stride, n);
    if (s->dtype == DD_F64) return reset_host<double>(s, p, nullptr, c, mask, obs, obs_stride, n);
    return DD_E_DTYPE;
}

int dd_step_host(const DDState* s, const DDParams* p, const DDEnvConfig* c, const uint8_t* actions, void* obs, int32_t obs_stride,
                 void* reward, uint8_t* done_flags, void* final_obs, uint64_t* stats, int64_t n)
{
    if (!s) return DD_E_NULL;
    if (int rc = check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32) return step_host<float>(s, p, nullptr, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n);
    if (s->dtype == DD_F64) return step_host<double>(s, p, nullptr, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n);
    return DD_E_DTYPE;
}

int dd_rollout_host(const DDState* s, const DDParams* p, const DDEnvConfig* c, int32_t policy, const uint8_t* actions_tn, uint32_t t0,
                    int32_t T, void* reward_tn, uint8_t* done_tn, void* obs_tn, int32_t obs_stride, void* shaped_tn, uint64_t* stats, int64_t n)
{
    if (!s) return DD_E_NULL;
    if (int rc = check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32)
        return rollout_host<float>(s, p, nullptr, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n);
    if (s->dtype == DD_F64)
        return rollout_host<double>(s, p, nullptr, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n);
    return DD_E_DTYPE;
}

int dd_param_sets_build_host(const DDParams* sets, int32_t count, int32_t dtype, void* host_out)
{
    return param_sets_build_checked(sets, count, dtype, host_out);
}

int dd_reset_sets_host(const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, const uint8_t* mask, void* obs,
                       int32_t obs_stride, int64_t n)
{
    if (!s) return DD_E_NULL;
    if (int rc = check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32) return reset_host<float>(s, nullptr, ps, c, mask, obs, obs_stride, n);
    if (s->dtype == DD_F64) return reset_host<double>(s, nullptr, ps, c, mask, obs, obs_stride, n);
    return DD_E_DTYPE;
}

int dd_step_sets_host(const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, const uint8_t* actions, void* obs,
                      int32_t obs_stride, void* reward, uint8_t* done_flags, void* final_obs, uint64_t* stats, int64_t n)
{
    if (!s) return DD_E_NULL;
    if (int rc = check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32) return step_host<float>(s, nullptr, ps, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n);
    if (s->dtype == DD_F64) return step_host<double>(s, nullptr, ps, c, actions, obs, obs_stride, reward, done_flags, final_obs, stats, n);
    return DD_E_DTYPE;
}

int dd_rollout_sets_host(const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, int32_t policy, const uint8_t* actions_tn,
                         uint32_t t0, int32_t T, void* reward_tn, uint8_t* done_tn, void* obs_tn, int32_t obs_stride,
                         void* shaped_tn, uint64_t* stats, int64_t n)
{
    if (!s) return DD_E_NULL;
    if (int rc = check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32)
        return rollout_host<float>(s, nullptr, ps, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n);
    if (s->dtype == DD_F64)
        return rollout_host<double>(s, nullptr, ps, c, policy, actions_tn, t0, T, reward_tn, done_tn, obs_tn, obs_stride, shaped_tn, stats, n);
    return DD_E_DTYPE;
}

int dd_obs16_convert_host(int32_t fmt, const float* x, uint16_t* out, int64_t n)
{
    if ((!x || !out) && n > 0) return DD_E_NULL;
    if ((fmt != DD_OBS_F16 && fmt != DD_OBS_BF16) || n < 0) return DD_E_RANGE;
    for (int64_t i = 0; i < n; ++i)
        out[i] = (uint16_t)(fmt == DD_OBS_F16 ? obs16_pack2<DD_OBS_F16>(x[i], 0.0f) : obs16_pack2<DD_OBS_BF16>(x[i], 0.0f));
    return 0;
}

}  // extern "C"
