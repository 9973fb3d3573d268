// env_abi.h -- host side of the env entry points of the C ABI (drone_kernels.cu, policy_rollout.cu): the argument checks
// of include/drone_b200.h that turn DDState / DDParams / DDParamSets / DDEnvConfig into a kernel argument block, and the
// helpers that turn a call's runtime choices into the template arguments of the kernel it runs.
#pragma once
#include <stdint.h>
#include <string.h>
#include <type_traits>
#include "drone_device.cuh"

namespace dd {

// Everything of the argument block but the constants.
template <typename R>
inline int fill_state(KArgs<R>& a, const DDState* s, const DDEnvConfig* c, int64_t n)
{
    if (!s || !c) return DD_E_NULL;
    if (n < 0 || n > (int64_t)DD_MAX_ENVS_PER_CALL) return DD_E_RANGE;
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
inline int fill_args(KArgs<R>& a, const DDState* s, const DDParams* p, const DDEnvConfig* c, int64_t n)
{
    if (!p) return DD_E_NULL;
    if (int rc = fill_state(a, s, c, n)) return rc;
    a.k = make_consts<R>(*p);
    return 0;
}

// The DDParamSets checks of include/drone_b200.h, then the argument block of the per-env kernels.
template <typename R>
inline int fill_args(KArgsPS<R>& a, const DDState* s, const DDParamSets* ps, const DDEnvConfig* c, int64_t n)
{
    if (!ps) return DD_E_NULL;
    if (int rc = fill_state(a, s, c, n)) return rc;
    if (n > 0 && (!ps->table || !ps->index)) return DD_E_NULL;
    if (ps->count < 1 || ps->count > DD_MAX_PARAM_SETS || (ps->flags & ~(DD_PARAM_SETS_RESAMPLE | DD_PARAM_SETS_STATS_BY_SET)))
        return DD_E_RANGE;
    if (ps->dtype != s->dtype) return DD_E_DTYPE;
    if (reinterpret_cast<uintptr_t>(ps->table) & 15u) return DD_E_ALIGN;
    a.ps_table = ps->table; a.ps_index = ps->index;
    a.ps_count = (uint32_t)ps->count; a.ps_resample = (ps->flags & DD_PARAM_SETS_RESAMPLE) ? 1 : 0;
    return 0;
}

inline int check_stride(int32_t stride) {
    return (stride == DD_OBS_DIM || stride == kMaxObsStride) ? 0 : DD_E_RANGE;
}

// DDEnvConfig.obs_format, checked before any CUDA call: DD_E_RANGE for an unknown value, DD_E_DTYPE for a 16-bit format
// with float64 state (the exact-parity instantiation writes its own precision only).  NULL structs are left to the
// callee's checks.
inline int check_obs_format(const DDState* s, const DDEnvConfig* c)
{
    if (!s || !c) return 0;
    if (c->obs_format < DD_OBS_NATIVE || c->obs_format > DD_OBS_BF16) return DD_E_RANGE;
    if (c->obs_format != DD_OBS_NATIVE && s->dtype != DD_F32) return DD_E_DTYPE;
    return 0;
}

// Whether a call may run the DEF kernels, which hold config.py's parameters as immediates.
inline bool params_are_default(const DDParams& p)
{
    const DDParams d = kDefaultParams;
    if (memcmp(&p, &d, sizeof d) != 0) return false;
    // the compile-time constants assume sqrt thresholds that the search confirms
    return speed2_threshold<float>((float)p.land_speed) == (float)p.land_speed * (float)p.land_speed &&
           speed2_threshold<double>(p.land_speed) == p.land_speed * p.land_speed;
}

// The preamble of the env entry points: a state, an obs_format that fits it, then f(R()) with the state's element type.
template <typename F>
inline int with_state_type(const DDState* s, const DDEnvConfig* c, F&& f)
{
    if (!s) return DD_E_NULL;
    if (int rc = check_obs_format(s, c)) return rc;
    if (s->dtype == DD_F32) return f(float());
    if (s->dtype == DD_F64) return f(double());
    return DD_E_DTYPE;
}

// ---- runtime choice -> template argument ------------------------------------------------------------------------------
// Both f(std::true_type()) and f(std::false_type()) are instantiated: a rule that excludes kernels must be applied to the
// constant with `if constexpr`, never to the runtime value.
template <typename F>
inline auto with_bool(bool b, F&& f) { return b ? f(std::true_type()) : f(std::false_type()); }

template <int V> using int_c = std::integral_constant<int, V>;

// f(std::bool_constant<BYSET>()): the statistics-per-set kernels exist for parameter-set calls only.
template <bool SETS, typename P, typename F>
inline auto with_by_set(const P& p, F&& f)
{
    if constexpr (SETS) return with_bool((p.flags & DD_PARAM_SETS_STATS_BY_SET) != 0, f);
    else return f(std::false_type());
}

// f(int_c<OF>()) for a DDEnvConfig.obs_format that check_obs_format accepted: the 16-bit formats exist for float only.
template <typename R, typename F>
inline auto with_obs_format(int32_t obs_format, F&& f)
{
    if constexpr (std::is_same<R, float>::value) {
        if (obs_format == DD_OBS_F16) return f(int_c<DD_OBS_F16>());
        if (obs_format == DD_OBS_BF16) return f(int_c<DD_OBS_BF16>());
    }
    return f(int_c<DD_OBS_NATIVE>());
}

}  // namespace dd
