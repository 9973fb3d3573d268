/*
 * drone_b200_host.h -- HOST twins of dd_reset / dd_step / dd_rollout_shaped (SURVEY.md 8b: "plus host
 * double/float twins of dd_step for tests").
 *
 * TEST INFRASTRUCTURE, not a product path and not a fallback: the twins live in their own library
 * (libdrone_b200_host.so, built by g++ -ffp-contract=off from csrc/host_twin.cpp), nothing under
 * reinforcement-learning-101_b200/ loads it, and BatchedDroneEnv refuses non-CUDA devices.  What they are for:
 * they instantiate the SAME per-environment source the kernels inline -- step_core, write_obs, spawn,
 * shaped_reward, philox4x32_10, action_block of csrc/drone_core.cuh -- for the host, so the kernel's own
 * arithmetic source is under test on a machine without a GPU, against the golden vectors recorded from the
 * unmodified reference (/root/reference/delivery_drone/game/game_engine.py:95-216).
 *
 * Same argument meaning as the device entry points of drone_b200.h, with these differences:
 *   - every pointer is HOST memory, there is no stream, the call is synchronous;
 *   - `stats` is ONE block uint64[DD_STATS_WORDS] (no contention slots), words 0-5 as on the device; under
 *     DD_PARAM_SETS_STATS_BY_SET (the _sets twins) uint64[count][DD_STATS_WORDS], attributed as on the device;
 *   - DD_F32: bit-identical to the device kernels except where sin / cos enter (the device uses sincospif,
 *     the host rounds a float64 libm result; <= 1 ulp apart) and expf of the `pg` shaping.
 *     DD_F64: every product and sum rounded separately like the device path; libm sin / cos.
 *   - c->obs_format is honoured as on the device: 16-bit rows are the fp32 rows converted by the portable
 *     round-to-nearest-even routine that stands in for the kernels' hardware conversion.
 */
#ifndef DRONE_B200_HOST_H
#define DRONE_B200_HOST_H

#include "drone_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

int dd_host_abi_version(void);      /* == DD_ABI_VERSION of the sources it was built from */

int dd_reset_host(const DDState *s, const DDParams *p, const DDEnvConfig *c, const uint8_t *mask,
                  void *obs, int32_t obs_stride, int64_t n);

int dd_step_host(const DDState *s, const DDParams *p, const DDEnvConfig *c, const uint8_t *actions,
                 void *obs, int32_t obs_stride, void *reward, uint8_t *done_flags, void *final_obs,
                 uint64_t *stats, int64_t n);

int dd_rollout_host(const DDState *s, const DDParams *p, const DDEnvConfig *c, int32_t policy,
                    const uint8_t *actions_tn, uint32_t t0, int32_t T,
                    void *reward_tn, uint8_t *done_tn, void *obs_tn, int32_t obs_stride, void *shaped_tn,
                    uint64_t *stats, int64_t n);

/* The _sets entry points of drone_b200.h over host memory: `ps->table` holds the bytes dd_param_sets_build_host (or
 * the device library's dd_param_sets_build) wrote, `ps->index` is host memory, written at resets under
 * DD_PARAM_SETS_RESAMPLE.  Same selection, resampling rule and argument codes as on the device. */
int dd_param_sets_build_host(const DDParams *sets, int32_t count, int32_t dtype, void *host_out);
int dd_reset_sets_host(const DDState *s, const DDParamSets *ps, const DDEnvConfig *c, const uint8_t *mask,
                       void *obs, int32_t obs_stride, int64_t n);
int dd_step_sets_host(const DDState *s, const DDParamSets *ps, const DDEnvConfig *c, const uint8_t *actions,
                      void *obs, int32_t obs_stride, void *reward, uint8_t *done_flags, void *final_obs,
                      uint64_t *stats, int64_t n);
int dd_rollout_sets_host(const DDState *s, const DDParamSets *ps, const DDEnvConfig *c, int32_t policy,
                         const uint8_t *actions_tn, uint32_t t0, int32_t T,
                         void *reward_tn, uint8_t *done_tn, void *obs_tn, int32_t obs_stride, void *shaped_tn,
                         uint64_t *stats, int64_t n);

/* out[i] = x[i] as DD_OBS_F16 / DD_OBS_BF16 bits (fmt): the conversion of the 16-bit observation formats. */
int dd_obs16_convert_host(int32_t fmt, const float *x, uint16_t *out, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* DRONE_B200_HOST_H */
