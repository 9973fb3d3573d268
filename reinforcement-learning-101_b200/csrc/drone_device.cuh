// drone_device.cuh -- device-side helpers shared by the kernels of drone_kernels.cu, policy_rollout.cu
// and ppo_kernels.cu: kernel argument block, 16-byte vector access, load pinning, programmatic
// dependent launch, warp sums, warp-aggregated episode statistics.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "drone_core.cuh"

namespace dd {

constexpr int kMaxObsStride = 16;

template <typename R>
struct KArgs {
    R *pos_vel, *att_fuel, *platform, *prev_dist;
    int32_t* steps;
    uint32_t* episode;
    uint8_t* flags;
    const uint8_t* actions;
    R *obs, *reward, *final_obs;
    uint8_t* done_flags;
    unsigned long long* stats;
    uint32_t n;
    uint64_t seed, env_id_base;
    int32_t max_steps, obs_stride;
    int32_t shaping;                      // DD_SHAPING_*
    int32_t rand_drone, rand_platform;
    Consts<R> k;
};

// The argument block of the per-env parameter-set kernels (SETS = true): KArgs (whose `k` they do not read) + the
// DDParamSets pointers.  Appended, so that the single-set kernels keep their argument layout.
template <typename R>
struct KArgsPS : KArgs<R> {
    const void* ps_table;                 // Consts<R> [word][set], drone_core.cuh param_set
    uint8_t* ps_index;
    uint32_t ps_count;
    int32_t ps_resample;                  // DD_PARAM_SETS_RESAMPLE
};
template <typename R, bool SETS> struct KArgsSel { using type = KArgs<R>; };
template <typename R> struct KArgsSel<R, true> { using type = KArgsPS<R>; };
template <typename R, bool SETS> using KArgsOf = typename KArgsSel<R, SETS>::type;

// DEF: the parameters are config.py's defaults -> compile-time constants (immediates); otherwise
// they come from the kernel argument (constant bank).
template <typename R, bool DEF>
__device__ __forceinline__ Consts<R> consts_of(const KArgs<R>& a) {
    if constexpr (DEF) {
        constexpr Consts<R> kc = make_consts_base<R>(kDefaultParams);
        return kc;
    } else {
        return a.k;
    }
}

// ---- 16-byte vector access ---------------------------------------------------------------
__device__ __forceinline__ void load4(const float* p, uint32_t i, float& a, float& b, float& c, float& d) {
    const float4 v = reinterpret_cast<const float4*>(p)[i];
    a = v.x; b = v.y; c = v.z; d = v.w;
}
__device__ __forceinline__ void load4(const double* p, uint32_t i, double& a, double& b, double& c, double& d) {
    const double2 u = reinterpret_cast<const double2*>(p)[2 * (size_t)i], v = reinterpret_cast<const double2*>(p)[2 * (size_t)i + 1];
    a = u.x; b = u.y; c = v.x; d = v.y;
}
__device__ __forceinline__ void store4(float* p, uint32_t i, float a, float b, float c, float d) {
    reinterpret_cast<float4*>(p)[i] = make_float4(a, b, c, d);
}
__device__ __forceinline__ void store4(double* p, uint32_t i, double a, double b, double c, double d) {
    reinterpret_cast<double2*>(p)[2 * (size_t)i] = make_double2(a, b);
    reinterpret_cast<double2*>(p)[2 * (size_t)i + 1] = make_double2(c, d);
}
__device__ __forceinline__ void load2(const float* p, uint32_t i, float& a, float& b) {
    const float2 v = reinterpret_cast<const float2*>(p)[i]; a = v.x; b = v.y;
}
__device__ __forceinline__ void load2(const double* p, uint32_t i, double& a, double& b) {
    const double2 v = reinterpret_cast<const double2*>(p)[i]; a = v.x; b = v.y;
}
__device__ __forceinline__ void store2(float* p, uint32_t i, float a, float b) {
    reinterpret_cast<float2*>(p)[i] = make_float2(a, b);
}
__device__ __forceinline__ void store2(double* p, uint32_t i, double a, double b) {
    reinterpret_cast<double2*>(p)[i] = make_double2(a, b);
}

// The optimiser may not sink a load below this point (e.g. into a branch that is the only user):
// all of a thread's loads must be in flight together.
__device__ __forceinline__ void pin(float v) { asm volatile("" :: "f"(v)); }
__device__ __forceinline__ void pin(double v) { asm volatile("" :: "d"(v)); }
__device__ __forceinline__ void pin(uint32_t v) { asm volatile("" :: "r"(v)); }
__device__ __forceinline__ void pin(int32_t v) { asm volatile("" :: "r"(v)); }

template <typename R>
__device__ __forceinline__ void load_env(const KArgs<R>& a, uint32_t i, Env<R>& e) {
    load4(a.pos_vel, i, e.x, e.y, e.vx, e.vy);
    load4(a.att_fuel, i, e.angle, e.angvel, e.fuel, e.ret);
    load2(a.platform, i, e.px, e.py);
    e.steps = a.steps[i];
    pin(e.x); pin(e.y); pin(e.vx); pin(e.vy); pin(e.angle); pin(e.angvel); pin(e.fuel); pin(e.ret);
    pin(e.px); pin(e.py); pin(e.steps);
}
template <typename R>
__device__ __forceinline__ void store_env(const KArgs<R>& a, uint32_t i, const Env<R>& e) {
    store4(a.pos_vel, i, e.x, e.y, e.vx, e.vy);
    store4(a.att_fuel, i, e.angle, e.angvel, e.fuel, e.ret);
    a.steps[i] = e.steps;
}

// Programmatic dependent launch (sm_90+): `wait` blocks until the preceding kernel in the stream
// has completed and flushed (no-op when the launch carried no such dependency); `launch` lets the
// next kernel's CTAs become resident as soon as every CTA of this one has got here.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- K3: episode statistics ------------------------------------------------------------------
// Words: 0 episodes, 1 landed, 2 crashed, 3 truncated, 4 sum_return (int64, 2^-20), 5 sum_length.
// (word 6, env_steps, is derived at collapse time: sum_length + steps of the live episodes.)
// Integer accumulation makes the totals independent of summation order, hence of grid shape and
// GPU count.
template <typename T>                                   // sum over the 32 lanes of a converged warp
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <typename R> __device__ __forceinline__ R nan_of();
template <> __device__ __forceinline__ float nan_of<float>() { return __int_as_float(0x7fc00000); }
template <> __device__ __forceinline__ double nan_of<double>() { return __longlong_as_double(0x7ff8000000000000ll); }

__device__ __forceinline__ long long return_fx(double ret) { return __double2ll_rn(ret * DD_RETURN_FIXED_SCALE); }
// fp32 state: scaling by 2^20 is exact in float, so this is the same integer as the double path, without
// touching the (slow on B200) FP64 pipe
__device__ __forceinline__ long long return_fx(float ret) { return __float2ll_rn(ret * (float)DD_RETURN_FIXED_SCALE); }

// Called by ALL 32 lanes of a warp (f == 0 in lanes whose episode goes on).  Costs one ballot in
// the common case; the reductions and the REDs run only in warps where some episode ended.
template <typename R>
__device__ __forceinline__ void stats_warp_commit(unsigned long long* stats, uint32_t f, R ret, int32_t steps) {
    const unsigned done = __ballot_sync(0xffffffffu, f != 0u);
    if (done == 0u) return;                                // warp-uniform
    const unsigned landed = __ballot_sync(0xffffffffu, (f & DD_LANDED) != 0u);
    const unsigned crashed = __ballot_sync(0xffffffffu, (f & DD_CRASHED) != 0u);
    const unsigned trunc = __ballot_sync(0xffffffffu, (f & DD_TRUNCATED) != 0u);
    const long long rsum = warp_sum(f ? return_fx(ret) : 0ll);
    const unsigned len = __reduce_add_sync(0xffffffffu, f ? (unsigned)steps : 0u);
    if ((threadIdx.x & 31) == 0) {
        const unsigned gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
        unsigned long long* s = stats + (gw % DD_STATS_SLOTS) * DD_STATS_WORDS;
        atomicAdd(s + 0, (unsigned long long)__popc(done));
        if (landed) atomicAdd(s + 1, (unsigned long long)__popc(landed));
        if (crashed) atomicAdd(s + 2, (unsigned long long)__popc(crashed));
        if (trunc) atomicAdd(s + 3, (unsigned long long)__popc(trunc));
        atomicAdd(s + 4, (unsigned long long)rsum);
        atomicAdd(s + 5, (unsigned long long)len);
    }
}

// ---- statistics per parameter set (DD_PARAM_SETS_STATS_BY_SET) ----------------------------------
// `stats` is uint64[count][DD_STATS_SLOTS][DD_STATS_WORDS]; an episode counts in the block of the set its ending step ran
// under.  Slot choice as above: only the sums are defined.
__device__ __forceinline__ unsigned long long* stats_set_slot(unsigned long long* stats, uint32_t set, unsigned slot) {
    return stats + ((size_t)set * DD_STATS_SLOTS + slot % DD_STATS_SLOTS) * DD_STATS_WORDS;
}

// stats_warp_commit with the ending lanes grouped by `set`: one pass of the same reductions per distinct set among them
// (usually one).  Called by ALL 32 lanes; the common case is still the one ballot.
template <typename R>
__device__ __forceinline__ void stats_warp_commit_by_set(unsigned long long* stats, uint32_t f, R ret, int32_t steps,
                                                         uint32_t set) {
    unsigned todo = __ballot_sync(0xffffffffu, f != 0u);
    if (todo == 0u) return;                                // warp-uniform
    const long long rfx = f ? return_fx(ret) : 0ll;
    const unsigned gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    do {
        const uint32_t s = __shfl_sync(0xffffffffu, set, __ffs(todo) - 1);
        const bool mine = f != 0u && set == s;
        const unsigned done = __ballot_sync(0xffffffffu, mine);
        todo &= ~done;
        const unsigned landed = __ballot_sync(0xffffffffu, mine && (f & DD_LANDED) != 0u);
        const unsigned crashed = __ballot_sync(0xffffffffu, mine && (f & DD_CRASHED) != 0u);
        const unsigned trunc = __ballot_sync(0xffffffffu, mine && (f & DD_TRUNCATED) != 0u);
        const long long rsum = warp_sum(mine ? rfx : 0ll);
        const unsigned len = __reduce_add_sync(0xffffffffu, mine ? (unsigned)steps : 0u);
        if ((threadIdx.x & 31) == 0) {
            unsigned long long* b = stats_set_slot(stats, s, gw);
            atomicAdd(b + 0, (unsigned long long)__popc(done));
            if (landed) atomicAdd(b + 1, (unsigned long long)__popc(landed));
            if (crashed) atomicAdd(b + 2, (unsigned long long)__popc(crashed));
            if (trunc) atomicAdd(b + 3, (unsigned long long)__popc(trunc));
            atomicAdd(b + 4, (unsigned long long)rsum);
            atomicAdd(b + 5, (unsigned long long)len);
        }
    } while (todo);
}

// The same statistics accumulated PER THREAD over a multi-step kernel and committed once at its end: integer sums, so
// the totals equal a stats_warp_commit per step.  (In the T-steps-per-launch kernels the per-step commit -- a ballot every
// step; three more ballots, ten shuffles and six atomics whenever a lane's episode ended -- was 1-6 % of the issue slots.)
struct StatsAcc {
    uint32_t done = 0, landed = 0, crashed = 0, trunc = 0, len = 0;
    long long ret = 0;
    template <typename R>
    __device__ __forceinline__ void add(uint32_t f, R ret_, int32_t steps) {
        if (f) {
            done += 1u; landed += (f & DD_LANDED) ? 1u : 0u; crashed += (f & DD_CRASHED) ? 1u : 0u; trunc += (f & DD_TRUNCATED) ? 1u : 0u;
            ret += return_fx(ret_); len += (uint32_t)steps;
        }
    }
    // called by ALL 32 lanes of a warp
    __device__ __forceinline__ void commit(unsigned long long* stats) const {
        const unsigned nd = __reduce_add_sync(0xffffffffu, done);
        if (nd == 0u) return;                              // warp-uniform
        const unsigned nl = __reduce_add_sync(0xffffffffu, landed), nc = __reduce_add_sync(0xffffffffu, crashed),
                       nt = __reduce_add_sync(0xffffffffu, trunc);
        const long long lsum = warp_sum((long long)len), rsum = warp_sum(ret);
        if ((threadIdx.x & 31) == 0) {
            const unsigned gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
            unsigned long long* s = stats + (gw % DD_STATS_SLOTS) * DD_STATS_WORDS;
            atomicAdd(s + 0, (unsigned long long)nd);
            if (nl) atomicAdd(s + 1, (unsigned long long)nl);
            if (nc) atomicAdd(s + 2, (unsigned long long)nc);
            if (nt) atomicAdd(s + 3, (unsigned long long)nt);
            atomicAdd(s + 4, (unsigned long long)rsum);
            atomicAdd(s + 5, (unsigned long long)lsum);
        }
    }
    // By-set mode.  commit with the lanes grouped by their (final) set, called by ALL 32 lanes.
    __device__ __forceinline__ void commit_by_set(unsigned long long* stats, uint32_t set) const {
        unsigned todo = __ballot_sync(0xffffffffu, done != 0u);
        if (todo == 0u) return;                            // warp-uniform
        const unsigned gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
        do {
            const uint32_t s = __shfl_sync(0xffffffffu, set, __ffs(todo) - 1);
            const bool mine = done != 0u && set == s;
            todo &= ~__ballot_sync(0xffffffffu, mine);
            const unsigned nd = __reduce_add_sync(0xffffffffu, mine ? done : 0u),
                           nl = __reduce_add_sync(0xffffffffu, mine ? landed : 0u),
                           nc = __reduce_add_sync(0xffffffffu, mine ? crashed : 0u),
                           nt = __reduce_add_sync(0xffffffffu, mine ? trunc : 0u);
            const long long lsum = warp_sum(mine ? (long long)len : 0ll), rsum = warp_sum(mine ? ret : 0ll);
            if ((threadIdx.x & 31) == 0) {
                unsigned long long* b = stats_set_slot(stats, s, gw);
                atomicAdd(b + 0, (unsigned long long)nd);
                if (nl) atomicAdd(b + 1, (unsigned long long)nl);
                if (nc) atomicAdd(b + 2, (unsigned long long)nc);
                if (nt) atomicAdd(b + 3, (unsigned long long)nt);
                atomicAdd(b + 4, (unsigned long long)rsum);
                atomicAdd(b + 5, (unsigned long long)lsum);
            }
        } while (todo);
    }
    // By-set mode, when a resampling reset moves the thread to another set: this thread's totals so far go to `set`'s
    // block on their own (a few REDs in the episode-end branch; no warp collective there) and the accumulator restarts.
    __device__ __forceinline__ void flush_thread(unsigned long long* stats, uint32_t set) {
        if (done) {
            unsigned long long* b = stats_set_slot(stats, set, blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
            atomicAdd(b + 0, (unsigned long long)done);
            if (landed) atomicAdd(b + 1, (unsigned long long)landed);
            if (crashed) atomicAdd(b + 2, (unsigned long long)crashed);
            if (trunc) atomicAdd(b + 3, (unsigned long long)trunc);
            atomicAdd(b + 4, (unsigned long long)ret);
            atomicAdd(b + 5, (unsigned long long)len);
        }
        *this = StatsAcc();
    }
};

}  // namespace dd
