// ppo_kernels.cu -- the three HBM-bound reductions / scans that sit right after a rollout:
//
//   K4 moments_kernel    n, sum x, sum x^2 of the advantage buffer (one read of [T*n] floats)
//      normalize_kernel  (x - mean) / (std + eps), unbiased std like torch.std
//                        (Actor_Critic_PPO.ipynb c21:L105, Policy_Gradients.ipynb c26:L33-36)
//   N3 gae_kernel        compute_gae backward scan, one thread per env, coalesced over n
//                        (Actor_Critic_PPO.ipynb c15:L49-53)
//
// Streaming float work: float4 loads, grid = a whole number of waves over the 148 SMs, double
// accumulation only in the per-thread / per-warp partials.
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/drone_b200.h"
#include "drone_device.cuh"
#include "host_guard.h"

namespace dd {

constexpr int kRedBlock = 256;
constexpr int kSMs = 148;

__global__ void __launch_bounds__(kRedBlock) moments_kernel(const float* __restrict__ x, int64_t n, double* out)
{
    __shared__ double s_s[kRedBlock / 32], s_q[kRedBlock / 32];
    double s = 0.0, q = 0.0;
    pdl_wait();
    pdl_launch_dependents();
    const int64_t tid = (int64_t)blockIdx.x * kRedBlock + threadIdx.x;
    const int64_t nthreads = (int64_t)gridDim.x * kRedBlock;
    // leading scalars until x is 16-byte aligned, then float4, then the tail
    int64_t head = (int64_t)((16u - (uint32_t)(reinterpret_cast<uintptr_t>(x) & 15u)) & 15u) / 4;
    if (head > n) head = n;
    const int64_t n4 = (n - head) / 4;
    const float4* x4 = reinterpret_cast<const float4*>(x + head);
    // four independent 16-byte loads in flight per thread per trip (one load at a time is latency-bound)
    for (int64_t j = tid; j < n4; j += 4 * nthreads) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t k = j + u * nthreads;
            v[u] = k < n4 ? __ldg(x4 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            // partial sums of 4 in float would lose bits; go to double per element
            s += (double)v[u].x + (double)v[u].y + (double)v[u].z + (double)v[u].w;
            q += (double)v[u].x * v[u].x + (double)v[u].y * v[u].y + (double)v[u].z * v[u].z + (double)v[u].w * v[u].w;
        }
    }
    if (tid < head) { const double v = x[tid]; s += v; q += v * v; }
    const int64_t tail0 = head + 4 * n4;
    if (tid < n - tail0) { const double v = x[tail0 + tid]; s += v; q += v * v; }

    s = warp_sum(s); q = warp_sum(q);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) { s_s[w] = s; s_q[w] = q; }
    __syncthreads();
    if (w == 0) {
        s = lane < kRedBlock / 32 ? s_s[lane] : 0.0;
        q = lane < kRedBlock / 32 ? s_q[lane] : 0.0;
        s = warp_sum(s); q = warp_sum(q);
        if (lane == 0) {
            atomicAdd(out + 1, s);
            atomicAdd(out + 2, q);
            if (blockIdx.x == 0) atomicAdd(out + 0, (double)n);
        }
    }
}

__global__ void __launch_bounds__(kRedBlock) normalize_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                               const double* __restrict__ m, double eps, int64_t n)
{
    pdl_wait();                                            // the moments (and x) come from the previous kernels
    pdl_launch_dependents();
    const double cnt = m[0], s = m[1], q = m[2];
    const double mean = cnt > 0 ? s / cnt : 0.0;
    double var = cnt > 1 ? (q - s * mean) / (cnt - 1.0) : 0.0;     // unbiased, torch.std default
    var = var > 0 ? var : 0.0;
    const float fmean = (float)mean;
    const float inv = (float)(1.0 / (sqrt(var) + eps));
    const int64_t tid = (int64_t)blockIdx.x * kRedBlock + threadIdx.x;
    const int64_t nthreads = (int64_t)gridDim.x * kRedBlock;
    const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0;
    if (vec) {
        const int64_t n4 = n / 4;
        const float4* x4 = reinterpret_cast<const float4*>(x);
        float4* y4 = reinterpret_cast<float4*>(y);
        for (int64_t j = tid; j < n4; j += 4 * nthreads) {      // four independent loads in flight per thread per trip
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t k = j + u * nthreads;
                if (k < n4) v[u] = __ldg(x4 + k);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t k = j + u * nthreads;
                if (k < n4) {
                    v[u].x = (v[u].x - fmean) * inv; v[u].y = (v[u].y - fmean) * inv;
                    v[u].z = (v[u].z - fmean) * inv; v[u].w = (v[u].w - fmean) * inv;
                    y4[k] = v[u];
                }
            }
        }
        if (tid < n - 4 * n4) y[4 * n4 + tid] = (x[4 * n4 + tid] - fmean) * inv;
    } else {
        for (int64_t j = tid; j < n; j += nthreads) y[j] = (x[j] - fmean) * inv;
    }
}

// delta_t = r_t + gamma * V_{t+1} * (1 - done_t) - V_t ;  A_t = delta_t + gamma * lambda * (1 - done_t) * A_{t+1}
// fp32 throughout, in the operation order of the torch original (python scalars gamma, gamma*lambda
// are combined in double and rounded to fp32 when they meet the tensors).  No FMA contraction, so
// the result is bit-identical to the eager torch loop.
// The scan is a dependent chain only through `gae` (4 dependent fp32 operations per step); the loads are not on
// it.  A thread-per-env scan has little parallelism at PPO sizes (65,536 envs = 443 threads per SM), so the
// loop works in chunks of kGaeUnroll steps whose 3 x kGaeUnroll loads are all issued before the first is used:
// the launch is bound by DRAM latency / kGaeUnroll instead of DRAM latency per step.
// Chunks are double-buffered in registers: the loads of chunk c+1 are issued BEFORE chunk c is scanned, so loads
// stay in flight during the dependent arithmetic and the stores (round 1 issued them only after the scan of the
// previous chunk: 4.4 TB/s).  A thread owns V adjacent envs: one 4V-byte load per array and step
// instead of V scalar ones, V independent scan chains per thread.  Measured on B200 at 65,536 envs x 250 steps
// (profiles/r02_gae_variants.jsonl, V = 1 / 2 / 4 x block x chunk): V = 2, 16-step chunks, 32-thread CTAs is the best
// register configuration (a thread then keeps 2 x 16 x 18 B in flight); V = 1 serves buffers that are not aligned
// to the pair or an odd number of envs.  A cp.async shared-memory ring with 4-6 stages per 64-env CTA
// was tried and is SLOWER (47 us against 39.5: at this size the kernel is a ~33 us stream plus a fixed ~4 us
// of launch ramp and drain; at 262,144 envs the same kernel runs at 89 % of the measured HBM bandwidth).
// The launches carry the programmatic-dependent-launch attribute: the CTAs become resident while the previous
// kernel of the stream drains and wait (griddepcontrol.wait) before their first global access.
// MOM: the advantage moments (n, sum, sum of squares; K4) are accumulated in the same pass -- the normalisation
// that follows (Actor_Critic_PPO.ipynb c21:L105) then needs no separate read of the advantage buffer.
constexpr int kGaeBlock = 32;     // threads per CTA
constexpr int kGaeUnroll = 16;    // steps per register chunk
constexpr int kGaeVec = 2;        // envs per thread when every row is aligned to the pair

template <int V> struct VecLd;
template <> struct VecLd<1> {
    static __device__ __forceinline__ void f(const float* p, float (&o)[1]) { o[0] = __ldg(p); }
    static __device__ __forceinline__ void b(const uint8_t* p, uint8_t (&o)[1]) { o[0] = __ldg(p); }
    static __device__ __forceinline__ void st(float* p, const float (&v)[1]) { *p = v[0]; }
};
template <> struct VecLd<2> {
    static __device__ __forceinline__ void f(const float* p, float (&o)[2]) { const float2 t = __ldg(reinterpret_cast<const float2*>(p)); o[0] = t.x; o[1] = t.y; }
    static __device__ __forceinline__ void b(const uint8_t* p, uint8_t (&o)[2]) { const uchar2 t = __ldg(reinterpret_cast<const uchar2*>(p)); o[0] = t.x; o[1] = t.y; }
    static __device__ __forceinline__ void st(float* p, const float (&v)[2]) { *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]); }
};

template <int V, int U>
struct GaeChunk {
    float r[U][V], v[U][V];
    uint8_t d[U][V];
    // steps t1-1 ... t1-U (clamped at 0: the surplus loads of the last chunk re-read row 0)
    __device__ __forceinline__ void load(const float* __restrict__ rew, const float* __restrict__ val,
                                         const uint8_t* __restrict__ done, int32_t t1, int64_t n, int64_t i) {
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int32_t t = t1 - 1 - j;
            const int64_t o = (int64_t)(t >= 0 ? t : 0) * n + i;
            VecLd<V>::f(rew + o, r[j]); VecLd<V>::f(val + o, v[j]); VecLd<V>::b(done + o, d[j]);
        }
    }
    template <bool MOM>
    __device__ __forceinline__ void scan(float* __restrict__ adv, float* __restrict__ ret, float g, float gl, int32_t t1,
                                         int64_t n, int64_t i, float (&gae)[V], float (&v_next)[V], double& s, double& q) const {
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int32_t t = t1 - 1 - j;
            if (t >= 0) {
                const int64_t o = (int64_t)t * n + i;
                float a[V], rt[V];
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    const float mask = d[j][e] ? 0.0f : 1.0f;
                    const float delta = __fsub_rn(__fadd_rn(r[j][e], __fmul_rn(__fmul_rn(g, v_next[e]), mask)), v[j][e]);
                    gae[e] = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, mask), gae[e]));
                    a[e] = gae[e];
                    rt[e] = __fadd_rn(gae[e], v[j][e]);
                    v_next[e] = v[j][e];
                    if (MOM) { const double x = (double)gae[e]; s += x; q = fma(x, x, q); }
                }
                VecLd<V>::st(adv + o, a);
                if (ret) VecLd<V>::st(ret + o, rt);
            }
        }
    }
};

template <int V, bool MOM>
__global__ void __launch_bounds__(kGaeBlock) gae_kernel(const float* __restrict__ rew, const float* __restrict__ val,
                                                        const uint8_t* __restrict__ done, float* __restrict__ adv,
                                                        float* __restrict__ ret, double* __restrict__ mom, float g, float gl,
                                                        int32_t T, int64_t n)
{
    const int64_t i = ((int64_t)blockIdx.x * kGaeBlock + threadIdx.x) * V;
    double s = 0.0, q = 0.0;
    pdl_wait();                                            // inputs may come from the previous kernel of the stream
    pdl_launch_dependents();
    if (i < n) {
        float gae[V], v_next[V];
#pragma unroll
        for (int e = 0; e < V; ++e) gae[e] = 0.0f;
        VecLd<V>::f(val + (int64_t)T * n + i, v_next);
        constexpr int U = kGaeUnroll;                                     // 2 x U x 9V bytes of registers per thread
        GaeChunk<V, U> a, b;
        a.load(rew, val, done, T, n, i);
        for (int32_t t1 = T; t1 > 0; t1 -= 2 * U) {                // two chunks per trip: a = [t1-U, t1), b = [t1-2U, t1-U)
            if (t1 - U > 0) b.load(rew, val, done, t1 - U, n, i);
            a.template scan<MOM>(adv, ret, g, gl, t1, n, i, gae, v_next, s, q);
            if (t1 - U <= 0) break;
            if (t1 - 2 * U > 0) a.load(rew, val, done, t1 - 2 * U, n, i);
            b.template scan<MOM>(adv, ret, g, gl, t1 - U, n, i, gae, v_next, s, q);
        }
    }
    if (MOM) {                                             // block-level sums, one atomic pair per CTA
        __shared__ double s_s[kGaeBlock / 32 > 0 ? kGaeBlock / 32 : 1], s_q[kGaeBlock / 32 > 0 ? kGaeBlock / 32 : 1];
        s = warp_sum(s); q = warp_sum(q);
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (lane == 0) { s_s[w] = s; s_q[w] = q; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double ts = 0.0, tq = 0.0;
            for (int k = 0; k < kGaeBlock / 32; ++k) { ts += s_s[k]; tq += s_q[k]; }
            atomicAdd(mom + 1, ts); atomicAdd(mom + 2, tq);
            if (blockIdx.x == 0) atomicAdd(mom + 0, (double)T * (double)n);
        }
    }
}

// compute_returns (Policy_Gradients.ipynb: G = r + gamma * G over reversed(rewards), python floats = float64),
// batched: G restarts after a step that ended an episode.  Accumulated in double like the original, written as
// fp32 (the notebook builds a float32 tensor from the list).  Same double-buffered chunk scheme as gae_kernel.
struct RetChunk {
    float r[kGaeUnroll];
    uint8_t d[kGaeUnroll];
    __device__ __forceinline__ void load(const float* __restrict__ rew, const uint8_t* __restrict__ done, int32_t t1, int64_t n, int64_t i) {
#pragma unroll
        for (int j = 0; j < kGaeUnroll; ++j) {
            const int32_t t = t1 - 1 - j;
            const int64_t o = (int64_t)(t >= 0 ? t : 0) * n + i;
            r[j] = __ldg(rew + o); d[j] = done ? __ldg(done + o) : (uint8_t)0;
        }
    }
    __device__ __forceinline__ void scan(float* __restrict__ out, double gamma, int32_t t1, int64_t n, int64_t i, double& G) const {
#pragma unroll
        for (int j = 0; j < kGaeUnroll; ++j) {
            const int32_t t = t1 - 1 - j;
            if (t >= 0) {
                if (d[j]) G = 0.0;                              // step t ended its episode: nothing flows back into it
                G = __dadd_rn((double)r[j], __dmul_rn(gamma, G));
                out[(int64_t)t * n + i] = (float)G;
            }
        }
    }
};

__global__ void __launch_bounds__(kGaeBlock) returns_kernel(const float* __restrict__ rew, const uint8_t* __restrict__ done,
                                                            float* __restrict__ out, double gamma, int32_t T, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * kGaeBlock + threadIdx.x;
    pdl_wait();
    pdl_launch_dependents();
    if (i >= n) return;
    double G = 0.0;
    RetChunk a, b;
    a.load(rew, done, T, n, i);
    for (int32_t t1 = T; t1 > 0; t1 -= 2 * kGaeUnroll) {
        if (t1 - kGaeUnroll > 0) b.load(rew, done, t1 - kGaeUnroll, n, i);
        a.scan(out, gamma, t1, n, i, G);
        if (t1 - kGaeUnroll <= 0) break;
        if (t1 - 2 * kGaeUnroll > 0) a.load(rew, done, t1 - 2 * kGaeUnroll, n, i);
        b.scan(out, gamma, t1 - kGaeUnroll, n, i, G);
    }
}

static inline int wave_grid(int64_t work_items, int per_block, int max_waves_ctas)
{
    int64_t g = (work_items + per_block - 1) / per_block;
    if (g > max_waves_ctas) g = max_waves_ctas;
    if (g < 1) g = 1;
    return (int)g;
}

}  // namespace dd

extern "C" {

int dd_moments(const float* x, int64_t n, double* out, void* stream)
{
    if (!x || !out) return DD_E_NULL;
    if (n < 0) return DD_E_RANGE;
    if ((reinterpret_cast<uintptr_t>(x) & 3u) || (reinterpret_cast<uintptr_t>(out) & 7u)) return DD_E_ALIGN;
    if (n == 0) return 0;
    const int grid = dd::wave_grid(n / 4 + 1, dd::kRedBlock * 4, dd::kSMs * 8);    // (4 CTAs per SM measured slower: 16.7 vs 15 us at 16.4 M elements)
    dd::DeviceGuard guard((cudaStream_t)stream, x);
    if (guard.err != cudaSuccess) return (int)guard.err;
    return dd::launch(dd::moments_kernel, grid, dd::kRedBlock, (cudaStream_t)stream, true, x, n, out);
}

int dd_normalize(const float* x, float* y, const double* moments, double eps, int64_t n, void* stream)
{
    if (!x || !y || !moments) return DD_E_NULL;
    if (n < 0) return DD_E_RANGE;
    if (n == 0) return 0;
    const int grid = dd::wave_grid(n / 4 + 1, dd::kRedBlock * 2, dd::kSMs * 8);
    dd::DeviceGuard guard((cudaStream_t)stream, x);
    if (guard.err != cudaSuccess) return (int)guard.err;
    return dd::launch(dd::normalize_kernel, grid, dd::kRedBlock, (cudaStream_t)stream, true, x, y, moments, eps, n);
}

int dd_gae_moments(const float* rewards_tn, const float* values_t1n, const uint8_t* dones_tn, float* adv_tn,
                   float* returns_tn, double* moments, double gamma, double lambda, int32_t T, int64_t n, void* stream)
{
    if (!rewards_tn || !values_t1n || !dones_tn || !adv_tn) return DD_E_NULL;
    if (n < 0 || T < 0) return DD_E_RANGE;
    if (moments && (reinterpret_cast<uintptr_t>(moments) & 7u)) return DD_E_ALIGN;
    if (n == 0 || T == 0) return 0;
    dd::DeviceGuard guard((cudaStream_t)stream, rewards_tn);
    if (guard.err != cudaSuccess) return (int)guard.err;
    const float g = (float)gamma, gl = (float)(gamma * lambda);
    cudaStream_t st = (cudaStream_t)stream;
    // V envs per thread need every row (stride n elements) of every array aligned to the vector width
    const uintptr_t fl = reinterpret_cast<uintptr_t>(rewards_tn) | reinterpret_cast<uintptr_t>(values_t1n) |
                         reinterpret_cast<uintptr_t>(adv_tn) | (returns_tn ? reinterpret_cast<uintptr_t>(returns_tn) : 0);
    int V = dd::kGaeVec;
    while (V > 1 && ((n % V) != 0 || (fl & (4u * V - 1)) != 0 || (reinterpret_cast<uintptr_t>(dones_tn) & (V - 1)) != 0)) V >>= 1;
    const int64_t threads = (n + V - 1) / V;
    const int grid = (int)((threads + dd::kGaeBlock - 1) / dd::kGaeBlock);
    double* const no_mom = nullptr;
#define GAE_LAUNCH(V_) (moments ? dd::launch(dd::gae_kernel<V_, true>, grid, dd::kGaeBlock, st, true, rewards_tn, values_t1n, dones_tn, adv_tn, returns_tn, moments, g, gl, T, n) \
                                : dd::launch(dd::gae_kernel<V_, false>, grid, dd::kGaeBlock, st, true, rewards_tn, values_t1n, dones_tn, adv_tn, returns_tn, no_mom, g, gl, T, n))
    return V == 2 ? GAE_LAUNCH(2) : GAE_LAUNCH(1);
#undef GAE_LAUNCH
}

int dd_gae(const float* rewards_tn, const float* values_t1n, const uint8_t* dones_tn, float* adv_tn,
           float* returns_tn, double gamma, double lambda, int32_t T, int64_t n, void* stream)
{
    return dd_gae_moments(rewards_tn, values_t1n, dones_tn, adv_tn, returns_tn, nullptr, gamma, lambda, T, n, stream);
}

int dd_discounted_returns(const float* rewards_tn, const uint8_t* dones_tn, float* returns_tn, double gamma,
                          int32_t T, int64_t n, void* stream)
{
    if (!rewards_tn || !returns_tn) return DD_E_NULL;
    if (n < 0 || T < 0) return DD_E_RANGE;
    if (n == 0 || T == 0) return 0;
    const int grid = (int)((n + dd::kGaeBlock - 1) / dd::kGaeBlock);
    dd::DeviceGuard guard((cudaStream_t)stream, rewards_tn);
    if (guard.err != cudaSuccess) return (int)guard.err;
    return dd::launch(dd::returns_kernel, grid, dd::kGaeBlock, (cudaStream_t)stream, true, rewards_tn, dones_tn, returns_tn, gamma, T, n);
}

}  // extern "C"
