// policy_rollout.cu -- K5: the PPO rollout inner loop fused into ONE persistent kernel.
//
// Replaces `collect_episodes_ppo`'s per-step work (Actor_Critic_PPO.ipynb c16:L42-108): stack the
// observations, run the policy `DroneGamerBoi` (c11:L5-17: Linear(15,128)-LN-ReLU-Linear(128,128)-LN-
// ReLU-Linear(128,64)-LN-ReLU-Linear(64,3)-Sigmoid), sample 3 independent Bernoulli actions
// (c16:L61-63) or threshold them (c18:L24-25), step every game, append to the rollout buffers.
//
// Mapping to sm_100a:
//   * one CTA per SM, 512 threads = 4 warpgroup "tiles" of 128 environments; a thread owns ONE
//     environment for the whole T-step rollout (state in registers) and the matching accumulator
//     row (TMEM lane) of its tile;
//   * the three dense layers run on the 5th-gen tensor cores: `tcgen05.mma.cta_group::1.kind::f16`
//     (SASS UTCHMMA), M = 128 (envs) x N = 128/128/64 x K = 16/128/128, bf16 operands from shared
//     memory (UMMA K-major, no-swizzle canonical layout), fp32 accumulators in TMEM (128 columns
//     per tile, 512 = the whole TMEM per CTA), issued by one elected thread per tile and tracked with
//     `tcgen05.commit` -> mbarrier;
//   * LayerNorm is folded into the GEMM operands by dd_policy_pack.  With C = I - 11^T/N (centring over
//     the N outputs), S = diag(sign gamma), g = |gamma| and g_prev the |gamma| of the PREVIOUS LayerNorm:
//     the weight image is f16(S C W diag(g_prev)), the bias S C b rides in an extra K = 16 block (a constant
//     "ones" A block x a [N][16] image holding the bias split into hi + lo), so the accumulator row is
//     x'_j = s_j (x_j - mean x).  relu(gamma n + beta) = g relu(s n + beta / g): the activation handed on is
//     a_j = relu(x'_j rstd + beta_j / g_j) and g_j is already in the next layer's image (in w3 for the last
//     hidden layer).  What is left for the CUDA cores is  var = 1/N sum_j x'_j^2  (pass 1: ONE FFMA2 per column
//     pair) and a_j (pass 2: one FFMA2, ReLU inside the 16-bit conversion): 3 instructions per pair; round 1
//     kept gamma in the image of its own layer and paid an FMUL2 by 1/gamma per pair in pass 1 (+160 FMUL2 and
//     80 LDCU per env-step, 14 % of the kernel's instructions);
//   * the 16-bit operand format is fp16 when the packed network fits its range (checked by dd_policy_pack from
//     the parameters: 10 mantissa bits, 8x lower rounding error than bf16 at the same MMA rate), bf16 otherwise;
//   * beta / g and the last Linear travel by value in the kernel argument (DDPolicyConsts): after
//     unrolling every access is c[0][imm] -> LDCU.128 -> a uniform-register operand of FFMA2, no
//     shared-memory loads in the epilogues;
//   * the first layer runs in split-bf16 precision: observation and layer-0 image are hi + lo bf16 pairs and
//     D = x_hi W_hi + x_hi W_lo + x_lo W_hi (three K = 16 MMAs instead of one, ~16 mantissa bits): the input
//     rounding was 3/4 of the whole network's bf16 error (positions quantised to 1/512) -- measured on the
//     reference checkpoints: max logit error 0.090 -> 0.020, critic value error 8.9 -> 2.4 (std 254);
//   * each thread reads its accumulator row with `tcgen05.ld.32x32b.x16` (SASS LDTM), twice,
//     double-buffered (chunk c+1 is in flight while chunk c is processed) and writes the next A tile
//     straight into the UMMA layout;
//   * the operand images (16-bit, already in UMMA layout; 64 KB with the head image) + the ones block (4 KB) live in shared
//     memory for the whole kernel, the A tiles take 32 KB per tile, the observation staging tiles
//     (one TMA bulk store per tile-step) 7.5 KB per tile: 224 KB of the 227 KB;
//   * the policy head (64 -> 3) is a FOURTH tcgen05.mma (TS form, N = 16: rows 0-2 / 3-5 of its image are the high / low
//     halves of w3 |gamma2|) fed from TMEM by the third epilogue -- the 96 FFMA2 + 64 FMNMX + 44 LDCU per env-step it took
//     on the CUDA cores cost more than the extra hand-off (1.220 -> 1.176 ms); the critic's one-row head (forward-only
//     instantiation) stays on the CUDA cores in fp32.  Sigmoid / Bernoulli / log-prob follow on the CUDA cores; the
//     environment step is `step_core` from drone_core.cuh, the same code as K1, so the environment side is bit-identical
//     to dd_rollout on the same actions.
//   * layer 3 takes its A operand from TENSOR memory (tcgen05.mma "TS" form): the second epilogue writes the packed
//     16-bit activations with tcgen05.st into columns [0, 64) of its own accumulator -- columns pass 2 has already
//     consumed -- and D3 accumulates in columns [64, 128).  That takes the 32 KB A2 store and the 32 KB A2 operand read
//     of every tile-step off shared memory (an SS-form K-block streams 4 KB of A + 4 KB of B through the 128 B/clk
//     port, as fast as the tensor pipe consumes them): -12..18 % on the forward-only kernels, -0.5 % on the rollout.
//     Layers 1 -> 2 cannot do the same: A1 (64 columns) + D2 (128) do not fit a tile's 128 columns;
//   * off the serial chain, in registers: the spawn of the env's NEXT episode is drawn ahead of time (a reset on the
//     chain is a few moves; the 10 Philox rounds of the spawn after it run under the second MMA of the following
//     step), and the landing test -- which a trained policy enters on most tile-steps -- decides from the angle-addition
//     formulas on the pre-update sin / cos already held, falling back to sincospif only within 1e-3 px of a platform
//     edge in config.py's world, a few float ulps of the coordinates in a larger one (step_core<.., PRE_SC>, pre_sc_margin:
//     same decisions bit for bit): 1.250 -> 1.220 ms.
// The four tiles of a CTA are independent pipelines, so while one waits for its MMAs the other three
// keep the CUDA cores busy; work that is not on the chain obs -> network -> action -> env step -> obs runs in
// the shadow of an MMA, where the warp would otherwise sleep: the previous step's log-prob / output stores
// under the first, the Philox draws under the second, sin / cos of the pre-update angle under the head MMA; the episode
// statistics are accumulated per thread and committed once per rollout.  Measured on B200, cfg 4 (DESIGN.md 4b,
// profiles/r02b_ncu_policy_rollout_summary.txt): 1.134 ms per 65,536 x 250 launch, 1,266 instructions per env-step, issue
// slots 63 % busy, tensor pipe 53 %.  Before the tensor-core head (1.22 ms, 1,445 instructions, 64 % / 47 %):  T(k tiles per SM) = 0.72 / 0.86 / 1.02 /
// 1.26 ms: one tile alone needs 5,500 cycles per step (its chain: 3 x {fence, barrier, MMA, mbarrier, TMEM read,
// two-pass LayerNorm}, sample, env step), four tiles overlap to 9,300.  Removing one part at a time (timing only)
// takes off: LayerNorm pass 2 + conversions + A stores + last Linear 0.49 ms, the MMAs 0.26, the env step 0.20,
// output stores 0.08, LayerNorm pass 1 0.02, the sampling Philox 0.00 -- the parts add up to the whole: a serial
// chain per tile.  Tried and rejected this round: deferred outputs under the second MMA (+1 %), all four warps
// waiting on the MMA mbarrier / suspend-time hints (+0.3..1.3 %), phase-shifted tile starts (0 %), and a warp-specialised
// rewrite (two tiles per warpgroup alternating phase by phase, MMA-issuer warps, mbarrier arrive instead of named barriers:
// bit-identical, but 1.435 ms -- two compute warps per scheduler hide less than four; profiles/r02_k5b_experiment.cu.txt).
// Later (profiles/r02_k5_experiments_session3.json): half-N MMA batches to start pass 1 early (+8.5 %: an SS-form K-block
// streams its 4 KB A block through the 128 B/clk shared-memory port whatever N is -- that port, ~170 KB per tile-step, is a
// co-limiter), and dynamic (tile, segment) work units over all 148 SMs (bit-identical, no gain on cfg 4: with the whole chip
// busy T(k) = 0.77 / 0.91 / 1.08 / 1.26 ms, so a 3 / 4 mix is bounded at 1.17 ms and the hand-offs eat it).  Kept from that
// work: the launcher spreads the tiles over the SMs up to 3 per SM (policy_launch).
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>
#include "drone_device.cuh"
#include "host_guard.h"

namespace dd {

constexpr int kTile = 128;                     // envs per tile == UMMA M == TMEM lanes
constexpr int kGroups = 4;                     // tiles per CTA: 4 x 128 columns = all 512 TMEM columns
constexpr int kPolThreads = kTile * kGroups;   // 512
constexpr int kH1 = 128, kH2 = 128, kH3 = 64, kIn = 15, kInPad = 16, kOut = 3;

// ---- parameter blob (device memory, produced by policy_pack_kernel; copied verbatim to smem) ----
// bf16 operand images in UMMA K-major no-swizzle layout: element (n, k) of a [N][K] matrix sits at
// byte (k / 8) * (N * 16) + n * 16 + (k % 8) * 2   (8x16-byte core matrices; LBO = N*16, SBO = 128)
constexpr int kW0Off = 0;                                  // [128][16]  G0 C0 [W0 | b0]  (obs[15] := 1), high halves
constexpr int kW1Off = kW0Off + kH1 * kInPad * 2;          // [128][128] G1 C1 W1
constexpr int kW1bOff = kW1Off + kH2 * kH1 * 2;            // [128][16]  col 0/1 = hi/lo of G1 C1 b1
constexpr int kW2Off = kW1bOff + kH2 * 16 * 2;             // [64][128]  G2 C2 W2
constexpr int kW2bOff = kW2Off + kH3 * kH2 * 2;            // [64][16]   col 0/1 = hi/lo of G2 C2 b2
constexpr int kW0loOff = kW2bOff + kH3 * 16 * 2;           // [128][16]  low halves of the layer-0 image (split bf16)
constexpr int kW3Off = kW0loOff + kH1 * kInPad * 2;        // [16][64]   the last Linear x |gamma2| for the tensor-core head: rows 0-2 = hi, 3-5 = lo, rest 0
constexpr int kW3Rows = 16;                                // UMMA N of the head MMA (the smallest N at M = 128)
constexpr int kParOff = kW3Off + kW3Rows * kH3 * 2;        // a DDPolicyConsts image (fp32 parameters + operand format)
// word offsets inside it: beta / |gamma| per LayerNorm, then the last Linear (x |gamma| of the last LayerNorm), format
constexpr int pBe0 = 0, pBe1 = 128, pBe2 = 256, pW3 = 320, pB3 = 512, pFmt = 516, kParWords = 520;
constexpr int kBlobBytes = kParOff + kParWords * 4;        // 67,616
static_assert(kBlobBytes == DD_POLICY_BLOB_BYTES, "header and kernel disagree on the blob size");
static_assert(kBlobBytes % 16 == 0, "blob must be a whole number of uint4");
static_assert(sizeof(DDPolicyConsts) == kParWords * 4, "the blob's parameter section is a DDPolicyConsts image");
static_assert(offsetof(DDPolicyConsts, beta1) == pBe1 * 4 && offsetof(DDPolicyConsts, beta2) == pBe2 * 4 &&
              offsetof(DDPolicyConsts, w3) == pW3 * 4 && offsetof(DDPolicyConsts, b3) == pB3 * 4 &&
              offsetof(DDPolicyConsts, operands) == pFmt * 4, "DDPolicyConsts layout");
constexpr float kGammaFloor = 1e-12f;                      // |gamma| below this is treated as +-1e-12
constexpr int kChunk = 16;                                 // accumulator columns per tcgen05.ld (8, 16 and 32 measured: 16 best)

constexpr int kABytes = kTile * kH1 * 2;                   // 32 KB: A tile of one group (A0 aliases its head)
constexpr int kSmemBlob = 0;
constexpr int kSmemOnes = ((kParOff + 1023) / 1024) * 1024;      // [128][16] bf16: columns 0, 1 = 1.0
constexpr int kOnesBytes = kTile * 16 * 2;
constexpr int kSmemA = kSmemOnes + kOnesBytes;
constexpr int kSmemBar = kSmemA + kGroups * kABytes;
constexpr int kObsTileBytes = kTile * kIn * 4;                      // one tile's [128][15] fp32 observations: 7,680 B,
constexpr int kSmemObs = kSmemBar + 80;                             //   contiguous in obs_tn -> one TMA bulk store
                                                                    //   (bar area: 4 MMA + 4 obs-load mbarriers, TMEM base)
constexpr int kSmemTotal = kSmemObs + kGroups * kObsTileBytes;      // 225,344 of the 232,448 B
static_assert(kSmemTotal <= 227 * 1024, "shared memory budget");

struct PArgs {
    DDPolicyConsts pc;     // per-column LN parameters + last layer: constant bank -> uniform operands
    KArgs<float> a;        // env state pointers etc.
    const uint8_t* blob;
    int32_t mode;              // DD_ACTION_*
    float inv_temperature;     // DD_ACTION_SAMPLE: actions ~ Bernoulli(sigmoid(logit * inv_temperature))
    uint32_t t0;
    int32_t T;
    uint8_t* actions_tn;
    float* logp_tn;
    float* reward_tn;
    uint8_t* done_tn;
    float* obs_tn;             // [T][n][15]
    float* probs_tn;           // [T][n][3] (optional)
    float* shaped_tn;          // [T][n] notebook training reward (optional)
    const float* obs_in;       // forward-only instantiation: [n][15], no env stepping
    int32_t auto_reset;
    int32_t head;              // forward-only: 3 = probs[n][3] (sigmoid, DroneGamerBoi), 1 = values[n] (DroneTeacherBoi)
    float pre_margin;          // dd::pre_sc_margin of the parameters (the DEF instantiations use its default-world 1e-3)
};

// ---- raw PTX wrappers -----------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// A lost MMA / TMA completion must fault, never hang the GPU -- but the bound is WALL TIME (%globaltimer, 20 s),
// not a poll count: under time-slicing, MPS preemption, ncu / compute-sanitizer replay or a debugger a healthy
// kernel can spend any number of polls waiting.  The clock is read once per 2^16 polls, off the fast path.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    uint64_t t_first = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 0xffffu) == 0u) {
            uint64_t now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t_first == 0) t_first = now;
            else if (now - t_first > 20000000000ull) __trap();
        }
    }
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// one lane of a converged warp (the same lane every time for the same mask)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void group_bar(int g) { asm volatile("bar.sync %0, %1;" :: "r"(g + 1), "n"(kTile) : "memory"); }
// (In front of an MMA issue only the issuing warp has to wait; `bar.arrive` for the other three measured no different: the
// MMA cannot start before the last warp has arrived either way.)
// Wait for the tile's committed MMAs.  (Round 2 measured the alternatives on B200 -- all four warps waiting on the
// mbarrier, with and without a suspend-time hint: 1.265 / 1.278 ms against 1.262 for this scheme.)  Only the issuing warp polls the mbarrier (try_wait returns after a short
// system-defined time, so a waiting warp keeps executing a poll loop that competes for issue slots: ~200
// instructions per thread-step when all four warps of a tile poll); the other three block on a second named
// barrier that the issuing warp joins once the phase has flipped.
__device__ __forceinline__ void wait_mma(uint32_t bar, uint32_t& phase, bool issuer_warp, int g) {
    if (issuer_warp) mbar_wait(bar, phase);
    phase ^= 1u;
    asm volatile("bar.sync %0, %1;" :: "r"(g + 1 + kGroups), "n"(kTile) : "memory");
    tc_fence_after();
}

// UMMA shared-memory matrix descriptor: K-major, no swizzle, 8x16-byte core matrices.
//   bits [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (next 16-byte K chunk)
//   | [32,46) stride byte offset >> 4 (next 8-row group) | [46,48) version = 1 | [61,64) layout = 0
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// Instruction descriptor, kind::f16: D fp32 (bit 4), A format at [7,10) and B format at [10,13) (0 = fp16, 1 = bf16),
// both K-major, N >> 3 at [17,23), M >> 4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, bool f16) {
    return (1u << 4) | (f16 ? 0u : ((1u << 7) | (1u << 10))) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// A operand from tensor memory ("TS" form): row r of the 128 x 16 A block is TMEM lane r, its 16 sixteen-bit elements are
// the 8 thirty-two-bit columns starting at `tmem_a` (element 2j in the low half of column j).
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// 8 thirty-two-bit columns of this thread's TMEM lane <- 8 registers (16 packed sixteen-bit activations)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&w)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "r"(taddr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
// CH (8 or 16) consecutive fp32 columns of this thread's TMEM lane.  Issue and wait are split so the next
// chunk can be in flight while this one is processed.  `tcgen05.wait::ld` covers every load the thread has
// issued; the registers are threaded through the wait statements as in/out operands so the compiler
// cannot schedule a consumer above the wait.
template <int CH> struct TmemChunk;
template <> struct TmemChunk<8> {
    uint32_t r[8];
    __device__ __forceinline__ void issue(uint32_t taddr) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                     : "r"(taddr) : "memory");
    }
    __device__ __forceinline__ void wait() {
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]) :: "memory");
    }
};
template <> struct TmemChunk<16> {
    uint32_t r[16];
    __device__ __forceinline__ void issue(uint32_t taddr) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                     "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                       "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                     : "r"(taddr) : "memory");
    }
    __device__ __forceinline__ void wait() {
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                       "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                     :: "memory");
    }
};
template <int CH>
__device__ __forceinline__ float2 f2_of(const TmemChunk<CH>& t, int pair) {
    return make_float2(__uint_as_float(t.r[2 * pair]), __uint_as_float(t.r[2 * pair + 1]));
}
// two fp32 -> one 32-bit word of two 16-bit operands (`lo` in the low half); F16: fp16, else bf16
template <bool F16>
__device__ __forceinline__ uint32_t pack16(float lo, float hi) {
    uint32_t d;
    if constexpr (F16) asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    else               asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
// max(x, 0) fused into the conversion (F2FP.RELU): the ReLU of the hidden layers is free
template <bool F16>
__device__ __forceinline__ uint32_t pack16_relu(float lo, float hi) {
    uint32_t d;
    if constexpr (F16) asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    else               asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
// the two halves of a packed word back as fp32 (for the split hi + lo first layer)
template <bool F16>
__device__ __forceinline__ float2 unpack16(uint32_t w) {
    if constexpr (F16) return __half22float2(*reinterpret_cast<const __half2*>(&w));
    else return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}

// ---- one hidden layer's epilogue: LayerNorm over the N columns of my accumulator row ----------------
// The accumulator holds x'_j = s_j (x_j - mean x) (see the header).  Pass 1: sum of x'_j^2 -> rstd (one FFMA2 per
// column pair).  Pass 2: y_j = x'_j rstd + beta_j / g_j, handed to sink(chunk, y[CH]) BEFORE the ReLU (the sink applies
// it: for free inside the 16-bit conversion for layers 1-2, as FMNMX for the last hidden layer).  All element-wise
// arithmetic is packed fp32x2 (FFMA2, new on sm_100).  The TMEM reads are double buffered: chunk c+1 (and pass 2's
// first chunk) is in flight while chunk c is processed.
template <int N, int CH, typename Sink>
__device__ __forceinline__ void ln_epilogue(uint32_t trow, const float (&beta)[N], Sink sink)
{
    constexpr int NC = N / CH;
    static_assert(NC % 2 == 0, "two buffers alternate over an even number of chunks");
    TmemChunk<CH> buf[2];
    float2 q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = make_float2(0.f, 0.f);
    buf[0].issue(trow);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        buf[c & 1].wait();
        buf[(c + 1) & 1].issue(trow + (uint32_t)(((c + 1) % NC) * CH));      // next chunk / pass 2's first
#pragma unroll
        for (int j = 0; j < CH / 2; ++j) {
            const float2 t = f2_of(buf[c & 1], j);
            q[j & 3] = __ffma2_rn(t, t, q[j & 3]);
        }
    }
    const float2 qs = __fadd2_rn(__fadd2_rn(q[0], q[1]), __fadd2_rn(q[2], q[3]));     // packed adds: 4 instructions instead of 7
    const float sq = qs.x + qs.y;
    float rstd;                                                            // biased variance, like nn.LayerNorm; the argument is
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rstd) : "f"(fmaf(sq, 1.0f / N, 1e-5f)));   //   >= 1e-5: one MUFU.RSQ, no denormal fix-up
    const float2 r2 = make_float2(rstd, rstd);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        buf[c & 1].wait();
        if (c + 1 < NC) buf[(c + 1) & 1].issue(trow + (uint32_t)((c + 1) * CH));
        float y[CH];
#pragma unroll
        for (int j = 0; j < CH / 4; ++j) {
            const int col = c * CH + 4 * j;                  // compile-time after unrolling: c[0][imm] -> uniform registers
            const float2 y0 = __ffma2_rn(f2_of(buf[c & 1], 2 * j), r2, make_float2(beta[col], beta[col + 1]));
            const float2 y1 = __ffma2_rn(f2_of(buf[c & 1], 2 * j + 1), r2, make_float2(beta[col + 2], beta[col + 3]));
            y[4 * j] = y0.x; y[4 * j + 1] = y0.y; y[4 * j + 2] = y1.x; y[4 * j + 3] = y1.y;
        }
        sink(c, y);
    }
}

// ReLU + write CH activations of my row (K columns CH*c .. CH*c+CH-1) as fp16 / bf16 into the A tile (UMMA layout)
template <int CH, bool F16>
__device__ __forceinline__ void store_a_chunk_relu(uint8_t* a_tile, int row, int c, const float (&y)[CH]) {
#pragma unroll
    for (int q = 0; q < CH / 8; ++q) {                      // 16-byte K chunks
        uint4 w;
        w.x = pack16_relu<F16>(y[8 * q + 0], y[8 * q + 1]); w.y = pack16_relu<F16>(y[8 * q + 2], y[8 * q + 3]);
        w.z = pack16_relu<F16>(y[8 * q + 4], y[8 * q + 5]); w.w = pack16_relu<F16>(y[8 * q + 6], y[8 * q + 7]);
        *reinterpret_cast<uint4*>(a_tile + ((CH / 8) * c + q) * (kTile * 16) + row * 16) = w;
    }
}

// ReLU + write CH activations of my row as fp16 / bf16 into the TMEM A operand of the next layer: K columns CH*c .. CH*c+CH-1
// are the CH/2 thirty-two-bit columns starting at ta + (CH/2)*c.
template <int CH, bool F16>
__device__ __forceinline__ void store_a_chunk_relu_tmem(uint32_t ta, int c, const float (&y)[CH]) {
    static_assert(CH % 16 == 0, "one tcgen05.st.x8 per 16 activations");
#pragma unroll
    for (int q = 0; q < CH / 16; ++q) {
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = pack16_relu<F16>(y[16 * q + 2 * j], y[16 * q + 2 * j + 1]);
        tmem_st8(ta + (uint32_t)((CH / 2) * c + 8 * q), w);
    }
}

// =================================================================================================
// FWD = false: the T-step rollout (a thread owns one environment).  FWD = true: the network alone over n rows of
// observations (parity hook for the policy; the critic's values over a rollout buffer), persistent over blocks of
// 512 rows: the "step" loop walks row blocks and the observation tile of the NEXT block is fetched by TMA
// (cp.async.bulk -> mbarrier) while the current one goes through the layers.
// HEAD: 3 = policy (probabilities); 1 = critic (FWD only): the two unused rows of the last Linear are not computed.
// FAST = true (rollout only): the PPO-collection configuration -- Bernoulli sampling at temperature 1, auto-reset,
// statistics, and exactly the action / log-prob / reward / done / observation buffers (no shaped reward, no
// probabilities) -- with every launch-constant switch a compile-time constant: predicated-off stores, their address
// arithmetic and the selects between modes still cost issue slots, and this kernel is bound by them.
// F16: the operand images in the blob and the activations are fp16 (else bf16); chosen by dd_policy_pack.
template <bool DEF, bool FWD, int HEAD = 3, bool FAST = false, bool F16 = false>
__global__ void __launch_bounds__(kPolThreads, 1) policy_rollout_kernel(const __grid_constant__ PArgs pa)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    const KArgs<float>& a = pa.a;
    const Consts<float> k = consts_of<float, DEF>(a);

    // The warp index is made warp-uniform FOR THE COMPILER (shfl from lane 0): everything derived from it --
    // tile index, TMEM / shared-memory addresses, UMMA descriptors -- then lives in uniform registers and
    // the MMA issue sequence needs no per-instruction lane election.
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), g = warp >> 2, row = tid & (kTile - 1);
    uint8_t* s_blob = smem + kSmemBlob;
    uint8_t* s_a = smem + kSmemA + g * kABytes;
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + kSmemBar);          // [kGroups] MMA done, [kGroups] obs tile landed
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + kSmemBar + 64);

    // ---- one-time setup: weights -> smem, mbarriers, TMEM ----
    {
        const uint4* src = reinterpret_cast<const uint4*>(pa.blob);
        uint4* dst = reinterpret_cast<uint4*>(s_blob);
        for (int j = tid; j < kParOff / 16; j += kPolThreads) dst[j] = __ldg(src + j);   // operand images only
    }
    {   // the constant A block that carries the biases: row r = [1, 1, 0 x 14] (K chunk 0), zeros (K chunk 1)
        uint4* ones = reinterpret_cast<uint4*>(smem + kSmemOnes);
        for (int j = tid; j < kOnesBytes / 16; j += kPolThreads)
            ones[j] = j < kTile ? make_uint4(F16 ? 0x3c003c00u : 0x3f803f80u, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
    }
    if (tid == 0) {
#pragma unroll
        for (int j = 0; j < 2 * kGroups; ++j) mbar_init(smem_u32(s_bar + j), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {                                        // one warp allocates the whole TMEM (512 columns)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(s_tmem)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();                                     // weight image (generic stores) -> async proxy (UMMA reads)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    const uint32_t tmem_d = tmem_base + (uint32_t)(g * 128);                         // my tile's accumulator columns
    const uint32_t trow = tmem_d + ((uint32_t)((warp & 3) * 32) << 16);              // my warp's 32 lanes
    const uint32_t bar = smem_u32(s_bar + g);
    const bool issuer_warp = (warp & 3) == g;   // tile g issues from its warp g: one issuing warp per scheduler
    const uint32_t a_addr = smem_u32(s_a);
    const uint32_t w0_addr = smem_u32(s_blob + kW0Off), w1_addr = smem_u32(s_blob + kW1Off), w2_addr = smem_u32(s_blob + kW2Off);
    const uint32_t w1b_addr = smem_u32(s_blob + kW1bOff), w2b_addr = smem_u32(s_blob + kW2bOff), ones_addr = smem_u32(smem + kSmemOnes);
    const uint32_t w0lo_addr = smem_u32(s_blob + kW0loOff), w3_addr = smem_u32(s_blob + kW3Off);
    uint32_t phase = 0;
    float* s_obs = reinterpret_cast<float*>(smem + kSmemObs + g * kObsTileBytes);
    const DDPolicyConsts& pc = pa.pc;

    // ---- my environment (FWD: my row of the current block, advanced in the loop) ----
    constexpr bool forward_only = FWD;
    // FWD: consecutive tiles per CTA (walked block by block).  Rollout: tile b + gridDim.x * g in slot g of CTA b -- the
    // launcher SPREADS the tiles over the SMs (policy_launch); a slot without a tile skips the step loop.
    uint32_t tile0 = FWD ? (blockIdx.x * kGroups + g) * kTile : (blockIdx.x + gridDim.x * g) * kTile;
    const int32_t T_mine = (FWD || tile0 < a.n) ? pa.T : 0;
    uint32_t i = tile0 + row;
    bool live = i < a.n;
    // FWD: a tile's [128][15] fp32 rows are contiguous: full 16-byte aligned tiles arrive by TMA into s_obs
    const bool in_aligned = FWD && (reinterpret_cast<uintptr_t>(pa.obs_in) & 15u) == 0u;
    const uint32_t obs_bar = smem_u32(s_bar + kGroups + g);
    uint32_t obs_phase = 0;
    auto tile_bulk_in = [&](uint32_t t0_) { return in_aligned && (uint64_t)t0_ + kTile <= (uint64_t)a.n; };
    auto fetch_tile = [&](uint32_t t0_) {                    // one elected thread
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(obs_bar), "n"(kObsTileBytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(smem_u32(s_obs)), "l"(pa.obs_in + (size_t)t0_ * kIn), "n"(kObsTileBytes), "r"(obs_bar) : "memory");
    };
    if (FWD && tile_bulk_in(tile0) && issuer_warp && elect_one()) fetch_tile(tile0);
    Env<float> e = {};
    uint32_t pflags = 0, ep = 0;
    bool platform_dirty = false;
    if (live && !forward_only) {
        load4(a.pos_vel, i, e.x, e.y, e.vx, e.vy);
        load4(a.att_fuel, i, e.angle, e.angvel, e.fuel, e.ret);
        load2(a.platform, i, e.px, e.py);
        e.steps = a.steps[i];
        pflags = a.flags[i];
        ep = a.episode[i];
    }
    const uint64_t gid = a.env_id_base + (uint64_t)i;
    float speed = 0.f, dist = 0.f;
    if (!forward_only) speed_dist(e, speed, dist);
    // The spawn of my env's NEXT episode (Philox(seed, env id, episode counter)) is drawn ahead of time and kept in
    // registers: a reset on the serial chain is then a handful of moves, and the 10 Philox rounds of the spawn after
    // it run under the second MMA of the following step (same spawn_draw as spawn(): bit-identical resets).
    float nsx = 0.f, nsy = 0.f, nspx = 0.f, nspy = 0.f, nsdist = 0.f;
    bool need_spawn = false;
    auto draw_next_spawn = [&]() {
        spawn_draw(k, a.seed, gid, ep, a.rand_drone != 0, a.rand_platform != 0, nsx, nsy, nspx, nspy);
        const float ddx = nspx - nsx, ddy = nspy - nsy;                       // speed_dist() of the fresh state
        nsdist = Arith<float>::sqrt_(Arith<float>::fma_(ddx, ddx, Arith<float>::mul(ddy, ddy)));
    };
    if (!forward_only && live) draw_next_spawn();
    const bool shaping = !FAST && pa.shaped_tn != nullptr;
    // The tile's observations of one step are 128 x 15 contiguous floats of obs_tn: full, 16-byte aligned tiles
    // are staged in shared memory (stride 15 words: conflict-free) and leave with one cp.async.bulk per step.
    // launch-constant switches, read from the argument block once
    const bool out_act = FAST || pa.actions_tn != nullptr, out_logp = FAST || pa.logp_tn != nullptr,
               out_rew = FAST || pa.reward_tn != nullptr, out_done = FAST || pa.done_tn != nullptr,
               out_probs = !FAST && pa.probs_tn != nullptr, do_stats = FAST || a.stats != nullptr,
               auto_reset = FAST || pa.auto_reset != 0, thresholded = !FAST && pa.mode == DD_ACTION_THRESHOLD,
               tempered = !FAST && pa.inv_temperature != 1.0f;
    const int32_t max_steps = a.max_steps;
    const bool obs_out = !forward_only && (FAST || pa.obs_tn != nullptr);
    // (a ragged last tile stores its live rows only: (n - tile0) * 60 bytes, a multiple of 16 when n % 4 == 0)
    const uint32_t obs_bytes = (tile0 < a.n ? (a.n - tile0 < (uint32_t)kTile ? a.n - tile0 : (uint32_t)kTile) : 0u) * (kIn * 4u);
    const bool obs_bulk = obs_out && tile0 < a.n && (a.n & 3u) == 0u &&
                          (reinterpret_cast<uintptr_t>(pa.obs_tn) & 15u) == 0u;
    float dprev = nan_of<float>(), dcur = dist * k.inv_width;
    if (live && shaping) dprev = a.prev_dist[i];

    // Outputs of a step that nothing in the NEXT step's network input depends on (log-prob, the action / log-prob /
    // reward / done / shaped stores, the statistics commit) are deferred: they run under the first MMA of the next
    // step, where the warp would otherwise sleep, instead of in front of it on the tile's serial chain.
    // Episode statistics are accumulated per thread over the rollout and committed once at its end (integer sums: the same
    // totals as a commit per step; the per-step warp commit -- a ballot every step, three more ballots, ten shuffles and six
    // atomics whenever a lane's episode ended, ~30 % of the warp-steps of a trained policy -- sat in the over-full shadow
    // of the first MMA, i.e. on the tile's chain: 1.173 -> 1.155 ms).
    StatsAcc st;
    struct Pending { float p0, p1, p2, reward, shaped; uint32_t act, oflags; } pend = {};
    auto flush_pending = [&](size_t o_prev) {
        if (live) {
            if (shaping) pa.shaped_tn[o_prev] = pend.shaped;
            if (out_act) pa.actions_tn[o_prev] = (uint8_t)pend.act;
            if (out_logp) {                                  // Bernoulli(probs).log_prob(a).sum(), probs clamped like torch
                const float eps = 1.1920929e-07f;
                const float q0 = fminf(fmaxf(pend.p0, eps), 1.f - eps), q1 = fminf(fmaxf(pend.p1, eps), 1.f - eps),
                            q2 = fminf(fmaxf(pend.p2, eps), 1.f - eps);
                // one logarithm of the product (each factor >= 1.19e-7: no underflow) instead of three
                pa.logp_tn[o_prev] = __logf((((pend.act & DD_ACT_MAIN) ? q0 : 1.f - q0) * ((pend.act & DD_ACT_LEFT) ? q1 : 1.f - q1)) *
                                            ((pend.act & DD_ACT_RIGHT) ? q2 : 1.f - q2));
            }
            if (out_rew) pa.reward_tn[o_prev] = pend.reward;
            if (out_done) pa.done_tn[o_prev] = (uint8_t)pend.oflags;
        }
    };

    for (int32_t t = 0; t < T_mine; ++t) {
        const size_t o = FWD ? (size_t)i : (size_t)t * a.n + i;
        // ---------------- observation -> A0 (bf16, K = 16: 15 inputs + constant 1 for the bias) -------
        float ob[16];
        const bool tile_in = FWD && tile_bulk_in(tile0);     // warp-uniform: this tile's rows are in s_obs (or on their way)
        if (forward_only) {
            if (tile_in) {
                mbar_wait(obs_bar, obs_phase); obs_phase ^= 1u;
#pragma unroll
                for (int j = 0; j < kIn; ++j) ob[j] = s_obs[row * kIn + j];
            } else {
#pragma unroll
                for (int j = 0; j < kIn; ++j) ob[j] = live ? pa.obs_in[(size_t)i * kIn + j] : 0.f;
            }
        } else {
            write_obs(e, pflags, speed, dist, k, [&](int j, float v) { ob[j] = v; });
        }
        ob[15] = 1.0f;
        // split 16-bit: hi = f16(x), lo = f16(x - hi); K chunks 0-1 = hi, 2-3 = lo
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float x0 = ob[8 * q + 2 * j], x1 = ob[8 * q + 2 * j + 1];
                hi[j] = pack16<F16>(x0, x1);
                // rollout: inputs 13, 14 (landed, crashed) are exactly 0 or 1 and input 15 is the constant 1: no low halves
                if (!FWD && q == 1 && j == 3) { lo[j] = 0u; continue; }
                const float2 h = unpack16<F16>(hi[j]);
                lo[j] = (!FWD && q == 1 && j == 2) ? pack16<F16>(x0 - h.x, 0.f) : pack16<F16>(x0 - h.x, x1 - h.y);
            }
            *reinterpret_cast<uint4*>(s_a + q * (kTile * 16) + row * 16) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(s_a + (2 + q) * (kTile * 16) + row * 16) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        // ---------------- layer 1: D[128x128] = A0[128x16] * W0''^T, split bf16 (3 MMAs) ---------------
        fence_async_smem(); tc_fence_before(); group_bar(g);
        if (issuer_warp && elect_one()) {
            tc_fence_after();
            umma_bf16(tmem_d, umma_desc(a_addr, kTile * 16, 128), umma_desc(w0_addr, kH1 * 16, 128), umma_idesc(128, kH1, F16), 0u);      // x_hi W_hi
            umma_bf16(tmem_d, umma_desc(a_addr, kTile * 16, 128), umma_desc(w0lo_addr, kH1 * 16, 128), umma_idesc(128, kH1, F16), 1u);    // x_hi W_lo
            umma_bf16(tmem_d, umma_desc(a_addr + 2 * (kTile * 16), kTile * 16, 128), umma_desc(w0_addr, kH1 * 16, 128), umma_idesc(128, kH1, F16), 1u);   // x_lo W_hi
            umma_commit(bar);
            if (FWD) {                                       // everyone has read s_obs: fetch the next block's tile
                const uint32_t next0 = tile0 + gridDim.x * (kGroups * kTile);
                if (t + 1 < pa.T && tile_bulk_in(next0)) fetch_tile(next0);
            }
        }
        // under the first MMA: the observation leaves (staged for the TMA store issued after the next barrier, or
        // directly for ragged / unaligned tiles), and the previous step's deferred outputs
        if (obs_bulk) {
#pragma unroll
            for (int j = 0; j < kIn; ++j) s_obs[row * kIn + j] = ob[j];
        }
        if (obs_out && !obs_bulk && live) {
            float* dst = pa.obs_tn + o * kIn;
#pragma unroll
            for (int j = 0; j < kIn; ++j) dst[j] = ob[j];
        }
        if (!forward_only && t > 0) flush_pending(o - a.n);   // (under the second MMA instead: measured slower, 1.270 vs 1.257 ms)
        wait_mma(bar, phase, issuer_warp, g);
        ln_epilogue<kH1, kChunk>(trow, pc.beta0,
                             [&](int c, const float (&y)[kChunk]) { store_a_chunk_relu<kChunk, F16>(s_a, row, c, y); });
        // ---------------- layer 2: D[128x128] = A1[128x128] * W1''^T + ones * bias1''^T -----------------
        fence_async_smem(); tc_fence_before(); group_bar(g);
        if (issuer_warp && elect_one()) {
            tc_fence_after();
            if (obs_bulk) {                                  // the staged observation tile is complete: one TMA store
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                             :: "l"(pa.obs_tn + ((size_t)t * a.n + tile0) * kIn), "r"(smem_u32(s_obs)), "r"(obs_bytes) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
#pragma unroll
            for (int j = 0; j < kH1 / 16; ++j)
                umma_bf16(tmem_d, umma_desc(a_addr + j * 2 * (kTile * 16), kTile * 16, 128),
                          umma_desc(w1_addr + j * 2 * (kH2 * 16), kH2 * 16, 128), umma_idesc(128, kH2, F16), j > 0 ? 1u : 0u);
            umma_bf16(tmem_d, umma_desc(ones_addr, kTile * 16, 128), umma_desc(w1b_addr, kH2 * 16, 128), umma_idesc(128, kH2, F16), 1u);
            umma_commit(bar);
        }
        U4 rnd = {0u, 0u, 0u, 0u};                           // under the second MMA: this step's Philox draws
        if (!forward_only && need_spawn) { draw_next_spawn(); need_spawn = false; }   // refill after a reset (off the chain)
        if (!forward_only && !thresholded) {
            // (7 Philox rounds instead of 10: -0.7 %, not taken; one block per pair of steps with 21-bit uniforms, or the ten
            // rounds under / split with MMA3: no gain; the log-prob under MMA2 instead of MMA1: +1.6 %)
            rnd = philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), pa.t0 + (uint32_t)t, 2u,
                                (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
            pin(rnd.a); pin(rnd.b); pin(rnd.c);
        }
        wait_mma(bar, phase, issuer_warp, g);
        // The activations of layer 2 go to TENSOR memory, not shared memory: A2 (128 lanes x 64 columns of packed 16-bit
        // pairs) overlays the columns [0, 64) of D2 that pass 2 has already consumed (chunk c reads D2 columns
        // [16c, 16c+16) and writes A2 columns [8c, 8c+8)), layer 3 reads its A operand from there (TS form) and
        // accumulates D3 in columns [64, 128).  Shared memory is what bounds this kernel (each SS-form K-block streams
        // 4 KB of A + 4 KB of B through the 128 B/clk port, on top of the epilogues' stores): this takes the 32 KB A2
        // store and the 32 KB A2 operand read of every tile-step off it.
        ln_epilogue<kH2, kChunk>(trow, pc.beta1,
                             [&](int c, const float (&y)[kChunk]) { store_a_chunk_relu_tmem<kChunk, F16>(trow, c, y); });
        tmem_st_wait();
        // ---------------- layer 3: D[128x64] = A2[128x128] (TMEM) * W2''^T + ones * bias2''^T --------------
        if (obs_bulk && issuer_warp && elect_one()) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging tile reusable after this barrier
        tc_fence_before(); group_bar(g);
        if (issuer_warp && elect_one()) {
            tc_fence_after();
#pragma unroll
            for (int j = 0; j < kH2 / 16; ++j)
                umma_ts(tmem_d + 64u, tmem_d + (uint32_t)(8 * j),
                        umma_desc(w2_addr + j * 2 * (kH3 * 16), kH3 * 16, 128), umma_idesc(128, kH3, F16), j > 0 ? 1u : 0u);
            umma_bf16(tmem_d + 64u, umma_desc(ones_addr, kTile * 16, 128), umma_desc(w2b_addr, kH3 * 16, 128), umma_idesc(128, kH3, F16), 1u);
            umma_commit(bar);
        }
        constexpr bool mma_head = HEAD == 3;                 // the critic's one-row head stays on the CUDA cores, in fp32
        float s_pre = 0.f, c_pre = 1.f;                      // under the third MMA (the fourth with the tensor-core head): sin / cos of the pre-update angle
        if (!forward_only && !mma_head) { Arith<float>::sincos_deg(e.angle, s_pre, c_pre); pin(s_pre); pin(c_pre); }   // (main thrust, drone.py:58-66)
        wait_mma(bar, phase, issuer_warp, g);
        float z0, z1, z2;
        if constexpr (mma_head) {
            // ---------------- epilogue 3, then the policy head as a fourth MMA ----------------------------------
            // The activations of the last hidden layer go to TMEM like those of layer 2 (packed 16-bit, ReLU inside the
            // conversion) into columns [0, 32) -- A2 is dead once MMA3 has completed --, the head D4[128 x 16] = A3 x W3''^T
            // accumulates in columns [32, 48): image rows 0-2 hold the high halves of w3 |gamma2|, rows 3-5 the low halves, so
            // logit_o = D4[o] + D4[3 + o] + b3[o] carries only the rounding of the activations.  That replaces 96 FFMA2 + 64
            // FMNMX + 48 LDCU per env-step (15 % of the kernel's instructions) with one more hand-off.
            ln_epilogue<kH3, kChunk>(trow + 64u, pc.beta2, [&](int c, const float (&y)[kChunk]) { store_a_chunk_relu_tmem<kChunk, F16>(trow, c, y); });
            tmem_st_wait();
            tc_fence_before(); group_bar(g);
            if (issuer_warp && elect_one()) {
                tc_fence_after();
#pragma unroll
                for (int j = 0; j < kH3 / 16; ++j)
                    umma_ts(tmem_d + 32u, tmem_d + (uint32_t)(8 * j),
                            umma_desc(w3_addr + j * 2 * (kW3Rows * 16), kW3Rows * 16, 128), umma_idesc(128, kW3Rows, F16), j > 0 ? 1u : 0u);
                umma_commit(bar);
            }
            if (!forward_only) { Arith<float>::sincos_deg(e.angle, s_pre, c_pre); pin(s_pre); pin(c_pre); }   // under the head MMA
            wait_mma(bar, phase, issuer_warp, g);             // (sin / cos under MMA3 instead, or all four warps on the mbarrier: measured equal or slower)
            TmemChunk<8> d4;
            d4.issue(trow + 32u);
            d4.wait();
            z0 = (__uint_as_float(d4.r[0]) + __uint_as_float(d4.r[3])) + pc.b3[0];
            z1 = (__uint_as_float(d4.r[1]) + __uint_as_float(d4.r[4])) + pc.b3[1];
            z2 = (__uint_as_float(d4.r[2]) + __uint_as_float(d4.r[5])) + pc.b3[2];
        } else {
        // ---------------- epilogue 3 + layer 4 (64 -> 3) on the CUDA cores ------------------------------
        float2 za = make_float2(0.f, 0.f), zb = za, zc = za;
        ln_epilogue<kH3, kChunk>(trow + 64u, pc.beta2, [&](int c, const float (&y)[kChunk]) {
#pragma unroll
            for (int j = 0; j < kChunk / 4; ++j) {
                const float2 h0 = make_float2(fmaxf(y[4 * j], 0.f), fmaxf(y[4 * j + 1], 0.f));      // ReLU
                const float2 h1 = make_float2(fmaxf(y[4 * j + 2], 0.f), fmaxf(y[4 * j + 3], 0.f));
                const int col = c * kChunk + 4 * j;
                za = __ffma2_rn(h0, make_float2(pc.w3[0][col], pc.w3[0][col + 1]), za); za = __ffma2_rn(h1, make_float2(pc.w3[0][col + 2], pc.w3[0][col + 3]), za);
                if (HEAD == 3) {
                    zb = __ffma2_rn(h0, make_float2(pc.w3[1][col], pc.w3[1][col + 1]), zb); zb = __ffma2_rn(h1, make_float2(pc.w3[1][col + 2], pc.w3[1][col + 3]), zb);
                    zc = __ffma2_rn(h0, make_float2(pc.w3[2][col], pc.w3[2][col + 1]), zc); zc = __ffma2_rn(h1, make_float2(pc.w3[2][col + 2], pc.w3[2][col + 3]), zc);
                }
            }
        });
        z0 = za.x + za.y + pc.b3[0]; z1 = zb.x + zb.y + pc.b3[1]; z2 = zc.x + zc.y + pc.b3[2];
        }
        tc_fence_before();                                   // my TMEM reads are done before the next MMA may overwrite
        // sigmoid with the approximate reciprocal (MUFU.RCP, ~1 ulp): the IEEE division sequence costs ~8 issue slots
        // per output on the chain; the same expression serves the rollout and the forward-only instantiation
        const float p0 = __fdividef(1.0f, 1.0f + __expf(-z0)), p1 = __fdividef(1.0f, 1.0f + __expf(-z1)),
                    p2 = __fdividef(1.0f, 1.0f + __expf(-z2));
        if (FWD && HEAD == 1) {                           // critic: the raw scalar (DroneTeacherBoi, c12)
            if (live) pa.probs_tn[o] = z0;
        } else if (out_probs && live) {
            float* dst = pa.probs_tn + o * kOut;
            dst[0] = p0; dst[1] = p1; dst[2] = p2;
        }
        if (forward_only) {                                  // next block of rows
            tile0 += gridDim.x * (kGroups * kTile);
            i = tile0 + row;
            live = i < a.n;
            continue;
        }

        // ---------------- action: threshold (c18:L24-25) or Bernoulli sample (c16:L61-63) --------------
        uint32_t act;
        if (thresholded) {
            act = (p0 > 0.5f ? DD_ACT_MAIN : 0u) | (p1 > 0.5f ? DD_ACT_LEFT : 0u) | (p2 > 0.5f ? DD_ACT_RIGHT : 0u);
        } else {
            const float u0 = (float)(rnd.a >> 8) * (1.0f / 16777216.0f), u1 = (float)(rnd.b >> 8) * (1.0f / 16777216.0f),
                        u2 = (float)(rnd.c >> 8) * (1.0f / 16777216.0f);
            // evaluate_policy_simple's temperature (c18): p^(1/tau) / (p^(1/tau) + (1-p)^(1/tau)) == sigmoid(logit / tau)
            const float s0 = tempered ? __fdividef(1.0f, 1.0f + __expf(-z0 * pa.inv_temperature)) : p0,
                        s1 = tempered ? __fdividef(1.0f, 1.0f + __expf(-z1 * pa.inv_temperature)) : p1,
                        s2 = tempered ? __fdividef(1.0f, 1.0f + __expf(-z2 * pa.inv_temperature)) : p2;
            act = (u0 < s0 ? DD_ACT_MAIN : 0u) | (u1 < s1 ? DD_ACT_LEFT : 0u) | (u2 < s2 ? DD_ACT_RIGHT : 0u);
        }

        // ---------------- environment step (same code as K1) -------------------------------------------
        uint32_t oflags = pflags;
        float reward = 0.f, shaped = 0.f;
        if (live && !(pflags & DD_DONE)) {
            uint32_t f = step_core<float, true, true>(e, act, k, reward, speed, dist, s_pre, c_pre, DEF ? 1e-3f : pa.pre_margin);
            if (!f && max_steps > 0 && e.steps >= max_steps) f = DD_DONE | DD_TRUNCATED;
            oflags = f;
            if (shaping) {
                shaped = shaped_reward(a.shaping, e, f, speed, dist, dprev, max_steps > 0 && e.steps >= max_steps, k);
                dprev = dcur;
                dcur = Arith<float>::div(dist, k.width, k.inv_width);
            }
            if (f) {
                if (do_stats) st.add(f, e.ret, e.steps);     // per-thread totals (a few predicated adds in the episode-end branch)
                if (auto_reset) {
                    spawn_apply(e, k, nsx, nsy, nspx, nspy);                   // == spawn(e, ..., ep): drawn ahead of time
                    ep += 1;
                    need_spawn = true;
                    platform_dirty = true;
                    f = 0;
                    speed = 0.f; dist = nsdist;                               // == speed_dist(e, ...) of a fresh episode (v = 0)
                    if (shaping) { dprev = nan_of<float>(); dcur = Arith<float>::div(dist, k.width, k.inv_width); }
                }
            }
            pflags = f;
        }
        pend.p0 = p0; pend.p1 = p1; pend.p2 = p2; pend.act = act; pend.reward = reward; pend.shaped = shaped;
        pend.oflags = oflags;
    }
    if (!forward_only && T_mine > 0) flush_pending((size_t)(T_mine - 1) * a.n + i);
    if (!forward_only && do_stats && T_mine > 0) st.commit(a.stats);            // one statistics commit per warp and rollout

    if (live && !forward_only) {
        store4(a.pos_vel, i, e.x, e.y, e.vx, e.vy);
        store4(a.att_fuel, i, e.angle, e.angvel, e.fuel, e.ret);
        a.steps[i] = e.steps;
        a.flags[i] = (uint8_t)pflags;
        a.episode[i] = ep;
        if (platform_dirty) store2(a.platform, i, e.px, e.py);
        if (shaping) a.prev_dist[i] = dprev;
    }
    if (obs_bulk && issuer_warp && elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    // ---- teardown: everyone is done with TMEM, then the allocating warp frees it ----
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(512) : "memory");
    }
}

// ---- fp32 torch parameters -> blob ---------------------------------------------------------------
// One CTA.  For a layer x = W a + b followed by LayerNorm(gamma, beta) over its N outputs, with s = sign(gamma),
// g = max(|gamma|, 1e-12) and g_prev the g of the previous LayerNorm (1 for the first layer):
//   image[n][k] = f16( s_n (W[n][k] - mean_n' W[n'][k]) g_prev_k ),  bias image = s_n (b[n] - mean b)  (hi + lo),
//   beta' = beta / g stays fp32 (DDPolicyConsts), the last Linear becomes w3[o][j] g_j.
// The floor changes a pre-activation by < 1.2e-11 (|normalised value| <= sqrt(N)), far below the 16-bit rounding.
// Operand format: fp16 if the network provably fits (see DD_OPERANDS_* in the header), else bf16.
__device__ __forceinline__ float gamma_abs(float g) { const float a = fabsf(g); return a < kGammaFloor ? kGammaFloor : a; }
__device__ __forceinline__ float gamma_sign(float g) { return g < 0.f ? -1.f : 1.f; }
__device__ __forceinline__ int img_at(int N, int n, int kk) { return (kk / 8) * (N * 8) + n * 8 + (kk % 8); }   // element index

template <bool F16> __device__ __forceinline__ float round16(float v) {
    if constexpr (F16) return __half2float(__float2half_rn(v));
    else return __bfloat162float(__float2bfloat16_rn(v));
}
template <bool F16> __device__ __forceinline__ void store16(uint8_t* img, int idx, float v) {
    if constexpr (F16) reinterpret_cast<__half*>(img)[idx] = __float2half_rn(v);
    else reinterpret_cast<__nv_bfloat16*>(img)[idx] = __float2bfloat16_rn(v);
}

struct PackLayer { const float *w, *b, *g, *gprev; int N, K; };   // K real inputs (15 or 128); gprev == nullptr: ones

__device__ __forceinline__ float pack_entry(const PackLayer& L, const float* mean, int n, int kk)
{   // kk == L.K: the bias column
    const float s = gamma_sign(L.g[n]);
    if (kk == L.K) return s * (L.b[n] - mean[L.K]);
    const float c = L.gprev ? gamma_abs(L.gprev[kk]) : 1.0f;
    return s * (L.w[n * L.K + kk] - mean[kk]) * c;
}

template <bool F16>
__device__ void pack_write_images(const PackLayer (&Ls)[3], const float (*mean)[129], uint8_t* blob, int tid, int nth)
{
    // layer 0: [W0 | b0] is one [128][16] matrix (obs[15] := 1), split hi + lo
    for (int j = tid; j < kH1 * kInPad; j += nth) {
        const int n = j / kInPad, kk = j % kInPad;
        const float v = pack_entry(Ls[0], mean[0], n, kk);
        const float hi = round16<F16>(v);
        store16<F16>(blob + kW0Off, img_at(kH1, n, kk), v);
        store16<F16>(blob + kW0loOff, img_at(kH1, n, kk), v - hi);
    }
    // layers 1, 2: K = 128 weight image + the bias block (col 0 = hi, col 1 = lo against the constant ones block)
    const int woff[3] = {0, kW1Off, kW2Off}, boff[3] = {0, kW1bOff, kW2bOff};
    for (int l = 1; l < 3; ++l) {
        const PackLayer& L = Ls[l];
        for (int j = tid; j < L.N * 128; j += nth) {
            const int n = j / 128, kk = j % 128;
            store16<F16>(blob + woff[l], img_at(L.N, n, kk), pack_entry(L, mean[l], n, kk));
        }
        for (int j = tid; j < L.N * 16; j += nth) {
            const int n = j / 16, kk = j % 16;
            const float v = pack_entry(L, mean[l], n, 128);
            const float hi = round16<F16>(v);
            store16<F16>(blob + boff[l], img_at(L.N, n, kk), kk == 0 ? v : (kk == 1 ? v - hi : 0.f));
        }
    }
}

__global__ void __launch_bounds__(256) policy_pack_kernel(DDPolicy p, int head, int operands, uint8_t* blob)
{
    __shared__ float s_mean[3][129];                       // per layer: column means over the outputs; [K] = mean of the bias
    __shared__ unsigned s_imax[3], s_bmax, s_gmin, s_gmax, s_w3max;  // maxima / minima as the bit patterns of non-negative floats
    __shared__ int s_fmt;
    const int tid = threadIdx.x, nth = blockDim.x;
    const PackLayer Ls[3] = {{p.w0, p.b0, p.g0, nullptr, kH1, kIn}, {p.w1, p.b1, p.g1, p.g0, kH2, kH1}, {p.w2, p.b2, p.g2, p.g1, kH3, kH2}};
    if (tid < 3) s_imax[tid] = 0u;
    if (tid == 0) { s_bmax = 0u; s_gmin = 0x7f800000u; s_gmax = 0u; s_w3max = 0u; }
    for (int l = 0; l < 3; ++l) {
        const PackLayer& L = Ls[l];
        for (int kk = tid; kk <= L.K; kk += nth) {
            double m = 0.0;
            for (int n = 0; n < L.N; ++n) m += (double)(kk < L.K ? L.w[n * L.K + kk] : L.b[n]);
            s_mean[l][kk] = (float)(m / L.N);
        }
    }
    __syncthreads();
    // ---- can the images and activations live in fp16?  (NaN / inf parameters fail every comparison -> bf16) ----
    for (int l = 0; l < 3; ++l) {
        const PackLayer& L = Ls[l];
        unsigned mx = 0u;
        for (int j = tid; j < L.N * (L.K + 1); j += nth) {
            const float v = fabsf(pack_entry(L, s_mean[l], j / (L.K + 1), j % (L.K + 1)));
            mx = max(mx, v == v ? __float_as_uint(v) : 0x7f800000u);
        }
        atomicMax(&s_imax[l], mx);
        const float* be = l == 0 ? p.be0 : (l == 1 ? p.be1 : p.be2);
        for (int j = tid; j < L.N; j += nth) {
            const float g = gamma_abs(L.g[j]), bp = fabsf(be[j] / g);
            atomicMax(&s_gmax, g == g ? __float_as_uint(g) : 0x7f800000u);
            atomicMin(&s_gmin, __float_as_uint(g));
            atomicMax(&s_bmax, bp == bp ? __float_as_uint(bp) : 0x7f800000u);
        }
    }
    for (int j = tid; j < head * kH3; j += nth) {            // the head image (tensor-core head): |w3 gamma2| must not overflow fp16
        const float v = fabsf(p.w3[j] * gamma_abs(p.g2[j % kH3]));
        atomicMax(&s_w3max, v == v ? __float_as_uint(v) : 0x7f800000u);
    }
    __syncthreads();
    if (tid == 0) {
        bool ok = __uint_as_float(s_w3max) <= 1024.f && __uint_as_float(s_gmin) >= 0.015625f && __uint_as_float(s_gmax) <= 64.f && __uint_as_float(s_bmax) <= 1024.f;
        for (int l = 0; l < 3; ++l) ok = ok && __uint_as_float(s_imax[l]) <= 1024.f && __uint_as_float(s_imax[l]) >= 0.00390625f;
        s_fmt = (operands != DD_OPERANDS_BF16 && ok) ? DD_OPERANDS_FP16 : DD_OPERANDS_BF16;
    }
    __syncthreads();
    if (s_fmt == DD_OPERANDS_FP16) pack_write_images<true>(Ls, s_mean, blob, tid, nth);
    else pack_write_images<false>(Ls, s_mean, blob, tid, nth);

    // the head image [16][64] for the tensor-core head: row o = hi, row 3 + o = lo of w3[o][k] |gamma2[k]|, the other rows 0
    for (int j = tid; j < kW3Rows * kH3; j += nth) {
        const int n = j / kH3, kk = j % kH3, o = n % 3;
        float v = 0.f;
        if (n < 6 && o < head) {
            const float w = p.w3[o * kH3 + kk] * gamma_abs(p.g2[kk]);
            const float hi = s_fmt == DD_OPERANDS_FP16 ? round16<true>(w) : round16<false>(w);
            v = n < 3 ? w : w - hi;
        }
        if (s_fmt == DD_OPERANDS_FP16) store16<true>(blob + kW3Off, img_at(kW3Rows, n, kk), v);
        else store16<false>(blob + kW3Off, img_at(kW3Rows, n, kk), v);
    }
    float* par = reinterpret_cast<float*>(blob + kParOff);
    for (int j = tid; j < 128; j += nth) {
        par[pBe0 + j] = p.be0[j] / gamma_abs(p.g0[j]);
        par[pBe1 + j] = p.be1[j] / gamma_abs(p.g1[j]);
    }
    for (int j = tid; j < 64; j += nth) par[pBe2 + j] = p.be2[j] / gamma_abs(p.g2[j]);
    for (int j = tid; j < kOut * kH3; j += nth) par[pW3 + j] = j < head * kH3 ? p.w3[j] * gamma_abs(p.g2[j % kH3]) : 0.f;   // head rows of [head][64]
    for (int j = tid; j < 4; j += nth) par[pB3 + j] = j < head ? p.b3[j] : 0.f;
    if (tid < 4) reinterpret_cast<int32_t*>(par)[pFmt + tid] = tid == 0 ? s_fmt : 0;
}

static bool pol_params_default(const DDParams& p)
{
    const DDParams d = kDefaultParams;
    return memcmp(&p, &d, sizeof d) == 0;
}

// CTAs of a rollout launch over n envs on a device with `sms` SMs; slot g (0..3) of CTA b runs tile b + grid * g.
// Per-SM throughput saturates with the number of resident tiles -- measured on B200 with every SM busy: 0.77 / 0.91 /
// 1.08 / 1.26 ms per 250 steps at 1 / 2 / 3 / 4 tiles per SM -- so up to 3 tiles per SM the tiles are SPREAD over the
// SMs (a 32,768-env batch runs 2 tiles on each of 128 SMs instead of 4 on 64), and above that they are packed four to
// a CTA (cfg 4, 512 tiles: 128 CTAs x 4 at 1.22 ms; 68 CTAs x 4 + 80 x 3 on all 148 SMs measured 1.26 -- the SMs with
// four tiles set the time and the busier chip clocks lower).
static int rollout_grid(int64_t n, int sms)
{
    const int64_t tiles = (n + kTile - 1) / kTile, blocks = (tiles + kGroups - 1) / kGroups;
    if (sms > 0 && tiles <= (int64_t)(kGroups - 1) * sms) return (int)(tiles < sms ? tiles : sms);
    return (int)blocks;
}

static int policy_launch(PArgs& pa, const DDParams& p, int64_t n, bool forward, cudaStream_t st)
{
    const int blocks = (int)((n + kTile * kGroups - 1) / (kTile * kGroups));
    const bool def = pol_params_default(p);
    void (*kern)(PArgs);
    int grid = blocks;
    DeviceGuard guard(st, pa.blob);                         // the device that owns the stream (or the blob)
    if (guard.err != cudaSuccess) return (int)guard.err;
    const bool f16 = pa.pc.operands == DD_OPERANDS_FP16;
    if (forward) {
        kern = pa.head == 1 ? (f16 ? policy_rollout_kernel<true, true, 1, false, true> : policy_rollout_kernel<true, true, 1, false, false>)
                            : (f16 ? policy_rollout_kernel<true, true, 3, false, true> : policy_rollout_kernel<true, true, 3, false, false>);
        int sms = 0;
        const cudaError_t e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, guard.dev);
        if (e != cudaSuccess) return (int)e;
        grid = blocks < sms ? blocks : sms;                 // persistent: one CTA per SM walks the row blocks
        pa.T = (blocks + grid - 1) / grid;
    } else {
        int sms = 0;
        const cudaError_t e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, guard.dev);
        if (e != cudaSuccess) return (int)e;
        grid = rollout_grid(n, sms);
        const bool fast = pa.mode == DD_ACTION_SAMPLE && pa.inv_temperature == 1.0f && pa.auto_reset && pa.a.stats &&
                          pa.actions_tn && pa.logp_tn && pa.reward_tn && pa.done_tn && pa.obs_tn && !pa.shaped_tn && !pa.probs_tn;
#define DD_K5(DEF_, FAST_) (f16 ? policy_rollout_kernel<DEF_, false, 3, FAST_, true> : policy_rollout_kernel<DEF_, false, 3, FAST_, false>)
        kern = def ? (fast ? DD_K5(true, true) : DD_K5(true, false)) : (fast ? DD_K5(false, true) : DD_K5(false, false));
#undef DD_K5
    }
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (err != cudaSuccess) return (int)err;
    kern<<<grid, kPolThreads, kSmemTotal, st>>>(pa);
    return (int)cudaGetLastError();
}

static int pack_common(const DDPolicy* p, int head, int operands, void* blob, DDPolicyConsts* consts, void* stream)
{
    if (!p || !blob || !consts) return DD_E_NULL;
    if (head != 1 && head != 3) return DD_E_RANGE;
    if (operands != DD_OPERANDS_AUTO && operands != DD_OPERANDS_BF16 && operands != DD_OPERANDS_FP16) return DD_E_RANGE;
    const float* const* q = reinterpret_cast<const float* const*>(p);
    for (int j = 0; j < 14; ++j) if (!q[j]) return DD_E_NULL;
    if (reinterpret_cast<uintptr_t>(blob) & 15u) return DD_E_ALIGN;
    DeviceGuard guard((cudaStream_t)stream, blob);
    if (guard.err != cudaSuccess) return (int)guard.err;
    policy_pack_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(*p, head, operands, (uint8_t*)blob);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return (int)err;
    err = cudaMemcpyAsync(consts, (const uint8_t*)blob + kParOff, sizeof(DDPolicyConsts), cudaMemcpyDeviceToHost, (cudaStream_t)stream);
    if (err != cudaSuccess) return (int)err;
    err = cudaStreamSynchronize((cudaStream_t)stream);
    if (err != cudaSuccess) return (int)err;
    // fp16 was demanded but the network does not fit its range: the blob holds bf16 images, say so
    if (operands == DD_OPERANDS_FP16 && consts->operands != DD_OPERANDS_FP16) return DD_E_RANGE;
    return 0;
}

static int forward_common(const void* blob, const DDPolicyConsts* consts, const float* obs, float* out, int head, int64_t n, void* stream)
{
    if (!blob || !consts || !obs || !out) return DD_E_NULL;
    if (n < 0 || n > (int64_t)DD_MAX_ENVS_PER_CALL) return DD_E_RANGE;
    if (consts->operands != DD_OPERANDS_BF16 && consts->operands != DD_OPERANDS_FP16) return DD_E_RANGE;   // not filled by dd_policy_pack
    if (reinterpret_cast<uintptr_t>(blob) & 15u) return DD_E_ALIGN;
    if (n == 0) return 0;
    PArgs pa{};
    pa.pc = *consts;
    pa.a.n = (uint32_t)n;
    pa.blob = (const uint8_t*)blob; pa.T = 1; pa.obs_in = obs; pa.probs_tn = out; pa.head = head;
    DDParams p = kDefaultParams;
    return policy_launch(pa, p, n, true, (cudaStream_t)stream);
}

}  // namespace dd

extern "C" {

int dd_policy_pack(const DDPolicy* p, void* blob, DDPolicyConsts* consts, void* stream)
{
    return dd::pack_common(p, 3, DD_OPERANDS_AUTO, blob, consts, stream);
}

int dd_policy_pack_ex(const DDPolicy* p, int32_t head, int32_t operands, void* blob, DDPolicyConsts* consts, void* stream)
{
    return dd::pack_common(p, head, operands, blob, consts, stream);
}

int dd_value_pack(const DDPolicy* p, void* blob, DDPolicyConsts* consts, void* stream)
{
    return dd::pack_common(p, 1, DD_OPERANDS_AUTO, blob, consts, stream);
}

int dd_policy_forward(const void* blob, const DDPolicyConsts* consts, const float* obs, float* probs, int64_t n, void* stream)
{
    return dd::forward_common(blob, consts, obs, probs, 3, n, stream);
}

int dd_value_forward(const void* blob, const DDPolicyConsts* consts, const float* obs, float* values, int64_t n, void* stream)
{
    return dd::forward_common(blob, consts, obs, values, 1, n, stream);
}

int dd_policy_rollout_grid(int64_t n, int32_t sms)
{
    if (n <= 0 || n > (int64_t)DD_MAX_ENVS_PER_CALL) return 0;
    return dd::rollout_grid(n, sms);
}

int dd_policy_rollout(const DDState* s, const DDParams* p, const DDEnvConfig* c, const void* blob,
                      const DDPolicyConsts* consts, int32_t mode, float temperature, uint32_t t0, int32_t T, uint8_t* actions_tn, float* logp_tn, float* reward_tn, uint8_t* done_tn,
                      float* obs_tn, float* probs_tn, float* shaped_tn, uint64_t* stats, int64_t n, void* stream)
{
    if (!s || !p || !c || !blob || !consts) return DD_E_NULL;
    if (s->dtype != DD_F32) return DD_E_DTYPE;                 // the fused kernel is the fp32 throughput path
    if (mode != DD_ACTION_THRESHOLD && mode != DD_ACTION_SAMPLE) return DD_E_RANGE;
    if (consts->operands != DD_OPERANDS_BF16 && consts->operands != DD_OPERANDS_FP16) return DD_E_RANGE;       // not filled by dd_policy_pack
    if (mode == DD_ACTION_SAMPLE && !(temperature > 0.0f)) return DD_E_RANGE;
    if (T < 0 || n < 0 || n > (int64_t)DD_MAX_ENVS_PER_CALL) return DD_E_RANGE;
    if (n > 0 && (!s->pos_vel || !s->att_fuel || !s->platform || !s->steps || !s->episode || !s->flags)) return DD_E_NULL;
    if ((reinterpret_cast<uintptr_t>(s->pos_vel) | reinterpret_cast<uintptr_t>(s->att_fuel) | reinterpret_cast<uintptr_t>(blob)) & 15u) return DD_E_ALIGN;
    if (reinterpret_cast<uintptr_t>(s->platform) & 7u) return DD_E_ALIGN;
    if (shaped_tn && !s->prev_dist && n > 0) return DD_E_NULL;
    if (shaped_tn && c->shaping != DD_SHAPING_PPO && c->shaping != DD_SHAPING_PG) return DD_E_RANGE;
    if (n == 0 || T == 0) return 0;
    dd::PArgs pa{};
    pa.pc = *consts;
    pa.a.prev_dist = (float*)s->prev_dist; pa.shaped_tn = shaped_tn;
    pa.a.pos_vel = (float*)s->pos_vel; pa.a.att_fuel = (float*)s->att_fuel; pa.a.platform = (float*)s->platform;
    pa.a.steps = s->steps; pa.a.episode = s->episode; pa.a.flags = s->flags;
    pa.a.stats = (unsigned long long*)stats;
    pa.a.n = (uint32_t)n; pa.a.seed = c->seed; pa.a.env_id_base = c->env_id_base; pa.a.max_steps = c->max_steps; pa.a.shaping = c->shaping;
    pa.a.rand_drone = c->randomize_drone; pa.a.rand_platform = c->randomize_platform;
    pa.a.k = dd::make_consts<float>(*p);
    pa.pre_margin = dd::pre_sc_margin(*p);
    pa.blob = (const uint8_t*)blob; pa.mode = mode; pa.t0 = t0; pa.T = T;
    pa.inv_temperature = mode == DD_ACTION_SAMPLE ? 1.0f / temperature : 1.0f;
    pa.actions_tn = actions_tn; pa.logp_tn = logp_tn; pa.reward_tn = reward_tn; pa.done_tn = done_tn;
    pa.obs_tn = obs_tn; pa.probs_tn = probs_tn; pa.obs_in = nullptr; pa.auto_reset = c->auto_reset;
    return dd::policy_launch(pa, *p, n, false, (cudaStream_t)stream);
}

}  // extern "C"
