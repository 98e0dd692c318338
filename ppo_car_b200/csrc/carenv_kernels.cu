// carenv_kernels.cu — sm_100a kernels and the C ABI of libcarenv_b200.so (include/carenv_b200.h).
//
//   k_rollout   one thread per environment, n_steps >= 1 CarEnv.step calls per launch with the
//               state held in registers between steps (carenv_step is the n_steps == 1 case).
//               Wall geometry lives in kernel-parameter (constant-bank) space so that every
//               segment coordinate is a uniform operand of the FMA-pipe instructions; the
//               per-thread-indexed tables (72 headings, gates) are staged once per block into
//               shared memory.
//   k_rollout_warp   small batches (<= 2,048 envs, <= 32 wall segments): one WARP per environment, lane = wall
//               segment, per-ray extrema by integer REDUX; bit-identical to k_rollout.
//   k_observe   observations recomputed from 32-byte pose records (compact rollout storage).
//   k_reset     CarEnv.reset for every environment.
//   k_gae       Buffer.calculate_advantages as a reverse scan, one thread per environment column.
//   k_rollout_tab   launches of 4,096 environments or more: the same step with the denominators cross(e, d) read
//               from a per-track shared-memory table (8 skewed, conflict-free copies), one 512-thread CTA per SM.
//   k_rollout_tab_sliced   the same for launches of >= 75,776 environments and >= 4 steps, with an SM's env-steps cut
//               into 16 equal per-warp intervals (jobs that straddle two warps are split in time): four warps per
//               scheduler until the launch ends.
//               Both table kernels also come as <U, NS> instantiations for the segment counts of the shipped tracks
//               (24 and 16): the segment loop fully unrolled, every segment record a constant-bank operand.
//   k_rollout_multi / k_reset_multi / k_render   a track id per environment in one launch; headless rgb_array frames.
//   csrc/policy_rollout.cuh (included below)   k_policy_rollout / k_policy_rollout_tc / _tc2 / _tc3: policy forward +
//               sampling + env step + Buffer rows in one launch (CUDA cores / tcgen05 tensor cores, policy_core.cuh,
//               tc_mlp.cuh); k_pack_policy packs the network parameters for them.
//   csrc/ppo_update.cuh, csrc/ppo_epoch.cuh   fused PPO minibatch update in three launches / all updates of an epoch
//               in one persistent launch with the gradient all-reduce over NVLink peer memory inside the kernel.
//   csrc/policy_abi.cuh (included below)   the C-ABI entry points of the policy / PPO kernels.
//   carenv_step_host   the host-buffer step: sub-range pipeline of narrowing, H2D, kernel and D2H copies.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 --shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <string>
#include <vector>

#include "../../include/carenv_b200.h"
#include "carenv_tables.h"
#include "policy_core.cuh"
#include "ppo_update.cuh"
#include "ppo_epoch.cuh"
#include "tc_mlp.cuh"

using namespace carenv;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char *what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return -1000 - (int)e;
}
#define CU(call)                                          \
    do {                                                  \
        cudaError_t _e = (call);                          \
        if (_e != cudaSuccess) return cuda_fail(_e, #call); \
    } while (0)

struct Handle {
    int device;
    HostTrack host;
    unsigned char *d_blob;    // trig64 | acc64 | gates | trig32 | trig32s | walls64 | segf | segd | den4
    const float4 *d_den4;     // [72][n_pairs] denominators of the pair kernels (null: track without pairs)
    CullGrid cull;            // candidate table of the culled table kernels (mask in d_blob after den4; null: none)
    int host_ranges;          // tuning hook: sub-ranges of the host-buffer step (0 = by size)
    float *cur_fobs;          // pre-reset ("final") observations for the launch being dispatched (else null)
    int4 *cur_rec;            // step records instead of reward / flag arrays for the launch being dispatched (else null)
    int tab;                  // 0 = k_rollout_tab for large launches, 1 = always (where the track allows), -1 = never
    Tables dev;               // device pointers into d_blob
    unsigned long long *d_stats;
    size_t smem_bytes;
    int force_generic;        // test hook: run the generic (not unrolled) kernel
    int max_unroll;           // tuning hook: cap the segment-loop unrolling (0 = no cap)
    int block;                // tuning hook: threads per block of k_rollout (0 = chosen per launch, see rollout_block)
    int smem_pad;             // tuning hook: extra dynamic shared memory per block (limits resident blocks per SM)
    int tc_tiles;             // tuning hook: 128-env groups per CTA of k_policy_rollout_tc (0 = chosen per launch)
    int tc_stagger;           // tuning hook: start delay of group 1 in k_policy_rollout_tc2, cycles (-1 = default)
    int pose_rows;            // fused rollout kernels: obs_buf holds 32-byte pose records instead of observations
    int warp_per_env;         // 0 = warp-per-environment kernel for small batches, 1 = always, -1 = never
    struct HostStep *hs;      // staging buffers / streams of carenv_step_host (allocated on first use)
    int *d_flags;             // k_rollout_tab_sliced: "head part done" flag per 32-environment job (allocated on first use)
    size_t flags_cap;         // ints in d_flags
    int tab_slice;            // 0 = time-sliced table kernel where it applies, 1 = wherever possible, -1 = never
};

// Resources of the host-buffer step path (carenv_step_host): device staging for one step of `cap` environments,
// a pinned byte buffer the caller's actions are narrowed into, side streams and events for the sub-range pipeline.
struct HostStep {
    static constexpr int kMaxRanges = 16;
    int cap = 0, flag_bytes = 0;
    unsigned char *d_act = nullptr, *h_act = nullptr;
    float *d_obs = nullptr, *d_rew = nullptr;
    unsigned char *d_term = nullptr, *d_trunc = nullptr;
    int32_t *d_info = nullptr;
    int4 *d_rec = nullptr;    // carenv_step_host_records: one 16-byte record per environment
    cudaStream_t streams[kMaxRanges] = {};
    cudaEvent_t ready = nullptr, done[kMaxRanges] = {};
    void release() {
        cudaFree(d_act); cudaFreeHost(h_act); cudaFree(d_obs); cudaFree(d_rew); cudaFree(d_term); cudaFree(d_trunc);
        cudaFree(d_info); cudaFree(d_rec);
        for (int i = 0; i < kMaxRanges; ++i) {
            if (streams[i]) cudaStreamDestroy(streams[i]);
            if (done[i]) cudaEventDestroy(done[i]);
        }
        if (ready) cudaEventDestroy(ready);
        *this = HostStep();
    }
};

// int64 actions (what train.py:185 passes) -> one byte each; anything outside 0..8 acts like 8 (lib/car_env.py:698-722).
// Runs on the host in front of every sub-range of carenv_step_host, so it is written for SSE2 (4 actions per
// iteration, ~0.3 ns each) instead of a scalar 64-bit compare-and-select loop (1 ns each).
static void narrow_actions_i64(const unsigned long long *a, unsigned char *d, int m) {
    int i = 0;
#if defined(__SSE2__)
    const __m128i sign = _mm_set1_epi32((int)0x80000000u), eight = _mm_set1_epi32(8), zero = _mm_setzero_si128();
    const __m128i eight_s = _mm_xor_si128(eight, sign);
    for (; i + 4 <= m; i += 4) {
        const __m128 x0 = _mm_castsi128_ps(_mm_loadu_si128(reinterpret_cast<const __m128i *>(a + i)));
        const __m128 x1 = _mm_castsi128_ps(_mm_loadu_si128(reinterpret_cast<const __m128i *>(a + i + 2)));
        const __m128i lo = _mm_castps_si128(_mm_shuffle_ps(x0, x1, 0x88));     // low halves of the four int64
        const __m128i hi = _mm_castps_si128(_mm_shuffle_ps(x0, x1, 0xDD));     // high halves
        const __m128i ok_hi = _mm_cmpeq_epi32(hi, zero);
        const __m128i bad_lo = _mm_cmpgt_epi32(_mm_xor_si128(lo, sign), eight_s);  // unsigned lo > 8
        const __m128i ok = _mm_andnot_si128(bad_lo, ok_hi);
        __m128i v = _mm_or_si128(_mm_and_si128(ok, lo), _mm_andnot_si128(ok, eight));
        v = _mm_packs_epi32(v, v);
        v = _mm_packus_epi16(v, v);
        const int w = _mm_cvtsi128_si32(v);
        memcpy(d + i, &w, 4);
    }
#endif
    for (; i < m; ++i) { const unsigned long long u = a[i]; d[i] = (unsigned char)(u < 8ull ? u : 8ull); }
}

struct DeviceGuard {
    int prev;
    bool ok;
    explicit DeviceGuard(int dev) : prev(-1), ok(false) {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = (prev == dev) || (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

#ifndef CARENV_BLOCK
#define CARENV_BLOCK 128
#endif
constexpr int kBlock = CARENV_BLOCK;
constexpr int kWarpPerEnvMax = 2048;   // n_envs up to which k_rollout_warp is launched (tracks with <= 32 segments)

// The action index of one element of the caller's action array.  An action outside 0..8 does nothing (decode_action);
// a 64-bit action must not be truncated into that range first (2^32 + 1 is not action 1).  The same rule as
// narrow_actions_i64 on the host path.
template <typename ActT> __device__ __forceinline__ int action_index(ActT a) { return (int)a; }
template <> __device__ __forceinline__ int action_index<int64_t>(int64_t a) {
    return (unsigned long long)a < 8ull ? (int)a : 8;
}

template <typename FlagT> __device__ __forceinline__ FlagT make_flag(int v);
template <> __device__ __forceinline__ uint8_t make_flag<uint8_t>(int v) { return (uint8_t)v; }
template <> __device__ __forceinline__ float make_flag<float>(int v) { return v ? 1.0f : 0.0f; }

// Reward / flags / info of one env-step: either the separate arrays of carenv_step / carenv_rollout or ONE 16-byte
// carenv_step_record (reward f64 | gates_passed i32 | time_passed u16 | terminated u8 | truncated u8) — what the
// host-buffer step path ships over PCIe, already in the reference's dtypes.
template <typename FlagT>
__device__ __forceinline__ void store_step(const StepResult &o, size_t idx, float *__restrict__ rew_out,
                                           FlagT *__restrict__ term_out, FlagT *__restrict__ trunc_out,
                                           int4 *__restrict__ info_out, int4 *__restrict__ rec_out) {
    if (rec_out) {
        rec_out[idx] = make_int4(__double2loint(o.reward64), __double2hiint(o.reward64), o.gates_passed,
                                 (o.time_passed & 0xffff) | (o.terminated << 16) | (o.truncated << 24));
    } else {
        rew_out[idx] = o.reward;
        term_out[idx] = make_flag<FlagT>(o.terminated);
        trunc_out[idx] = make_flag<FlagT>(o.truncated);
    }
    if (info_out) info_out[idx] = make_int4(o.gates_passed, o.time_passed, o.next_gate, o.gate_hit | (o.lap << 1));
}

// Stage the per-thread-indexed tables into shared memory (all sizes are multiples of 8 bytes).
__device__ __forceinline__ Tables stage_tables(const Tables &G, int n_gates, int n_seg, unsigned char *smem) {
    D2 *s_trig64 = reinterpret_cast<D2 *>(smem);
    D2 *s_acc64 = s_trig64 + kHeadings;
    GateRec *s_gates = reinterpret_cast<GateRec *>(s_acc64 + kHeadings);
    F2 *s_trig32 = reinterpret_cast<F2 *>(s_gates + n_gates);
    F2 *s_trig32s = s_trig32 + kHeadings;
    double *s_walls = reinterpret_cast<double *>(s_trig32s + kHeadings);   // float64 walls for the exact path: a
    const int n64a = kHeadings * 2, n64g = n_gates * (int)(sizeof(GateRec) / 8);   // global-memory copy costs ~10 k cycles per fallback
    double *d0 = reinterpret_cast<double *>(s_trig64);
    double *d1 = reinterpret_cast<double *>(s_acc64);
    double *d2 = reinterpret_cast<double *>(s_gates);
    double *d3 = reinterpret_cast<double *>(s_trig32);
    const double *g0 = reinterpret_cast<const double *>(G.trig64);
    const double *g1 = reinterpret_cast<const double *>(G.acc64);
    const double *g2 = reinterpret_cast<const double *>(G.gates);
    const double *g3 = reinterpret_cast<const double *>(G.trig32);
    for (int i = threadIdx.x; i < n64a; i += blockDim.x) { d0[i] = g0[i]; d1[i] = g1[i]; }
    for (int i = threadIdx.x; i < n64g; i += blockDim.x) d2[i] = g2[i];
    for (int i = threadIdx.x; i < 2 * kHeadings; i += blockDim.x) d3[i] = g3[i];   // trig32 | trig32s (contiguous in the blob)
    for (int i = threadIdx.x; i < 4 * n_seg; i += blockDim.x) s_walls[i] = G.walls64[i];
    const SegF *s_segf = nullptr;
    const SegD *s_segd = nullptr;
    if (n_seg > kMaxSeg) {                                  // big track: the segment records live in shared memory too
        static_assert(sizeof(SegF) == 48 && sizeof(SegD) == 24, "staging below copies 6 / 3 doubles per record");
        double *d4 = s_walls + 4 * n_seg, *d5 = d4 + 6 * n_seg;            // SegF = 6 doubles, SegD = 3 doubles
        const double *g4 = reinterpret_cast<const double *>(G.segf), *g5 = reinterpret_cast<const double *>(G.segd);
        for (int i = threadIdx.x; i < 6 * n_seg; i += blockDim.x) d4[i] = g4[i];
        for (int i = threadIdx.x; i < 3 * n_seg; i += blockDim.x) d5[i] = g5[i];
        s_segf = reinterpret_cast<const SegF *>(d4);
        s_segd = reinterpret_cast<const SegD *>(d5);
    }
    __syncthreads();
    return Tables{s_trig32, s_trig32s, s_trig64, s_acc64, s_gates, s_walls, s_segf, s_segd};
}

// What k_rollout writes per env-step besides reward and flags (SURVEY §8 f-3: rollout storage format).
enum { kObsNone = 0, kObsFull = 1, kObsPose = 2 };

// The pose behind an observation: `s` is the state the observation was computed from, obs2 / obs3 its velocity
// entries.  time_step == 0 only in the start state (after reset or autoreset), whose observation is the reset
// observation (evaluated with the literal float64 formulas, not recomputable by the float32 path).
__device__ __forceinline__ void store_pose(PoseRec *dst, const EnvState &s, float obs2, float obs3) {
    double2 *d2 = reinterpret_cast<double2 *>(dst);
    d2[0] = make_double2(s.px, s.py);
    reinterpret_cast<float4 *>(dst)[1] = make_float4(obs2, obs3, __int_as_float(s.k), __int_as_float(s.t == 0 ? 1 : 0));
}

// Observations from pose records (optionally gathered through `index`): the same cast_walls / normalisation
// code as env_step, so the result is bit-identical to the observation the rollout would have written.
template <int U>
__global__ void __launch_bounds__(kBlock)
k_observe(const __grid_constant__ TrackParams P, const Tables G, long long n, const PoseRec *__restrict__ poses,
          const long long *__restrict__ index, float *__restrict__ obs_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    const Tables T = stage_tables(G, P.n_gates, P.n_seg, smem);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const PoseRec *src = poses + (index ? index[i] : i);
    const double2 p = reinterpret_cast<const double2 *>(src)[0];
    const float4 q = reinterpret_cast<const float4 *>(src)[1];
    float obs[kObsDim];
    if (__float_as_int(q.w) != 0) {
#pragma unroll
        for (int k = 0; k < kObsDim; ++k) obs[k] = P.reset_obs[k];
    } else {
        EnvState s;
        s.px = p.x; s.py = p.y; s.vx = 0.0; s.vy = 0.0;
        s.k = __float_as_int(q.z); s.t = 0; s.next_gate = 0; s.passed = 0;
        float dist[kNumRays];
        cast_walls<U>(s, P, T, dist, nullptr);
        pose_observation(s, q.x, q.y, dist, T, obs);
    }
    float2 *dst = reinterpret_cast<float2 *>(obs_out + (size_t)i * kObsDim);
#pragma unroll
    for (int k = 0; k < kObsDim / 2; ++k) dst[k] = make_float2(obs[2 * k], obs[2 * k + 1]);
}

#ifndef CARENV_MIN_BLOCKS
#define CARENV_MIN_BLOCKS 4
#endif
template <typename ActT, typename FlagT, int U>
__global__ void __launch_bounds__(kBlock, CARENV_MIN_BLOCKS)
k_rollout(const __grid_constant__ TrackParams P, const Tables G, int n_envs, int n_steps, double2 *__restrict__ pos,
          double2 *__restrict__ vel, int4 *__restrict__ ints, const ActT *__restrict__ actions, double reward_scale,
          float *__restrict__ obs_out, float *__restrict__ rew_out, FlagT *__restrict__ term_out,
          FlagT *__restrict__ trunc_out, int4 *__restrict__ info_out, int4 *__restrict__ rec_out,
          float *__restrict__ fobs_out, unsigned long long *stats, int obs_mode) {
    extern __shared__ __align__(16) unsigned char smem[];
    const Tables T = stage_tables(G, P.n_gates, P.n_seg, smem);
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;

    EnvState s;
    {
        const double2 p = pos[e], v = vel[e];
        const int4 q = ints[e];
        s.px = p.x; s.py = p.y; s.vx = v.x; s.vy = v.y;
        s.k = q.x; s.t = q.y; s.next_gate = q.z; s.passed = q.w;
    }
    int a_next = action_index(actions[e]);
    for (int t = 0; t < n_steps; ++t) {
        const size_t idx = (size_t)t * (size_t)n_envs + (size_t)e;
        const int a = a_next;
        if (t + 1 < n_steps) a_next = action_index(actions[idx + (size_t)n_envs]);   // next step's action is in flight during this step
        StepResult o;
        env_step<U>(s, a, reward_scale, P, T, o, stats, nullptr, nullptr, fobs_out ? fobs_out + idx * kObsDim : nullptr);
        if (obs_mode == kObsFull) {
            float2 *dst = reinterpret_cast<float2 *>(obs_out + idx * kObsDim);
#pragma unroll
            for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(o.obs[2 * i], o.obs[2 * i + 1]);
        } else if (obs_mode == kObsPose) {                   // 32-byte pose record instead of the 72-byte observation
            store_pose(reinterpret_cast<PoseRec *>(obs_out) + idx, s, o.obs[2], o.obs[3]);
        }
        store_step(o, idx, rew_out, term_out, trunc_out, info_out, rec_out);
    }
    pos[e] = make_double2(s.px, s.py);
    vel[e] = make_double2(s.vx, s.vy);
    ints[e] = make_int4(s.k, s.t, s.next_gate, s.passed);
}

// Large launches on tracks the pair kernels take (<= 128 segments, even chain lengths): thread per environment
// like k_rollout, but the 144 denominators cross(e, d) a step needs come from a per-track table in shared memory
// (TabView, carenv_core.cuh) instead of 144 FMUL2 / FFMA2 — the values are the same bit for bit.  One CTA of up to
// 512 threads per SM owns the table copies (72 headings x n_pairs x 16 B, x 8 skewed copies = 147 KB on big_track)
// and walks over blocks of environments; the block sizes are chosen on the host (launch_rollout_tab) so that every
// SM gets the same number of blocks and the last round is as short as its remainder allows.
#ifndef CARENV_TAB_THREADS
#define CARENV_TAB_THREADS 512
#endif
constexpr int kTabThreads = CARENV_TAB_THREADS;
template <typename ActT, typename FlagT, int U, int NS = 0, bool CULL = false>
__global__ void __launch_bounds__(kTabThreads, 1)
k_rollout_tab(const __grid_constant__ TrackParams P, const Tables G, const float4 *__restrict__ den4, const CullGrid cull,
              int n_pairs,
              int row_f4, int copies, int table_bytes, int n_envs, int n_steps, int epb_main, int n_main, int epb_last,
              int n_blocks,
              double2 *__restrict__ pos, double2 *__restrict__ vel, int4 *__restrict__ ints,
              const ActT *__restrict__ actions, double reward_scale, float *__restrict__ obs_out,
              float *__restrict__ rew_out, FlagT *__restrict__ term_out, FlagT *__restrict__ trunc_out,
              int4 *__restrict__ info_out, int4 *__restrict__ rec_out, unsigned long long *stats, int obs_mode) {
    extern __shared__ __align__(16) unsigned char smem[];
    // [tables | pad to 128 B | copy 0 | copy 1 (+16 B) | ...]: copy c starts at c * (72 * row + 1) float4
    const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(smem);
    const int t_off = (int)(((s0 + (uint32_t)table_bytes + 127u) & ~127u) - s0);
    float4 *tab = reinterpret_cast<float4 *>(smem + t_off);
    const int copy_f4 = kHeadings * row_f4 + 1;
    for (int i = threadIdx.x; i < kHeadings * n_pairs; i += blockDim.x) {
        const float4 v = den4[i];
        const int k = i / n_pairs, jp = i - k * n_pairs;
        for (int c = 0; c < copies; ++c) tab[c * copy_f4 + k * row_f4 + jp] = v;
    }
    const Tables T = stage_tables(G, P.n_gates, P.n_seg, smem);      // ends with __syncthreads()
    const TabView tv{tab + (threadIdx.x & (copies - 1)) * copy_f4, row_f4, cull};

    // blocks [0, n_main) hold epb_main environments each (full rounds: four warps per scheduler), the blocks of the
    // last round epb_last (a multiple of 128: every scheduler of the SM gets the same number of warps)
    for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        // (a last-round block is its CTA's final block, so leaving the loop is the same as skipping the block — and
        // `break` keeps the loop body provably convergent, which the uniform-register operands of the wall tests need)
        const bool last = blk >= n_main;
        if ((int)threadIdx.x >= (last ? epb_last : epb_main)) break;
        const int e = last ? n_main * epb_main + (blk - n_main) * epb_last + threadIdx.x : blk * epb_main + threadIdx.x;
        if (e >= n_envs) break;
        EnvState s;
        {
            const double2 p = pos[e], v = vel[e];
            const int4 q = ints[e];
            s.px = p.x; s.py = p.y; s.vx = v.x; s.vy = v.y;
            s.k = q.x; s.t = q.y; s.next_gate = q.z; s.passed = q.w;
        }
        int a_next = action_index(actions[e]);
        for (int t = 0; t < n_steps; ++t) {
            const size_t idx = (size_t)t * (size_t)n_envs + (size_t)e;
            const int a = a_next;
            if (t + 1 < n_steps) a_next = action_index(actions[idx + (size_t)n_envs]);
            StepResult o;
            env_step<U, true, NS, CULL>(s, a, reward_scale, P, T, o, stats, nullptr, &tv);
            if (obs_mode == kObsFull) {
                float2 *dst = reinterpret_cast<float2 *>(obs_out + idx * kObsDim);
#pragma unroll
                for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(o.obs[2 * i], o.obs[2 * i + 1]);
            } else if (obs_mode == kObsPose) {
                store_pose(reinterpret_cast<PoseRec *>(obs_out) + idx, s, o.obs[2], o.obs[3]);
            }
            store_step(o, idx, rew_out, term_out, trunc_out, info_out, rec_out);
        }
        pos[e] = make_double2(s.px, s.py);
        vel[e] = make_double2(s.vx, s.vy);
        ints[e] = make_int4(s.k, s.t, s.next_gate, s.passed);
    }
}

// k_rollout_tab with the work of an SM spread EVENLY over its 16 warps in units of env-STEPS instead of whole blocks
// of environments.  With blocks, an SM that owns W warps' worth of environments runs ceil(W / 16) rounds and the last
// round is short-handed: 131,072 envs on 148 SMs (the 8-GPU shard of the 1 M-env job) = 27.7 warps per SM = a round
// with four warps per scheduler and one with three, which run at 0.98 and 0.84 warp-steps/us — 6 % lost.  Here a
// "job" is 32 consecutive environments x n_steps steps; the W jobs of an SM are laid end to end (W x n_steps
// warp-steps) and cut into 16 equal intervals, one per warp (McNaughton's wrap-around rule for preemptible jobs on
// identical machines).  A job that straddles the boundary between warp w and warp w + 1 is split IN TIME: warp w + 1
// runs its first steps at the start of its interval, stores the state (the pos / vel / ints arrays themselves are the
// hand-over buffer) and raises the job's flag; warp w runs the remaining steps at the END of its interval (an interval
// is at least n_steps long, so the first part has finished by then; the flag makes it safe).  Every warp is busy for
// the same number of steps and every scheduler keeps four warps until the very end.  Per-environment arithmetic is
// untouched: results are bit-identical to k_rollout_tab / k_rollout.
template <typename ActT, typename FlagT, int U, int NS = 0, bool CULL = false>
__global__ void __launch_bounds__(kTabThreads, 1)
k_rollout_tab_sliced(const __grid_constant__ TrackParams P, const Tables G, const float4 *__restrict__ den4,
                     const CullGrid cull, int n_pairs,
                     int row_f4, int copies, int table_bytes, int n_envs, int n_steps, int *__restrict__ flags,
                     double2 *__restrict__ pos, double2 *__restrict__ vel, int4 *__restrict__ ints,
                     const ActT *__restrict__ actions, double reward_scale, float *__restrict__ obs_out,
                     float *__restrict__ rew_out, FlagT *__restrict__ term_out, FlagT *__restrict__ trunc_out,
                     int4 *__restrict__ info_out, int4 *__restrict__ rec_out, unsigned long long *stats, int obs_mode) {
    extern __shared__ __align__(16) unsigned char smem[];
    const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(smem);
    const int t_off = (int)(((s0 + (uint32_t)table_bytes + 127u) & ~127u) - s0);
    float4 *tab = reinterpret_cast<float4 *>(smem + t_off);
    const int copy_f4 = kHeadings * row_f4 + 1;
    for (int i = threadIdx.x; i < kHeadings * n_pairs; i += blockDim.x) {
        const float4 v = den4[i];
        const int k = i / n_pairs, jp = i - k * n_pairs;
        for (int c = 0; c < copies; ++c) tab[c * copy_f4 + k * row_f4 + jp] = v;
    }
    const Tables T = stage_tables(G, P.n_gates, P.n_seg, smem);      // ends with __syncthreads()
    const TabView tv{tab + (threadIdx.x & (copies - 1)) * copy_f4, row_f4, cull};

    // (the warp index through a shuffle: the compiler then knows that it — and with it every item bound below, the
    // trip count of the step loop included — is warp-uniform; derived from threadIdx alone the loop counted as
    // divergent and the wall tests lost their uniform-register operands: 8 % slower)
    const int slot = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31, n_slots = blockDim.x >> 5;
    const int jobs_total = (n_envs + 31) >> 5;
    const int job_lo = (int)((long long)blockIdx.x * jobs_total / gridDim.x);
    const int job_hi = (int)((long long)(blockIdx.x + 1) * jobs_total / gridDim.x);
    // This warp's interval [lo, hi) of the SM's job_count x n_steps warp-steps, as a list of items:
    //   the job cut by lo (the previous warp holds its LAST steps): its first steps   [item first_job, steps 0 .. head_len)
    //   whole jobs                                                                    [first_job + has_head .. last_full]
    //   the job cut by hi (the next warp runs its first steps): its last steps        [item tail_job, steps n - tail_len .. n)
    const SliceItems items = slice_items(job_hi - job_lo, n_steps, slot, n_slots);   // carenv_core.cuh (tested on the host)
    const int first_job = items.first_job, head_len = items.head_len, last_full = items.last_full, tail_len = items.tail_len;
    // (item bookkeeping in shared memory instead of registers was measured: fewer spills, 1.5 % slower)
    const int n_items = (last_full + 1 - first_job) + (tail_len > 0 ? 1 : 0);     // the head item is job first_job itself
    for (int it = 0; it < n_items; ++it) {
        const int job = first_job + it;
        const bool head = it == 0 && head_len > 0, tail = job > last_full;
        const int t0 = tail ? n_steps - tail_len : 0, t1 = head ? head_len : n_steps;
        const int e = ((job_lo + job) << 5) + lane;
        // (only the grid's very last job can have lanes past the end, and it is the last item of every warp that touches
        // it — `break` keeps the loop body provably convergent, which the uniform-register operands of the wall tests need)
        if (e >= n_envs) break;
        int *flag = flags + job_lo + job;
        if (tail) {                                          // the first part's state must be in memory
            int spins = 0;
            while (*reinterpret_cast<volatile int *>(flag) == 0)
                if (++spins > (1 << 28)) __trap();           // a scheduling error must not hang the GPU box
            __threadfence();
        }
        EnvState s;
        {
            const double2 pp = __ldcg(pos + e), v = __ldcg(vel + e);
            const int4 qq = __ldcg(ints + e);
            s.px = pp.x; s.py = pp.y; s.vx = v.x; s.vy = v.y;
            s.k = qq.x; s.t = qq.y; s.next_gate = qq.z; s.passed = qq.w;
        }
        int a_next = action_index(actions[(size_t)t0 * (size_t)n_envs + (size_t)e]);
        for (int t = t0; t < t1; ++t) {
            const size_t idx = (size_t)t * (size_t)n_envs + (size_t)e;
            const int a = a_next;
            if (t + 1 < t1) a_next = action_index(actions[idx + (size_t)n_envs]);
            StepResult o;
            env_step<U, true, NS, CULL>(s, a, reward_scale, P, T, o, stats, nullptr, &tv);
            if (obs_mode == kObsFull) {
                float2 *dst = reinterpret_cast<float2 *>(obs_out + idx * kObsDim);
#pragma unroll
                for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(o.obs[2 * i], o.obs[2 * i + 1]);
            } else if (obs_mode == kObsPose) {
                store_pose(reinterpret_cast<PoseRec *>(obs_out) + idx, s, o.obs[2], o.obs[3]);
            }
            store_step(o, idx, rew_out, term_out, trunc_out, info_out, rec_out);
        }
        __stcg(pos + e, make_double2(s.px, s.py));
        __stcg(vel + e, make_double2(s.vx, s.vy));
        __stcg(ints + e, make_int4(s.k, s.t, s.next_gate, s.passed));
        if (head) {                                          // publish: every lane's state first, then the flag
            __threadfence();
            __syncwarp();
            if (lane == 0) *reinterpret_cast<volatile int *>(flag) = 1;
        }
    }
}

// Small batches: one WARP per environment, lane j = wall segment j (tracks with at most 32 segments), per-ray
// extrema by warp-level integer REDUX (carenv_core.cuh: cast_walls_warp).  A lone thread-per-environment warp
// needs ~1.9 us per step (1,700 dependent-ish instructions); here the 24 segments are evaluated side by side
// and a step is ~600 warp-instructions.  Every lane carries the (identical) environment state and runs the scalar
// part of the step redundantly; lane 0 writes the outputs.  Bit-identical to k_rollout.
template <typename ActT, typename FlagT>
__global__ void __launch_bounds__(128)
k_rollout_warp(const __grid_constant__ TrackParams P, const Tables G, int n_envs, int n_steps, double2 *__restrict__ pos,
               double2 *__restrict__ vel, int4 *__restrict__ ints, const ActT *__restrict__ actions,
               double reward_scale, float *__restrict__ obs_out, float *__restrict__ rew_out,
               FlagT *__restrict__ term_out, FlagT *__restrict__ trunc_out, int4 *__restrict__ info_out,
               int4 *__restrict__ rec_out, float *__restrict__ fobs_out, unsigned long long *stats, int obs_mode) {
    extern __shared__ __align__(16) unsigned char smem[];
    const Tables T = stage_tables(G, P.n_gates, P.n_seg, smem);
    const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (e >= n_envs) return;

    WarpSeg ws;
    ws.active = lane < P.n_seg;
    ws.f = G.segf[ws.active ? lane : 0];
    ws.g = G.segd[ws.active ? lane : 0];
    EnvState s;
    {
        const double2 p = pos[e], v = vel[e];
        const int4 q = ints[e];
        s.px = p.x; s.py = p.y; s.vx = v.x; s.vy = v.y;
        s.k = q.x; s.t = q.y; s.next_gate = q.z; s.passed = q.w;
    }
    unsigned long long *my_stats = lane == 0 ? stats : nullptr;
    int a_next = action_index(actions[e]);
    for (int t = 0; t < n_steps; ++t) {
        const size_t idx = (size_t)t * (size_t)n_envs + (size_t)e;
        const int a = a_next;
        if (t + 1 < n_steps) a_next = action_index(actions[idx + (size_t)n_envs]);
        StepResult o;
        env_step<kWarpPerEnv>(s, a, reward_scale, P, T, o, my_stats, &ws, nullptr,
                              (fobs_out && lane == 0) ? fobs_out + idx * kObsDim : nullptr);
        if (lane == 0) {
            if (obs_mode == kObsFull) {
                float2 *dst = reinterpret_cast<float2 *>(obs_out + idx * kObsDim);
#pragma unroll
                for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(o.obs[2 * i], o.obs[2 * i + 1]);
            } else if (obs_mode == kObsPose) {
                store_pose(reinterpret_cast<PoseRec *>(obs_out) + idx, s, o.obs[2], o.obs[3]);
            }
            store_step(o, idx, rew_out, term_out, trunc_out, info_out, rec_out);
        }
    }
    if (lane == 0) {
        pos[e] = make_double2(s.px, s.py);
        vel[e] = make_double2(s.vx, s.vy);
        ints[e] = make_int4(s.k, s.t, s.next_gate, s.passed);
    }
}

#include "policy_rollout.cuh"   // k_policy_rollout, k_policy_rollout_tc, k_pack_policy, k_tc_gemm_test

__global__ void __launch_bounds__(kBlock)
k_reset(const __grid_constant__ TrackParams P, int n_envs, double2 *__restrict__ pos, double2 *__restrict__ vel,
        int4 *__restrict__ ints, float *__restrict__ obs_out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;
    pos[e] = make_double2(P.start_x, P.start_y);
    vel[e] = make_double2(0.0, 0.0);
    ints[e] = make_int4(0, 0, 0, 0);
    if (obs_out) {
        float2 *dst = reinterpret_cast<float2 *>(obs_out + (size_t)e * kObsDim);
#pragma unroll
        for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(P.reset_obs[2 * i], P.reset_obs[2 * i + 1]);
    }
}

// GAE(lambda), lib/buffer.py:51-63.  The recurrence is serial in t but the loads are not: timesteps are
// processed in batches of kGaeUnroll with the NEXT batch's 4 * kGaeUnroll loads issued before the
// current batch is consumed (register double buffering), so every thread keeps loads in flight while
// it walks the dependent chain.  Streaming loads/stores: every byte is touched once.
template <int kGaeUnroll> struct GaeBatch { float r[kGaeUnroll], v[kGaeUnroll], te[kGaeUnroll], tr[kGaeUnroll]; };

template <int kGaeUnroll>
__device__ __forceinline__ void gae_load(GaeBatch<kGaeUnroll> &b, const float *__restrict__ rew, const float *__restrict__ val,
                                         const float *__restrict__ term, const float *__restrict__ trunc, int t,
                                         size_t N, size_t e) {
#pragma unroll
    for (int i = 0; i < kGaeUnroll; ++i) {
        const size_t k = (size_t)(t - i) * N + e;
        b.r[i] = __ldcs(rew + k); b.v[i] = __ldcs(val + k); b.te[i] = __ldcs(term + k); b.tr[i] = __ldcs(trunc + k);
    }
}

// kGaeUnroll = 8 (80 registers) is best up to ~65 k columns, 16 (164 registers, more loads in flight per
// thread) beyond: 5.92 vs 4.69 TB/s at [1024, 65536], 5.30 vs 5.45 at [1024, 131072], 5.81 vs 5.94 at [128, 1 M].
template <int kGaeUnroll>
__global__ void __launch_bounds__(128)
k_gae(const float *__restrict__ rew, const float *__restrict__ val, const float *__restrict__ term,
      const float *__restrict__ trunc, const float *__restrict__ last_val, const float *__restrict__ last_term,
      const float *__restrict__ last_trunc, float *__restrict__ adv, float *__restrict__ ret, int T, int N, float g,
      float gl) {
  // grid-stride over the columns: the launch sizes the grid to ONE balanced wave of resident threads
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < N; e += gridDim.x * blockDim.x) {
    float nv = last_val[e];
    float tm = __fadd_rn(1.0f, -last_term[e]);
    float um = __fadd_rn(1.0f, -last_trunc[e]);
    float a = 0.0f;
    int t = T - 1;
    GaeBatch<kGaeUnroll> cur, nxt;
    if (t >= kGaeUnroll - 1) gae_load(cur, rew, val, term, trunc, t, (size_t)N, (size_t)e);
    for (; t >= kGaeUnroll - 1; t -= kGaeUnroll) {
        const bool more = (t - kGaeUnroll) >= kGaeUnroll - 1;
        if (more) gae_load(nxt, rew, val, term, trunc, t - kGaeUnroll, (size_t)N, (size_t)e);
#pragma unroll
        for (int i = 0; i < kGaeUnroll; ++i) {
            const size_t k = (size_t)(t - i) * (size_t)N + (size_t)e;
            const float delta = __fadd_rn(__fadd_rn(cur.r[i], __fmul_rn(__fmul_rn(g, nv), tm)), -cur.v[i]);
            a = __fadd_rn(delta, __fmul_rn(__fmul_rn(__fmul_rn(gl, tm), um), a));
            __stcs(adv + k, a);
            __stcs(ret + k, __fadd_rn(a, cur.v[i]));
            nv = cur.v[i];
            tm = __fadd_rn(1.0f, -cur.te[i]);
            um = __fadd_rn(1.0f, -cur.tr[i]);
        }
        if (more) cur = nxt;
    }
    for (; t >= 0; --t) {
        const size_t k = (size_t)t * (size_t)N + (size_t)e;
        const float r = __ldcs(rew + k), v = __ldcs(val + k);
        const float delta = __fadd_rn(__fadd_rn(r, __fmul_rn(__fmul_rn(g, nv), tm)), -v);
        a = __fadd_rn(delta, __fmul_rn(__fmul_rn(__fmul_rn(gl, tm), um), a));
        __stcs(adv + k, a);
        __stcs(ret + k, __fadd_rn(a, v));
        nv = v;
        tm = __fadd_rn(1.0f, -__ldcs(term + k));
        um = __fadd_rn(1.0f, -__ldcs(trunc + k));
    }
  }
}

// ---- several tracks in ONE launch (SURVEY §8 f-4: reset(options={"track_path": ...}) per environment,
// lib/car_env.py:621-628).  Every environment carries a track id; the per-track constants (TrackParams) and tables
// live in global memory (concatenated in the multi-track handle) and each thread reads ITS track's through a
// pointer, so environments on different tracks may share a warp.  The arithmetic is the generic segment loop
// (env_step<0>: geometry read through Tables::segf / segd), bit-identical to the single-track kernels.
struct MultiTrack {
    int n_tracks, device;
    TrackParams *d_params;    // [n_tracks]
    Tables *d_tables;         // [n_tracks] pointers into the single-track handles' blobs
    unsigned long long *d_stats;
};

template <typename ActT, typename FlagT>
__global__ void __launch_bounds__(128)
k_rollout_multi(const TrackParams *__restrict__ params, const Tables *__restrict__ tables, int n_tracks,
                const int *__restrict__ track_ids, int n_envs, int n_steps, double2 *__restrict__ pos,
                double2 *__restrict__ vel, int4 *__restrict__ ints, const ActT *__restrict__ actions,
                double reward_scale, float *__restrict__ obs_out, float *__restrict__ rew_out,
                FlagT *__restrict__ term_out, FlagT *__restrict__ trunc_out, int4 *__restrict__ info_out,
                unsigned long long *stats) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;
    int tr = track_ids[e];
    tr = tr < 0 ? 0 : (tr >= n_tracks ? n_tracks - 1 : tr);
    const TrackParams &P = params[tr];
    const Tables T = tables[tr];
    EnvState s;
    {
        const double2 p = pos[e], v = vel[e];
        const int4 q = ints[e];
        s.px = p.x; s.py = p.y; s.vx = v.x; s.vy = v.y;
        s.k = q.x; s.t = q.y; s.next_gate = q.z; s.passed = q.w;
    }
    for (int t = 0; t < n_steps; ++t) {
        const size_t idx = (size_t)t * (size_t)n_envs + (size_t)e;
        StepResult o;
        env_step<0>(s, action_index(actions[idx]), reward_scale, P, T, o, stats);
        if (obs_out) {
            float2 *dst = reinterpret_cast<float2 *>(obs_out + idx * kObsDim);
#pragma unroll
            for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(o.obs[2 * i], o.obs[2 * i + 1]);
        }
        store_step(o, idx, rew_out, term_out, trunc_out, info_out, (int4 *)nullptr);
    }
    pos[e] = make_double2(s.px, s.py);
    vel[e] = make_double2(s.vx, s.vy);
    ints[e] = make_int4(s.k, s.t, s.next_gate, s.passed);
}

__global__ void __launch_bounds__(128)
k_reset_multi(const TrackParams *__restrict__ params, int n_tracks, const int *__restrict__ track_ids, int n_envs,
              double2 *__restrict__ pos, double2 *__restrict__ vel, int4 *__restrict__ ints, float *__restrict__ obs_out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;
    int tr = track_ids[e];
    tr = tr < 0 ? 0 : (tr >= n_tracks ? n_tracks - 1 : tr);
    const TrackParams &P = params[tr];
    pos[e] = make_double2(P.start_x, P.start_y);
    vel[e] = make_double2(0.0, 0.0);
    ints[e] = make_int4(0, 0, 0, 0);
    if (obs_out)
        for (int i = 0; i < kObsDim; ++i) obs_out[(size_t)e * kObsDim + i] = P.reset_obs[i];
}

// ---- headless rgb_array frames (lib/car_env.py:762-812, consumer train.py:23-50): one thread per pixel.
// Background (11,102,35), the corridor between the outer and the inner polygon gray, walls black 5 px, active gates
// green 5 px (the next one yellow), the rays as thin lines to their hit points, the car as a rotated 40 x 20 px box
// (the reference blits lib/assets/car.png there; the sprite is not part of this repository).  A diagnostic picture
// for videos of a handful of environments — not a pixel-exact restatement of pygame's rasteriser.
__device__ __forceinline__ float seg_dist2(float px, float py, float ax, float ay, float bx, float by) {
    const float ex = bx - ax, ey = by - ay, wx = px - ax, wy = py - ay;
    const float l2 = ex * ex + ey * ey;
    float t = l2 > 0.0f ? (wx * ex + wy * ey) / l2 : 0.0f;
    t = fminf(fmaxf(t, 0.0f), 1.0f);
    const float dx = wx - t * ex, dy = wy - t * ey;
    return dx * dx + dy * dy;
}

__global__ void __launch_bounds__(256)
k_render(const __grid_constant__ TrackParams P, const Tables G, int n_outer, int n_frames, const int *__restrict__ env_index,
         const double2 *__restrict__ pos, const int4 *__restrict__ ints, const float *__restrict__ obs, int width,
         int height, unsigned char *__restrict__ rgb) {
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    const int f = blockIdx.y;
    if (pix >= width * height || f >= n_frames) return;
    const int e = env_index[f];
    const float x = (float)(pix % width) + 0.5f, y = (float)(pix / width) + 0.5f;
    const double2 cp = pos[e];
    const int4 st = ints[e];
    const float cx = (float)cp.x, cy = (float)cp.y;
    const F2 hd = G.trig32[st.x];
    // crossing number of the two closed border polylines; distance to the nearest wall
    bool in_outer = false, in_inner = false;
    float wall2 = 1.0e30f;
    for (int j = 0; j < P.n_seg; ++j) {
        const float ax = (float)G.walls64[4 * j], ay = (float)G.walls64[4 * j + 1];
        const float bx = (float)G.walls64[4 * j + 2], by = (float)G.walls64[4 * j + 3];
        if ((ay > y) != (by > y) && x < ax + (y - ay) * (bx - ax) / (by - ay)) {
            if (j < n_outer) in_outer = !in_outer; else in_inner = !in_inner;
        }
        wall2 = fminf(wall2, seg_dist2(x, y, ax, ay, bx, by));
    }
    unsigned char r = 11, g = 102, b = 35;                                   // canvas.fill((11, 102, 35))
    if (in_outer && !in_inner) { r = 190; g = 190; b = 190; }                // "gray" polygon minus the inner one
    if (wall2 <= 6.25f) { r = 0; g = 0; b = 0; }                             // boundary.draw(canvas, "black", 5)
    for (int q = st.z; q < P.n_gates; ++q) {                                 // gates below next_gate_index are inactive
        const GateRec gt = G.gates[q];
        if (seg_dist2(x, y, (float)gt.x1, (float)gt.y1, (float)gt.x2, (float)gt.y2) <= 6.25f) {
            if (q == st.z) { r = 255; g = 255; b = 0; } else { r = 0; g = 255; b = 0; }
        }
    }
    for (int i = 0; i < kNumRays; ++i) {                                     // car.draw_rays: origin -> hit point
        const F2 d = G.trig32[wrap72(st.x + 6 * i)];
        const float len = obs[(size_t)e * kObsDim + 6 + i] * 1000.0f;
        if (seg_dist2(x, y, cx, cy, cx + d.x * len, cy + d.y * len) <= 0.6f) { r = 255; g = 255; b = 255; }
    }
    {   // the car: 40 x 20 px box along the heading
        const float dx = x - cx, dy = y - cy;
        const float u = dx * hd.x + dy * hd.y, v = -dx * hd.y + dy * hd.x;
        if (fabsf(u) <= 20.0f && fabsf(v) <= 10.0f) { r = 200; g = 30; b = 30; if (u > 12.0f) { r = 250; g = 220; b = 60; } }
    }
    unsigned char *dst = rgb + ((size_t)f * width * height + pix) * 3;
    dst[0] = r; dst[1] = g; dst[2] = b;
}

// FP32-pipe peak probe: kFfmaChains independent FFMA chains per thread, no memory traffic.
// SURVEY §8(d): MEASURED_PEAKS.json has no FP32 entry, so bench.py measures one beside the nominal.
constexpr int kFfmaChains = 8;
__global__ void __launch_bounds__(256) k_ffma_peak(float *out, int iters, float a, float b) {
    float acc[kFfmaChains];
#pragma unroll
    for (int i = 0; i < kFfmaChains; ++i) acc[i] = (float)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int i = 0; i < kFfmaChains; ++i) acc[i] = __fmaf_rn(acc[i], a, b);
    }
    float sum = 0.0f;
#pragma unroll
    for (int i = 0; i < kFfmaChains; ++i) sum += acc[i];
    if (sum == 12345.678f) out[0] = sum;   // keeps the chains alive without storing
}

template <typename ActT, typename FlagT, int U>
int launch_rollout_t(Handle *h, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints, const void *actions,
                   double reward_scale, float *obs_out, float *reward_out, void *term_out, void *trunc_out,
                   int32_t *info_out, cudaStream_t stream, int obs_mode) {
    auto kern = k_rollout<ActT, FlagT, U>;
    const int block = h->block > 0 ? h->block : kBlock;
    const size_t smem = h->smem_bytes + (size_t)h->smem_pad;
    if (smem > 48 * 1024)
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = (n_envs + block - 1) / block;
    kern<<<grid, block, smem, stream>>>(
        h->host.P, h->dev, n_envs, n_steps, reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel),
        reinterpret_cast<int4 *>(ints), static_cast<const ActT *>(actions), reward_scale, obs_out, reward_out,
        static_cast<FlagT *>(term_out), static_cast<FlagT *>(trunc_out), reinterpret_cast<int4 *>(info_out),
        h->cur_rec, h->cur_fobs, h->d_stats, obs_mode);
    CU(cudaGetLastError());
    return 0;
}

// k_rollout_tab: table geometry, balanced block size, launch.  Returns 1 if the table does not fit in shared memory.
template <typename ActT, typename FlagT>
int launch_rollout_tab(Handle *h, int U, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints,
                       const void *actions, double reward_scale, float *obs_out, float *reward_out, void *term_out,
                       void *trunc_out, int32_t *info_out, cudaStream_t stream, int obs_mode) {
    // The segment loop fully unrolled (NS = n_seg) for the segment counts of the shipped tracks, big_track (24) and
    // track.json (16): no indexed constant loads and no loop overhead (DESIGN.md §3).  Other tracks run the U loop.
    // big_track's unroll skips the segment pairs the candidate table culls (CULL, cast_walls): 3.7 of 12 pairs per
    // warp-step, 5 % faster.  track.json's does not: it culls 1 of 8 and the lookup costs more (3 % slower, §3).
    const int n_seg = h->host.P.n_seg;
    const int n_pairs = h->host.n_pairs;
    const int row_f4 = (n_pairs + 7) / 8 * 8;                // rows are multiples of 128 bytes
    const int table_bytes = (int)((h->smem_bytes + 15) / 16 * 16);
    int copies = 8;
    auto total = [&](int c) { return (size_t)table_bytes + 128 + (size_t)c * (kHeadings * row_f4 + 1) * 16; };
    while (copies > 1 && total(copies) > 200 * 1024) copies >>= 1;
    if (total(copies) > 200 * 1024) return 1;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    const int block = h->block > 0 ? h->block * 4 : kTabThreads;           // tuning hook (block is 0..128: x4)
    // Time-sliced distribution (k_rollout_tab_sliced) when every SM gets at least one 32-environment job per warp, so
    // that no job is cut twice; not for the final-observation variant (cur_fobs never reaches this function).
    {
        const long long jobs = (n_envs + 31) / 32;
        // (single steps — the host-buffer step's sub-ranges — stay with the block scheme: nothing to balance over time
        // and its prologue is shorter; measured 7 % on the end-to-end rate)
        const bool fits = jobs / sms >= block / 32 && block == kTabThreads && n_steps >= 4;
        if (h->tab_slice >= 0 && fits) {
            const size_t need = (size_t)jobs;
            bool ok = true;
            {
                if (h->flags_cap < need) {
                    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
                    cudaStreamIsCapturing(stream, &cap);
                    if (cap != cudaStreamCaptureStatusNone) {
                        ok = false;                          // no allocation inside a graph capture: block scheme
                    } else {
                        if (h->d_flags) cudaFree(h->d_flags);
                        h->d_flags = nullptr; h->flags_cap = 0;
                        CU(cudaMalloc(reinterpret_cast<void **>(&h->d_flags), need * sizeof(int)));
                        h->flags_cap = need;
                    }
                }
                if (ok) CU(cudaMemsetAsync(h->d_flags, 0, need * sizeof(int), stream));
            }
            if (ok) {
                const size_t smem_s = total(copies);
                auto launch_s = [&](auto kern) -> int {
                    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s));
                    kern<<<sms, block, smem_s, stream>>>(
                        h->host.P, h->dev, h->d_den4, h->cull, n_pairs, row_f4, copies, table_bytes, n_envs, n_steps, h->d_flags,
                        reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel), reinterpret_cast<int4 *>(ints),
                        static_cast<const ActT *>(actions), reward_scale, obs_out, reward_out, static_cast<FlagT *>(term_out),
                        static_cast<FlagT *>(trunc_out), reinterpret_cast<int4 *>(info_out), h->cur_rec, h->d_stats, obs_mode);
                    CU(cudaGetLastError());
                    return 0;
                };
                if (U == 6 && n_seg == 24) return launch_s(k_rollout_tab_sliced<ActT, FlagT, 6, 24, true>);
                if (U == 4 && n_seg == 16) return launch_s(k_rollout_tab_sliced<ActT, FlagT, 4, 16>);
                if (U == 6) return launch_s(k_rollout_tab_sliced<ActT, FlagT, 6>);
                if (U == 4) return launch_s(k_rollout_tab_sliced<ActT, FlagT, 4>);
                return launch_s(k_rollout_tab_sliced<ActT, FlagT, 2>);
            }
        }
    }
    // A round = one block per SM.  Its duration is set by the warps per SCHEDULER (a block of 448 environments takes as
    // long as one of 512), so all rounds but the last are full blocks and the last round's blocks are the smallest
    // multiple of 128 environments that covers the remainder: 131,072 envs on 148 SMs = 148 x 512 + 148 x 384.
    const long long per_round = (long long)sms * block;
    const int rounds = (int)((n_envs + per_round - 1) / per_round);
    const int n_main = (rounds - 1) * sms, epb_main = block;
    const int rem = n_envs - n_main * epb_main;
    int epb_last = ((rem + sms - 1) / sms + 127) / 128 * 128;
    if (epb_last > block) epb_last = block;
    const int n_blocks = n_main + (rem + epb_last - 1) / epb_last;
    const int grid = n_blocks < sms ? n_blocks : sms;
    const size_t smem = total(copies);
    auto launch = [&](auto kern) -> int {
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, block, smem, stream>>>(
            h->host.P, h->dev, h->d_den4, h->cull, n_pairs, row_f4, copies, table_bytes, n_envs, n_steps, epb_main, n_main,
            epb_last,
            n_blocks,
            reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel), reinterpret_cast<int4 *>(ints),
            static_cast<const ActT *>(actions), reward_scale, obs_out, reward_out, static_cast<FlagT *>(term_out),
            static_cast<FlagT *>(trunc_out), reinterpret_cast<int4 *>(info_out), h->cur_rec, h->d_stats, obs_mode);
        CU(cudaGetLastError());
        return 0;
    };
    if (U == 6 && n_seg == 24) return launch(k_rollout_tab<ActT, FlagT, 6, 24, true>);
    if (U == 4 && n_seg == 16) return launch(k_rollout_tab<ActT, FlagT, 4, 16>);
    if (U == 6) return launch(k_rollout_tab<ActT, FlagT, 6>);
    if (U == 4) return launch(k_rollout_tab<ActT, FlagT, 4>);
    return launch(k_rollout_tab<ActT, FlagT, 2>);
}

// Segment-loop unrolling is chosen per track (TrackParams::unroll); all variants give identical results.
template <typename ActT, typename FlagT>
int launch_rollout(Handle *h, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints, const void *actions,
                   double reward_scale, float *obs_out, float *reward_out, void *term_out, void *trunc_out,
                   int32_t *info_out, cudaStream_t stream, int obs_mode) {
    // small batches on small tracks: one warp per environment (crossover measured by benchmarks/small_batch.py)
    const bool warp_ok = h->host.P.n_seg <= 32 && !h->force_generic;
    if (warp_ok && (h->warp_per_env == 1 || (h->warp_per_env == 0 && n_envs <= kWarpPerEnvMax))) {
        auto kern = k_rollout_warp<ActT, FlagT>;
        if (h->smem_bytes > 48 * 1024)                       // tracks with more than ~900 gates
            CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes));
        const int grid = (n_envs + 3) / 4;
        kern<<<grid, 128, h->smem_bytes, stream>>>(
            h->host.P, h->dev, n_envs, n_steps, reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel),
            reinterpret_cast<int4 *>(ints), static_cast<const ActT *>(actions), reward_scale, obs_out, reward_out,
            static_cast<FlagT *>(term_out), static_cast<FlagT *>(trunc_out), reinterpret_cast<int4 *>(info_out),
            h->cur_rec, h->cur_fobs, h->d_stats, obs_mode);
        CU(cudaGetLastError());
        return 0;
    }
    int U = h->force_generic ? 1 : h->host.P.unroll;
    if (h->max_unroll > 0 && U > h->max_unroll) U = (U % h->max_unroll == 0) ? h->max_unroll : 1;
    if (h->host.P.n_seg > kMaxSeg) U = 0;                   // geometry from shared memory
    // 4,096 environments or more: denominators from the shared-memory table (k_rollout_tab) — measured equal or faster
    // than k_rollout from there on for every launch length, single steps included (benchmarks/ab_step.py: 1 M envs x 1
    // step 92 vs 120 us; the arithmetic kernels evaluate the denominators on the FP64 pipe).
    if (U >= 2 && h->d_den4 && h->tab >= 0 && !h->cur_fobs && (h->tab == 1 || n_envs >= 4096)) {
        const int rc = launch_rollout_tab<ActT, FlagT>(h, U, n_envs, n_steps, pos, vel, ints, actions, reward_scale,
                                                       obs_out, reward_out, term_out, trunc_out, info_out, stream,
                                                       obs_mode);
        if (rc != 1) return rc;                              // 1: the table does not fit, fall through to k_rollout
    }
#define ARGS h, n_envs, n_steps, pos, vel, ints, actions, reward_scale, obs_out, reward_out, term_out, trunc_out, info_out, stream, obs_mode
    if (U == 6) return launch_rollout_t<ActT, FlagT, 6>(ARGS);
    if (U == 4) return launch_rollout_t<ActT, FlagT, 4>(ARGS);
    if (U == 2) return launch_rollout_t<ActT, FlagT, 2>(ARGS);
    if (U == 0) return launch_rollout_t<ActT, FlagT, 0>(ARGS);
    return launch_rollout_t<ActT, FlagT, 1>(ARGS);
#undef ARGS
}

int dispatch_rollout(void *handle, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints,
                     const void *actions, int action_dtype, double reward_scale, float *obs_out, float *reward_out,
                     void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out, void *stream,
                     int obs_mode) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0 || n_steps < 0) return fail(CARENV_E_INVAL, "negative n_envs / n_steps");
    if (n_envs == 0 || n_steps == 0) return 0;
    if (!obs_out) obs_mode = kObsNone;
    if (!pos || !vel || !ints || !actions || (!h->cur_rec && (!reward_out || !term_out || !trunc_out)))
        return fail(CARENV_E_INVAL, "null state / action / output pointer");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define CASE(A, AT, F, FT)                                                                                       \
    if (action_dtype == A && flag_dtype == F)                                                                    \
        return launch_rollout<AT, FT>(h, n_envs, n_steps, pos, vel, ints, actions, reward_scale, obs_out,       \
                                      reward_out, term_out, trunc_out, info_out, st, obs_mode);
    CASE(CARENV_ACT_U8, uint8_t, CARENV_FLAG_U8, uint8_t)
    CASE(CARENV_ACT_U8, uint8_t, CARENV_FLAG_F32, float)
    CASE(CARENV_ACT_I32, int32_t, CARENV_FLAG_U8, uint8_t)
    CASE(CARENV_ACT_I32, int32_t, CARENV_FLAG_F32, float)
    CASE(CARENV_ACT_I64, int64_t, CARENV_FLAG_U8, uint8_t)
    CASE(CARENV_ACT_I64, int64_t, CARENV_FLAG_F32, float)
#undef CASE
    return fail(CARENV_E_INVAL, "unknown action_dtype / flag_dtype");
}

}  // namespace

extern "C" {

int carenv_abi_version(void) { return CARENV_ABI_VERSION; }
const char *carenv_last_error(void) { return g_err.c_str(); }

int carenv_create(const double *walls, int n_walls, const double *gates, int n_gates, double init_x, double init_y,
                  double init_angle_deg, int device, void **handle) {
    if (!handle) return fail(CARENV_E_INVAL, "null handle pointer");
    *handle = nullptr;
    if (!walls || !gates) return fail(CARENV_E_INVAL, "null geometry pointer");
    if (n_walls < 1 || n_walls > CARENV_MAX_SEGMENTS)
        return fail(CARENV_E_TRACK, "number of wall segments must be in 1.." + std::to_string(CARENV_MAX_SEGMENTS));
    static_assert(CARENV_MAX_SEGMENTS == kMaxBigSeg, "header and kernel limits differ");
    if (n_gates < 1 || n_gates > 4000) return fail(CARENV_E_TRACK, "number of gates must be in 1..4000");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1) return fail(CARENV_E_NOGPU, "no CUDA device");
    if (device < 0 || device >= n_dev) return fail(CARENV_E_INVAL, "device index out of range");
    Handle *h = new Handle();
    h->device = device;
    h->d_blob = nullptr; h->d_stats = nullptr; h->force_generic = 0; h->max_unroll = 0; h->block = 0; h->smem_pad = 0; h->tc_tiles = 0; h->tc_stagger = -1; h->pose_rows = 0; h->warp_per_env = 0; h->hs = nullptr; h->d_den4 = nullptr; h->tab = 0; h->cur_rec = nullptr; h->cur_fobs = nullptr; h->host_ranges = 0; h->d_flags = nullptr; h->flags_cap = 0; h->tab_slice = 0;
    if (build_host_track(walls, n_walls, gates, n_gates, init_x, init_y, init_angle_deg, h->host) != 0) {
        delete h;
        return fail(CARENV_E_TRACK, "malformed track");
    }
    DeviceGuard guard(device);
    if (!guard.ok) { delete h; return fail(CARENV_E_NOGPU, "cannot select CUDA device"); }
    const size_t b_trig64 = sizeof(D2) * kHeadings, b_acc = sizeof(D2) * kHeadings;
    const size_t b_gates = sizeof(GateRec) * (size_t)n_gates, b_trig32 = 2 * sizeof(F2) * kHeadings;   // trig32 | trig32s
    const size_t b_walls = sizeof(double) * 4 * (size_t)n_walls;
    const size_t b_segf = sizeof(SegF) * (size_t)n_walls, b_segd = sizeof(SegD) * (size_t)n_walls;
    const size_t o_acc = b_trig64, o_gates = o_acc + b_acc, o_trig32 = o_gates + b_gates, o_walls = o_trig32 + b_trig32;
    const size_t o_segf = o_walls + b_walls, o_segd = o_segf + b_segf;
    const bool big = n_walls > kMaxSeg;
    // staged to shared memory: everything up to the walls, plus the segment records for big tracks
    h->smem_bytes = big ? o_segd + b_segd : o_walls + b_walls;
    if (h->smem_bytes > 200 * 1024) { delete h; return fail(CARENV_E_TRACK, "track tables do not fit in shared memory"); }
    const size_t o_den4 = (o_segd + b_segd + 15) / 16 * 16, b_den4 = sizeof(float) * h->host.den4.size();
    const size_t o_cull = o_den4 + b_den4, b_cull = sizeof(uint16_t) * h->host.cull.size();
    cudaError_t e = cudaMalloc(&h->d_blob, o_cull + b_cull + 16);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_stats, sizeof(unsigned long long) * kNumStats);
    if (e == cudaSuccess) e = cudaMemset(h->d_stats, 0, sizeof(unsigned long long) * kNumStats);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob, h->host.trig64.data(), b_trig64, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob + o_acc, h->host.acc64.data(), b_acc, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob + o_gates, h->host.gates.data(), b_gates, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob + o_trig32, h->host.trig32.data(), b_trig32 / 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob + o_trig32 + b_trig32 / 2, h->host.trig32s.data(), b_trig32 / 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && b_den4) e = cudaMemcpy(h->d_blob + o_den4, h->host.den4.data(), b_den4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && b_cull) e = cudaMemcpy(h->d_blob + o_cull, h->host.cull.data(), b_cull, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob + o_walls, h->host.walls64.data(), b_walls, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob + o_segf, h->host.segf.data(), b_segf, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_blob + o_segd, h->host.segd.data(), b_segd, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cudaFree(h->d_blob); cudaFree(h->d_stats);
        delete h;
        return cuda_fail(e, "carenv_create: device allocation / upload");
    }
    h->dev.trig64 = reinterpret_cast<const D2 *>(h->d_blob);
    h->dev.acc64 = reinterpret_cast<const D2 *>(h->d_blob + o_acc);
    h->dev.gates = reinterpret_cast<const GateRec *>(h->d_blob + o_gates);
    h->dev.trig32 = reinterpret_cast<const F2 *>(h->d_blob + o_trig32);
    h->dev.trig32s = h->dev.trig32 + kHeadings;
    h->d_den4 = b_den4 ? reinterpret_cast<const float4 *>(h->d_blob + o_den4) : nullptr;
    h->cull = h->host.cull_grid;
    h->cull.mask = b_cull ? reinterpret_cast<const uint16_t *>(h->d_blob + o_cull) : nullptr;
    h->dev.walls64 = reinterpret_cast<const double *>(h->d_blob + o_walls);
    h->dev.segf = reinterpret_cast<const SegF *>(h->d_blob + o_segf);
    h->dev.segd = reinterpret_cast<const SegD *>(h->d_blob + o_segd);
    *handle = h;
    return 0;
}

int carenv_destroy(void *handle) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return 0;
    {
        DeviceGuard guard(h->device);
        cudaFree(h->d_blob);
        cudaFree(h->d_stats);
        if (h->d_flags) cudaFree(h->d_flags);
        if (h->hs) { h->hs->release(); delete h->hs; }
    }
    delete h;
    return 0;
}

int carenv_reset_obs(void *handle, float *obs18_host) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h || !obs18_host) return fail(CARENV_E_INVAL, "null argument");
    for (int i = 0; i < kObsDim; ++i) obs18_host[i] = h->host.P.reset_obs[i];
    return 0;
}

int carenv_reset(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, float *obs_out, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0) return fail(CARENV_E_INVAL, "negative n_envs");
    if (n_envs == 0) return 0;
    if (!pos || !vel || !ints) return fail(CARENV_E_INVAL, "null state pointer");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const int grid = (n_envs + kBlock - 1) / kBlock;
    k_reset<<<grid, kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
        h->host.P, n_envs, reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel),
        reinterpret_cast<int4 *>(ints), obs_out);
    CU(cudaGetLastError());
    return 0;
}

int carenv_step(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions,
                int action_dtype, double reward_scale, float *obs_out, float *reward_out, void *term_out,
                void *trunc_out, int flag_dtype, int32_t *info_out, void *stream) {
    if (!obs_out) return fail(CARENV_E_INVAL, "carenv_step needs obs_out");
    return dispatch_rollout(handle, n_envs, 1, pos, vel, ints, actions, action_dtype, reward_scale, obs_out,
                            reward_out, term_out, trunc_out, flag_dtype, info_out, stream, kObsFull);
}

int carenv_step_final(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions,
                      int action_dtype, double reward_scale, float *obs_out, float *final_obs_out, float *reward_out,
                      void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (!obs_out || !final_obs_out) return fail(CARENV_E_INVAL, "carenv_step_final needs obs_out and final_obs_out");
    h->cur_fobs = final_obs_out;
    const int rc = dispatch_rollout(handle, n_envs, 1, pos, vel, ints, actions, action_dtype, reward_scale, obs_out,
                                    reward_out, term_out, trunc_out, flag_dtype, info_out, stream, kObsFull);
    h->cur_fobs = nullptr;
    return rc;
}

int carenv_rollout(void *handle, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints,
                   const void *actions, int action_dtype, double reward_scale, float *obs_out, float *reward_out,
                   void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out, void *stream) {
    return dispatch_rollout(handle, n_envs, n_steps, pos, vel, ints, actions, action_dtype, reward_scale, obs_out,
                            reward_out, term_out, trunc_out, flag_dtype, info_out, stream, kObsFull);
}

int carenv_rollout_poses(void *handle, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints,
                         const void *actions, int action_dtype, double reward_scale, void *pose_out, float *reward_out,
                         void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out, void *stream) {
    if (!pose_out) return fail(CARENV_E_INVAL, "carenv_rollout_poses needs pose_out");
    static_assert(sizeof(PoseRec) == CARENV_POSE_BYTES, "header and kernel disagree on the pose record");
    return dispatch_rollout(handle, n_envs, n_steps, pos, vel, ints, actions, action_dtype, reward_scale,
                            static_cast<float *>(pose_out), reward_out, term_out, trunc_out, flag_dtype, info_out,
                            stream, kObsPose);
}

int carenv_host_alloc(size_t bytes, void **ptr) {
    if (!ptr) return fail(CARENV_E_INVAL, "null pointer");
    *ptr = nullptr;
    CU(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return 0;
}

int carenv_host_free(void *ptr) {
    if (ptr) CU(cudaFreeHost(ptr));
    return 0;
}

// Shared implementation of the host-buffer steps.  `rec_host` != null: record mode (one 16-byte record per environment
// instead of the reward / flag arrays).
static int step_host_impl(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions_host,
                          int action_dtype, double reward_scale, float *obs_host, float *reward_host, void *term_host,
                          void *trunc_host, int flag_dtype, int32_t *info_host, carenv_step_record *rec_host,
                          void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0) return fail(CARENV_E_INVAL, "negative n_envs");
    if (n_envs == 0) return 0;
    if (!pos || !vel || !ints || !actions_host || !obs_host || (!rec_host && (!reward_host || !term_host || !trunc_host)))
        return fail(CARENV_E_INVAL, "null state / action / output pointer");
    if (action_dtype != CARENV_ACT_U8 && action_dtype != CARENV_ACT_I32 && action_dtype != CARENV_ACT_I64)
        return fail(CARENV_E_INVAL, "unknown action_dtype");
    if (flag_dtype != CARENV_FLAG_U8 && flag_dtype != CARENV_FLAG_F32) return fail(CARENV_E_INVAL, "unknown flag_dtype");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const int fb = flag_dtype == CARENV_FLAG_F32 ? 4 : 1;
    if (!h->hs) h->hs = new HostStep();
    HostStep &S = *h->hs;
    if (S.cap < n_envs || S.flag_bytes != fb) {               // (re)allocate the staging for this batch size
        S.release();
        const size_t n = (size_t)n_envs;
        cudaError_t e = cudaMalloc(&S.d_act, n);
        if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void **>(&S.h_act), n, cudaHostAllocDefault);
        if (e == cudaSuccess) e = cudaMalloc(&S.d_obs, n * kObsDim * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&S.d_rew, n * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&S.d_term, n * fb);
        if (e == cudaSuccess) e = cudaMalloc(&S.d_trunc, n * fb);
        if (e == cudaSuccess) e = cudaMalloc(&S.d_info, n * 4 * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc(&S.d_rec, n * sizeof(int4));
        for (int i = 0; i < HostStep::kMaxRanges && e == cudaSuccess; ++i) {
            e = cudaStreamCreateWithFlags(&S.streams[i], cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&S.done[i], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&S.ready, cudaEventDisableTiming);
        if (e != cudaSuccess) { S.release(); return cuda_fail(e, "carenv_step_host: staging allocation"); }
        S.cap = n_envs; S.flag_bytes = fb;
    }
    // Sub-ranges sized by bytes (16,384 environments = 1.4 MB of results, at most 8 ranges): the narrowing + H2D +
    // kernel of range i + 1 overlap the D2H copies of range i, which are the bottleneck (88 B per environment over
    // PCIe in record mode).  A 131,072-environment shard of an 8-GPU job gets an 8-deep pipeline, not a 2-deep one.
    // Measured at 1,048,576 envs (benchmarks/e2e_breakdown.py): 2 ranges 2.05 ms, 4: 1.84, 8: 1.82, 16: 1.85.
    int n_ranges = n_envs / 16384;
    n_ranges = n_ranges < 1 ? 1 : (n_ranges > 8 ? 8 : n_ranges);
    if (h->host_ranges > 0) n_ranges = h->host_ranges > HostStep::kMaxRanges ? HostStep::kMaxRanges : h->host_ranges;
    if (n_ranges > n_envs) n_ranges = n_envs;
    cudaStream_t user = static_cast<cudaStream_t>(stream);
    CU(cudaEventRecord(S.ready, user));                       // earlier work on the caller's stream (reset, device steps)
    // With four or more ranges the first one is split 1 : 3 (one more range): the device->host copies — the
    // bottleneck — then start after a quarter-size narrowing + H2D + kernel instead of a full-size one.
    int lo_of[HostStep::kMaxRanges + 2];
    if (n_ranges >= 4 && h->host_ranges == 0) {
        const int first = (int)((long long)n_envs / n_ranges);
        lo_of[0] = 0; lo_of[1] = first / 4;
        for (int r = 1; r <= n_ranges; ++r) lo_of[r + 1] = (int)((long long)n_envs * r / n_ranges);
        n_ranges += 1;
    } else {
        for (int r = 0; r <= n_ranges; ++r) lo_of[r] = (int)((long long)n_envs * r / n_ranges);
    }
    for (int r = 0; r < n_ranges; ++r) {
        const int lo = lo_of[r], m = lo_of[r + 1] - lo;
        if (action_dtype == CARENV_ACT_I64) {
            narrow_actions_i64(static_cast<const unsigned long long *>(actions_host) + lo, S.h_act + lo, m);
        } else if (action_dtype == CARENV_ACT_I32) {
            const uint32_t *a = static_cast<const uint32_t *>(actions_host) + lo;
            unsigned char *d = S.h_act + lo;
            for (int i = 0; i < m; ++i) { const uint32_t u = a[i]; d[i] = (unsigned char)(u < 8u ? u : 8u); }
        } else {
            memcpy(S.h_act + lo, static_cast<const unsigned char *>(actions_host) + lo, (size_t)m);
        }
        cudaStream_t st = S.streams[r];
        CU(cudaStreamWaitEvent(st, S.ready, 0));
        CU(cudaMemcpyAsync(S.d_act + lo, S.h_act + lo, (size_t)m, cudaMemcpyHostToDevice, st));
        h->cur_rec = rec_host ? reinterpret_cast<int4 *>(S.d_rec) + lo : nullptr;
        const int rc = dispatch_rollout(h, m, 1, pos + 2 * (size_t)lo, vel + 2 * (size_t)lo, ints + 4 * (size_t)lo,
                                        S.d_act + lo, CARENV_ACT_U8, reward_scale, S.d_obs + (size_t)lo * kObsDim,
                                        S.d_rew + lo, S.d_term + (size_t)lo * fb, S.d_trunc + (size_t)lo * fb, flag_dtype,
                                        info_host ? S.d_info + 4 * (size_t)lo : nullptr, st, kObsFull);
        h->cur_rec = nullptr;
        if (rc != 0) return rc;
        CU(cudaMemcpyAsync(obs_host + (size_t)lo * kObsDim, S.d_obs + (size_t)lo * kObsDim,
                           (size_t)m * kObsDim * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (rec_host) {
            CU(cudaMemcpyAsync(rec_host + lo, S.d_rec + lo, (size_t)m * sizeof(int4), cudaMemcpyDeviceToHost, st));
        } else {
            CU(cudaMemcpyAsync(reward_host + lo, S.d_rew + lo, (size_t)m * sizeof(float), cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(static_cast<unsigned char *>(term_host) + (size_t)lo * fb, S.d_term + (size_t)lo * fb,
                               (size_t)m * fb, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(static_cast<unsigned char *>(trunc_host) + (size_t)lo * fb, S.d_trunc + (size_t)lo * fb,
                               (size_t)m * fb, cudaMemcpyDeviceToHost, st));
        }
        if (info_host)
            CU(cudaMemcpyAsync(info_host + 4 * (size_t)lo, S.d_info + 4 * (size_t)lo, (size_t)m * 4 * sizeof(int32_t),
                               cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(S.done[r], st));
    }
    for (int r = 0; r < n_ranges; ++r) CU(cudaStreamWaitEvent(user, S.done[r], 0));   // later device work sees the new state
    for (int r = 0; r < n_ranges; ++r) CU(cudaEventSynchronize(S.done[r]));           // results are in the host buffers
    return 0;
}

int carenv_step_host(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions_host,
                     int action_dtype, double reward_scale, float *obs_host, float *reward_host, void *term_host,
                     void *trunc_host, int flag_dtype, int32_t *info_host, void *stream) {
    return step_host_impl(handle, n_envs, pos, vel, ints, actions_host, action_dtype, reward_scale, obs_host, reward_host,
                          term_host, trunc_host, flag_dtype, info_host, nullptr, stream);
}

int carenv_step_host_records(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions_host,
                             int action_dtype, double reward_scale, float *obs_host, carenv_step_record *rec_host,
                             int32_t *debug_info_host, void *stream) {
    if (!rec_host) return fail(CARENV_E_INVAL, "carenv_step_host_records needs rec_host");
    static_assert(sizeof(carenv_step_record) == 16, "record layout");
    return step_host_impl(handle, n_envs, pos, vel, ints, actions_host, action_dtype, reward_scale, obs_host, nullptr,
                          nullptr, nullptr, CARENV_FLAG_U8, debug_info_host, rec_host, stream);
}

int carenv_step_records(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions,
                        int action_dtype, double reward_scale, float *obs_out, carenv_step_record *rec_out,
                        int32_t *debug_info_out, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (!obs_out || !rec_out) return fail(CARENV_E_INVAL, "carenv_step_records needs obs_out and rec_out");
    h->cur_rec = reinterpret_cast<int4 *>(rec_out);
    const int rc = dispatch_rollout(handle, n_envs, 1, pos, vel, ints, actions, action_dtype, reward_scale, obs_out, nullptr,
                                    nullptr, nullptr, CARENV_FLAG_U8, debug_info_out, stream, kObsFull);
    h->cur_rec = nullptr;
    return rc;
}

int carenv_observe(void *handle, long long n, const void *poses, const long long *index, float *obs_out,
                   void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n < 0 || n > 0x7fffffffLL * 128) return fail(CARENV_E_INVAL, "bad record count");
    if (n == 0) return 0;
    if (!poses || !obs_out) return fail(CARENV_E_INVAL, "null pointer");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    int U = h->force_generic ? 1 : h->host.P.unroll4;
    if (h->host.P.n_seg > kMaxSeg) U = 0;
    const unsigned grid = (unsigned)((n + kBlock - 1) / kBlock);
    auto launch = [&](auto kern) -> int {
        if (h->smem_bytes > 48 * 1024)
            CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes));
        kern<<<grid, kBlock, h->smem_bytes, static_cast<cudaStream_t>(stream)>>>(
            h->host.P, h->dev, n, static_cast<const PoseRec *>(poses), index, obs_out);
        CU(cudaGetLastError());
        return 0;
    };
    if (U == 4) return launch(k_observe<4>);
    if (U == 2) return launch(k_observe<2>);
    if (U == 0) return launch(k_observe<0>);
    return launch(k_observe<1>);
}

#include "policy_abi.cuh"       // carenv_pack_policy, carenv_ppo_*, carenv_policy_rollout*, carenv_tc_gemm_test

/* ---- several tracks in one launch ---- */
int carenv_multi_create(void *const *handles, int n_tracks, void **multi) {
    if (!multi) return fail(CARENV_E_INVAL, "null pointer");
    *multi = nullptr;
    if (!handles || n_tracks < 1 || n_tracks > 4096) return fail(CARENV_E_INVAL, "need 1..4096 track handles");
    std::vector<TrackParams> params((size_t)n_tracks);
    std::vector<Tables> tabs((size_t)n_tracks);
    int device = -1;
    for (int i = 0; i < n_tracks; ++i) {
        const Handle *h = static_cast<const Handle *>(handles[i]);
        if (!h) return fail(CARENV_E_INVAL, "null track handle");
        if (device >= 0 && h->device != device) return fail(CARENV_E_INVAL, "all track handles must be on one device");
        device = h->device;
        params[i] = h->host.P;
        tabs[i] = h->dev;
    }
    DeviceGuard guard(device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select CUDA device");
    MultiTrack *m = new MultiTrack{n_tracks, device, nullptr, nullptr, nullptr};
    cudaError_t e = cudaMalloc(&m->d_params, sizeof(TrackParams) * n_tracks);
    if (e == cudaSuccess) e = cudaMalloc(&m->d_tables, sizeof(Tables) * n_tracks);
    if (e == cudaSuccess) e = cudaMalloc(&m->d_stats, sizeof(unsigned long long) * kNumStats);
    if (e == cudaSuccess) e = cudaMemset(m->d_stats, 0, sizeof(unsigned long long) * kNumStats);
    if (e == cudaSuccess) e = cudaMemcpy(m->d_params, params.data(), sizeof(TrackParams) * n_tracks, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(m->d_tables, tabs.data(), sizeof(Tables) * n_tracks, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cudaFree(m->d_params); cudaFree(m->d_tables); cudaFree(m->d_stats);
        delete m;
        return cuda_fail(e, "carenv_multi_create");
    }
    *multi = m;
    return 0;
}

int carenv_multi_destroy(void *multi) {
    MultiTrack *m = static_cast<MultiTrack *>(multi);
    if (!m) return 0;
    {
        DeviceGuard guard(m->device);
        cudaFree(m->d_params); cudaFree(m->d_tables); cudaFree(m->d_stats);
    }
    delete m;
    return 0;
}

int carenv_multi_reset(void *multi, int n_envs, const int32_t *track_ids, double *pos, double *vel, int32_t *ints,
                       float *obs_out, void *stream) {
    MultiTrack *m = static_cast<MultiTrack *>(multi);
    if (!m) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0) return fail(CARENV_E_INVAL, "negative n_envs");
    if (n_envs == 0) return 0;
    if (!track_ids || !pos || !vel || !ints) return fail(CARENV_E_INVAL, "null pointer");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    k_reset_multi<<<(n_envs + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
        m->d_params, m->n_tracks, track_ids, n_envs, reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel),
        reinterpret_cast<int4 *>(ints), obs_out);
    CU(cudaGetLastError());
    return 0;
}

int carenv_multi_rollout(void *multi, int n_envs, int n_steps, const int32_t *track_ids, double *pos, double *vel,
                         int32_t *ints, const void *actions, int action_dtype, double reward_scale, float *obs_out,
                         float *reward_out, void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out,
                         void *stream) {
    MultiTrack *m = static_cast<MultiTrack *>(multi);
    if (!m) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0 || n_steps < 0) return fail(CARENV_E_INVAL, "negative n_envs / n_steps");
    if (n_envs == 0 || n_steps == 0) return 0;
    if (!track_ids || !pos || !vel || !ints || !actions || !reward_out || !term_out || !trunc_out)
        return fail(CARENV_E_INVAL, "null pointer");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int grid = (n_envs + 127) / 128;
#define MCASE(A, AT, F, FT)                                                                                         \
    if (action_dtype == A && flag_dtype == F) {                                                                     \
        k_rollout_multi<AT, FT><<<grid, 128, 0, st>>>(                                                              \
            m->d_params, m->d_tables, m->n_tracks, track_ids, n_envs, n_steps, reinterpret_cast<double2 *>(pos),    \
            reinterpret_cast<double2 *>(vel), reinterpret_cast<int4 *>(ints), static_cast<const AT *>(actions),     \
            reward_scale, obs_out, reward_out, static_cast<FT *>(term_out), static_cast<FT *>(trunc_out),           \
            reinterpret_cast<int4 *>(info_out), m->d_stats);                                                        \
        CU(cudaGetLastError());                                                                                     \
        return 0;                                                                                                   \
    }
    MCASE(CARENV_ACT_U8, uint8_t, CARENV_FLAG_U8, uint8_t)
    MCASE(CARENV_ACT_U8, uint8_t, CARENV_FLAG_F32, float)
    MCASE(CARENV_ACT_I32, int32_t, CARENV_FLAG_U8, uint8_t)
    MCASE(CARENV_ACT_I32, int32_t, CARENV_FLAG_F32, float)
    MCASE(CARENV_ACT_I64, int64_t, CARENV_FLAG_U8, uint8_t)
    MCASE(CARENV_ACT_I64, int64_t, CARENV_FLAG_F32, float)
#undef MCASE
    return fail(CARENV_E_INVAL, "unknown action_dtype / flag_dtype");
}

/* ---- headless rgb_array frames ---- */
int carenv_render(void *handle, int n_outer_segments, int n_frames, const int32_t *env_index, const double *pos,
                  const int32_t *ints, const float *obs, int width, int height, unsigned char *rgb_out, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_frames < 0 || n_frames > 65535) return fail(CARENV_E_INVAL, "n_frames must be in 0..65535");
    if (n_frames == 0) return 0;
    if (width < 1 || height < 1 || (long long)width * height > (1LL << 26)) return fail(CARENV_E_INVAL, "bad frame size");
    if (!env_index || !pos || !ints || !obs || !rgb_out) return fail(CARENV_E_INVAL, "null pointer");
    if (n_outer_segments < 0 || n_outer_segments > h->host.P.n_seg) return fail(CARENV_E_INVAL, "bad n_outer_segments");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const dim3 grid((unsigned)((width * height + 255) / 256), (unsigned)n_frames);
    k_render<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        h->host.P, h->dev, n_outer_segments, n_frames, env_index, reinterpret_cast<const double2 *>(pos),
        reinterpret_cast<const int4 *>(ints), obs, width, height, rgb_out);
    CU(cudaGetLastError());
    return 0;
}

int carenv_set_option(void *handle, const char *name, int value) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h || !name) return fail(CARENV_E_INVAL, "null argument");
    if (std::string(name) == "force_generic") { h->force_generic = value ? 1 : 0; return 0; }
    if (std::string(name) == "max_unroll") { h->max_unroll = value; return 0; }
    if (std::string(name) == "block") {
        if (value < 0 || value > kBlock || value % 32) return fail(CARENV_E_INVAL, "block must be 0, 32, 64, 96 or 128");
        h->block = value; return 0;
    }
    if (std::string(name) == "pose_rows") { h->pose_rows = value ? 1 : 0; return 0; }
    if (std::string(name) == "host_ranges") { h->host_ranges = value < 0 ? 0 : value; return 0; }
    if (std::string(name) == "tab") { h->tab = value > 0 ? 1 : (value < 0 ? -1 : 0); return 0; }
    if (std::string(name) == "warp_per_env") { h->warp_per_env = value > 0 ? 1 : (value < 0 ? -1 : 0); return 0; }
    if (std::string(name) == "tc_stagger") { h->tc_stagger = value; return 0; }
    if (std::string(name) == "tab_slice") { h->tab_slice = value; return 0; }
    if (std::string(name) == "tc_tiles") {
        if (value != 0 && (value < 2 || value > 5)) return fail(CARENV_E_INVAL, "tc_tiles must be 0 or 2..5");
        h->tc_tiles = value; return 0;
    }
    if (std::string(name) == "smem_pad") {
        if (value < 0 || value > 100 * 1024) return fail(CARENV_E_INVAL, "smem_pad must be in 0..102400");
        h->smem_pad = value; return 0;
    }
    return fail(CARENV_E_INVAL, std::string("unknown option ") + name);
}

int carenv_stats(void *handle, unsigned long long out[4], int reset_counters) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h || !out) return fail(CARENV_E_INVAL, "null argument");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out, h->d_stats, sizeof(unsigned long long) * kNumStats, cudaMemcpyDeviceToHost));
    if (reset_counters) CU(cudaMemset(h->d_stats, 0, sizeof(unsigned long long) * kNumStats));
    return 0;
}

int gae_reverse_scan(const float *rew, const float *val, const float *term, const float *trunc,
                     const float *last_val, const float *last_term, const float *last_trunc, float *adv, float *ret,
                     int T, int N, double gamma, double gae_lambda, void *stream) {
    if (T < 0 || N < 0) return fail(CARENV_E_INVAL, "negative T / N");
    if (T == 0 || N == 0) return 0;
    if (!rew || !val || !term || !trunc || !last_val || !last_term || !last_trunc || !adv || !ret)
        return fail(CARENV_E_INVAL, "null pointer");
    const float g = (float)gamma;
    const float gl = (float)(gamma * gae_lambda);   // evaluated in double first (lib/buffer.py:61)
    // 64-thread blocks (1,024 blocks at N = 65,536 balance over 148 SMs better than 512 blocks of 128: 6.05 vs 5.93
    // TB/s) and one wave: when there are more columns than resident threads every thread takes k columns, so that
    // no SM idles through a partial last wave (N = 131,072: 2 columns per thread)
    const int block = 64;
    // long scans (T >= 512): unroll 8 and one wave; short, very wide ones ([128, 1 M]): one column per thread and the
    // 16-deep variant, whose per-column fill / drain is amortised by the many waves (6.07 vs 5.23 TB/s)
    const bool one_wave = T >= 512;
    const bool wide = !one_wave && N >= 100000;
    int threads = N;
    if (one_wave) {
        int dev = 0, sms = 148, per_sm = 8;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gae<8>, block, 0);
        const long long cap = (long long)(per_sm > 0 ? per_sm : 1) * sms * block;
        const int k = (int)((N + cap - 1) / cap);
        threads = (N + k - 1) / k;
    }
    const int grid = (threads + block - 1) / block;
    if (wide)
        k_gae<16><<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(rew, val, term, trunc, last_val, last_term,
                                                                       last_trunc, adv, ret, T, N, g, gl);
    else
        k_gae<8><<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(rew, val, term, trunc, last_val, last_term,
                                                                      last_trunc, adv, ret, T, N, g, gl);
    CU(cudaGetLastError());
    return 0;
}

/* Measurement helper: launches blocks x 256 threads, each doing iters * 64 FFMA (2 flop each). */
int carenv_bench_ffma(int blocks, int iters, float *scratch, void *stream) {
    if (blocks < 1 || iters < 1 || !scratch) return fail(CARENV_E_INVAL, "bad argument");
    k_ffma_peak<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(scratch, iters, 0.999f, 0.001f);
    CU(cudaGetLastError());
    return 0;
}

}  // extern "C"
