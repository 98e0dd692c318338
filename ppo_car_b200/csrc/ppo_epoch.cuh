// ppo_epoch.cuh — ALL minibatch updates of one PPO epoch in ONE persistent cooperative launch, with the gradient
// all-reduce across GPUs done inside the kernel over NVLink peer memory (SURVEY §8 f-1: the caller of the hot path,
// train.py:223-261; network lib/model.py:10-26).
//
// The three-launch update of ppo_update.cuh (k_ppo_forward / k_ppo_backward / k_ppo_adam + an NCCL all-reduce
// between two launches) costs 49 us per minibatch on one GPU, 79 us on eight, and the reference schedule has 80
// minibatches per epoch (this kernel: 10.7 / 14.7 us, profiles/r2_ppo_epoch_kernel.jsonl).  Here a
// grid of G CTAs x 256 threads stays resident for the whole epoch and walks over the updates:
//
//   phase A   CTA c owns samples [c*S, c*S + S) of the minibatch (S = ceil(B / G)); thread j owns hidden unit j of
//             BOTH nets (its W1 rows, b1 and W2 columns live in registers: 48 parameters).  Forward for the CTA's
//             samples, logits folded over the 256 threads (transposing warp butterfly + 8-way smem fold, fixed
//             order), loss terms and d loss / d logits by thread = sample, then backward: every thread accumulates
//             the gradients of ITS 48 parameters over the CTA's samples in registers and writes them as one
//             coalesced row of the partial-gradient matrix [G][12,298].
//   barrier 1 (grid)
//   phase B   CTA c owns parameter slice c (193 parameters at G = 64): sums the G partials in a fixed order; with
//             several GPUs every thread PUSHES its element into the peers' exchange buffers (IPC-mapped, NVLink) as
//             one 8-byte store {value, update number}, polls its own buffer for the peers' elements of this update
//             (low-latency protocol: no fences, no flags) and sums them in RANK order — every rank gets the same
//             bits.  Slice sum of squares -> global.
//   barrier 2 (grid)
//   phase C   global norm from the G slice sums (fixed order), clip coefficient, Adam step (torch.optim.Adam, eps
//             outside the square root as in ppo_update.cuh; hardware square root / reciprocal, see adam_quotient).  EVERY CTA keeps a full copy of the parameters (thread
//             j: the 48 of unit j in registers) and of the Adam moments (shared memory) for the whole launch and
//             applies the same step to its copy — same operations on the same reduced gradient, same bits — so
//             the next forward needs neither a parameter reload nor a third grid barrier.  CTA 0 writes the
//             parameters and moments back when the launch ends.
//
// The gathers of update u + 1 (observation rows, advantages, ...) are issued before barrier 1 of update u.
// No atomics on data, fixed summation orders: results are deterministic and identical on every rank.  Every wait is
// bounded (a missing peer sets *err and the grid drains instead of hanging the GPU).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "ppo_update.cuh"

namespace carenv {
namespace ppo {

constexpr int kEpochThreads = kH;                    // 256: thread j = hidden unit j of both nets
constexpr int kLocalK = 48;                          // parameters owned by a thread
constexpr int kLocal = kLocalK * kH + kQ + 1;        // 12,298 (= kNumParams), "local" order: e = k * 256 + j, then b2
constexpr int kLocalPad = 12320;                     // row stride of the partial-gradient matrix (multiple of 32)
constexpr int kXStride = 12416;                      // floats per exchange-buffer half
constexpr int kMaxCtas = 160;
constexpr int kMinCtas = 49;                         // a slice must fit one CTA: ceil(12,298 / G) <= 256
constexpr int kMaxWorld = 8;
static_assert(kLocal == kNumParams, "local layout is a permutation of the flat parameter layout");

// One per rank, in device memory that every peer maps (cudaIpc).  Low-latency exchange: a slot is 8 bytes — the
// float and the 32-bit sequence number of the update it belongs to — written by the peer with ONE 64-bit store and
// polled locally until the sequence number matches, so no fence and no separate flag is needed (single 8-byte
// accesses are atomic).  ll[parity][source rank][local element]; the parity double-buffers consecutive updates.
struct Exchange {
    uint2 ll[2][kMaxWorld][kXStride];
};

struct EpochArgs {
    MutableParams P;
    const float *obs;                 // [.][18]
    const long long *idx;             // [n_updates][B] rows of obs / act / ...
    const float *act, *old_logp, *adv, *ret;
    int B, n_updates;
    float clip_ratio, vf_coef, ent_coef, max_grad_norm, beta1, beta2, eps;
    float *m, *v;                     // Adam moments, flat parameter layout
    const float *lr;
    int *step;
    float *sums4;
    float *partial;                   // [gridDim.x][kLocalPad]
    float *ssq;                       // [2][kMaxCtas]
    float *stat;                      // [2][kMaxCtas] float4: slice sum of squares, policy loss, entropy, value loss partial sums; then [kLocalPad]: the reduced gradient
    unsigned int *bar;                // grid barrier counter, zero at launch
    int *err;                         // set to 1 by a wait that ran out of time
    int world, rank;
    Exchange *peer[kMaxWorld];        // peer[rank] is the local buffer
    unsigned long long seq_base;      // updates completed by earlier launches (same on every rank)
    long long *prof;                  // optional [n_updates][4] globaltimer stamps of CTA 0: start, barrier 1, 2, 3
    // k_ppo_epoch<SMAX, true> only: statistics and early stop
    double target_kl;                 // stop at the first update whose approx KL exceeds it (+inf: never)
    float *kl_out;                    // [n_updates][2] approx KL, clip fraction; NaN after the stopping update
    int *n_done;                      // updates that applied a step
    unsigned long long *seq_dev;      // world > 1: the exchanged-update count, read at launch and advanced at exit
};

// local element e -> index in the flat layout W1a b1a W2a b2a W1c b1c W2c b2c
__host__ __device__ inline int local_to_flat(int e) {
    if (e >= kLocalK * kH) { const int q = e - kLocalK * kH; return q < kQ ? kOffB2a + q : kOffB2c; }
    const int k = e / kH, j = e % kH;
    if (k < kIn) return kOffW1a + j * kIn + k;
    if (k == kIn) return kOffB1a + j;
    if (k < kIn + 1 + kQ) return kOffW2a + (k - kIn - 1) * kH + j;
    if (k < 2 * kIn + 1 + kQ) return kOffW1c + j * kIn + (k - kIn - 1 - kQ);
    if (k == 2 * kIn + 1 + kQ) return kOffB1c + j;
    return kOffW2c + j;
}

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_slot_sys(uint2 *p, uint2 v) {
    asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};\n" :: "l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ uint2 ld_slot_sys(const uint2 *p) {
    uint2 v;
    asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];\n" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_volatile_int(const int *p) {
    int v;
    asm volatile("ld.volatile.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ long long global_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
    return t;
}

constexpr long long kWaitCycles = 40000000000ll;     // ~20 s at 1.9 GHz: a wait this long means a peer is gone

// Grid-wide barrier on a monotonic counter (the launch is cooperative: all CTAs are resident).  Returns non-zero
// when the grid must drain (timeout here or an error raised elsewhere).
__device__ __forceinline__ int grid_barrier(unsigned int *bar, unsigned int &target, int *err, int *s_flag) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        atomicAdd(bar, 1u);
        const long long t0 = clock64();
        int bad = 0;
        while (ld_acquire_gpu(bar) < target) {
            if (ld_volatile_int(err) != 0) { bad = 1; break; }
            if (clock64() - t0 > kWaitCycles) { atomicExch(err, 1); bad = 1; break; }
        }
        if (!bad) bad = ld_volatile_int(err);
        *s_flag = bad;
    }
    __syncthreads();
    return *s_flag;
}

// 256-thread block sum in a fixed order (warp butterfly, then the 8 warp sums in order).
__device__ __forceinline__ float block_sum_256(float v, float *red8) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red8[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = red8[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) t += red8[w];
    return t;
}

// Transposing warp fold: every lane holds N values; afterwards the warp-wide sums are spread over the lanes, lane
// l holding fold_rem<N,16>() consecutive sums starting at fold_base<N,16>(l).  N/2 + N/4 + ... shuffles instead
// of 5 N.
template <int N, int OFF, int NMAX>
__device__ __forceinline__ void warp_fold(float (&v)[NMAX], const int lane) {
    if constexpr (OFF >= 1) {
        if constexpr (N % 2 == 0) {
            constexpr int H = N / 2;
            const bool up = (lane & OFF) != 0;
#pragma unroll
            for (int i = 0; i < H; ++i) {
                const float send = up ? v[i] : v[i + H];
                const float keep = up ? v[i + H] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);
            }
            warp_fold<H, OFF / 2, NMAX>(v, lane);
        } else {
#pragma unroll
            for (int i = 0; i < N; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], OFF);
            warp_fold<N, OFF / 2, NMAX>(v, lane);
        }
    }
}
template <int N, int OFF> __device__ __forceinline__ int fold_base(const int lane) {
    if constexpr (OFF >= 1) {
        if constexpr (N % 2 == 0) return ((lane & OFF) ? N / 2 : 0) + fold_base<N / 2, OFF / 2>(lane);
        else return fold_base<N, OFF / 2>(lane);
    } else {
        return 0;
    }
}
template <int N, int OFF> __host__ __device__ constexpr int fold_rem() {
    if constexpr (OFF >= 1) {
        if constexpr (N % 2 == 0) return fold_rem<N / 2, OFF / 2>();
        else return fold_rem<N, OFF / 2>();
    } else {
        return N;
    }
}

// num / (sqrt(v) / sqrt(bc2) + eps) with the hardware square root and reciprocal (MUFU.SQRT, MUFU.RCP: about two
// units in the last place each) instead of the IEEE-rounded sequences: every CTA applies the Adam step to ALL 12,298
// parameters, and the IEEE sqrt + divide (Newton iterations and slow-path calls) cost 9.7 us per update there against
// 0.7 us for everything else in the phase.  The denominator is at least eps = 1e-5, far from the reciprocal's edge cases.
__device__ __forceinline__ float adam_quotient(float num, float v, float inv_sqrt_bc2, float eps) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;\n" : "=f"(r) : "f"(v));
    return __fdividef(num, r * inv_sqrt_bc2 + eps);
}

constexpr int kEpochSamples = 8;                     // samples per CTA: G = max(64, ceil(B / 8)) CTAs cover B <= 1,024
constexpr int kEpochSmemBytes = 2 * kLocalK * kH * (int)sizeof(float);   // Adam moments of the 48 x 256 unit parameters
constexpr int kZ = kQ + 1;                           // 9 logits + the value per sample
constexpr int kAdvPer = kMaxBatch / kEpochThreads;   // 4 advantage values per thread (whole minibatch)

// The per-CTA arithmetic of an epoch update, shared by k_ppo_epoch and k_ppo_epoch_pop (population.cuh): thread j
// owns hidden unit j of both nets, its 48 parameters w in registers (local order: W1a row, b1a, W2a column, W1c row,
// b1c, W2c), their Adam moments in s_m / s_v ([48][256]); threads j < kZ also own second-layer bias j (s_b2, moments
// s_b2m / s_b2v).  Every helper keeps the operation order the kernels had when each held its own copy, and both
// kernels compile to the same instructions as they did then.  Two pieces are still written out in both kernels,
// because moving them into a helper changed the machine code: the per-sample loss (softmax, clipped surrogate,
// d loss / d logits: 1 to 130 instructions of each of the four instantiations; shared with k_ppo_forward as well, 1,223
// of its instructions and 4 more registers) and the Adam step of phase C (about 1,000 instructions of each, 16 more
// registers in k_ppo_epoch<8, false>; read from the argument struct inside the helper, 31 and 26 in k_ppo_epoch).

// parameters and moments of unit j (and bias j) from the flat layout of P, m, v
__device__ __forceinline__ void stage_unit(const MutableParams &P, const float *m, const float *v, const int j,
                                           float (&w)[kLocalK], float *s_m, float *s_v, float (&s_b2)[kZ],
                                           float (&s_b2m)[kZ], float (&s_b2v)[kZ]) {
#pragma unroll
    for (int k = 0; k < kLocalK; ++k) {
        const int f = local_to_flat(k * kH + j);
        w[k] = *param_ptr(P, f);
        s_m[k * kH + j] = m[f];
        s_v[k * kH + j] = v[f];
    }
    if (j < kZ) {
        const int f = local_to_flat(kLocalK * kH + j);
        s_b2[j] = *param_ptr(P, f); s_b2m[j] = m[f]; s_b2v[j] = v[f];
    }
}

// the inverse of stage_unit
__device__ __forceinline__ void write_back_unit(const MutableParams &P, float *m, float *v, const int j,
                                                const float (&w)[kLocalK], const float *s_m, const float *s_v,
                                                const float (&s_b2)[kZ], const float (&s_b2m)[kZ],
                                                const float (&s_b2v)[kZ]) {
#pragma unroll
    for (int k = 0; k < kLocalK; ++k) {
        const int f = local_to_flat(k * kH + j);
        *param_ptr(P, f) = w[k];
        m[f] = s_m[k * kH + j];
        v[f] = s_v[k * kH + j];
    }
    if (j < kZ) {
        const int f = local_to_flat(kLocalK * kH + j);
        *param_ptr(P, f) = s_b2[j]; m[f] = s_b2m[j]; v[f] = s_b2v[j];
    }
}

// advantage mean and 1 / max(std, 1e-5) of the whole minibatch (train.py:236-237, unbiased std) from the values
// thread j holds (element j + i * 256): the same bits in every CTA
__device__ __forceinline__ void advantage_stats(const float (&al)[kAdvPer], const int j, const int B, const float invB,
                                                float *red8, float &a_mean, float &a_inv) {
    float sum = 0.0f;
#pragma unroll
    for (int i = 0; i < kAdvPer; ++i) sum += al[i];
    a_mean = block_sum_256(sum, red8) * invB;
    float s2 = 0.0f;
#pragma unroll
    for (int i = 0; i < kAdvPer; ++i) {
        const float d = j + i * kEpochThreads < B ? al[i] - a_mean : 0.0f;
        s2 += d * d;
    }
    const float var = block_sum_256(s2, red8) / (float)(B > 1 ? B - 1 : 1);
    a_inv = 1.0f / fmaxf(sqrtf(var), 1.0e-5f);
}

__device__ __forceinline__ void load_row(const float (&row)[20], float (&x)[20]) {
    const float4 *xv = reinterpret_cast<const float4 *>(row);
#pragma unroll
    for (int i = 0; i < 5; ++i) { const float4 t = xv[i]; x[4 * i] = t.x; x[4 * i + 1] = t.y; x[4 * i + 2] = t.z; x[4 * i + 3] = t.w; }
}

// Forward of unit j for the SMAX observation rows of s_x (rows s >= n count as absent): pre-activations of both nets,
// then the second-layer products folded over the 256 threads (transposing warp butterfly + 8-way smem fold, fixed
// order) into s_z[s] = 9 logits | value, second-layer biases not added.  Ends with the block synchronised.
template <int SMAX>
__device__ __forceinline__ void unit_forward(const float (&w)[kLocalK], const float (&s_x)[SMAX][20], const int n,
                                             const int j, const int lane, const int warp, float (&pre_a)[SMAX], float (&pre_c)[SMAX],
                                             float (&s_red)[8][kZ * SMAX], float (&s_z)[SMAX][12]) {
    constexpr int kFold = kZ * SMAX;
    {
        float contrib[kFold];
#pragma unroll
        for (int s = 0; s < SMAX; ++s) {
            float x[20];
            load_row(s_x[s], x);
            float pa = w[kIn], pb = 0.0f, pc = 0.0f, qa = w[2 * kIn + 1 + kQ], qb = 0.0f, qc = 0.0f;   // ppo_update.cuh's order
#pragma unroll
            for (int k = 0; k < kIn; k += 3) {
                pa = fmaf(w[k], x[k], pa); pb = fmaf(w[k + 1], x[k + 1], pb); pc = fmaf(w[k + 2], x[k + 2], pc);
                qa = fmaf(w[kIn + 1 + kQ + k], x[k], qa); qb = fmaf(w[kIn + 2 + kQ + k], x[k + 1], qb);
                qc = fmaf(w[kIn + 3 + kQ + k], x[k + 2], qc);
            }
            const bool on = s < n;
            pre_a[s] = on ? (pa + pb) + pc : 0.0f;
            pre_c[s] = on ? (qa + qb) + qc : 0.0f;
            const float ha = fmaxf(pre_a[s], 0.0f), hc = fmaxf(pre_c[s], 0.0f);
#pragma unroll
            for (int q = 0; q < kQ; ++q) contrib[s * kZ + q] = w[kIn + 1 + q] * ha;
            contrib[s * kZ + kQ] = w[kLocalK - 1] * hc;
        }
        warp_fold<kFold, 16, kFold>(contrib, lane);
        constexpr int kRem = fold_rem<kFold, 16>();
        const int base = fold_base<kFold, 16>(lane);
#pragma unroll
        for (int i = 0; i < kRem; ++i) s_red[warp][base + i] = contrib[i];   // lanes holding copies write the same bits
    }
    __syncthreads();
    if (j < kFold) {
        float t = s_red[0][j];
#pragma unroll
        for (int w8 = 1; w8 < 8; ++w8) t += s_red[w8][j];
        s_z[j / kZ][j % kZ] = t;
    }
    __syncthreads();
}

// Backward of unit j over the SMAX rows: adds to g the gradients of its 48 parameters, given s_z[s] = d loss / d logits
// | d loss / d value and unit_forward's pre-activations
template <int SMAX>
__device__ __forceinline__ void unit_backward(const float (&w)[kLocalK], const float (&s_x)[SMAX][20],
                                              const float (&s_z)[SMAX][12], const float (&pre_a)[SMAX],
                                              const float (&pre_c)[SMAX], float (&g)[kLocalK]) {
#pragma unroll
    for (int s = 0; s < SMAX; ++s) {
        float x[20];
        load_row(s_x[s], x);
        const float4 *zv = reinterpret_cast<const float4 *>(s_z[s]);
        const float4 d0 = zv[0], d1 = zv[1], d2 = zv[2];
        const float dz[kQ] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w, d2.x};
        const float dv = d2.y;
        const float ha = fmaxf(pre_a[s], 0.0f), hc = fmaxf(pre_c[s], 0.0f);
        float dh = 0.0f;
#pragma unroll
        for (int q = 0; q < kQ; ++q) { g[kIn + 1 + q] = fmaf(dz[q], ha, g[kIn + 1 + q]); dh = fmaf(dz[q], w[kIn + 1 + q], dh); }
        dh = pre_a[s] > 0.0f ? dh : 0.0f;                        // ReLU'(pre), zero at pre == 0 like torch
        const float dc = pre_c[s] > 0.0f ? dv * w[kLocalK - 1] : 0.0f;
        g[kLocalK - 1] = fmaf(dv, hc, g[kLocalK - 1]);
#pragma unroll
        for (int k = 0; k < kIn; ++k) {
            g[k] = fmaf(dh, x[k], g[k]);
            g[kIn + 1 + kQ + k] = fmaf(dc, x[k], g[kIn + 1 + kQ + k]);
        }
        g[kIn] += dh;
        g[2 * kIn + 1 + kQ] += dc;
    }
}

// Adam bias corrections of step t: s_bias = {lr / (1 - beta1^t), 1 / sqrt(1 - beta2^t)}.  powf is ~150 instructions,
// so one thread forms them while a barrier is pending.
__device__ __forceinline__ void adam_bias_corrections(float (&s_bias)[2], const int t, const float lr,
                                                      const float beta1, const float beta2) {
    const float bc1 = 1.0f - powf(beta1, (float)t), bc2 = 1.0f - powf(beta2, (float)t);
    s_bias[0] = lr / bc1; s_bias[1] = rsqrtf(bc2);
}

// KL = true adds the PPO diagnostics and the early stop (carenv_ppo_epoch_kl): phase A also sums each sample's
// (ratio - 1) - log ratio and |ratio - 1| > clip_ratio; the two CTA sums ride in the partial-gradient row at columns
// kLocal, kLocal + 1 and are reduced (over the CTAs, then the ranks) by two extra threads of CTA 0 in phase B, outside
// the slice sum of squares, so the parameter arithmetic keeps its bits.  Phase C divides them by the sample count,
// CTA 0 records them, and when the KL exceeds target_kl every CTA of every rank (the totals are the same bits
// everywhere) skips that update's step and leaves the loop.  With several GPUs the exchange sequence base lives in
// device memory (seq_dev), because only the device knows how many updates a launch exchanged.
template <int SMAX, bool KL = false>
__global__ void __launch_bounds__(kEpochThreads, 1) k_ppo_epoch(const EpochArgs A) {
    static_assert(SMAX * kIn <= kEpochThreads, "one thread per staged observation element");
    constexpr int kParts = KL ? 5 : 3;                  // policy loss, entropy, value loss (, KL term, clipped)
    extern __shared__ __align__(16) float s_dyn[];       // m [48][256] | v [48][256]: this CTA's copy of the Adam moments
    float *const s_m = s_dyn, *const s_v = s_dyn + kLocalK * kH;
    __shared__ __align__(16) float s_x[SMAX][20];        // observation rows of the CTA's samples
    __shared__ float s_red[8][kZ * SMAX];                // per-warp sums of the second layer
    __shared__ __align__(16) float s_z[SMAX][12];        // logits | value, then d loss / d logits | d loss / d value
    __shared__ float s_part[SMAX][kParts];               // per-sample policy loss, entropy, value loss
    __shared__ float s_red8[8];
    __shared__ float4 s_fold[8];
    __shared__ float s_bias[2];
    __shared__ float s_b2[kZ], s_b2m[kZ], s_b2v[kZ];     // second-layer biases (b2a[0..8], b2c) and their moments
    __shared__ int s_flag;

    const int j = threadIdx.x, lane = j & 31, warp = j >> 5;
    const int c = blockIdx.x, G = gridDim.x;
    const int B = A.B;
    const int S = (B + G - 1) / G;                       // samples per CTA (<= SMAX, checked by the launcher)
    const int s0 = c * S;
    const int nS = max(0, min(S, B - s0));
    const int slice = (kLocal + G - 1) / G;              // parameters per CTA in phase B (<= 256)
    const int e_mine = c * slice + j;
    const bool own = j < slice && e_mine < kLocal;
    // KL: threads slice, slice + 1 of CTA 0 (slice <= 251, so they exist) reduce the two statistic sums, elements
    // kLocal and kLocal + 1; own_b / e_b are phase B's owner and element, own alone feeds the sum of squares
    const bool own_b = KL ? own || (c == 0 && j >= slice && j < slice + 2) : own;
    const int e_b = KL ? (own ? e_mine : kLocal + j - slice) : e_mine;
    const float invB = 1.0f / (float)B;
    const int step0 = *A.step;
    const float lr = A.lr[0];
    float *const gfull = A.ssq + 2 * kMaxCtas + 8 * kMaxCtas;       // [kLocalPad] reduced gradient (workspace tail)
    unsigned int bar_target = 0;
    // KL with several GPUs: the sequence base comes from the device (A.seq_base is read in place otherwise: a copy
    // would change k_ppo_epoch<8>'s machine code)
    unsigned long long seq_kl = 0;
    if constexpr (KL) seq_kl = A.world > 1 ? *A.seq_dev : A.seq_base;
    int n_run = A.n_updates;                             // KL: updates that applied a step
    int n_eval = A.n_updates;                            // KL: updates whose statistics were formed (and exchanged)

    // ---- every CTA keeps ALL parameters and Adam moments for the whole launch: thread j the 48 of hidden unit j
    // (parameters in registers, moments in shared memory), threads 0..9 the second-layer biases.  Every CTA applies
    // the same Adam step to its copy (same operations on the same reduced gradient: same bits), so the next forward
    // needs neither a reload nor a third grid barrier; CTA 0 writes the result back at the end.
    float w[kLocalK];
    stage_unit(A.P, A.m, A.v, j, w, s_m, s_v, s_b2, s_b2m, s_b2v);
    for (int i = j; i < SMAX * 20; i += kEpochThreads) (&s_x[0][0])[i] = 0.0f;   // rows >= nS and the padding stay zero

    // ---- gathers of the next update are issued before the grid barriers and land while the CTA waits
    float x_pf = 0.0f, al_pf[kAdvPer], l_act = 0.0f, l_olp = 0.0f, l_adv = 0.0f, l_ret = 0.0f;
    auto prefetch = [&](int u2) {
        const long long *idx = A.idx + (size_t)u2 * (size_t)B;
        if (j < nS * kIn) x_pf = A.obs[(size_t)idx[s0 + j / kIn] * kIn + j % kIn];
#pragma unroll
        for (int i = 0; i < kAdvPer; ++i) {
            const int t = j + i * kEpochThreads;
            al_pf[i] = t < B ? A.adv[idx[t]] : 0.0f;
        }
        if (j < nS) {
            const long long row = idx[s0 + j];
            l_act = A.act[row]; l_olp = A.old_logp[row]; l_adv = A.adv[row]; l_ret = A.ret[row];
        }
    };
    prefetch(0);
    __syncthreads();

    for (int u = 0; u < A.n_updates; ++u) {
        const bool stamp = A.prof != nullptr && c == 0 && j == 0;
        if (stamp) A.prof[4 * u] = global_ns();
        const int par = (int)(((KL ? seq_kl : A.seq_base) + (unsigned long long)u) & 1ull);     // continues across launches (odd n_updates)

        // ---- this CTA's observation rows
        if (j < nS * kIn) s_x[j / kIn][j % kIn] = x_pf;

        // ---- advantage statistics of the whole minibatch (train.py:236-237), the same bits in every CTA
        float a_mean, a_inv;
        advantage_stats(al_pf, j, B, invB, s_red8, a_mean, a_inv);
        __syncthreads();                                              // s_x complete

        // ---- forward: pre-activations of unit j for the CTA's samples, second-layer products
        float pre_a[SMAX], pre_c[SMAX];
        unit_forward(w, s_x, nS, j, lane, warp, pre_a, pre_c, s_red, s_z);

        // ---- loss terms and their derivatives, thread = sample (ppo_update.cuh: k_ppo_forward)
        if (j < SMAX) {
            float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f;
            if (j < nS) {
                float z[kQ];
                float mx = -1.0e30f;
#pragma unroll
                for (int q = 0; q < kQ; ++q) { z[q] = s_z[j][q] + s_b2[q]; mx = fmaxf(mx, z[q]); }
                float ex[kQ], se = 0.0f;
#pragma unroll
                for (int q = 0; q < kQ; ++q) { ex[q] = expf(z[q] - mx); se += ex[q]; }
                const float lse = logf(se);
                float H = 0.0f, p[kQ], lp[kQ];
#pragma unroll
                for (int q = 0; q < kQ; ++q) { lp[q] = (z[q] - mx) - lse; p[q] = expf(lp[q]); H -= p[q] * lp[q]; }
                const int a = (int)l_act;
                float new_lp = lp[0];
#pragma unroll
                for (int q = 1; q < kQ; ++q) new_lp = (a == q) ? lp[q] : new_lp;
                const float ratio = expf(new_lp - l_olp);
                const float an = (l_adv - a_mean) * a_inv;
                const float lo = 1.0f - A.clip_ratio, hi = 1.0f + A.clip_ratio;
                const float t1 = -an * ratio, t2 = -an * fminf(fmaxf(ratio, lo), hi);
                const bool inside = ratio >= lo && ratio <= hi;
                const float g_ratio = (inside || t1 > t2) ? -an : 0.0f;     // torch.max / clamp subgradients
                const float g_lp = g_ratio * ratio * invB;
                const float val = s_z[j][kQ] + s_b2[kQ];
                const float d = val - l_ret;
#pragma unroll
                for (int q = 0; q < kQ; ++q)
                    s_z[j][q] = g_lp * ((a == q ? 1.0f : 0.0f) - p[q]) + A.ent_coef * invB * p[q] * (lp[q] + H);
                s_z[j][kQ] = A.vf_coef * d * invB;
                p0 = fmaxf(t1, t2); p1 = H; p2 = 0.5f * d * d;
                if constexpr (KL) {
                    const float log_r = new_lp - l_olp;
                    s_part[j][3] = (ratio - 1.0f) - log_r;
                    s_part[j][4] = fabsf(ratio - 1.0f) > A.clip_ratio ? 1.0f : 0.0f;
                }
            } else {
#pragma unroll
                for (int q = 0; q < kZ; ++q) s_z[j][q] = 0.0f;
                if constexpr (KL) { s_part[j][3] = 0.0f; s_part[j][4] = 0.0f; }
            }
            s_part[j][0] = p0; s_part[j][1] = p1; s_part[j][2] = p2;
        }
        __syncthreads();

        // ---- backward: gradients of the 48 parameters of unit j over the CTA's samples
        {
            float g[kLocalK];
#pragma unroll
            for (int k = 0; k < kLocalK; ++k) g[k] = 0.0f;
            unit_backward(w, s_x, s_z, pre_a, pre_c, g);
            float *row = A.partial + (size_t)c * kLocalPad;
#pragma unroll
            for (int k = 0; k < kLocalK; ++k) __stcg(row + k * kH + j, g[k]);
            if (j < kZ) {                                            // second-layer biases: sum of dz over the samples
                float t = 0.0f;
#pragma unroll
                for (int s = 0; s < SMAX; ++s) t += s_z[s][j];
                __stcg(row + kLocalK * kH + j, t);
            }
            if constexpr (KL) {                                      // the CTA's KL and clip sums, sample order
                if (j == kZ) {
                    float tk = 0.0f, tc = 0.0f;
#pragma unroll
                    for (int s = 0; s < SMAX; ++s) { tk += s_part[s][3]; tc += s_part[s][4]; }
                    __stcg(row + kLocal, tk);
                    __stcg(row + kLocal + 1, tc);
                }
            }
        }
        if (u + 1 < A.n_updates) prefetch(u + 1);
        if (grid_barrier(A.bar, bar_target, A.err, &s_flag)) return;
        if (stamp) A.prof[4 * u + 1] = global_ns();

        // ---- phase B: slice c of the gradient, summed over the CTAs (and over the GPUs)
        float gsum = 0.0f;
        if (own_b) {
            const float *col = A.partial + e_b;
            constexpr int kInFlight = 32;
            float t[kInFlight];
            for (int c2 = 0; c2 < G; c2 += kInFlight) {              // 32 loads in flight, summed in CTA order
#pragma unroll
                for (int i = 0; i < kInFlight; ++i) t[i] = c2 + i < G ? __ldcg(col + (size_t)(c2 + i) * kLocalPad) : 0.0f;
#pragma unroll
                for (int i = 0; i < kInFlight; ++i) gsum += t[i];
            }
        }
        if (A.world > 1 && own_b) {
            // push this rank's value of the element to every peer, then collect theirs: one-way NVLink latency
            const unsigned int seq = (unsigned int)((KL ? seq_kl : A.seq_base) + (unsigned long long)u + 1ull);
            const uint2 mine = make_uint2(__float_as_uint(gsum), seq);
            float val[kMaxWorld];
            unsigned int pending = 0;
#pragma unroll
            for (int r = 0; r < kMaxWorld; ++r) {
                val[r] = 0.0f;
                if (r < A.world && r != A.rank) {
                    st_slot_sys(&A.peer[r]->ll[par][A.rank][e_b], mine);
                    pending |= 1u << r;
                }
            }
            const Exchange *me = A.peer[A.rank];
            const long long t0 = clock64();
            int spins = 0;
            while (pending) {
                uint2 got[kMaxWorld];
#pragma unroll
                for (int r = 0; r < kMaxWorld; ++r)
                    if (pending & (1u << r)) got[r] = ld_slot_sys(&me->ll[par][r][e_b]);
#pragma unroll
                for (int r = 0; r < kMaxWorld; ++r)
                    if ((pending & (1u << r)) && got[r].y == seq) { val[r] = __uint_as_float(got[r].x); pending &= ~(1u << r); }
                if (pending && (++spins & 1023) == 0) {
                    if (ld_volatile_int(A.err) != 0) break;
                    if (clock64() - t0 > kWaitCycles) { atomicExch(A.err, 1); break; }
                }
            }
            float t = 0.0f;
#pragma unroll
            for (int r = 0; r < kMaxWorld; ++r)                       // rank order: the same bits on every rank
                if (r < A.world) t += (r == A.rank) ? gsum : val[r];
            gsum = t * (1.0f / (float)A.world);
        }
        if (own_b) __stcg(gfull + e_b, gsum);
        {   // this CTA's line of the norm / statistics table: slice sum of squares, loss partial sums of its samples
            const float ss = block_sum_256(own ? gsum * gsum : 0.0f, s_red8);
            if (j == 0) {
                float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f;
#pragma unroll
                for (int s = 0; s < SMAX; ++s) { p0 += s_part[s][0]; p1 += s_part[s][1]; p2 += s_part[s][2]; }
                __stcg(reinterpret_cast<float4 *>(A.stat) + par * kMaxCtas + c, make_float4(ss, p0, p1, p2));
            }
        }
        if (j == 64) adam_bias_corrections(s_bias, step0 + u + 1, lr, A.beta1, A.beta2);
        if (grid_barrier(A.bar, bar_target, A.err, &s_flag)) return;
        const float step_size = s_bias[0], inv_sqrt_bc2 = s_bias[1];
        if (stamp) A.prof[4 * u + 2] = global_ns();

        // ---- phase C: clip_grad_norm_ + Adam on this CTA's copy of every parameter, statistics
        {
            float g[kLocalK];
#pragma unroll
            for (int k = 0; k < kLocalK; ++k) g[k] = __ldcg(gfull + k * kH + j);
            const float gb = j < kZ ? __ldcg(gfull + kLocalK * kH + j) : 0.0f;
            const float4 line = j < G ? __ldcg(reinterpret_cast<const float4 *>(A.stat) + par * kMaxCtas + j)
                                      : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            float4 tot = line;                                        // fixed-order fold over the CTAs' lines
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                tot.x += __shfl_xor_sync(0xffffffffu, tot.x, o); tot.y += __shfl_xor_sync(0xffffffffu, tot.y, o);
                tot.z += __shfl_xor_sync(0xffffffffu, tot.z, o); tot.w += __shfl_xor_sync(0xffffffffu, tot.w, o);
            }
            __syncthreads();
            if (lane == 0) s_fold[warp] = tot;
            __syncthreads();
            tot = s_fold[0];
#pragma unroll
            for (int w8 = 1; w8 < 8; ++w8) { const float4 o = s_fold[w8]; tot.x += o.x; tot.y += o.y; tot.z += o.z; tot.w += o.w; }
            if constexpr (KL) {                                       // same bits in every CTA and on every rank
                const float kl = __ldcg(gfull + kLocal) * invB, clip_frac = __ldcg(gfull + kLocal + 1) * invB;
                if (c == 0 && j == 0) { A.kl_out[2 * u] = kl; A.kl_out[2 * u + 1] = clip_frac; }
                if ((double)kl > A.target_kl) { n_run = u; n_eval = u + 1; break; }
            }
            const float coef = fminf(A.max_grad_norm / (sqrtf(tot.x) + 1.0e-6f), 1.0f);    // clip_grad_norm_
#ifdef CARENV_EPOCH_PROF2
            if (stamp) A.prof[4 * A.n_updates + 4 * u] = global_ns();
#endif
            if (c == 0 && j == 0) {
                const float pol = tot.y * invB, ent = tot.z * invB, vl = tot.w * invB;
                A.sums4[0] += pol; A.sums4[1] += vl; A.sums4[2] += ent; A.sums4[3] += pol + A.vf_coef * vl - A.ent_coef * ent;
            }
            // eight parameters at a time with the moments staged in registers: the shared-memory stores of one
            // parameter must not serialise the (long: sqrt, divide) dependent chain of the next
#pragma unroll
            for (int k0 = 0; k0 < kLocalK; k0 += 8) {
                float mm[8], vv[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { mm[i] = s_m[(k0 + i) * kH + j]; vv[i] = s_v[(k0 + i) * kH + j]; }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float gc = g[k0 + i] * coef;
                    mm[i] = A.beta1 * mm[i] + (1.0f - A.beta1) * gc;
                    vv[i] = A.beta2 * vv[i] + (1.0f - A.beta2) * gc * gc;
                    w[k0 + i] = w[k0 + i] - adam_quotient(step_size * mm[i], vv[i], inv_sqrt_bc2, A.eps);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) { s_m[(k0 + i) * kH + j] = mm[i]; s_v[(k0 + i) * kH + j] = vv[i]; }
            }
#ifdef CARENV_EPOCH_PROF2
            if (stamp) A.prof[4 * A.n_updates + 4 * u + 1] = global_ns();
#endif
            if (j < kZ) {
                const float gc = gb * coef;
                const float mi = A.beta1 * s_b2m[j] + (1.0f - A.beta1) * gc;
                const float vi = A.beta2 * s_b2v[j] + (1.0f - A.beta2) * gc * gc;
                s_b2m[j] = mi; s_b2v[j] = vi;
                s_b2[j] = s_b2[j] - adam_quotient(step_size * mi, vi, inv_sqrt_bc2, A.eps);
            }
        }
        __syncthreads();                                              // s_b2 before the next loss pass
        if (stamp) A.prof[4 * u + 3] = global_ns();
    }
    // ---- write the parameters and moments back (every CTA holds the same bits; CTA 0 writes)
    if (c == 0) {
        write_back_unit(A.P, A.m, A.v, j, w, s_m, s_v, s_b2, s_b2m, s_b2v);
        if constexpr (KL) {
            for (int i = 2 * n_eval + j; i < 2 * A.n_updates; i += kEpochThreads) A.kl_out[i] = __int_as_float(0x7fc00000);
            if (j == 0) {
                *A.step = step0 + n_run;
                *A.n_done = n_run;
                if (A.world > 1) *A.seq_dev = seq_kl + (unsigned long long)n_eval;
            }
        } else {
            if (j == 0) *A.step = step0 + A.n_updates;
        }
    }
}

}  // namespace ppo
}  // namespace carenv
