// population.cuh — P independent PPO training runs ("members") advanced together: the member-batched forms of the
// fused rollouts and of the policy packing (C ABI carenv_*_pop over the POP instantiations of policy_rollout.cuh) and
// the population epoch update k_ppo_epoch_pop below.  Members never exchange data: member p owns its parameters,
// Adam moments, step count, hyperparameters, seed and n environments, which are columns p * n .. p * n + n - 1 of
// every [N] and [T, N] array (N = P * n).
//
// Textually included at the end of policy_abi.cuh, i.e. inside the extern "C" block of carenv_kernels.cu; the kernel
// sits in an extern "C++" block of the anonymous namespace, as in policy_eval.cuh.
//
// k_ppo_epoch_pop: all n_updates minibatch updates of an epoch for all P members in ONE ordinary cluster launch.
// Member p is one thread-block cluster of kPopCluster CTAs x 256 threads (grid P x kPopCluster); clusters never wait
// for each other, so P may exceed the number of co-resident clusters.  Inside a cluster the plan and the arithmetic are
// k_ppo_epoch's, with the grid replaced by the cluster.  The two kernels share one copy of the parameter staging and
// write-back, the advantage statistics, the forward with its warp fold, the backward and the Adam bias corrections
// (the helpers in ppo_epoch.cuh); the per-sample loss and the Adam step are still written out in both, since moving
// them into helpers changed the machine code (ppo_epoch.cuh says by how much):
//
//   phase A   thread j owns hidden unit j's 48 parameters in registers; CTA r takes samples [r*S, r*S + S) of the
//             member's minibatch (S = ceil(B / kPopCluster)) in chunks of kEpochSamples and accumulates its partial
//             gradient (one fma chain per parameter over all its samples) in ITS OWN shared memory.  The advantage
//             mean and standard deviation are computed redundantly over the whole minibatch by every CTA.
//   barrier   barrier.cluster.arrive.release / wait.acquire
//   phase B   CTA r sums slice r of the kPopCluster partials through distributed shared memory (mapa +
//             ld.shared::cluster) in rank order, keeps the reduced slice in its shared memory, and the slice's sum
//             of squares and its loss partial sums in one float4.
//   barrier
//   phase C   every CTA reads the reduced slices and the kPopCluster float4 lines over DSMEM in a fixed order, computes
//             the clip coefficient and applies the same Adam step to its full copy (moments in shared memory), so all
//             CTAs of the cluster hold the same bits.  CTA 0 writes parameters and moments back at the end.
//
// Two full cluster barriers per update leave nothing to double-buffer: a CTA rewrites its partial (phase A of update
// u + 1) only after barrier 2 of update u, which every peer reaches after its last phase-B read of it, and rewrites its
// reduced slice (phase B of u + 1) only after barrier 1 of u + 1, which every peer reaches after its phase-C reads of
// update u.  One more barrier before exit keeps a CTA's shared memory alive until its peers' last reads.
//
// The reduction order differs from k_ppo_epoch's (kPopCluster partials of S samples instead of G of 8), so results are
// not bit-identical to it; they are deterministic and do not depend on the other members or on the launch's P.
#pragma once

#ifndef CARENV_POP_CLUSTER
#define CARENV_POP_CLUSTER 8
#endif

extern "C++" {
namespace {

constexpr int kPopCluster = CARENV_POP_CLUSTER;   // CTAs per member: a compile-time constant, the bits depend on it
static_assert(kPopCluster >= 2 && kPopCluster <= 16, "cluster size 2..16");
constexpr int kPopSlice = (ppo::kLocal + kPopCluster - 1) / kPopCluster;           // parameters reduced by one CTA
constexpr int kPopSlicePer = (kPopSlice + ppo::kEpochThreads - 1) / ppo::kEpochThreads;
constexpr int kPopSliceFloats = (kPopSlice + 3) / 4 * 4;
// dynamic shared memory: m [48][256] | v [48][256] | partial gradient [kLocalPad] | reduced slice [kPopSliceFloats]
constexpr int kPopSmemBytes = (2 * ppo::kLocalK * ppo::kH + ppo::kLocalPad + kPopSliceFloats) * (int)sizeof(float);
static_assert(kPopSmemBytes + 8 * 1024 <= 227 * 1024, "shared memory of the population update");

struct PopEpochArgs {
    ppo::MutableParams P;             // stacked [P][...] parameters (member 0's addresses)
    const float *obs;                 // [.][18]
    const long long *idx;             // [P][n_updates][B] rows of obs / act / ...
    const float *act, *old_logp, *adv, *ret;
    int B, n_updates;
    const float *lr, *clip_ratio, *vf_coef, *ent_coef, *max_grad_norm;   // [P] each
    float beta1, beta2, eps;
    float *m, *v;                     // [P][12,298] Adam moments, flat parameter layout
    int *step;                        // [P]
    float *sums4;                     // [P][4]
    // k_ppo_epoch_pop<true> only: statistics and early stop, per member
    double target_kl;                 // a member stops at its first update whose approx KL exceeds it (+inf: never)
    float *kl_out;                    // [P][n_updates][2] approx KL, clip fraction; NaN after the stopping update
    int *n_done;                      // [P] updates that applied a step
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t dsmem_map(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ float dsmem_ld(uint32_t addr) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];\n" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ float4 dsmem_ld4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];\n"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// KL = true: k_ppo_epoch<8, true>'s statistics and stop rule per member (carenv_ppo_epoch_pop_kl).  Each CTA's KL and
// clip sums form a second float4 of its stats line, read over DSMEM and folded in the same fixed order as the first,
// so every CTA of the cluster sees the same totals, takes the same exit and still reaches the final cluster barrier.
template <bool KL = false>
__global__ void __launch_bounds__(ppo::kEpochThreads, 1) k_ppo_epoch_pop(const PopEpochArgs A) {
    using namespace ppo;
    constexpr int SMAX = kEpochSamples;
    constexpr int kParts = KL ? 5 : 3;                   // policy loss, entropy, value loss (, KL term, clipped)
    static_assert(SMAX * kIn <= kEpochThreads, "one thread per staged observation element");
    extern __shared__ __align__(16) float s_dyn[];
    float *const s_m = s_dyn, *const s_v = s_dyn + kLocalK * kH;
    float *const s_g = s_v + kLocalK * kH;               // this CTA's partial gradient, local order
    float *const s_slice = s_g + kLocalPad;              // reduced slice r of the gradient
    __shared__ __align__(16) float s_x[SMAX][20];
    __shared__ float s_red[8][kZ * SMAX];
    __shared__ __align__(16) float s_z[SMAX][12];
    __shared__ float s_part[SMAX][kParts];
    __shared__ float s_red8[8];
    __shared__ __align__(16) float4 s_line;              // slice sum of squares, loss partial sums of the CTA's samples
    __shared__ float4 s_tot;
    __shared__ __align__(16) float4 s_line_kl;           // KL: KL and clip sums of the CTA's samples
    __shared__ float2 s_tot_kl;
    __shared__ float s_bias[2];
    __shared__ float s_b2[kZ], s_b2m[kZ], s_b2v[kZ];

    const int j = threadIdx.x, lane = j & 31, warp = j >> 5;
    const int r = (int)cluster_ctarank();
    const int p = blockIdx.x / kPopCluster;
    const int B = A.B;
    const int S = (B + kPopCluster - 1) / kPopCluster;
    const int s0 = r * S;
    const int nS = max(0, min(S, B - s0));
    const int n_chunks = max(1, (nS + SMAX - 1) / SMAX);
    const float invB = 1.0f / (float)B;
    const size_t pq = (size_t)p;
    const MutableParams P{A.P.w1a + pq * kH * kIn, A.P.b1a + pq * kH, A.P.w2a + pq * kQ * kH, A.P.b2a + pq * kQ,
                          A.P.w1c + pq * kH * kIn, A.P.b1c + pq * kH, A.P.w2c + pq * kH, A.P.b2c + pq};
    float *const gm = A.m + pq * kLocal, *const gv = A.v + pq * kLocal;
    const long long *const idx_p = A.idx + pq * (size_t)A.n_updates * (size_t)B;
    const int step0 = A.step[p];
    const float lr = A.lr[p], clip_ratio = A.clip_ratio[p], vf_coef = A.vf_coef[p], ent_coef = A.ent_coef[p];
    const float max_grad_norm = A.max_grad_norm[p];
    int n_run = A.n_updates, n_eval = A.n_updates;      // KL: updates that applied a step / formed statistics
    const uint32_t a_g = tc::smem_u32(s_g), a_slice = tc::smem_u32(s_slice), a_line = tc::smem_u32(&s_line);

    float w[kLocalK];
    stage_unit(P, gm, gv, j, w, s_m, s_v, s_b2, s_b2m, s_b2v);
    for (int i = j; i < SMAX * 20; i += kEpochThreads) (&s_x[0][0])[i] = 0.0f;   // the padding columns stay zero

    // gathers of the next chunk (or of the next update's first chunk and advantages) are issued a chunk ahead
    float x_pf = 0.0f, al_pf[kAdvPer], l_act = 0.0f, l_olp = 0.0f, l_adv = 0.0f, l_ret = 0.0f;
    auto load_adv = [&](int u2) {
        const long long *idx = idx_p + (size_t)u2 * (size_t)B;
#pragma unroll
        for (int i = 0; i < kAdvPer; ++i) {
            const int t = j + i * kEpochThreads;
            al_pf[i] = t < B ? A.adv[idx[t]] : 0.0f;
        }
    };
    auto load_chunk = [&](int u2, int ch) {
        const long long *idx = idx_p + (size_t)u2 * (size_t)B;
        const int c_lo = s0 + ch * SMAX, nc = max(0, min(SMAX, s0 + nS - c_lo));
        x_pf = j < nc * kIn ? A.obs[(size_t)idx[c_lo + j / kIn] * kIn + j % kIn] : 0.0f;
        if (j < nc) {
            const long long row = idx[c_lo + j];
            l_act = A.act[row]; l_olp = A.old_logp[row]; l_adv = A.adv[row]; l_ret = A.ret[row];
        }
    };
    load_adv(0);
    load_chunk(0, 0);
    __syncthreads();

    for (int u = 0; u < A.n_updates; ++u) {
        // ---- advantage statistics of the member's whole minibatch, the same bits in every CTA
        float a_mean, a_inv;
        advantage_stats(al_pf, j, B, invB, s_red8, a_mean, a_inv);
        float lp0 = 0.0f, lp1 = 0.0f, lp2 = 0.0f;       // loss partial sums of the CTA's samples (thread 0)
        float lp3 = 0.0f, lp4 = 0.0f;                   // KL: KL and clip sums of the CTA's samples (thread 0)

        // ---- phase A: the CTA's samples, chunk by chunk
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int nc = max(0, min(SMAX, s0 + nS - (s0 + ch * SMAX)));
            if (j < SMAX * kIn) s_x[j / kIn][j % kIn] = x_pf;
            const float c_act = l_act, c_olp = l_olp, c_adv = l_adv, c_ret = l_ret;
            __syncthreads();                                          // s_x complete
            if (ch + 1 < n_chunks) load_chunk(u, ch + 1);
            else if (u + 1 < A.n_updates) { load_chunk(u + 1, 0); load_adv(u + 1); }

            float pre_a[SMAX], pre_c[SMAX];
            unit_forward(w, s_x, nc, j, lane, warp, pre_a, pre_c, s_red, s_z);

            // ---- loss terms and their derivatives, thread = sample
            if (j < SMAX) {
                float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f;
                if (j < nc) {
                    float z[kQ];
                    float mx = -1.0e30f;
#pragma unroll
                    for (int q = 0; q < kQ; ++q) { z[q] = s_z[j][q] + s_b2[q]; mx = fmaxf(mx, z[q]); }
                    float ex[kQ], se = 0.0f;
#pragma unroll
                    for (int q = 0; q < kQ; ++q) { ex[q] = expf(z[q] - mx); se += ex[q]; }
                    const float lse = logf(se);
                    float H = 0.0f, pr[kQ], lp[kQ];
#pragma unroll
                    for (int q = 0; q < kQ; ++q) { lp[q] = (z[q] - mx) - lse; pr[q] = expf(lp[q]); H -= pr[q] * lp[q]; }
                    const int a = (int)c_act;
                    float new_lp = lp[0];
#pragma unroll
                    for (int q = 1; q < kQ; ++q) new_lp = (a == q) ? lp[q] : new_lp;
                    const float ratio = expf(new_lp - c_olp);
                    const float an = (c_adv - a_mean) * a_inv;
                    const float lo = 1.0f - clip_ratio, hi = 1.0f + clip_ratio;
                    const float t1 = -an * ratio, t2 = -an * fminf(fmaxf(ratio, lo), hi);
                    const bool inside = ratio >= lo && ratio <= hi;
                    const float g_ratio = (inside || t1 > t2) ? -an : 0.0f;
                    const float g_lp = g_ratio * ratio * invB;
                    const float val = s_z[j][kQ] + s_b2[kQ];
                    const float d = val - c_ret;
#pragma unroll
                    for (int q = 0; q < kQ; ++q)
                        s_z[j][q] = g_lp * ((a == q ? 1.0f : 0.0f) - pr[q]) + ent_coef * invB * pr[q] * (lp[q] + H);
                    s_z[j][kQ] = vf_coef * d * invB;
                    p0 = fmaxf(t1, t2); p1 = H; p2 = 0.5f * d * d;
                    if constexpr (KL) {
                        const float log_r = new_lp - c_olp;
                        s_part[j][3] = (ratio - 1.0f) - log_r;
                        s_part[j][4] = fabsf(ratio - 1.0f) > clip_ratio ? 1.0f : 0.0f;
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < kZ; ++q) s_z[j][q] = 0.0f;
                    if constexpr (KL) { s_part[j][3] = 0.0f; s_part[j][4] = 0.0f; }
                }
                s_part[j][0] = p0; s_part[j][1] = p1; s_part[j][2] = p2;
            }
            __syncthreads();
            if (j == 0) {
#pragma unroll
                for (int s = 0; s < SMAX; ++s) { lp0 += s_part[s][0]; lp1 += s_part[s][1]; lp2 += s_part[s][2]; }
                if constexpr (KL) {
#pragma unroll
                    for (int s = 0; s < SMAX; ++s) { lp3 += s_part[s][3]; lp4 += s_part[s][4]; }
                }
            }

            // ---- backward: the 48 parameters of unit j, one fma chain over all of the CTA's samples
            {
                float g[kLocalK];
#pragma unroll
                for (int k = 0; k < kLocalK; ++k) g[k] = ch == 0 ? 0.0f : s_g[k * kH + j];
                unit_backward(w, s_x, s_z, pre_a, pre_c, g);
#pragma unroll
                for (int k = 0; k < kLocalK; ++k) s_g[k * kH + j] = g[k];
                if (j < kZ) {                                        // second-layer biases: sum of dz over the samples
                    float t = ch == 0 ? 0.0f : s_g[kLocalK * kH + j];
#pragma unroll
                    for (int s = 0; s < SMAX; ++s) t += s_z[s][j];
                    s_g[kLocalK * kH + j] = t;
                }
            }
            __syncthreads();                                          // s_x / s_z are rewritten by the next chunk
        }
        cluster_sync_all();                                           // every partial of the cluster is complete

        // ---- phase B: slice r of the member's gradient, summed over the CTAs in rank order
        float ss = 0.0f;
#pragma unroll
        for (int i = 0; i < kPopSlicePer; ++i) {
            const int loc = j + i * kEpochThreads, e = r * kPopSlice + loc;
            if (loc < kPopSlice && e < kLocal) {
                float t[kPopCluster];
#pragma unroll
                for (int c2 = 0; c2 < kPopCluster; ++c2) t[c2] = dsmem_ld(dsmem_map(a_g + 4u * (uint32_t)e, (uint32_t)c2));
                float gsum = t[0];
#pragma unroll
                for (int c2 = 1; c2 < kPopCluster; ++c2) gsum += t[c2];
                s_slice[loc] = gsum;
                ss = fmaf(gsum, gsum, ss);
            }
        }
        {
            const float ssum = block_sum_256(ss, s_red8);
            if (j == 0) s_line = make_float4(ssum, lp0, lp1, lp2);
            if constexpr (KL) {
                if (j == 0) s_line_kl = make_float4(lp3, lp4, 0.0f, 0.0f);
            }
        }
        if (j == 64) adam_bias_corrections(s_bias, step0 + u + 1, lr, A.beta1, A.beta2);
        cluster_sync_all();                                           // every reduced slice of the cluster is complete
        const float step_size = s_bias[0], inv_sqrt_bc2 = s_bias[1];

        // ---- phase C: clip_grad_norm_ + Adam on this CTA's copy of every parameter, statistics
        {
            float g[kLocalK];
#pragma unroll
            for (int k = 0; k < kLocalK; ++k) {
                const int e = k * kH + j, rk = e / kPopSlice;
                g[k] = dsmem_ld(dsmem_map(a_slice + 4u * (uint32_t)(e - rk * kPopSlice), (uint32_t)rk));
            }
            float gb = 0.0f;
            if (j < kZ) {
                const int e = kLocalK * kH + j, rk = e / kPopSlice;
                gb = dsmem_ld(dsmem_map(a_slice + 4u * (uint32_t)(e - rk * kPopSlice), (uint32_t)rk));
            }
            if (warp == 0) {                                          // fixed-order fold over the CTAs' lines
                float4 tot = lane < kPopCluster ? dsmem_ld4(dsmem_map(a_line, (uint32_t)lane))
                                                : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    tot.x += __shfl_xor_sync(0xffffffffu, tot.x, o); tot.y += __shfl_xor_sync(0xffffffffu, tot.y, o);
                    tot.z += __shfl_xor_sync(0xffffffffu, tot.z, o); tot.w += __shfl_xor_sync(0xffffffffu, tot.w, o);
                }
                if (lane == 0) s_tot = tot;
                if constexpr (KL) {
                    const float4 l2 = lane < kPopCluster ? dsmem_ld4(dsmem_map(tc::smem_u32(&s_line_kl), (uint32_t)lane))
                                                         : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    float2 t2 = make_float2(l2.x, l2.y);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        t2.x += __shfl_xor_sync(0xffffffffu, t2.x, o); t2.y += __shfl_xor_sync(0xffffffffu, t2.y, o);
                    }
                    if (lane == 0) s_tot_kl = t2;
                }
            }
            __syncthreads();
            const float4 tot = s_tot;
            if constexpr (KL) {                                       // the same bits in every CTA of the cluster
                const float kl = s_tot_kl.x * invB, clip_frac = s_tot_kl.y * invB;
                if (r == 0 && j == 0) {
                    float *row = A.kl_out + 2 * (pq * (size_t)A.n_updates + (size_t)u);
                    row[0] = kl; row[1] = clip_frac;
                }
                if ((double)kl > A.target_kl) { n_run = u; n_eval = u + 1; break; }
            }
            const float coef = fminf(max_grad_norm / (sqrtf(tot.x) + 1.0e-6f), 1.0f);    // clip_grad_norm_
            if (r == 0 && j == 0) {
                float *sums = A.sums4 + 4 * pq;
                const float pol = tot.y * invB, ent = tot.z * invB, vl = tot.w * invB;
                sums[0] += pol; sums[1] += vl; sums[2] += ent; sums[3] += pol + vf_coef * vl - ent_coef * ent;
            }
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
            if (j < kZ) {
                const float gc = gb * coef;
                const float mi = A.beta1 * s_b2m[j] + (1.0f - A.beta1) * gc;
                const float vi = A.beta2 * s_b2v[j] + (1.0f - A.beta2) * gc * gc;
                s_b2m[j] = mi; s_b2v[j] = vi;
                s_b2[j] = s_b2[j] - adam_quotient(step_size * mi, vi, inv_sqrt_bc2, A.eps);
            }
        }
        __syncthreads();                                              // s_b2 and s_tot before the next update
    }
    cluster_sync_all();                                               // the peers' last DSMEM reads of this CTA
    if (r == 0) {
        write_back_unit(P, gm, gv, j, w, s_m, s_v, s_b2, s_b2m, s_b2v);
        if constexpr (KL) {
            float *rows = A.kl_out + 2 * pq * (size_t)A.n_updates;
            for (int i = 2 * n_eval + j; i < 2 * A.n_updates; i += kEpochThreads) rows[i] = __int_as_float(0x7fc00000);
            if (j == 0) { A.step[p] = step0 + n_run; A.n_done[p] = n_run; }
        } else {
            if (j == 0) A.step[p] = step0 + A.n_updates;
        }
    }
}

}  // namespace
}  // extern "C++"

/* ---- C ABI ------------------------------------------------------------------------------------------------------ */

static int pop_sizes_ok(int n_members, int n_envs, int max_members) {
    return n_members > 0 && n_envs > 0 && n_members <= max_members && (long long)n_members * n_envs <= 0x7fffffffll;
}

int carenv_pack_policy_pop(int tensor_cores, int n_members, const float *w1a, const float *b1a, const float *w2a,
                           const float *b2a, const float *w1c, const float *b1c, const float *w2c, const float *b2c,
                           float *packed_out, void *stream) {
    if (n_members <= 0 || n_members > 65535) return fail(CARENV_E_INVAL, "n_members must be in 1..65535");
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !packed_out)
        return fail(CARENV_E_INVAL, "null pointer");
    const int n = tensor_cores ? kTcWeightFloats : kPolicyFloats;
    const dim3 grid((n + 255) / 256, n_members);
    if (tensor_cores)
        k_pack_policy<true, true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(w1a, b1a, w2a, b2a, w1c, b1c,
                                                                                      w2c, b2c, packed_out);
    else
        k_pack_policy<false, true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(w1a, b1a, w2a, b2a, w1c, b1c,
                                                                                       w2c, b2c, packed_out);
    CU(cudaGetLastError());
    return 0;
}

// checks shared by the two member-batched rollouts
static int rollout_pop_args_ok(Handle *h, int n_members, int n_envs, int n_steps, const unsigned long long *seeds,
                               const void *const *ptrs, int n_ptrs) {
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (!pop_sizes_ok(n_members, n_envs, 65535) || n_steps < 0)
        return fail(CARENV_E_INVAL, "n_members must be in 1..65535, n_envs_per_member positive, n_members * n_envs "
                                    "below 2^31 and n_steps non-negative");
    if (!seeds) return fail(CARENV_E_INVAL, "null pointer");
    for (int i = 0; i < n_ptrs; ++i)
        if (!ptrs[i]) return fail(CARENV_E_INVAL, "null pointer");
    if (h->pose_rows) return fail(CARENV_E_INVAL, "a population writes full observation rows: pose_rows must be 0");
    return 0;
}

static int policy_rollout_warp_pop_impl(void *handle, int n_members, const float *w1a, const float *b1a,
                                        const float *w2a, const float *b2a, const float *w1c, const float *b1c,
                                        const float *w2c, const float *b2c, int n_envs, int n_steps,
                                        const unsigned long long *seeds, unsigned long long step0, double *pos,
                                        double *vel, int32_t *ints, float *cur_obs, float *cur_term, float *cur_trunc,
                                        double reward_scale, float *obs_buf, float *act_buf, float *rew_buf,
                                        float *val_buf, float *term_buf, float *trunc_buf, float *logp_buf,
                                        float *last_val, float *u_dbg, void *stream, const SlotArgs &fs) {
    Handle *h = static_cast<Handle *>(handle);
    const void *ptrs[] = {w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c, pos, vel, ints, cur_obs, cur_term, cur_trunc,
                          obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf};
    if (const int rc = rollout_pop_args_ok(h, n_members, n_envs, n_steps, seeds, ptrs, (int)(sizeof(ptrs) / sizeof(ptrs[0]))))
        return rc;
    return policy_rollout_warp_launch(h, ppo::Params{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c}, n_members, n_envs,
                                      n_steps, 0, 0, seeds, step0, pos, vel, ints, cur_obs, cur_term, cur_trunc,
                                      reward_scale, obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf,
                                      last_val, u_dbg, stream, fs);
}

int carenv_policy_rollout_warp_pop(void *handle, int n_members, const float *w1a, const float *b1a, const float *w2a,
                                   const float *b2a, const float *w1c, const float *b1c, const float *w2c,
                                   const float *b2c, int n_envs, int n_steps, const unsigned long long *seeds,
                                   unsigned long long step0, double *pos, double *vel, int32_t *ints, float *cur_obs,
                                   float *cur_term, float *cur_trunc, double reward_scale, float *obs_buf,
                                   float *act_buf, float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                   float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    return policy_rollout_warp_pop_impl(handle, n_members, w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c, n_envs, n_steps,
                                        seeds, step0, pos, vel, ints, cur_obs, cur_term, cur_trunc, reward_scale,
                                        obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf, last_val,
                                        u_dbg, stream, SlotArgs{});
}

int carenv_policy_rollout_warp_pop_final(void *handle, int n_members, const float *w1a, const float *b1a,
                                         const float *w2a, const float *b2a, const float *w1c, const float *b1c,
                                         const float *w2c, const float *b2c, int n_envs, int n_steps,
                                         const unsigned long long *seeds, unsigned long long step0, double *pos,
                                         double *vel, int32_t *ints, float *cur_obs, float *cur_term,
                                         float *cur_trunc, double reward_scale, float *obs_buf, float *act_buf,
                                         float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                         float *logp_buf, float *last_val, float *u_dbg, void *stream,
                                         float *final_obs, int32_t *final_row, int n_slots) {
    const SlotArgs fs{final_obs, final_row, n_slots};
    if (const int rc = slot_args_ok(fs, n_steps)) return rc;
    return policy_rollout_warp_pop_impl(handle, n_members, w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c, n_envs, n_steps,
                                        seeds, step0, pos, vel, ints, cur_obs, cur_term, cur_trunc, reward_scale,
                                        obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf, last_val,
                                        u_dbg, stream, fs);
}

static int policy_rollout_tc_pop_impl(void *handle, int n_members, const float *packed_weights, int n_envs,
                                      int n_steps, const unsigned long long *seeds, unsigned long long step0,
                                      double *pos, double *vel, int32_t *ints, float *cur_obs, float *cur_term,
                                      float *cur_trunc, double reward_scale, float *obs_buf, float *act_buf,
                                      float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                      float *logp_buf, float *last_val, float *u_dbg, void *stream,
                                      const SlotArgs &fs) {
    Handle *h = static_cast<Handle *>(handle);
    const void *ptrs[] = {packed_weights, pos, vel, ints, cur_obs, cur_term, cur_trunc, obs_buf, act_buf, rew_buf,
                          val_buf, term_buf, trunc_buf, logp_buf};
    if (const int rc = rollout_pop_args_ok(h, n_members, n_envs, n_steps, seeds, ptrs, (int)(sizeof(ptrs) / sizeof(ptrs[0]))))
        return rc;
    return policy_rollout_tc_launch(h, packed_weights, n_members, n_envs, n_steps, 0, 0, seeds, step0, pos, vel, ints,
                                    cur_obs, cur_term, cur_trunc, reward_scale, obs_buf, act_buf, rew_buf, val_buf,
                                    term_buf, trunc_buf, logp_buf, last_val, u_dbg, stream, fs);
}

int carenv_policy_rollout_tc_pop(void *handle, int n_members, const float *packed_weights, int n_envs, int n_steps,
                                 const unsigned long long *seeds, unsigned long long step0, double *pos, double *vel,
                                 int32_t *ints, float *cur_obs, float *cur_term, float *cur_trunc, double reward_scale,
                                 float *obs_buf, float *act_buf, float *rew_buf, float *val_buf, float *term_buf,
                                 float *trunc_buf, float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    return policy_rollout_tc_pop_impl(handle, n_members, packed_weights, n_envs, n_steps, seeds, step0, pos, vel, ints,
                                      cur_obs, cur_term, cur_trunc, reward_scale, obs_buf, act_buf, rew_buf, val_buf,
                                      term_buf, trunc_buf, logp_buf, last_val, u_dbg, stream, SlotArgs{});
}

int carenv_policy_rollout_tc_pop_final(void *handle, int n_members, const float *packed_weights, int n_envs,
                                       int n_steps, const unsigned long long *seeds, unsigned long long step0,
                                       double *pos, double *vel, int32_t *ints, float *cur_obs, float *cur_term,
                                       float *cur_trunc, double reward_scale, float *obs_buf, float *act_buf,
                                       float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                       float *logp_buf, float *last_val, float *u_dbg, void *stream, float *final_obs,
                                       int32_t *final_row, int n_slots) {
    const SlotArgs fs{final_obs, final_row, n_slots};
    if (const int rc = slot_args_ok(fs, n_steps)) return rc;
    return policy_rollout_tc_pop_impl(handle, n_members, packed_weights, n_envs, n_steps, seeds, step0, pos, vel, ints,
                                      cur_obs, cur_term, cur_trunc, reward_scale, obs_buf, act_buf, rew_buf, val_buf,
                                      term_buf, trunc_buf, logp_buf, last_val, u_dbg, stream, fs);
}

int carenv_ppo_epoch_pop_cluster_size(void) { return kPopCluster; }

static void ppo_epoch_pop_config(cudaLaunchConfig_t *cfg, cudaLaunchAttribute *attr, int n_members, cudaStream_t st) {
    memset(cfg, 0, sizeof(*cfg));
    memset(attr, 0, sizeof(*attr));
    attr->id = cudaLaunchAttributeClusterDimension;
    attr->val.clusterDim.x = kPopCluster; attr->val.clusterDim.y = 1; attr->val.clusterDim.z = 1;
    cfg->gridDim = dim3((unsigned)(n_members * kPopCluster));
    cfg->blockDim = dim3(ppo::kEpochThreads);
    cfg->dynamicSmemBytes = kPopSmemBytes;
    cfg->stream = st;
    cfg->attrs = attr;
    cfg->numAttrs = 1;
}

static int ppo_epoch_pop_attributes(bool kl) {
    const void *kern = kl ? reinterpret_cast<const void *>(k_ppo_epoch_pop<true>)
                          : reinterpret_cast<const void *>(k_ppo_epoch_pop<false>);
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kPopSmemBytes));
    if (kPopCluster > 8) CU(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    return 0;
}

int carenv_ppo_epoch_pop_resident_clusters(int *n_clusters) {
    if (!n_clusters) return fail(CARENV_E_INVAL, "null pointer");
    if (const int rc = ppo_epoch_pop_attributes(false)) return rc;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    ppo_epoch_pop_config(&cfg, &attr, 1, nullptr);
    CU(cudaOccupancyMaxActiveClusters(n_clusters, k_ppo_epoch_pop<false>, &cfg));
    return 0;
}

// carenv_ppo_epoch_pop and carenv_ppo_epoch_pop_kl: kl_out == nullptr launches k_ppo_epoch_pop<false>
static int ppo_epoch_pop_launch(int n_members, float *w1a, float *b1a, float *w2a, float *b2a, float *w1c, float *b1c,
                                float *w2c, float *b2c, const float *obs, const long long *idx, const float *act,
                                const float *old_logp, const float *adv, const float *ret, int batch, int n_updates,
                                const float *lr, const float *clip_ratio, const float *vf_coef, const float *ent_coef,
                                const float *max_grad_norm, double beta1, double beta2, double eps, float *exp_avg,
                                float *exp_avg_sq, int *step, float *sums4, void *stream, double target_kl,
                                float *kl_out, int *n_done) {
    if (n_members <= 0 || n_members > 0x7fffffff / kPopCluster)
        return fail(CARENV_E_INVAL, "n_members must be positive (and n_members * cluster size below 2^31)");
    if (batch < 2 || batch > ppo::kMaxBatch) return fail(CARENV_E_INVAL, "batch must be in 2..1024");
    if (n_updates < 0) return fail(CARENV_E_INVAL, "negative n_updates");
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !obs || !idx || !act || !old_logp || !adv ||
        !ret || !lr || !clip_ratio || !vf_coef || !ent_coef || !max_grad_norm || !exp_avg || !exp_avg_sq || !step ||
        !sums4)
        return fail(CARENV_E_INVAL, "null pointer");
    const bool kl = kl_out != nullptr;
    if (n_updates == 0) {
        if (kl) CU(cudaMemsetAsync(n_done, 0, sizeof(int) * (size_t)n_members, static_cast<cudaStream_t>(stream)));
        return 0;
    }
    PopEpochArgs A;
    memset(&A, 0, sizeof(A));
    A.P = ppo::MutableParams{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c};
    A.obs = obs; A.idx = idx; A.act = act; A.old_logp = old_logp; A.adv = adv; A.ret = ret;
    A.B = batch; A.n_updates = n_updates;
    A.lr = lr; A.clip_ratio = clip_ratio; A.vf_coef = vf_coef; A.ent_coef = ent_coef; A.max_grad_norm = max_grad_norm;
    A.beta1 = (float)beta1; A.beta2 = (float)beta2; A.eps = (float)eps;
    A.m = exp_avg; A.v = exp_avg_sq; A.step = step; A.sums4 = sums4;
    A.target_kl = target_kl; A.kl_out = kl_out; A.n_done = n_done;
    if (const int rc = ppo_epoch_pop_attributes(kl)) return rc;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    ppo_epoch_pop_config(&cfg, &attr, n_members, static_cast<cudaStream_t>(stream));
    if (kl) CU(cudaLaunchKernelEx(&cfg, k_ppo_epoch_pop<true>, A));
    else CU(cudaLaunchKernelEx(&cfg, k_ppo_epoch_pop<false>, A));
    return 0;
}

int carenv_ppo_epoch_pop(int n_members, float *w1a, float *b1a, float *w2a, float *b2a, float *w1c, float *b1c,
                         float *w2c, float *b2c, const float *obs, const long long *idx, const float *act,
                         const float *old_logp, const float *adv, const float *ret, int batch, int n_updates,
                         const float *lr, const float *clip_ratio, const float *vf_coef, const float *ent_coef,
                         const float *max_grad_norm, double beta1, double beta2, double eps, float *exp_avg,
                         float *exp_avg_sq, int *step, float *sums4, void *stream) {
    return ppo_epoch_pop_launch(n_members, w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c, obs, idx, act, old_logp, adv, ret,
                                batch, n_updates, lr, clip_ratio, vf_coef, ent_coef, max_grad_norm, beta1, beta2, eps,
                                exp_avg, exp_avg_sq, step, sums4, stream, 0.0, nullptr, nullptr);
}

int carenv_ppo_epoch_pop_kl(int n_members, float *w1a, float *b1a, float *w2a, float *b2a, float *w1c, float *b1c,
                            float *w2c, float *b2c, const float *obs, const long long *idx, const float *act,
                            const float *old_logp, const float *adv, const float *ret, int batch, int n_updates,
                            const float *lr, const float *clip_ratio, const float *vf_coef, const float *ent_coef,
                            const float *max_grad_norm, double beta1, double beta2, double eps, float *exp_avg,
                            float *exp_avg_sq, int *step, float *sums4, void *stream, double target_kl,
                            float *kl_out, int *n_done) {
    if (!kl_out || !n_done) return fail(CARENV_E_INVAL, "null pointer");
    if (!(target_kl > 0.0)) return fail(CARENV_E_INVAL, "target_kl must be positive (+inf: statistics only)");
    return ppo_epoch_pop_launch(n_members, w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c, obs, idx, act, old_logp, adv, ret,
                                batch, n_updates, lr, clip_ratio, vf_coef, ent_coef, max_grad_norm, beta1, beta2, eps,
                                exp_avg, exp_avg_sq, step, sums4, stream, target_kl, kl_out, n_done);
}
