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
// k_ppo_epoch's (ppo_epoch.cuh), with the grid replaced by the cluster:
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

__global__ void __launch_bounds__(ppo::kEpochThreads, 1) k_ppo_epoch_pop(const PopEpochArgs A) {
    using namespace ppo;
    constexpr int SMAX = kEpochSamples;
    constexpr int kZ = 10;                               // 9 logits + the value per sample
    constexpr int kFold = kZ * SMAX;
    static_assert(SMAX * kIn <= kEpochThreads, "one thread per staged observation element");
    extern __shared__ __align__(16) float s_dyn[];
    float *const s_m = s_dyn, *const s_v = s_dyn + kLocalK * kH;
    float *const s_g = s_v + kLocalK * kH;               // this CTA's partial gradient, local order
    float *const s_slice = s_g + kLocalPad;              // reduced slice r of the gradient
    __shared__ __align__(16) float s_x[SMAX][20];
    __shared__ float s_red[8][kFold];
    __shared__ __align__(16) float s_z[SMAX][12];
    __shared__ float s_part[SMAX][3];
    __shared__ float s_red8[8];
    __shared__ __align__(16) float4 s_line;              // slice sum of squares, loss partial sums of the CTA's samples
    __shared__ float4 s_tot;
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
    const uint32_t a_g = tc::smem_u32(s_g), a_slice = tc::smem_u32(s_slice), a_line = tc::smem_u32(&s_line);

    float w[kLocalK];
#pragma unroll
    for (int k = 0; k < kLocalK; ++k) {
        const int f = local_to_flat(k * kH + j);
        w[k] = *param_ptr(P, f);
        s_m[k * kH + j] = gm[f];
        s_v[k * kH + j] = gv[f];
    }
    if (j < kZ) {
        const int f = local_to_flat(kLocalK * kH + j);
        s_b2[j] = *param_ptr(P, f); s_b2m[j] = gm[f]; s_b2v[j] = gv[f];
    }
    for (int i = j; i < SMAX * 20; i += kEpochThreads) (&s_x[0][0])[i] = 0.0f;   // the padding columns stay zero

    // gathers of the next chunk (or of the next update's first chunk and advantages) are issued a chunk ahead
    constexpr int kPer = kMaxBatch / kEpochThreads;
    float x_pf = 0.0f, al_pf[kPer], l_act = 0.0f, l_olp = 0.0f, l_adv = 0.0f, l_ret = 0.0f;
    auto load_adv = [&](int u2) {
        const long long *idx = idx_p + (size_t)u2 * (size_t)B;
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
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
        // ---- advantage statistics of the member's whole minibatch (train.py:236-237), the same bits in every CTA
        float a_mean, a_inv;
        {
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < kPer; ++i) sum += al_pf[i];
            a_mean = block_sum_256(sum, s_red8) * invB;
            float s2 = 0.0f;
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                const float d = j + i * kEpochThreads < B ? al_pf[i] - a_mean : 0.0f;
                s2 += d * d;
            }
            const float var = block_sum_256(s2, s_red8) / (float)(B > 1 ? B - 1 : 1);
            a_inv = 1.0f / fmaxf(sqrtf(var), 1.0e-5f);
        }
        float lp0 = 0.0f, lp1 = 0.0f, lp2 = 0.0f;       // loss partial sums of the CTA's samples (thread 0)

        // ---- phase A: the CTA's samples, chunk by chunk
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int nc = max(0, min(SMAX, s0 + nS - (s0 + ch * SMAX)));
            if (j < SMAX * kIn) s_x[j / kIn][j % kIn] = x_pf;
            const float c_act = l_act, c_olp = l_olp, c_adv = l_adv, c_ret = l_ret;
            __syncthreads();                                          // s_x complete
            if (ch + 1 < n_chunks) load_chunk(u, ch + 1);
            else if (u + 1 < A.n_updates) { load_chunk(u + 1, 0); load_adv(u + 1); }

            float pre_a[SMAX], pre_c[SMAX];
            {
                float contrib[kFold];
#pragma unroll
                for (int s = 0; s < SMAX; ++s) {
                    const float4 *xv = reinterpret_cast<const float4 *>(s_x[s]);
                    float x[20];
#pragma unroll
                    for (int i = 0; i < 5; ++i) { const float4 t = xv[i]; x[4 * i] = t.x; x[4 * i + 1] = t.y; x[4 * i + 2] = t.z; x[4 * i + 3] = t.w; }
                    float pa = w[kIn], pb = 0.0f, pc = 0.0f, qa = w[2 * kIn + 1 + kQ], qb = 0.0f, qc = 0.0f;
#pragma unroll
                    for (int k = 0; k < kIn; k += 3) {
                        pa = fmaf(w[k], x[k], pa); pb = fmaf(w[k + 1], x[k + 1], pb); pc = fmaf(w[k + 2], x[k + 2], pc);
                        qa = fmaf(w[kIn + 1 + kQ + k], x[k], qa); qb = fmaf(w[kIn + 2 + kQ + k], x[k + 1], qb);
                        qc = fmaf(w[kIn + 3 + kQ + k], x[k + 2], qc);
                    }
                    const bool on = s < nc;
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
                for (int i = 0; i < kRem; ++i) s_red[warp][base + i] = contrib[i];
            }
            __syncthreads();
            if (j < kFold) {
                float t = s_red[0][j];
#pragma unroll
                for (int w8 = 1; w8 < 8; ++w8) t += s_red[w8][j];
                s_z[j / kZ][j % kZ] = t;
            }
            __syncthreads();

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
                } else {
#pragma unroll
                    for (int q = 0; q < kZ; ++q) s_z[j][q] = 0.0f;
                }
                s_part[j][0] = p0; s_part[j][1] = p1; s_part[j][2] = p2;
            }
            __syncthreads();
            if (j == 0) {
#pragma unroll
                for (int s = 0; s < SMAX; ++s) { lp0 += s_part[s][0]; lp1 += s_part[s][1]; lp2 += s_part[s][2]; }
            }

            // ---- backward: the 48 parameters of unit j, one fma chain over all of the CTA's samples
            {
                float g[kLocalK];
#pragma unroll
                for (int k = 0; k < kLocalK; ++k) g[k] = ch == 0 ? 0.0f : s_g[k * kH + j];
#pragma unroll
                for (int s = 0; s < SMAX; ++s) {
                    const float4 *xv = reinterpret_cast<const float4 *>(s_x[s]);
                    float x[20];
#pragma unroll
                    for (int i = 0; i < 5; ++i) { const float4 t = xv[i]; x[4 * i] = t.x; x[4 * i + 1] = t.y; x[4 * i + 2] = t.z; x[4 * i + 3] = t.w; }
                    const float4 *zv = reinterpret_cast<const float4 *>(s_z[s]);
                    const float4 d0 = zv[0], d1 = zv[1], d2 = zv[2];
                    const float dz[kQ] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w, d2.x};
                    const float dv = d2.y;
                    const float ha = fmaxf(pre_a[s], 0.0f), hc = fmaxf(pre_c[s], 0.0f);
                    float dh = 0.0f;
#pragma unroll
                    for (int q = 0; q < kQ; ++q) { g[kIn + 1 + q] = fmaf(dz[q], ha, g[kIn + 1 + q]); dh = fmaf(dz[q], w[kIn + 1 + q], dh); }
                    dh = pre_a[s] > 0.0f ? dh : 0.0f;
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
        }
        if (j == 64) {                                                // bias corrections of this step
            const int t_step = step0 + u + 1;
            const float bc1 = 1.0f - powf(A.beta1, (float)t_step), bc2 = 1.0f - powf(A.beta2, (float)t_step);
            s_bias[0] = lr / bc1; s_bias[1] = rsqrtf(bc2);
        }
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
            }
            __syncthreads();
            const float4 tot = s_tot;
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
#pragma unroll
        for (int k = 0; k < kLocalK; ++k) {
            const int f = local_to_flat(k * kH + j);
            *param_ptr(P, f) = w[k];
            gm[f] = s_m[k * kH + j];
            gv[f] = s_v[k * kH + j];
        }
        if (j < kZ) {
            const int f = local_to_flat(kLocalK * kH + j);
            *param_ptr(P, f) = s_b2[j]; gm[f] = s_b2m[j]; gv[f] = s_b2v[j];
        }
        if (j == 0) A.step[p] = step0 + A.n_updates;
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

int carenv_policy_rollout_warp_pop(void *handle, int n_members, const float *w1a, const float *b1a, const float *w2a,
                                   const float *b2a, const float *w1c, const float *b1c, const float *w2c,
                                   const float *b2c, int n_envs, int n_steps, const unsigned long long *seeds,
                                   unsigned long long step0, double *pos, double *vel, int32_t *ints, float *cur_obs,
                                   float *cur_term, float *cur_trunc, double reward_scale, float *obs_buf,
                                   float *act_buf, float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                   float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    const void *ptrs[] = {w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c, pos, vel, ints, cur_obs, cur_term, cur_trunc,
                          obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf};
    if (const int rc = rollout_pop_args_ok(h, n_members, n_envs, n_steps, seeds, ptrs, (int)(sizeof(ptrs) / sizeof(ptrs[0]))))
        return rc;
    return policy_rollout_warp_launch(h, ppo::Params{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c}, n_members, n_envs,
                                      n_steps, 0, 0, seeds, step0, pos, vel, ints, cur_obs, cur_term, cur_trunc,
                                      reward_scale, obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf,
                                      last_val, u_dbg, stream);
}

int carenv_policy_rollout_tc_pop(void *handle, int n_members, const float *packed_weights, int n_envs, int n_steps,
                                 const unsigned long long *seeds, unsigned long long step0, double *pos, double *vel,
                                 int32_t *ints, float *cur_obs, float *cur_term, float *cur_trunc, double reward_scale,
                                 float *obs_buf, float *act_buf, float *rew_buf, float *val_buf, float *term_buf,
                                 float *trunc_buf, float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    const void *ptrs[] = {packed_weights, pos, vel, ints, cur_obs, cur_term, cur_trunc, obs_buf, act_buf, rew_buf,
                          val_buf, term_buf, trunc_buf, logp_buf};
    if (const int rc = rollout_pop_args_ok(h, n_members, n_envs, n_steps, seeds, ptrs, (int)(sizeof(ptrs) / sizeof(ptrs[0]))))
        return rc;
    return policy_rollout_tc_launch(h, packed_weights, n_members, n_envs, n_steps, 0, 0, seeds, step0, pos, vel, ints,
                                    cur_obs, cur_term, cur_trunc, reward_scale, obs_buf, act_buf, rew_buf, val_buf,
                                    term_buf, trunc_buf, logp_buf, last_val, u_dbg, stream);
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

static int ppo_epoch_pop_attributes() {
    CU(cudaFuncSetAttribute(k_ppo_epoch_pop, cudaFuncAttributeMaxDynamicSharedMemorySize, kPopSmemBytes));
    if (kPopCluster > 8) CU(cudaFuncSetAttribute(k_ppo_epoch_pop, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    return 0;
}

int carenv_ppo_epoch_pop_resident_clusters(int *n_clusters) {
    if (!n_clusters) return fail(CARENV_E_INVAL, "null pointer");
    if (const int rc = ppo_epoch_pop_attributes()) return rc;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    ppo_epoch_pop_config(&cfg, &attr, 1, nullptr);
    CU(cudaOccupancyMaxActiveClusters(n_clusters, k_ppo_epoch_pop, &cfg));
    return 0;
}

int carenv_ppo_epoch_pop(int n_members, float *w1a, float *b1a, float *w2a, float *b2a, float *w1c, float *b1c,
                         float *w2c, float *b2c, const float *obs, const long long *idx, const float *act,
                         const float *old_logp, const float *adv, const float *ret, int batch, int n_updates,
                         const float *lr, const float *clip_ratio, const float *vf_coef, const float *ent_coef,
                         const float *max_grad_norm, double beta1, double beta2, double eps, float *exp_avg,
                         float *exp_avg_sq, int *step, float *sums4, void *stream) {
    if (n_members <= 0 || n_members > 0x7fffffff / kPopCluster)
        return fail(CARENV_E_INVAL, "n_members must be positive (and n_members * cluster size below 2^31)");
    if (batch < 2 || batch > ppo::kMaxBatch) return fail(CARENV_E_INVAL, "batch must be in 2..1024");
    if (n_updates < 0) return fail(CARENV_E_INVAL, "negative n_updates");
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !obs || !idx || !act || !old_logp || !adv ||
        !ret || !lr || !clip_ratio || !vf_coef || !ent_coef || !max_grad_norm || !exp_avg || !exp_avg_sq || !step ||
        !sums4)
        return fail(CARENV_E_INVAL, "null pointer");
    if (n_updates == 0) return 0;
    PopEpochArgs A;
    memset(&A, 0, sizeof(A));
    A.P = ppo::MutableParams{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c};
    A.obs = obs; A.idx = idx; A.act = act; A.old_logp = old_logp; A.adv = adv; A.ret = ret;
    A.B = batch; A.n_updates = n_updates;
    A.lr = lr; A.clip_ratio = clip_ratio; A.vf_coef = vf_coef; A.ent_coef = ent_coef; A.max_grad_norm = max_grad_norm;
    A.beta1 = (float)beta1; A.beta2 = (float)beta2; A.eps = (float)eps;
    A.m = exp_avg; A.v = exp_avg_sq; A.step = step; A.sums4 = sums4;
    if (const int rc = ppo_epoch_pop_attributes()) return rc;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    ppo_epoch_pop_config(&cfg, &attr, n_members, static_cast<cudaStream_t>(stream));
    CU(cudaLaunchKernelEx(&cfg, k_ppo_epoch_pop, A));
    return 0;
}
