// policy_rollout.cuh — the fused policy + environment rollout kernels (SURVEY §8 f-2) and the tcgen05 bring-up test.
// Textually included by carenv_kernels.cu inside its anonymous namespace (after the step kernels, whose helpers
// stage_tables / store_pose / env_step it uses); kept in its own file so that the step path (carenv_core.cuh,
// carenv_tables.h, carenv_kernels.cu) can be hashed on its own by bench.py / profiles/make_traffic.py.
#pragma once
// tcgen05 bring-up / unit test: D[128,256] = A[128,24] * B[256,24]^T with kind::tf32, accumulators in TMEM.
__global__ void __launch_bounds__(128) k_tc_gemm_test(const float *__restrict__ A, const float *__restrict__ B,
                                                      float *__restrict__ D) {
    extern __shared__ __align__(16) unsigned char smem[];
    unsigned char *tsm = smem + ((128u - (tc::smem_u32(smem) & 127u)) & 127u);
    unsigned char *sA = tsm, *sB = tsm + tc::kABytes;
    __shared__ __align__(8) unsigned long long mbar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < tc::kTileM * tc::kK; i += blockDim.x)
        *reinterpret_cast<float *>(sA + tc::operand_offset(i / tc::kK, i % tc::kK)) = A[i];
    for (int i = tid; i < tc::kTileN * tc::kK; i += blockDim.x)
        *reinterpret_cast<float *>(sB + tc::operand_offset(i / tc::kK, i % tc::kK)) = B[i];
    if (tid == 0) tc::mbar_init(tc::smem_u32(&mbar), 1);
    if (warp == 0) tc::tmem_alloc<256>(&tmem_slot);
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tbase = tmem_slot;
    if (tid == 0) {
        const uint32_t idesc = tc::make_idesc_tf32(128, 256);
        for (int ks = 0; ks < tc::kK / 8; ++ks) {
            const uint64_t da = tc::make_smem_desc(tc::smem_u32(sA) + ks * 2 * tc::kLBO);
            const uint64_t db = tc::make_smem_desc(tc::smem_u32(sB) + ks * 2 * tc::kLBO);
            tc::mma_tf32(tbase, da, db, idesc, ks > 0);
        }
        tc::mma_commit(tc::smem_u32(&mbar));
    }
    tc::mbar_wait(tc::smem_u32(&mbar), 0);
    tc::tc_fence_after();
    const uint32_t lane_base = tbase + ((uint32_t)(warp * 32) << 16);
    for (int c = 0; c < 256; c += 16) {
        float v[16];
        tc::tmem_ld16(lane_base + c, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) D[(size_t)tid * 256 + c + i] = v[i];
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<256>(tbase);
}

// Fused rollout (SURVEY §8 f-2): actor/critic forward, categorical sampling, CarEnv.step and the Buffer
// row writes of train.py:173-195 for n_steps steps in ONE launch.  One thread per environment; the packed
// policy weights (53 KB) and the per-thread-indexed track tables live in shared memory.
#ifndef CARENV_POLICY_BLOCK
#define CARENV_POLICY_BLOCK 128
#endif
#ifndef CARENV_POLICY_MIN_BLOCKS
#define CARENV_POLICY_MIN_BLOCKS 3
#endif
constexpr int kPolicyBlock = CARENV_POLICY_BLOCK;

// ---- final-observation slots (FINAL instantiations, C ABI carenv_policy_rollout*_final) ---------------------------
// An environment truncates at most S = ceil(n_steps / kTimeLimit) times in a launch, whatever its starting time step.
// Its k-th truncation writes the observation the episode ended in (before the autoreset) to final_obs[k][e] and the
// row t of that step to final_row[k][e] ([S][stride](,18) arrays); when the rollout ends, the slots it did not use get
// row -1.  The writes sit in the autoreset branch of env_step (about once per 1000 env-steps); the step loop carries
// the two slot pointers and a count.  obs == nullptr: this thread writes nothing (idle or non-leader threads).
struct FinalSlots {
    float *obs;
    int *row;
    int used;
};
__device__ __forceinline__ FinalSlots final_slots_begin(bool writer, float *final_obs, int *final_row, int n_slots,
                                                        int e) {
    return FinalSlots{writer && n_slots > 0 ? final_obs + (size_t)e * kObsDim : nullptr,
                      writer ? final_row + e : nullptr, 0};
}
// after the step of row t: a truncation takes the slot just written and moves to the next one
__device__ __forceinline__ void final_slots_step(FinalSlots &f, int truncated, int t, int n_slots, int stride) {
    if (truncated) {
        if (f.obs) {
            *f.row = t;
            f.row += stride;
            f.obs += (size_t)stride * kObsDim;
        }
        if (++f.used >= n_slots) f.obs = nullptr;            // n_slots >= S (checked by the launchers): never taken
    }
}
__device__ __forceinline__ void final_slots_end(FinalSlots &f, int n_slots, int stride) {
    if (f.row)
        for (int k = f.used; k < n_slots; ++k, f.row += stride) *f.row = -1;
}

template <int U, bool FINAL = false>
__global__ void __launch_bounds__(kPolicyBlock, CARENV_POLICY_MIN_BLOCKS)
k_policy_rollout(const __grid_constant__ TrackParams P, const Tables G, const float *__restrict__ weights,
                 int n_envs, int n_steps, int env_offset, unsigned long long seed, unsigned long long step0,
                 double2 *__restrict__ pos, double2 *__restrict__ vel, int4 *__restrict__ ints,
                 float *__restrict__ cur_obs, float *__restrict__ cur_term, float *__restrict__ cur_trunc,
                 double reward_scale, float *__restrict__ obs_buf, float *__restrict__ act_buf,
                 float *__restrict__ rew_buf, float *__restrict__ val_buf, float *__restrict__ term_buf,
                 float *__restrict__ trunc_buf, float *__restrict__ logp_buf, float *__restrict__ last_val,
                 float *__restrict__ u_dbg, unsigned long long *stats, int table_bytes, int obs_mode,
                 float *__restrict__ final_obs, int *__restrict__ final_row, int n_slots) {
    extern __shared__ __align__(16) unsigned char smem[];
    float *sw = reinterpret_cast<float *>(smem + table_bytes);
    for (int i = threadIdx.x; i < kPolicyFloats / 4; i += blockDim.x)
        reinterpret_cast<float4 *>(sw)[i] = reinterpret_cast<const float4 *>(weights)[i];
    const Tables T = stage_tables(G, P.n_gates, P.n_seg, smem);      // ends with __syncthreads()
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;

    EnvState s;
    {
        const double2 p = pos[e], v = vel[e];
        const int4 q = ints[e];
        s.px = p.x; s.py = p.y; s.vx = v.x; s.vy = v.y;
        s.k = q.x; s.t = q.y; s.next_gate = q.z; s.passed = q.w;
    }
    float obs[kObsDim];
    {
        const float2 *src = reinterpret_cast<const float2 *>(cur_obs + (size_t)e * kObsDim);
#pragma unroll
        for (int i = 0; i < kObsDim / 2; ++i) { const float2 v = src[i]; obs[2 * i] = v.x; obs[2 * i + 1] = v.y; }
    }
    float tc = cur_term[e], uc = cur_trunc[e];
    const uint32_t gid = (uint32_t)(env_offset + e);
    FinalSlots fs{};
    if constexpr (FINAL) fs = final_slots_begin(true, final_obs, final_row, n_slots, e);
    PolicyOut po;
    for (int t = 0; t < n_steps; ++t) {
        const size_t idx = (size_t)t * (size_t)n_envs + (size_t)e;
        policy_forward(obs, sw, po);
        const unsigned long long gs = step0 + (unsigned long long)t;
        const uint32_t bits = philox_uniform_bits((uint32_t)seed, (uint32_t)(seed >> 32), gid, (uint32_t)gs,
                                                  (uint32_t)(gs >> 32), 0x43415245u);
        const float u = (float)(bits >> 8) * (1.0f / 16777216.0f);
        float logp, us;
        const int a = sample_action(po, u, logp, us);
        if (obs_mode == kObsPose) {
            store_pose(reinterpret_cast<PoseRec *>(obs_buf) + idx, s, obs[2], obs[3]);
        } else {
            float2 *dst = reinterpret_cast<float2 *>(obs_buf + idx * kObsDim);
#pragma unroll
            for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(obs[2 * i], obs[2 * i + 1]);
        }
        act_buf[idx] = (float)a;
        val_buf[idx] = po.value;
        logp_buf[idx] = logp;
        term_buf[idx] = tc;
        trunc_buf[idx] = uc;
        if (u_dbg) u_dbg[idx] = u;
        StepResult o;
        if constexpr (FINAL) {
            env_step<U>(s, a, reward_scale, P, T, o, stats, nullptr, nullptr, nullptr, fs.obs);
            final_slots_step(fs, o.truncated, t, n_slots, n_envs);
        } else {
            env_step<U>(s, a, reward_scale, P, T, o, stats);
        }
        rew_buf[idx] = o.reward;
#pragma unroll
        for (int i = 0; i < kObsDim; ++i) obs[i] = o.obs[i];
        tc = o.terminated ? 1.0f : 0.0f;
        uc = o.truncated ? 1.0f : 0.0f;
    }
    pos[e] = make_double2(s.px, s.py);
    vel[e] = make_double2(s.vx, s.vy);
    ints[e] = make_int4(s.k, s.t, s.next_gate, s.passed);
    {
        float2 *dst = reinterpret_cast<float2 *>(cur_obs + (size_t)e * kObsDim);
#pragma unroll
        for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(obs[2 * i], obs[2 * i + 1]);
    }
    cur_term[e] = tc;
    cur_trunc[e] = uc;
    if constexpr (FINAL) final_slots_end(fs, n_slots, n_envs);
    if (last_val) {                                          // bootstrap value of the state after the rollout
        policy_forward(obs, sw, po);
        last_val[e] = po.value;
    }
}

// ---- fused rollout, tensor-core version: packed weights ----------------------------------------------------------
// k_policy_rollout_tc3 (below) runs the two 18->256 layers (23.6 of the 29 kflop per env-step) on the 5th-gen tensor
// cores.  Its packed weights hold the first layer of each net as a K-major UMMA B operand (256 units x 24 K, the bias
// in column 18), split into TF32 hi and lo parts for 3xTF32 products, followed by the second layers for the CUDA cores.
constexpr int kTcBFloats = tc::kTileN * tc::kK;              // 6,144 floats per B operand
constexpr int kTcW2Off = 4 * kTcBFloats;                     // [actor hi | actor lo | critic hi | critic lo]
constexpr int kTcW2cOff = kTcW2Off + kHidden * 10;           // W2 actor as [j][5] pairs, then w2c[j]
constexpr int kTcTailOff = kTcW2cOff + kHidden;              // b2[0..9], b2c, pad
constexpr int kTcWeightFloats = kTcTailOff + 12;             // 27,404 floats

// ---- populations of independent members (POP instantiations, carenv_policy_rollout_*_pop) ----------------------
// Member p's parameters in stacked nn.Linear-layout tensors [P][256][18], [P][256], [P][9][256], [P][9], ...
__device__ __forceinline__ ppo::Params member_params(const ppo::Params &W, int p) {
    const size_t q = (size_t)p;
    return ppo::Params{W.w1a + q * kHidden * kObsDim, W.b1a + q * kHidden, W.w2a + q * kActions * kHidden,
                       W.b2a + q * kActions,          W.w1c + q * kHidden * kObsDim, W.b1c + q * kHidden,
                       W.w2c + q * kHidden,           W.b2c + q};
}

// Critic pass over the final-observation slots (carenv_final_values): thread i = slot k * N + column c; a used slot
// (0 <= final_row[k][c] < n_rows) gets boot[final_row[k][c]][c] = critic(final_obs[k][c]), float32 CUDA cores.  Column c
// belongs to member c / n_per_member of stacked nn.Linear critic tensors (one policy: n_per_member = N), and each
// thread reads only its member's parameters, so a member's values do not depend on the others.
__global__ void __launch_bounds__(128)
k_final_values(const ppo::Params W, const float *__restrict__ final_obs, const int *__restrict__ final_row, int n_slots,
               int N, int n_per_member, int n_rows, float *__restrict__ boot) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n_slots * N) return;
    const int row = final_row[i];
    if (row < 0 || row >= n_rows) return;
    const int c = (int)(i % N);
    const ppo::Params m = member_params(W, c / n_per_member);
    float x[kObsDim];
    {
        const float2 *src = reinterpret_cast<const float2 *>(final_obs + (size_t)i * kObsDim);
#pragma unroll
        for (int k = 0; k < kObsDim / 2; ++k) { const float2 v = src[k]; x[2 * k] = v.x; x[2 * k + 1] = v.y; }
    }
    float v0 = 0.0f, v1 = 0.0f;
#pragma unroll 2
    for (int j = 0; j < kHidden; ++j) {
        const float *w = m.w1c + j * kObsDim;
        float h = __ldg(m.b1c + j);
#pragma unroll
        for (int k = 0; k < kObsDim; ++k) h = fmaf(__ldg(w + k), x[k], h);
        if (j & 1) v1 = fmaf(__ldg(m.w2c + j), fmaxf(h, 0.0f), v1);
        else v0 = fmaf(__ldg(m.w2c + j), fmaxf(h, 0.0f), v0);
    }
    boot[(size_t)row * N + c] = (v0 + v1) + __ldg(m.b2c);
}

// Moves every per-environment pointer to column col0 (the member's first environment): afterwards the kernel indexes
// them with the member-local env e and, for the [T, N] rows, with the population's row stride N.  FINAL: the
// final-observation slots [S][N](,18) as well.
template <bool FINAL>
__device__ __forceinline__ void pop_shift_columns(int col0, double2 *__restrict__ &pos, double2 *__restrict__ &vel,
                                                  int4 *__restrict__ &ints, float *__restrict__ &cur_obs,
                                                  float *__restrict__ &cur_term, float *__restrict__ &cur_trunc,
                                                  float *__restrict__ &last_val, float *__restrict__ &obs_buf,
                                                  float *__restrict__ &act_buf, float *__restrict__ &rew_buf,
                                                  float *__restrict__ &val_buf, float *__restrict__ &term_buf,
                                                  float *__restrict__ &trunc_buf, float *__restrict__ &logp_buf,
                                                  float *__restrict__ &u_dbg, float *__restrict__ &final_obs,
                                                  int *__restrict__ &final_row) {
    const size_t c = (size_t)col0;
    pos += c; vel += c; ints += c;
    cur_obs += c * kObsDim; cur_term += c; cur_trunc += c;
    if (last_val) last_val += c;
    obs_buf += c * kObsDim;                                  // full observation rows only (the launchers refuse poses)
    act_buf += c; rew_buf += c; val_buf += c; term_buf += c; trunc_buf += c; logp_buf += c;
    if (u_dbg) u_dbg += c;
    if constexpr (FINAL) {
        final_obs += c * kObsDim;
        final_row += c;
    }
}

// Packing of the reference network's parameters (nn.Linear layout: weight [out][in], lib/model.py:10-26) into the
// two layouts above, one thread per packed float: runs after every optimiser epoch, so it is one launch and not
// forty small tensor operations (13 ms per epoch in PyTorch, as much as the rollout of 32,768 envs x 1,024 steps).
// POP (carenv_pack_policy_pop): blockIdx.y = member p of stacked parameters [P][...], output block p of [P][floats].
template <bool TC, bool POP = false>
__global__ void __launch_bounds__(256)
k_pack_policy(const float *__restrict__ w1a, const float *__restrict__ b1a, const float *__restrict__ w2a,
              const float *__restrict__ b2a, const float *__restrict__ w1c, const float *__restrict__ b1c,
              const float *__restrict__ w2c, const float *__restrict__ b2c, float *__restrict__ out) {
    if constexpr (POP) {
        const ppo::Params m = member_params(ppo::Params{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c}, blockIdx.y);
        w1a = m.w1a; b1a = m.b1a; w2a = m.w2a; b2a = m.b2a; w1c = m.w1c; b1c = m.b1c; w2c = m.w2c; b2c = m.b2c;
        out += (size_t)blockIdx.y * (TC ? kTcWeightFloats : kPolicyFloats);
    }
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float v = 0.0f;
    if (TC) {
        if (i >= kTcWeightFloats) return;
        if (i < 4 * kTcBFloats) {                            // [actor hi | actor lo | critic hi | critic lo], UMMA layout
            const int which = i / kTcBFloats, r = i % kTcBFloats;
            const int j = (r / 192) * 8 + (r % 32) / 4, k = ((r % 192) / 32) * 4 + r % 4;
            const float *w1 = which < 2 ? w1a : w1c, *b1 = which < 2 ? b1a : b1c;
            const float x = k < kObsDim ? w1[j * kObsDim + k] : (k == kObsDim ? b1[j] : 0.0f);
            const float hi = tc::to_tf32(x);
            v = (which & 1) ? tc::to_tf32(x - hi) : hi;
        } else if (i < kTcW2cOff) {                          // actor second layer as [j][10] (q = 9 is padding)
            const int r = i - kTcW2Off, j = r / 10, q = r % 10;
            v = q < kActions ? w2a[q * kHidden + j] : 0.0f;
        } else if (i < kTcTailOff) {
            v = w2c[i - kTcW2cOff];
        } else {
            const int r = i - kTcTailOff;                    // b2[0..8], 0, b2c, 0
            v = r < kActions ? b2a[r] : (r == 10 ? b2c[0] : 0.0f);
        }
    } else {
        if (i >= kPolicyFloats) return;
        constexpr int kBody = (kHidden / 2) * kPairFloats;
        if (i < kBody) {
            const int p = i / kPairFloats, r = i % kPairFloats;   // pair of hidden units (2p, 2p + 1)
            const bool critic = r >= kActorPairFloats;
            const int c = critic ? r - kActorPairFloats : r;
            const float *w1 = critic ? w1c : w1a, *b1 = critic ? b1c : b1a;
            if (c < 36) v = w1[(2 * p + (c & 1)) * kObsDim + (c >> 1)];
            else if (c < 38) v = b1[2 * p + (c - 36)];
            else if (c >= 40) {
                const int d = c - 40;
                if (!critic) {                               // (W2[2q][j], W2[2q+1][j]) for j = 2p, 2p + 1
                    const int q = d >> 2, sft = (d >> 1) & 1, rr = d & 1, row = 2 * q + rr;
                    v = row < kActions ? w2a[row * kHidden + 2 * p + sft] : 0.0f;
                } else if (d < 2) {
                    v = w2c[2 * p + d];
                }
            }
        } else {
            const int r = i - kBody;
            v = r < kActions ? b2a[r] : (r == 10 ? b2c[0] : 0.0f);
        }
    }
    out[i] = v;
}

// Two hidden units (h0, h1) of the actor through the 256 -> 9 layer: w = their ten weight pairs as five float4
// ([unit][5] float2 layout), L[q] = logits (2q, 2q + 1).
__device__ __forceinline__ void second_layer_pair(float h0, float h1, const float4 (&w)[5], float2 (&L)[5]) {
    L[0] = __ffma2_rn(make_float2(h0, h0), make_float2(w[0].x, w[0].y), L[0]);
    L[1] = __ffma2_rn(make_float2(h0, h0), make_float2(w[0].z, w[0].w), L[1]);
    L[2] = __ffma2_rn(make_float2(h0, h0), make_float2(w[1].x, w[1].y), L[2]);
    L[3] = __ffma2_rn(make_float2(h0, h0), make_float2(w[1].z, w[1].w), L[3]);
    L[4] = __ffma2_rn(make_float2(h0, h0), make_float2(w[2].x, w[2].y), L[4]);
    L[0] = __ffma2_rn(make_float2(h1, h1), make_float2(w[2].z, w[2].w), L[0]);
    L[1] = __ffma2_rn(make_float2(h1, h1), make_float2(w[3].x, w[3].y), L[1]);
    L[2] = __ffma2_rn(make_float2(h1, h1), make_float2(w[3].z, w[3].w), L[2]);
    L[3] = __ffma2_rn(make_float2(h1, h1), make_float2(w[4].x, w[4].y), L[3]);
    L[4] = __ffma2_rn(make_float2(h1, h1), make_float2(w[4].z, w[4].w), L[4]);
}

// ---- fused rollout, tensor cores, every second-layer weight load shared by TWO environments --------------------
// Same contract as k_policy_rollout.  Per step every environment thread writes its observation row (hi/lo TF32 split,
// a constant 1 in column 18 carries the bias) into the K-major UMMA operand tile of its 128-env group, one elected
// thread issues tcgen05.mma kind::tf32 — D = A_hi*B_hi + A_lo*B_hi + A_hi*B_lo (3xTF32: float32-level accuracy) — into
// tensor memory, and the threads read their rows of pre-activations back with tcgen05.ld and run ReLU and the second
// layers on the CUDA cores (FFMA2).
// The 256 -> 9 layer is bound by the shared-memory RETURN path (ncu, DESIGN.md §7 "Round 2"): a broadcast
// LDS.128 delivers 16 bytes to 32 lanes in two wavefronts, i.e. the weights of ONE packed FFMA2 per cycle and SM, half
// of what the FMA pipes take — and all warps run that phase together because their MMAs complete together (with one
// environment per weight load the pipe is ~100 % busy for 11k of a step's 29k cycles).  So here every weight load
// feeds two environments: the environment thread of lane r in group 0 runs hidden units 0..127 for BOTH environments
// on TMEM lane r (group 0's and group 1's columns), its twin in group 1 runs units 128..255 for both, and the two
// exchange the partial logits of each other's environment through shared memory.  The loads are software-pipelined
// by hand (the next pair of hidden units' weights in flight as ordered volatile loads; left to itself the compiler
// issues each load right before its first use).  The critic is done by 128 critic threads, lane r for both
// environments of the lane as well, off the critical path.  One CTA = 256 environment threads + 128 critic threads +
// the issuer warp (13 warps, 128 registers each at launch; the critic warps hand 64 of theirs to the environment
// warps).  Logits = (units 0..127) + (units 128..255) + bias, the same operands in the same order on both threads of
// a lane; value = (even units + odd units) + bias.
// U == 0 is the multi-track instantiation (carenv_policy_rollout_tc_multi): each environment thread reads
// track_ids[e] once and steps with env_step<0> on that track's TrackParams / Tables in global memory (the arrays of
// the multi-track handle), as k_rollout_multi does; no track tables are staged and P / G are unused.  Tracks may
// differ within a warp: the barrier protocol does not care, every environment thread still arrives once per phase.
__device__ __forceinline__ void second_layer_chunk16_x2(uint32_t a, const float (&va)[16], const float (&vb)[16],
                                                        float2 (&La)[5], float2 (&Lb)[5]) {
    float4 wa[5], wb[5];
#pragma unroll
    for (int r = 0; r < 5; ++r) wa[r] = tc::lds128(a + 16u * r);
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
#pragma unroll
        for (int r = 0; r < 5; ++r) wb[r] = tc::lds128(a + 80u * (i + 1) + 16u * r);
        second_layer_pair(fmaxf(va[2 * i], 0.0f), fmaxf(va[2 * i + 1], 0.0f), wa, La);
        second_layer_pair(fmaxf(vb[2 * i], 0.0f), fmaxf(vb[2 * i + 1], 0.0f), wa, Lb);
        if (i + 2 < 8) {
#pragma unroll
            for (int r = 0; r < 5; ++r) wa[r] = tc::lds128(a + 80u * (i + 2) + 16u * r);
        }
        second_layer_pair(fmaxf(va[2 * i + 2], 0.0f), fmaxf(va[2 * i + 3], 0.0f), wb, La);
        second_layer_pair(fmaxf(vb[2 * i + 2], 0.0f), fmaxf(vb[2 * i + 3], 0.0f), wb, Lb);
    }
}

// POP (carenv_policy_rollout_tc_pop, single-track U only): blockIdx.y = member p, as in k_policy_rollout_warp<true>:
// packed weights [P][kTcWeightFloats], seeds[p], n_envs environments per member at columns p * n_envs + e of arrays
// with row_stride columns.
// FINAL: final-observation slots (final_slots_begin above); only active threads write.
template <int U, bool TAB, bool POP = false, bool FINAL = false>
__global__ void __launch_bounds__(256 + 128 + 32, 1)
k_policy_rollout_tc3(const __grid_constant__ TrackParams P, const Tables G, const float *__restrict__ weights,
                     int n_envs, int n_steps, int env_offset, unsigned long long seed, unsigned long long step0,
                     double2 *__restrict__ pos, double2 *__restrict__ vel, int4 *__restrict__ ints,
                     float *__restrict__ cur_obs, float *__restrict__ cur_term, float *__restrict__ cur_trunc,
                     double reward_scale, float *__restrict__ obs_buf, float *__restrict__ act_buf,
                     float *__restrict__ rew_buf, float *__restrict__ val_buf, float *__restrict__ term_buf,
                     float *__restrict__ trunc_buf, float *__restrict__ logp_buf, float *__restrict__ last_val,
                     float *__restrict__ u_dbg, unsigned long long *stats, int table_bytes, int obs_mode,
                     const float4 *__restrict__ den4, int n_pairs, int row_f4, const TrackParams *__restrict__ mt_params,
                     const Tables *__restrict__ mt_tables, int n_tracks, const int *__restrict__ track_ids,
                     const unsigned long long *__restrict__ seeds, int row_stride, float *__restrict__ final_obs,
                     int *__restrict__ final_row, int n_slots) {
    static_assert(!POP || U != 0, "populations run on one track");
    constexpr int kGroups = 2, kCols = 256, kHalf = 128, kEnvThreads = kGroups * 128, kCriticThreads = 128;
    extern __shared__ __align__(16) unsigned char smem[];
    int stride = n_envs;
    if constexpr (POP) {
        const int p = blockIdx.y;
        weights += (size_t)p * kTcWeightFloats;
        seed = seeds[p];
        stride = row_stride;
        pop_shift_columns<FINAL>(p * n_envs, pos, vel, ints, cur_obs, cur_term, cur_trunc, last_val, obs_buf, act_buf, rew_buf,
                          val_buf, term_buf, trunc_buf, logp_buf, u_dbg, final_obs, final_row);
    }
    // [tables | pad to a 128-byte boundary | weights | A tiles (hi, lo per group) | exchanged partial logits [group][128][12]
    //  | TAB: the denominator table of k_rollout_tab, ONE copy whose rows are skewed by 16 bytes (row_f4 is odd in
    //    16-byte units): threads of a quarter warp with different headings mostly hit different bank groups (about
    //    2.6 instead of 1 wavefront per quarter — there is no room for the eight conflict-free copies) — this replaces
    //    the 144 x (DMUL + DFMA + F2F) per env-step that the arithmetic kernels spend on the same values]
    const int w_off = (int)((tc::smem_u32(smem) + (uint32_t)table_bytes + 127u) / 128u * 128u - tc::smem_u32(smem));
    float *sw = reinterpret_cast<float *>(smem + w_off);
    unsigned char *sA = smem + w_off + ((kTcWeightFloats * 4 + 127) / 128 * 128);
    float *s_xchg = reinterpret_cast<float *>(sA + kGroups * 2 * tc::kABytes);
    float4 *s_tab = reinterpret_cast<float4 *>(s_xchg + kGroups * 128 * 12);
    if (TAB)
        for (int i = threadIdx.x; i < kHeadings * n_pairs; i += blockDim.x) {
            const int k = i / n_pairs, jp = i - k * n_pairs;
            s_tab[k * row_f4 + jp] = den4[i];
        }
    const TabView tv{s_tab, row_f4};
    __shared__ __align__(8) unsigned long long mb_rows, mb_full_lo, mb_full_hi, mb_cons_a, mb_full_c, mb_cons_c, mb_xchg;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    for (int i = tid; i < kTcWeightFloats / 4; i += blockDim.x)
        reinterpret_cast<float4 *>(sw)[i] = reinterpret_cast<const float4 *>(weights)[i];
    if (tid == 0) {
        tc::mbar_init(tc::smem_u32(&mb_rows), kEnvThreads);
        tc::mbar_init(tc::smem_u32(&mb_full_lo), 1);
        tc::mbar_init(tc::smem_u32(&mb_full_hi), 1);
        tc::mbar_init(tc::smem_u32(&mb_cons_a), kEnvThreads);
        tc::mbar_init(tc::smem_u32(&mb_full_c), 1);
        tc::mbar_init(tc::smem_u32(&mb_cons_c), kCriticThreads);
        tc::mbar_init(tc::smem_u32(&mb_xchg), kEnvThreads);
    }
    if (warp == 0) tc::tmem_alloc<512>(&tmem_slot);
    // U == 0 (several tracks): nothing is staged, every environment thread reads its own track's tables
    const Tables T = U == 0 ? Tables{} : stage_tables(G, P.n_gates, P.n_seg, smem);   // ends with __syncthreads()
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tbase = tmem_slot;
    const int n_forward = n_steps + (last_val ? 1 : 0);
    const uint32_t b_rows = tc::smem_u32(&mb_rows), b_full_lo = tc::smem_u32(&mb_full_lo), b_full_hi = tc::smem_u32(&mb_full_hi);
    const uint32_t b_cons_a = tc::smem_u32(&mb_cons_a), b_full_c = tc::smem_u32(&mb_full_c), b_cons_c = tc::smem_u32(&mb_cons_c);
    const uint32_t b_xchg = tc::smem_u32(&mb_xchg);

    if (warp == (kEnvThreads + kCriticThreads) / 32) {
        // ===== MMA issuer (one lane); both groups advance together (their threads share the weight loads) =====
        if ((tid & 31) == 0) {
            const uint32_t sB = tc::smem_u32(sw);
            const uint32_t idesc_half = tc::make_idesc_tf32(128, kHalf), idesc_full = tc::make_idesc_tf32(128, kCols);
            auto issue = [&](uint32_t d, uint32_t ah, uint32_t bh, uint32_t idesc) {     // D = Ah*Bh + Al*Bh + Ah*Bl
                const uint32_t al = ah + tc::kABytes, bl = bh + (uint32_t)(kTcBFloats * 4);
#pragma unroll
                for (int pr = 0; pr < 3; ++pr) {
                    const uint32_t a0 = (pr == 1) ? al : ah, b0 = (pr == 2) ? bl : bh;
#pragma unroll
                    for (int ks = 0; ks < tc::kK / 8; ++ks)
                        tc::mma_tf32(d, tc::make_smem_desc(a0 + ks * 2 * tc::kLBO), tc::make_smem_desc(b0 + ks * 2 * tc::kLBO),
                                     idesc, (pr | ks) != 0);
                }
            };
            const uint32_t a0 = tc::smem_u32(sA), a1 = a0 + 2 * tc::kABytes;
            const uint32_t b_hi_half = sB + (uint32_t)((kHalf / 8) * tc::kSBO), b_critic = sB + (uint32_t)(2 * kTcBFloats * 4);
            for (int f = 0; f < n_forward; ++f) {
                const uint32_t par = (uint32_t)(f & 1);
                tc::mbar_wait(b_rows, par);                          // this pass's operand rows are written
                if (f > 0) tc::mbar_wait(b_cons_c, par ^ 1u);        // the previous pass's critic columns are read out
                tc::tc_fence_after();
                issue(tbase, a0, sB, idesc_half);                    // actor units 0..127, both groups
                issue(tbase + kCols, a1, sB, idesc_half);
                tc::mma_commit(b_full_lo);
                issue(tbase + kHalf, a0, b_hi_half, idesc_half);     // actor units 128..255, both groups
                issue(tbase + kCols + kHalf, a1, b_hi_half, idesc_half);
                tc::mma_commit(b_full_hi);
                tc::mbar_wait(b_cons_a, par);                        // the actor columns are read out
                tc::tc_fence_after();
                issue(tbase, a0, b_critic, idesc_full);              // critic, 256 units, both groups
                issue(tbase + kCols, a1, b_critic, idesc_full);
                tc::mma_commit(b_full_c);
            }
        }
    } else if (warp >= kEnvThreads / 32) {
        // ===== critic threads: lane r's two environments, every weight load used twice =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 64;\n");
        const int row = tid - kEnvThreads;
        const uint32_t lane_tmem = tbase + ((uint32_t)((warp & 3) * 32) << 16);
        const int ea_raw = blockIdx.x * kEnvThreads + row, eb_raw = ea_raw + 128;
        const float4 *wc = reinterpret_cast<const float4 *>(sw + kTcW2cOff);
        const float bias = sw[kTcTailOff + 10];
        for (int f = 0; f < n_forward; ++f) {
            tc::mbar_wait(b_full_c, (uint32_t)(f & 1));
            tc::tc_fence_after();
            float2 Va = make_float2(0.0f, 0.0f), Vb = make_float2(0.0f, 0.0f);
#pragma unroll 1
            for (int c = 0; c < kCols; c += 16) {
                float va[16], vb[16];
                tc::tmem_ld16(lane_tmem + c, va);
                tc::tmem_ld16(lane_tmem + kCols + c, vb);
                if (c + 16 == kCols) { tc::tc_fence_before(); tc::mbar_arrive(b_cons_c); }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 w = wc[c / 4 + i];
                    Va = __ffma2_rn(make_float2(fmaxf(va[4 * i], 0.0f), fmaxf(va[4 * i + 1], 0.0f)), make_float2(w.x, w.y), Va);
                    Vb = __ffma2_rn(make_float2(fmaxf(vb[4 * i], 0.0f), fmaxf(vb[4 * i + 1], 0.0f)), make_float2(w.x, w.y), Vb);
                    Va = __ffma2_rn(make_float2(fmaxf(va[4 * i + 2], 0.0f), fmaxf(va[4 * i + 3], 0.0f)), make_float2(w.z, w.w), Va);
                    Vb = __ffma2_rn(make_float2(fmaxf(vb[4 * i + 2], 0.0f), fmaxf(vb[4 * i + 3], 0.0f)), make_float2(w.z, w.w), Vb);
                }
            }
            const float value_a = (Va.x + Va.y) + bias, value_b = (Vb.x + Vb.y) + bias;
            if (f < n_steps) {
                if (ea_raw < n_envs) val_buf[(size_t)f * (size_t)stride + (size_t)ea_raw] = value_a;
                if (eb_raw < n_envs) val_buf[(size_t)f * (size_t)stride + (size_t)eb_raw] = value_b;
            } else {                                                 // bootstrap values of the final observations
                if (ea_raw < n_envs) last_val[ea_raw] = value_a;
                if (eb_raw < n_envs) last_val[eb_raw] = value_b;
            }
        }
    } else {
        // ===== environment threads =====
        asm volatile("setmaxnreg.inc.sync.aligned.u32 160;\n");
        const int group = tid >> 7, row = tid & 127;
        const int e_raw = blockIdx.x * kEnvThreads + tid;
        const bool active = e_raw < n_envs;
        const int e = active ? e_raw : n_envs - 1;           // idle threads shadow the last env (no stores)
        // U == 0: this environment's track, its constants and tables read through pointers as in k_rollout_multi
        const int tr = U == 0 ? min(max(track_ids[e], 0), n_tracks - 1) : 0;
        const TrackParams &PE = U == 0 ? mt_params[tr] : P;
        const Tables TE = U == 0 ? mt_tables[tr] : T;
        const uint32_t lane_tmem = tbase + ((uint32_t)((warp & 3) * 32) << 16);
        const uint32_t w2s = tc::smem_u32(sw + kTcW2Off) + (uint32_t)(group * kHalf) * 40u;   // this thread's 128 hidden units
        const uint32_t b_full_mine = group == 0 ? b_full_lo : b_full_hi;
        float *xchg_out = s_xchg + (size_t)((1 - group) * 128 + row) * 12;    // partial logits of the OTHER group's lane-r env
        const float *xchg_in = s_xchg + (size_t)(group * 128 + row) * 12;
        unsigned char *myA = sA + group * 2 * tc::kABytes;   // hi tile, then lo tile
        const float *tail = sw + kTcTailOff;
        EnvState s;
        {
            const double2 p = pos[e], v = vel[e];
            const int4 q = ints[e];
            s.px = p.x; s.py = p.y; s.vx = v.x; s.vy = v.y;
            s.k = q.x; s.t = q.y; s.next_gate = q.z; s.passed = q.w;
        }
        float obs[kObsDim];
        {
            const float2 *src = reinterpret_cast<const float2 *>(cur_obs + (size_t)e * kObsDim);
#pragma unroll
            for (int i = 0; i < kObsDim / 2; ++i) { const float2 v = src[i]; obs[2 * i] = v.x; obs[2 * i + 1] = v.y; }
        }
        float tc_ = cur_term[e], uc = cur_trunc[e];
        const uint32_t gid = (uint32_t)(env_offset + e);
        FinalSlots fs{};
        if constexpr (FINAL) fs = final_slots_begin(active, final_obs, final_row, n_slots, e);

        auto write_row = [&](int f) {
            if (f > 0) tc::mbar_wait(b_full_c, (uint32_t)((f - 1) & 1));   // the previous pass's MMAs have read the tile
#pragma unroll
            for (int c = 0; c < tc::kKChunks; ++c) {
                float hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int k = 4 * c + j;
                    const float x = k < kObsDim ? obs[k < kObsDim ? k : 0] : (k == kObsDim ? 1.0f : 0.0f);
                    hi[j] = tc::to_tf32(x);
                    lo[j] = tc::to_tf32(x - hi[j]);
                }
                const int off = tc::operand_offset(row, 4 * c);
                *reinterpret_cast<float4 *>(myA + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<float4 *>(myA + tc::kABytes + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
            }
            tc::fence_async_smem();
            tc::mbar_arrive(b_rows);
        };

        for (int t = 0; t < n_steps; ++t) {
            const size_t idx = (size_t)t * (size_t)stride + (size_t)e;
            const uint32_t par = (uint32_t)(t & 1);
            write_row(t);
            const unsigned long long gs = step0 + (unsigned long long)t;
            const uint32_t bits = philox_uniform_bits((uint32_t)seed, (uint32_t)(seed >> 32), gid, (uint32_t)gs,
                                                      (uint32_t)(gs >> 32), 0x43415245u);
            const float u = (float)(bits >> 8) * (1.0f / 16777216.0f);
            if (active) {
                if (obs_mode == kObsPose) {
                    store_pose(reinterpret_cast<PoseRec *>(obs_buf) + idx, s, obs[2], obs[3]);
                } else {
                    float2 *dst = reinterpret_cast<float2 *>(obs_buf + idx * kObsDim);
#pragma unroll
                    for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(obs[2 * i], obs[2 * i + 1]);
                }
                term_buf[idx] = tc_;
                trunc_buf[idx] = uc;
                if (u_dbg) u_dbg[idx] = u;
            }
            // my 128 hidden units for the two environments of TMEM lane r (a = group 0's, b = group 1's)
            float2 La[5], Lb[5];
#pragma unroll
            for (int q = 0; q < 5; ++q) { La[q] = make_float2(0.0f, 0.0f); Lb[q] = make_float2(0.0f, 0.0f); }
            tc::mbar_wait(b_full_mine, par);
            tc::tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < kHalf; c += 16) {
                float va[16], vb[16];
                tc::tmem_ld16(lane_tmem + group * kHalf + c, va);
                tc::tmem_ld16(lane_tmem + kCols + group * kHalf + c, vb);
                if (c + 16 == kHalf) { tc::tc_fence_before(); tc::mbar_arrive(b_cons_a); }   // my columns are read out
                second_layer_chunk16_x2(w2s + (uint32_t)c * 40u, va, vb, La, Lb);
            }
            {   // hand the other environment's partial logits to its thread, take mine
                const float2 *o = group == 0 ? Lb : La;
                reinterpret_cast<float4 *>(xchg_out)[0] = make_float4(o[0].x, o[0].y, o[1].x, o[1].y);
                reinterpret_cast<float4 *>(xchg_out)[1] = make_float4(o[2].x, o[2].y, o[3].x, o[3].y);
                reinterpret_cast<float2 *>(xchg_out)[4] = o[4];
            }
            tc::mbar_arrive(b_xchg);
            tc::mbar_wait(b_xchg, par);
            PolicyOut po;
            {
                const float2 *m = group == 0 ? La : Lb;
                const float4 p0 = reinterpret_cast<const float4 *>(xchg_in)[0], p1 = reinterpret_cast<const float4 *>(xchg_in)[1];
                const float2 p2 = reinterpret_cast<const float2 *>(xchg_in)[4];
                const float r[10] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w, p2.x, p2.y};
#pragma unroll
                for (int q = 0; q < 5; ++q) {
                    // (units 0..127) + (units 128..255): the same operands in the same order on both threads
                    const float lo0 = group == 0 ? m[q].x : r[2 * q], hi0 = group == 0 ? r[2 * q] : m[q].x;
                    const float lo1 = group == 0 ? m[q].y : r[2 * q + 1], hi1 = group == 0 ? r[2 * q + 1] : m[q].y;
                    po.logit[2 * q] = (lo0 + hi0) + tail[2 * q];
                    po.logit[2 * q + 1] = (lo1 + hi1) + tail[2 * q + 1];
                }
                po.value = 0.0f;
            }
            float logp, us;
            const int a = sample_action(po, u, logp, us);
            if (active) {
                act_buf[idx] = (float)a;
                logp_buf[idx] = logp;
            }
            StepResult o;
            if constexpr (FINAL) {
                env_step<U, TAB>(s, a, reward_scale, PE, TE, o, active ? stats : nullptr, nullptr, TAB ? &tv : nullptr,
                                 nullptr, fs.obs);
                final_slots_step(fs, o.truncated, t, n_slots, stride);
            } else {
                env_step<U, TAB>(s, a, reward_scale, PE, TE, o, active ? stats : nullptr, nullptr, TAB ? &tv : nullptr);
            }
            if (active) rew_buf[idx] = o.reward;
#pragma unroll
            for (int i = 0; i < kObsDim; ++i) obs[i] = o.obs[i];
            tc_ = o.terminated ? 1.0f : 0.0f;
            uc = o.truncated ? 1.0f : 0.0f;
        }
        if (last_val) {                                          // one more pass: the critic threads write the bootstrap values
            write_row(n_steps);
            tc::mbar_wait(b_full_mine, (uint32_t)(n_steps & 1));
            tc::tc_fence_before();
            tc::mbar_arrive(b_cons_a);
        }
        if (active) {
            pos[e] = make_double2(s.px, s.py);
            vel[e] = make_double2(s.vx, s.vy);
            ints[e] = make_int4(s.k, s.t, s.next_gate, s.passed);
            float2 *dst = reinterpret_cast<float2 *>(cur_obs + (size_t)e * kObsDim);
#pragma unroll
            for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(obs[2 * i], obs[2 * i + 1]);
            cur_term[e] = tc_;
            cur_trunc[e] = uc;
        }
        if constexpr (FINAL) final_slots_end(fs, n_slots, stride);
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tbase);
}

// ---- fused rollout for small batches: one WARP per environment --------------------------------------------------
// The reference's own training shape is 24 environments (README: "about 35 minutes" for 200 epochs).  There a
// thread-per-environment kernel is one long dependent chain on a nearly empty GPU (12 us per step in
// k_policy_rollout_tc3).  Here a warp owns one environment, as in k_rollout_warp: lane j carries wall segment j
// through the env step (per-ray extrema by integer REDUX) and, for the policy, hidden units j, j + 32, ... of both
// nets (16 units per lane: first layer from shared-memory rows [unit][20] — conflict-free for consecutive lanes —,
// ReLU, its share of the 256 -> 9 / 256 -> 1 sums), the ten partial sums are folded over the warp by an xor
// butterfly (every lane ends with the same bits), every lane samples the same action.  Float32 CUDA cores only:
// at 24 environments the tensor core has nothing to amortise its latency over.  The network parameters are read in
// nn.Linear layout (no packing launch).
constexpr int kWpRow = 20;                                   // first-layer row: 18 weights, bias, pad
constexpr int kWpW2 = 12;                                    // actor second-layer row: W2[0..8][j], pad
constexpr int kWpFloats = 2 * kHidden * kWpRow + kHidden * kWpW2 + kHidden + 12;   // 13,580 floats = 54,320 B

// POP (carenv_policy_rollout_warp_pop): a population of independent members, blockIdx.y = member p.  W points at the
// stacked parameters [P][...] of all members, seeds[p] keys member p's random stream, n_envs is the member's
// environment count and env e of member p is global column p * n_envs + e of every [N] and [T, N] array
// (row_stride = N).  The CTA stages member p's parameters and otherwise runs the single-policy code unchanged, so
// member p's rows are those of k_policy_rollout_warp<false> on that member alone with env_offset = 0.
// FINAL: final-observation slots (final_slots_begin above), written by lane 0.
template <bool POP, bool FINAL = false>
__global__ void __launch_bounds__(128)
k_policy_rollout_warp(const __grid_constant__ TrackParams P, const Tables G, const ppo::Params W, int n_envs, int n_steps,
                      int env_offset, unsigned long long seed, unsigned long long step0, double2 *__restrict__ pos,
                      double2 *__restrict__ vel, int4 *__restrict__ ints, float *__restrict__ cur_obs,
                      float *__restrict__ cur_term, float *__restrict__ cur_trunc, double reward_scale,
                      float *__restrict__ obs_buf, float *__restrict__ act_buf, float *__restrict__ rew_buf,
                      float *__restrict__ val_buf, float *__restrict__ term_buf, float *__restrict__ trunc_buf,
                      float *__restrict__ logp_buf, float *__restrict__ last_val, float *__restrict__ u_dbg,
                      unsigned long long *stats, int table_bytes, int obs_mode, const unsigned long long *__restrict__ seeds,
                      int row_stride, float *__restrict__ final_obs, int *__restrict__ final_row, int n_slots) {
    extern __shared__ __align__(16) unsigned char smem[];
    ppo::Params Wm = W;
    int stride = n_envs;
    if constexpr (POP) {
        const int p = blockIdx.y;
        Wm = member_params(W, p);
        seed = seeds[p];
        stride = row_stride;
        pop_shift_columns<FINAL>(p * n_envs, pos, vel, ints, cur_obs, cur_term, cur_trunc, last_val, obs_buf, act_buf, rew_buf,
                          val_buf, term_buf, trunc_buf, logp_buf, u_dbg, final_obs, final_row);
    }
    float *sw1 = reinterpret_cast<float *>(smem + table_bytes);   // [512][20]: rows 0..255 actor, 256..511 critic
    float *sw2 = sw1 + 2 * kHidden * kWpRow;                      // [256][12]
    float *swc = sw2 + kHidden * kWpW2;                           // [256]
    float *stail = swc + kHidden;                                 // b2a[0..8], 0, b2c, 0
    for (int i = threadIdx.x; i < 2 * kHidden * kWpRow; i += blockDim.x) {
        const int r = i / kWpRow, c = i - r * kWpRow, j = r & (kHidden - 1);
        const float *w1 = r < kHidden ? Wm.w1a : Wm.w1c, *b1 = r < kHidden ? Wm.b1a : Wm.b1c;
        sw1[i] = c < kObsDim ? w1[j * kObsDim + c] : (c == kObsDim ? b1[j] : 0.0f);
    }
    for (int i = threadIdx.x; i < kHidden * kWpW2; i += blockDim.x) {
        const int j = i / kWpW2, q = i - j * kWpW2;
        sw2[i] = q < kActions ? Wm.w2a[q * kHidden + j] : 0.0f;
    }
    for (int i = threadIdx.x; i < kHidden; i += blockDim.x) swc[i] = Wm.w2c[i];
    if (threadIdx.x < 12) stail[threadIdx.x] = threadIdx.x < kActions ? Wm.b2a[threadIdx.x] : (threadIdx.x == 10 ? Wm.b2c[0] : 0.0f);
    const Tables T = stage_tables(G, P.n_gates, P.n_seg, smem);      // ends with __syncthreads()
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
    float obs[kObsDim];
    {
        const float2 *src = reinterpret_cast<const float2 *>(cur_obs + (size_t)e * kObsDim);
#pragma unroll
        for (int i = 0; i < kObsDim / 2; ++i) { const float2 v = src[i]; obs[2 * i] = v.x; obs[2 * i + 1] = v.y; }
    }
    float tc_ = cur_term[e], uc = cur_trunc[e];
    const uint32_t gid = (uint32_t)(env_offset + e);
    unsigned long long *my_stats = lane == 0 ? stats : nullptr;
    FinalSlots fs{};
    if constexpr (FINAL) fs = final_slots_begin(lane == 0, final_obs, final_row, n_slots, e);

    // pre-activation of one hidden unit (row of sw1) for the observation in `obs`
    auto unit = [&](const float *row) {
        const float4 *r4 = reinterpret_cast<const float4 *>(row);
        const float4 w0 = r4[0], w1 = r4[1], w2 = r4[2], w3 = r4[3], w4 = r4[4];
        float pa = w4.z, pb = 0.0f, pc = 0.0f;                                   // bias; three chains
        pa = fmaf(w0.x, obs[0], pa); pb = fmaf(w0.y, obs[1], pb); pc = fmaf(w0.z, obs[2], pc);
        pa = fmaf(w0.w, obs[3], pa); pb = fmaf(w1.x, obs[4], pb); pc = fmaf(w1.y, obs[5], pc);
        pa = fmaf(w1.z, obs[6], pa); pb = fmaf(w1.w, obs[7], pb); pc = fmaf(w2.x, obs[8], pc);
        pa = fmaf(w2.y, obs[9], pa); pb = fmaf(w2.z, obs[10], pb); pc = fmaf(w2.w, obs[11], pc);
        pa = fmaf(w3.x, obs[12], pa); pb = fmaf(w3.y, obs[13], pb); pc = fmaf(w3.z, obs[14], pc);
        pa = fmaf(w3.w, obs[15], pa); pb = fmaf(w4.x, obs[16], pb); pc = fmaf(w4.y, obs[17], pc);
        return fmaxf((pa + pb) + pc, 0.0f);
    };
    // both nets for `obs`: logits (+ bias) and value in every lane
    auto forward = [&](PolicyOut &po, bool actor) {
        float part[10];
#pragma unroll
        for (int q = 0; q < 10; ++q) part[q] = 0.0f;
#pragma unroll 2
        for (int i = 0; i < kHidden / 32; ++i) {
            const int j = lane + 32 * i;
            if (actor) {
                const float h = unit(sw1 + j * kWpRow);
                const float4 *v4 = reinterpret_cast<const float4 *>(sw2 + j * kWpW2);
                const float4 v0 = v4[0], v1 = v4[1], v2 = v4[2];
                part[0] = fmaf(v0.x, h, part[0]); part[1] = fmaf(v0.y, h, part[1]); part[2] = fmaf(v0.z, h, part[2]);
                part[3] = fmaf(v0.w, h, part[3]); part[4] = fmaf(v1.x, h, part[4]); part[5] = fmaf(v1.y, h, part[5]);
                part[6] = fmaf(v1.z, h, part[6]); part[7] = fmaf(v1.w, h, part[7]); part[8] = fmaf(v2.x, h, part[8]);
            }
            part[9] = fmaf(swc[j], unit(sw1 + (kHidden + j) * kWpRow), part[9]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int q = 0; q < 10; ++q) part[q] += __shfl_xor_sync(0xffffffffu, part[q], o);
        }
#pragma unroll
        for (int q = 0; q < kActions; ++q) po.logit[q] = part[q] + stail[q];
        po.logit[9] = 0.0f;
        po.value = part[9] + stail[10];
    };

    PolicyOut po;
    for (int t = 0; t < n_steps; ++t) {
        const size_t idx = (size_t)t * (size_t)stride + (size_t)e;
        forward(po, true);
        const unsigned long long gs = step0 + (unsigned long long)t;
        const uint32_t bits = philox_uniform_bits((uint32_t)seed, (uint32_t)(seed >> 32), gid, (uint32_t)gs,
                                                  (uint32_t)(gs >> 32), 0x43415245u);
        const float u = (float)(bits >> 8) * (1.0f / 16777216.0f);
        float logp, us;
        const int a = sample_action(po, u, logp, us);
        if (lane == 0) {
            if (obs_mode == kObsPose) {
                store_pose(reinterpret_cast<PoseRec *>(obs_buf) + idx, s, obs[2], obs[3]);
            } else {
                float2 *dst = reinterpret_cast<float2 *>(obs_buf + idx * kObsDim);
#pragma unroll
                for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(obs[2 * i], obs[2 * i + 1]);
            }
            act_buf[idx] = (float)a;
            val_buf[idx] = po.value;
            logp_buf[idx] = logp;
            term_buf[idx] = tc_;
            trunc_buf[idx] = uc;
            if (u_dbg) u_dbg[idx] = u;
        }
        StepResult o;
        if constexpr (FINAL) {
            env_step<kWarpPerEnv>(s, a, reward_scale, P, T, o, my_stats, &ws, nullptr, nullptr, fs.obs);
            final_slots_step(fs, o.truncated, t, n_slots, stride);
        } else {
            env_step<kWarpPerEnv>(s, a, reward_scale, P, T, o, my_stats, &ws);
        }
        if (lane == 0) rew_buf[idx] = o.reward;
#pragma unroll
        for (int i = 0; i < kObsDim; ++i) obs[i] = o.obs[i];
        tc_ = o.terminated ? 1.0f : 0.0f;
        uc = o.truncated ? 1.0f : 0.0f;
    }
    if (last_val) forward(po, false);                        // bootstrap value of the final observation (critic only)
    if (lane == 0) {
        pos[e] = make_double2(s.px, s.py);
        vel[e] = make_double2(s.vx, s.vy);
        ints[e] = make_int4(s.k, s.t, s.next_gate, s.passed);
        float2 *dst = reinterpret_cast<float2 *>(cur_obs + (size_t)e * kObsDim);
#pragma unroll
        for (int i = 0; i < kObsDim / 2; ++i) dst[i] = make_float2(obs[2 * i], obs[2 * i + 1]);
        cur_term[e] = tc_;
        cur_trunc[e] = uc;
        if (last_val) last_val[e] = po.value;
    }
    if constexpr (FINAL) final_slots_end(fs, n_slots, stride);
}
