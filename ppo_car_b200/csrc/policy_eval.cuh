// policy_eval.cuh — policy evaluation: whole episodes of one actor played in ONE launch, one record per episode
// (returns, lengths, gates, laps, crashes).  The greedy / sampled play of the reference's video logger
// (train.py:23-50) without the Python loop around an eager actor and VecCarEnv.step.
//
// Textually included by policy_abi.cuh, i.e. inside the extern "C" block of carenv_kernels.cu, after the step and
// rollout kernels whose helpers (stage_tables, env_step, policy_core.cuh) it uses.  The kernel is a template, so it
// sits in an extern "C++" block of the same anonymous namespace.
//
//   k_policy_eval<U>   one thread = one episode SLOT of a persistent grid.  Slots claim episode indices i from a
//               per-call device counter (one warp-aggregated atomicAdd per warp and claim round); episode i has the
//               global id episode0 + i, which alone (with the weights, the seed and `greedy`) decides its
//               result: the random stream is keyed by the id and the step within the episode, every episode starts
//               from the start pose (the first claim of a slot starts there, later claims follow env_step's own
//               autoreset).  So the records do not depend on the grid, the slot count or n_episodes.
//               Actor only, float32 CUDA cores: the weights are staged from nn.Linear layout into the actor half of
//               pack_policy_weights' pair layout (128 pairs x 60 floats) and the logits are formed by the same FFMA2
//               chains, in the same order, as the actor part of policy_forward — the CUDA-core rollout's logits.
//               The step loop's trip count is warp-uniform (lanes without an episode step along and discard their
//               results) so that the wall tests keep their uniform constant-bank operands (DESIGN §3).
//   k_policy_eval<0>   several tracks (carenv_policy_eval_multi): a slot that claims episode i moves to the start pose
//               and reset observation of track episode_tracks[i] (as k_reset_multi) and steps with env_step<0> on that
//               track's TrackParams / Tables in global memory (as k_rollout_multi); nothing else changes, so episode i
//               on track k gives the record k_policy_eval gives on track k alone.
//   k_policy_eval<U, true>   a population (carenv_policy_eval_pop): blockIdx.y = member p.  The CTA stages member p's
//               actor from the stacked [P][...] tensors and keys its random stream with seeds[p]; member p claims from
//               counter[p] and writes its own blocks of the records and traces.  The rest is the single-member code,
//               so member p's records are those of k_policy_eval<U> on member p alone.
#pragma once

extern "C++" {
namespace {

constexpr int kEvalBlock = 128;
constexpr int kEvalTail = 12;                                              // b2a[0..8], 0, 0, 0
constexpr int kEvalFloats = (kHidden / 2) * kActorPairFloats + kEvalTail;  // 7,692 floats = 30,768 B
constexpr uint32_t kEvalStream = 0x4556414Cu;                              // "EVAL": 4th Philox counter word

// Actor logits for `obs` from the actor pair blocks `w` (stride kActorPairFloats): the actor half of
// policy_forward (policy_core.cuh), operation for operation.
__device__ __forceinline__ void actor_forward(const float (&obs)[kPolicyObs], const float *__restrict__ w,
                                              PolicyOut &out) {
    float2 L[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) L[q] = make_float2(0.0f, 0.0f);
#pragma unroll 2
    for (int p = 0; p < kHidden / 2; ++p) {
        const float4 *a4 = reinterpret_cast<const float4 *>(w + p * kActorPairFloats);
        const float4 t = a4[9];                             // (b1[j], b1[j+1], pad, pad)
        float2 H = make_float2(t.x, t.y);
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            const float4 ww = a4[i];
            H = __ffma2_rn(make_float2(obs[2 * i], obs[2 * i]), make_float2(ww.x, ww.y), H);
            H = __ffma2_rn(make_float2(obs[2 * i + 1], obs[2 * i + 1]), make_float2(ww.z, ww.w), H);
        }
        const float h0 = fmaxf(H.x, 0.0f), h1 = fmaxf(H.y, 0.0f);
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            const float4 ww = a4[10 + q];
            L[q] = __ffma2_rn(make_float2(h0, h0), make_float2(ww.x, ww.y), L[q]);
            L[q] = __ffma2_rn(make_float2(h1, h1), make_float2(ww.z, ww.w), L[q]);
        }
    }
    const float *tail = w + (kHidden / 2) * kActorPairFloats;
#pragma unroll
    for (int q = 0; q < 5; ++q) {
        out.logit[2 * q] = L[q].x + tail[2 * q];
        out.logit[2 * q + 1] = L[q].y + tail[2 * q + 1];
    }
    out.value = 0.0f;
}

// U == 0 keeps its 16 table pointers and the track pointer in registers (the single-track tables are shared-memory
// offsets): 3 CTAs per SM, 168 registers, where 4 CTAs (128 registers) spill.
template <int U, bool POP = false>
__global__ void __launch_bounds__(kEvalBlock, U == 0 ? 3 : 4)
k_policy_eval(const __grid_constant__ TrackParams P, const Tables G, const ppo::Params W, long long n_episodes,
              unsigned long long episode0, int greedy, unsigned long long seed,
              carenv_eval_record *__restrict__ records, int n_trace, unsigned char *__restrict__ trace_actions,
              float *__restrict__ trace_u, unsigned long long *counter, unsigned long long *stats, int table_bytes,
              const TrackParams *__restrict__ mt_params, const Tables *__restrict__ mt_tables, int n_tracks,
              const int *__restrict__ episode_tracks, const unsigned long long *__restrict__ seeds) {
    static_assert(!POP || U != 0, "populations play on one track");
    extern __shared__ __align__(16) unsigned char smem[];
    const float *w1a = W.w1a, *b1a = W.b1a, *w2a = W.w2a, *b2a = W.b2a;
    // POP: member p's block of a [P][per] array starts at p * per.  The record, trace and counter offsets are formed
    // where they are used, not added to the base pointers up front: held across the step loop, those pointers made
    // k_policy_eval<4, true> spill at the 128 registers of 4 CTAs per SM.
    auto member_block = [&](size_t per) -> size_t {
        if constexpr (POP) return (size_t)blockIdx.y * per;
        else return 0;
    };
    if constexpr (POP) {
        const size_t p = blockIdx.y;           // the actor only: the critic pointers are null
        w1a += p * kHidden * kObsDim; b1a += p * kHidden; w2a += p * kActions * kHidden; b2a += p * kActions;
        seed = seeds[p];
    }
    float *sw = reinterpret_cast<float *>(smem + table_bytes);
    for (int i = threadIdx.x; i < (kHidden / 2) * kActorPairFloats; i += blockDim.x) {
        const int p = i / kActorPairFloats, c = i - p * kActorPairFloats;   // as k_pack_policy<false>, actor half
        float v = 0.0f;
        if (c < 36) v = w1a[(2 * p + (c & 1)) * kObsDim + (c >> 1)];
        else if (c < 38) v = b1a[2 * p + (c - 36)];
        else if (c >= 40) {
            const int d = c - 40, q = d >> 2, sft = (d >> 1) & 1, row = 2 * q + (d & 1);
            v = row < kActions ? w2a[row * kHidden + 2 * p + sft] : 0.0f;
        }
        sw[i] = v;
    }
    if (threadIdx.x < kEvalTail)
        sw[(kHidden / 2) * kActorPairFloats + threadIdx.x] = threadIdx.x < kActions ? b2a[threadIdx.x] : 0.0f;
    // U == 0 (several tracks): nothing is staged, every lane reads its episode's track tables
    const Tables T = U == 0 ? Tables{} : stage_tables(G, P.n_gates, P.n_seg, smem);   // ends with __syncthreads()
    if constexpr (U == 0) __syncthreads();

    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    EnvState s;                                                     // the start pose (what carenv_reset writes)
    s.px = P.start_x; s.py = P.start_y; s.vx = 0.0; s.vy = 0.0;
    s.k = 0; s.t = 0; s.next_gate = 0; s.passed = 0;
    float obs[kObsDim];
#pragma unroll
    for (int i = 0; i < kObsDim; ++i) obs[i] = P.reset_obs[i];

    int tr = 0;                            // U == 0: the track of the lane's episode
    // U == 0: the start pose and reset observation of track `tr` (k_reset_multi); env_step's autoreset would go back
    // to the previous episode's track
    auto start_on_track = [&]() {
        const TrackParams &Q = mt_params[tr];
        s.px = Q.start_x; s.py = Q.start_y; s.vx = 0.0; s.vy = 0.0;
        s.k = 0; s.t = 0; s.next_gate = 0; s.passed = 0;
#pragma unroll
        for (int i = 0; i < kObsDim; ++i) obs[i] = Q.reset_obs[i];
    };
    if constexpr (U == 0) start_on_track();
    long long ep = -1;                     // episode index i of this call held by the lane (-1: none)
    bool drained = false;                  // the counter has run past n_episodes: the lane claims nothing more
    double ret = 0.0;
    int laps = 0, first_lap = -1;
    // Lanes with `want` take the next indices, in lane order, with one atomicAdd per warp.  Called by all 32 lanes.
    auto claim = [&](bool want) {
        const unsigned m = __ballot_sync(0xffffffffu, want);
        if (!m) return;
        const int leader = __ffs(m) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(counter + member_block(1), (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (want) {
            const unsigned long long i = base + (unsigned long long)__popc(m & lt_mask);
            if (i < (unsigned long long)n_episodes) {
                ep = (long long)i; ret = 0.0; laps = 0; first_lap = -1;
                if constexpr (U == 0) {
                    tr = min(max(episode_tracks[i], 0), n_tracks - 1);
                    start_on_track();
                }
            } else {
                drained = true;
            }
        }
    };
    claim(true);

    PolicyOut po;
    while (__any_sync(0xffffffffu, ep >= 0)) {
        const bool live = ep >= 0;
        const unsigned long long id = episode0 + (unsigned long long)(live ? ep : 0);
        const int step = s.t;                                       // steps already taken in this episode
        actor_forward(obs, sw, po);
        int a;
        float u = 0.0f;
        if (greedy) {
            a = 0;
            float m = po.logit[0];
#pragma unroll
            for (int i = 1; i < kActions; ++i)
                if (po.logit[i] > m) { m = po.logit[i]; a = i; }    // ties: the lowest index
        } else {
            const uint32_t bits = philox_uniform_bits((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)id,
                                                      (uint32_t)step, (uint32_t)(id >> 32), kEvalStream);
            u = (float)(bits >> 8) * (1.0f / 16777216.0f);
            float logp, us;
            a = sample_action(po, u, logp, us);
        }
        StepResult o;
        if constexpr (U == 0) env_step<0>(s, a, 1.0, mt_params[tr], mt_tables[tr], o, stats);
        else env_step<U>(s, a, 1.0, P, T, o, stats);
        if (live) {
            if (ep < n_trace) {
                const size_t ti = member_block((size_t)n_trace * kTimeLimit) + (size_t)ep * kTimeLimit + (size_t)step;
                trace_actions[ti] = (unsigned char)a;
                if (trace_u && !greedy) trace_u[ti] = u;
            }
            ret = __dadd_rn(ret, o.reward64);
            if (o.lap) {
                laps += 1;
                if (first_lap < 0) first_lap = o.time_passed;
            }
            if (o.terminated | o.truncated) {
                carenv_eval_record r;
                r.ret = ret;
                r.length = o.time_passed; r.gates = o.gates_passed; r.laps = laps; r.first_lap = first_lap;
                r.outcome = o.terminated ? 1 : 2; r.pad = 0;
                records[member_block((size_t)n_episodes) + ep] = r;
                ep = -1;
            }
        }
#pragma unroll
        for (int i = 0; i < kObsDim; ++i) obs[i] = o.obs[i];       // after an episode's end: the start pose
        claim(ep < 0 && !drained);
    }
}

}  // namespace
}  // extern "C++"

/* ---- C ABI (include/carenv_b200.h) ---- */
// One launch of an evaluation kernel: a persistent grid (ctas_per_member, n_members) of at most one wave in all
// (CARENV_EVAL_CTAS > 0 caps ctas_per_member further, a test hook so that a few slots play many episodes each) and one
// claim counter per member that lives for the call.  With more members than one wave holds, each member gets one CTA
// and the later CTAs wait to become resident: CTAs never wait for each other.  `m` and `episode_tracks` only for the
// multi-track instantiation, `seeds` only for the population instantiations (else null).
static int launch_eval(void (*kern)(const TrackParams, const Tables, const ppo::Params, long long, unsigned long long,
                                    int, unsigned long long, carenv_eval_record *, int, unsigned char *, float *,
                                    unsigned long long *, unsigned long long *, int, const TrackParams *,
                                    const Tables *, int, const int *, const unsigned long long *),
                       int device, const TrackParams &P, const Tables &G, int table_bytes, const MultiTrack *m,
                       const int32_t *episode_tracks, const ppo::Params &W, int n_members, long long n_episodes,
                       unsigned long long episode0, int greedy, unsigned long long seed,
                       const unsigned long long *seeds, carenv_eval_record *records, int n_trace,
                       unsigned char *trace_actions, float *trace_u, unsigned long long *stats, cudaStream_t st) {
    const size_t smem = (size_t)table_bytes + sizeof(float) * kEvalFloats;
    const char *cap_env = getenv("CARENV_EVAL_CTAS");
    const long long cap = cap_env ? atoll(cap_env) : 0;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int sms = 0, per_sm = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kEvalBlock, smem));
    long long grid = (n_episodes + kEvalBlock - 1) / kEvalBlock;
    const long long resident = (long long)sms * (per_sm > 0 ? per_sm : 1);
    const long long wave = resident / n_members > 1 ? resident / n_members : 1;
    if (grid > wave) grid = wave;
    if (cap > 0 && grid > cap) grid = cap;
    // The claim counters live for one call, allocated and freed in stream order: calls on one handle may run
    // concurrently on different streams.
    const size_t counter_bytes = sizeof(unsigned long long) * (size_t)n_members;
    unsigned long long *counter = nullptr;
    CU(cudaMallocAsync(reinterpret_cast<void **>(&counter), counter_bytes, st));
    cudaError_t e = cudaMemsetAsync(counter, 0, counter_bytes, st);
    if (e == cudaSuccess) {
        kern<<<dim3((unsigned)grid, (unsigned)n_members), kEvalBlock, smem, st>>>(
            P, G, W, n_episodes, episode0, greedy ? 1 : 0, seed, records, n_trace, trace_actions, trace_u, counter,
            stats, table_bytes, m ? m->d_params : nullptr, m ? m->d_tables : nullptr, m ? m->n_tracks : 0,
            episode_tracks, seeds);
        e = cudaGetLastError();
    }
    const cudaError_t ef = cudaFreeAsync(counter, st);
    if (e != cudaSuccess) return cuda_fail(e, "k_policy_eval launch");
    CU(ef);
    return 0;
}

// The instantiation for the handle's track, as carenv_policy_rollout chooses it: U = 4, 2 or 1.
static int eval_unroll(const Handle *h) {
    int U = h->force_generic ? 1 : h->host.P.unroll4;
    if (h->max_unroll > 0 && U > h->max_unroll) U = (U % h->max_unroll == 0) ? h->max_unroll : 1;
    return U;
}

int carenv_policy_eval(void *handle, const float *w1a, const float *b1a, const float *w2a, const float *b2a,
                       long long n_episodes, unsigned long long episode0, int greedy, unsigned long long seed,
                       carenv_eval_record *records, int n_trace, unsigned char *trace_actions, float *trace_u,
                       void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_episodes < 0) return fail(CARENV_E_INVAL, "negative n_episodes");
    if (!w1a || !b1a || !w2a || !b2a || !records) return fail(CARENV_E_INVAL, "null pointer");
    if (n_trace < 0) return fail(CARENV_E_INVAL, "negative n_trace");
    if (n_trace > 0 && !trace_actions) return fail(CARENV_E_INVAL, "n_trace > 0 needs trace_actions");
    if (h->host.P.n_seg > kMaxSeg)
        return fail(CARENV_E_TRACK, "policy evaluation supports tracks with at most 128 wall segments");
    if (n_episodes == 0) return 0;
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const int table_bytes = (int)((h->smem_bytes + 15) / 16 * 16);
    const int U = eval_unroll(h);
    const ppo::Params W{w1a, b1a, w2a, b2a, nullptr, nullptr, nullptr, nullptr};
    auto kern = U == 4 ? k_policy_eval<4> : (U == 2 ? k_policy_eval<2> : k_policy_eval<1>);
    return launch_eval(kern, h->device, h->host.P, h->dev, table_bytes, nullptr, nullptr, W, 1, n_episodes, episode0,
                       greedy, seed, nullptr, records, n_trace, trace_actions, trace_u, h->d_stats,
                       static_cast<cudaStream_t>(stream));
}

/* carenv_policy_eval for a population (k_policy_eval<U, true>): n_episodes episodes of each of n_members actors
 * stacked [P][...] in one launch; member p plays with seeds[p] and writes records [p][n_episodes] and traces
 * [p][n_trace][1000], the records and traces carenv_policy_eval gives for member p alone with seeds[p]. */
int carenv_policy_eval_pop(void *handle, int n_members, const float *w1a, const float *b1a, const float *w2a,
                           const float *b2a, long long n_episodes, unsigned long long episode0, int greedy,
                           const unsigned long long *seeds, carenv_eval_record *records, int n_trace,
                           unsigned char *trace_actions, float *trace_u, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_members <= 0 || n_members > 65535) return fail(CARENV_E_INVAL, "n_members must be in 1..65535");
    if (n_episodes < 0) return fail(CARENV_E_INVAL, "negative n_episodes");
    if (!w1a || !b1a || !w2a || !b2a || !seeds || !records) return fail(CARENV_E_INVAL, "null pointer");
    if (n_trace < 0) return fail(CARENV_E_INVAL, "negative n_trace");
    if (n_trace > 0 && !trace_actions) return fail(CARENV_E_INVAL, "n_trace > 0 needs trace_actions");
    if (h->host.P.n_seg > kMaxSeg)
        return fail(CARENV_E_TRACK, "policy evaluation supports tracks with at most 128 wall segments");
    if (n_episodes == 0) return 0;
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const int table_bytes = (int)((h->smem_bytes + 15) / 16 * 16);
    const int U = eval_unroll(h);
    const ppo::Params W{w1a, b1a, w2a, b2a, nullptr, nullptr, nullptr, nullptr};
    auto kern = U == 4 ? k_policy_eval<4, true> : (U == 2 ? k_policy_eval<2, true> : k_policy_eval<1, true>);
    return launch_eval(kern, h->device, h->host.P, h->dev, table_bytes, nullptr, nullptr, W, n_members, n_episodes,
                       episode0, greedy, 0, seeds, records, n_trace, trace_actions, trace_u, h->d_stats,
                       static_cast<cudaStream_t>(stream));
}

/* carenv_policy_eval on several tracks (k_policy_eval<0>): episode i of the call plays on track episode_tracks[i] of
 * the multi-track handle (clamped to 0..n_tracks - 1) and gives the record carenv_policy_eval gives on that track. */
int carenv_policy_eval_multi(void *multi, const int32_t *episode_tracks, const float *w1a, const float *b1a,
                             const float *w2a, const float *b2a, long long n_episodes, unsigned long long episode0,
                             int greedy, unsigned long long seed, carenv_eval_record *records, int n_trace,
                             unsigned char *trace_actions, float *trace_u, void *stream) {
    MultiTrack *m = static_cast<MultiTrack *>(multi);
    if (!m) return fail(CARENV_E_INVAL, "null handle");
    if (n_episodes < 0) return fail(CARENV_E_INVAL, "negative n_episodes");
    if (!episode_tracks || !w1a || !b1a || !w2a || !b2a || !records) return fail(CARENV_E_INVAL, "null pointer");
    if (n_trace < 0) return fail(CARENV_E_INVAL, "negative n_trace");
    if (n_trace > 0 && !trace_actions) return fail(CARENV_E_INVAL, "n_trace > 0 needs trace_actions");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int max_seg = 0;
    if (const int rc = multi_max_seg(m, st, &max_seg)) return rc;
    if (max_seg > kMaxSeg) return fail(CARENV_E_TRACK, "policy evaluation supports tracks with at most 128 wall segments");
    if (n_episodes == 0) return 0;
    static const TrackParams kNoTrack{};                     // P and G of the single-track instantiations: unused
    const ppo::Params W{w1a, b1a, w2a, b2a, nullptr, nullptr, nullptr, nullptr};
    return launch_eval(k_policy_eval<0>, m->device, kNoTrack, Tables{}, 0, m, episode_tracks, W, 1, n_episodes,
                       episode0, greedy, seed, nullptr, records, n_trace, trace_actions, trace_u, m->d_stats, st);
}
