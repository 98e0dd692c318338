// policy_abi.cuh — C-ABI entry points of the policy / PPO-update kernels (declared in include/carenv_b200.h).
// Textually included by carenv_kernels.cu inside its extern "C" block.
#pragma once
int carenv_pack_policy(int tensor_cores, const float *w1a, const float *b1a, const float *w2a, const float *b2a,
                       const float *w1c, const float *b1c, const float *w2c, const float *b2c, float *packed_out,
                       void *stream) {
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !packed_out)
        return fail(CARENV_E_INVAL, "null pointer");
    const int n = tensor_cores ? kTcWeightFloats : kPolicyFloats;
    if (tensor_cores)
        k_pack_policy<true><<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(w1a, b1a, w2a, b2a, w1c, b1c,
                                                                                           w2c, b2c, packed_out);
    else
        k_pack_policy<false><<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(w1a, b1a, w2a, b2a, w1c, b1c,
                                                                                            w2c, b2c, packed_out);
    CU(cudaGetLastError());
    return 0;
}

int carenv_ppo_num_params(void) { return ppo::kNumParams; }
int carenv_ppo_scratch_floats(int batch) { return batch > 0 && batch <= ppo::kMaxBatch ? ppo::scratch_floats(batch) : -1; }

int carenv_ppo_grad(const float *w1a, const float *b1a, const float *w2a, const float *b2a, const float *w1c,
                    const float *b1c, const float *w2c, const float *b2c, const float *obs, int obs_is_gathered,
                    const long long *idx, const float *act, const float *old_logp, const float *adv, const float *ret,
                    int batch, double clip_ratio, double vf_coef, double ent_coef, float *scratch, float *grads,
                    void *stream) {
    if (batch < 2 || batch > ppo::kMaxBatch) return fail(CARENV_E_INVAL, "batch must be in 2..1024");
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !obs || !idx || !act || !old_logp || !adv ||
        !ret || !scratch || !grads)
        return fail(CARENV_E_INVAL, "null pointer");
    const ppo::Params P{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int nb = (batch + ppo::kFwdThreads - 1) / ppo::kFwdThreads;
    const size_t smem_f = sizeof(float) * (ppo::kH * 20 + ppo::kH * ppo::kDz + 4);
    ppo::k_ppo_forward<<<dim3(nb, 2), ppo::kFwdThreads, smem_f, st>>>(P, obs, obs_is_gathered, idx, act, old_logp, adv,
                                                                      ret, batch, (float)clip_ratio, (float)vf_coef,
                                                                      (float)ent_coef, scratch);
    CU(cudaGetLastError());
    const size_t smem_b = sizeof(float) * ((size_t)batch * (20 + ppo::kDz) +
                                           (size_t)ppo::kBwdSlices * ppo::kBwdUnits * (ppo::kIn + 1 + ppo::kQ + 1));
    CU(cudaFuncSetAttribute(ppo::k_ppo_backward, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    ppo::k_ppo_backward<<<dim3(ppo::kH / ppo::kBwdUnits, 2), ppo::kBwdUnits * ppo::kBwdSlices, smem_b, st>>>(P, batch,
                                                                                                          scratch, grads);
    CU(cudaGetLastError());
    return 0;
}

int carenv_ppo_adam(float *w1a, float *b1a, float *w2a, float *b2a, float *w1c, float *b1c, float *w2c, float *b2c,
                    float *grads, double grad_scale, float *exp_avg, float *exp_avg_sq, const float *lr, int *step,
                    double beta1, double beta2, double eps, double max_grad_norm, const float *scratch, int batch,
                    double vf_coef, double ent_coef, float *sums4, void *stream) {
    if (batch < 2 || batch > ppo::kMaxBatch) return fail(CARENV_E_INVAL, "batch must be in 2..1024");
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !grads || !exp_avg || !exp_avg_sq || !lr ||
        !step || !scratch || !sums4)
        return fail(CARENV_E_INVAL, "null pointer");
    const ppo::MutableParams P{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c};
    ppo::k_ppo_adam<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(
        P, grads, (float)grad_scale, exp_avg, exp_avg_sq, lr, step, (float)beta1, (float)beta2, (float)eps,
        (float)max_grad_norm, scratch, batch, (float)vf_coef, (float)ent_coef, sums4);
    CU(cudaGetLastError());
    return 0;
}

/* ---- all minibatch updates of an epoch in one persistent launch (csrc/ppo_epoch.cuh) ---- */
struct PpoComm {
    int world = 1, rank = 0, device = 0;
    ppo::Exchange *local = nullptr;
    ppo::Exchange *peer[ppo::kMaxWorld] = {};
    unsigned long long seq = 0;           // updates completed so far (advances identically on every rank)
};

int carenv_ppo_comm_create(int world, int rank, void **comm, unsigned char *ipc_handle_out) {
    if (!comm || !ipc_handle_out) return fail(CARENV_E_INVAL, "null pointer");
    *comm = nullptr;
    if (world < 1 || world > ppo::kMaxWorld || rank < 0 || rank >= world)
        return fail(CARENV_E_INVAL, "world must be 1..8 and rank in [0, world)");
    static_assert(sizeof(cudaIpcMemHandle_t) == CARENV_IPC_HANDLE_BYTES, "handle size");
    PpoComm *c = new PpoComm();
    c->world = world; c->rank = rank;
    if (cudaGetDevice(&c->device) != cudaSuccess) { delete c; return fail(CARENV_E_NOGPU, "no CUDA device"); }
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&c->local), sizeof(ppo::Exchange));
    if (e == cudaSuccess) e = cudaMemset(c->local, 0, sizeof(ppo::Exchange));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, c->local);
    if (e != cudaSuccess) {
        if (c->local) cudaFree(c->local);
        delete c;
        return cuda_fail(e, "carenv_ppo_comm_create");
    }
    memcpy(ipc_handle_out, &h, sizeof(h));
    c->peer[rank] = c->local;
    *comm = c;
    return 0;
}

int carenv_ppo_comm_connect(void *comm, const unsigned char *all_handles) {
    PpoComm *c = static_cast<PpoComm *>(comm);
    if (!c || !all_handles) return fail(CARENV_E_INVAL, "null pointer");
    DeviceGuard guard(c->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the communicator's CUDA device");
    for (int r = 0; r < c->world; ++r) {
        if (r == c->rank || c->peer[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, all_handles + (size_t)r * sizeof(h), sizeof(h));
        void *p = nullptr;
        CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        c->peer[r] = static_cast<ppo::Exchange *>(p);
    }
    return 0;
}

int carenv_ppo_comm_destroy(void *comm) {
    PpoComm *c = static_cast<PpoComm *>(comm);
    if (!c) return 0;
    DeviceGuard guard(c->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < c->world; ++r)
        if (r != c->rank && c->peer[r]) cudaIpcCloseMemHandle(c->peer[r]);
    if (c->local) cudaFree(c->local);
    delete c;
    return 0;
}

int carenv_ppo_epoch_workspace_floats(void) { return ppo::kMaxCtas * ppo::kLocalPad + 2 * ppo::kMaxCtas + 8 * ppo::kMaxCtas + ppo::kLocalPad; }

int carenv_ppo_epoch(float *w1a, float *b1a, float *w2a, float *b2a, float *w1c, float *b1c, float *w2c, float *b2c,
                     const float *obs, const long long *idx, const float *act, const float *old_logp,
                     const float *adv, const float *ret, int batch, int n_updates, double clip_ratio, double vf_coef,
                     double ent_coef, float *exp_avg, float *exp_avg_sq, const float *lr, int *step, double beta1,
                     double beta2, double eps, double max_grad_norm, float *sums4, float *workspace, int *sync_words,
                     void *comm, int n_ctas, long long *prof, void *stream) {
    if (batch < 2 || batch > ppo::kMaxBatch) return fail(CARENV_E_INVAL, "batch must be in 2..1024");
    if (n_updates < 0) return fail(CARENV_E_INVAL, "negative n_updates");
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !obs || !idx || !act || !old_logp || !adv ||
        !ret || !exp_avg || !exp_avg_sq || !lr || !step || !sums4 || !workspace || !sync_words)
        return fail(CARENV_E_INVAL, "null pointer");
    if (n_updates == 0) return 0;
    PpoComm *c = static_cast<PpoComm *>(comm);
    int G = n_ctas > 0 ? n_ctas : 64;
    const int need = (batch + ppo::kEpochSamples - 1) / ppo::kEpochSamples;
    if (G < need) G = need;
    if (G < ppo::kMinCtas || G > ppo::kMaxCtas) return fail(CARENV_E_INVAL, "n_ctas must be in 49..160");
    int dev = 0, sms = 0, coop = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CU(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop || G > sms) return fail(CARENV_E_INVAL, "the device cannot keep the update grid resident");
    ppo::EpochArgs A;
    memset(&A, 0, sizeof(A));
    A.P = ppo::MutableParams{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c};
    A.obs = obs; A.idx = idx; A.act = act; A.old_logp = old_logp; A.adv = adv; A.ret = ret;
    A.B = batch; A.n_updates = n_updates;
    A.clip_ratio = (float)clip_ratio; A.vf_coef = (float)vf_coef; A.ent_coef = (float)ent_coef;
    A.max_grad_norm = (float)max_grad_norm; A.beta1 = (float)beta1; A.beta2 = (float)beta2; A.eps = (float)eps;
    A.m = exp_avg; A.v = exp_avg_sq; A.lr = lr; A.step = step; A.sums4 = sums4;
    A.partial = workspace;
    A.ssq = workspace + (size_t)ppo::kMaxCtas * ppo::kLocalPad;
    A.stat = A.ssq + 2 * ppo::kMaxCtas;
    A.bar = reinterpret_cast<unsigned int *>(sync_words);
    A.err = sync_words + 1;
    A.world = 1; A.rank = 0;
    A.prof = prof;
    if (c && c->world > 1) {
        if (c->device != dev) return fail(CARENV_E_INVAL, "the communicator belongs to another device");
        for (int r = 0; r < c->world; ++r)
            if (!c->peer[r]) return fail(CARENV_E_INVAL, "communicator not connected (carenv_ppo_comm_connect)");
        A.world = c->world; A.rank = c->rank; A.seq_base = c->seq;
        for (int r = 0; r < c->world; ++r) A.peer[r] = c->peer[r];
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CU(cudaMemsetAsync(sync_words, 0, sizeof(int), st));
    void *args[] = {&A};
    CU(cudaFuncSetAttribute(ppo::k_ppo_epoch<ppo::kEpochSamples>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            ppo::kEpochSmemBytes));
    CU(cudaLaunchCooperativeKernel(reinterpret_cast<void *>(ppo::k_ppo_epoch<ppo::kEpochSamples>), dim3(G),
                                   dim3(ppo::kEpochThreads), args, ppo::kEpochSmemBytes, st));
    if (c) c->seq += (unsigned long long)n_updates;
    return 0;
}

int carenv_policy_weights_floats(void) { return kPolicyFloats; }

int carenv_policy_rollout(void *handle, const float *packed_weights, int n_envs, int n_steps, int env_offset,
                          unsigned long long seed, unsigned long long step0, double *pos, double *vel, int32_t *ints,
                          float *cur_obs, float *cur_term, float *cur_trunc, double reward_scale, float *obs_buf,
                          float *act_buf, float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                          float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0 || n_steps < 0) return fail(CARENV_E_INVAL, "negative n_envs / n_steps");
    if (n_envs == 0) return 0;
    if (!packed_weights || !pos || !vel || !ints || !cur_obs || !cur_term || !cur_trunc || !obs_buf || !act_buf ||
        !rew_buf || !val_buf || !term_buf || !trunc_buf || !logp_buf)
        return fail(CARENV_E_INVAL, "null pointer");
    if (h->host.P.n_seg > kMaxSeg)
        return fail(CARENV_E_TRACK, "the fused rollout kernels support tracks with at most 128 wall segments");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const int table_bytes = (int)((h->smem_bytes + 15) / 16 * 16);
    const size_t smem = (size_t)table_bytes + sizeof(float) * kPolicyFloats;
    if (smem > 227 * 1024) return fail(CARENV_E_TRACK, "track tables too large for the CUDA-core rollout kernel");
    const int grid = (n_envs + kPolicyBlock - 1) / kPolicyBlock;
    int U = h->force_generic ? 1 : h->host.P.unroll4;   // the fused kernels are instantiated for 4, 2, 1
    if (h->max_unroll > 0 && U > h->max_unroll) U = (U % h->max_unroll == 0) ? h->max_unroll : 1;
    auto launch = [&](auto kern) -> int {
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, kPolicyBlock, smem, static_cast<cudaStream_t>(stream)>>>(
            h->host.P, h->dev, packed_weights, n_envs, n_steps, env_offset, seed, step0,
            reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel), reinterpret_cast<int4 *>(ints), cur_obs,
            cur_term, cur_trunc, reward_scale, obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf,
            last_val, u_dbg, h->d_stats, table_bytes, h->pose_rows ? kObsPose : kObsFull);
        CU(cudaGetLastError());
        return 0;
    };
    if (U == 4) return launch(k_policy_rollout<4>);
    if (U == 2) return launch(k_policy_rollout<2>);
    return launch(k_policy_rollout<1>);
}

/* Small batches: one warp per environment, network parameters in nn.Linear layout (k_policy_rollout_warp). */
// n_members == 0: one policy (k_policy_rollout_warp<false>); otherwise n_members stacked policies with n_envs
// environments each and seeds[p] (k_policy_rollout_warp<true>, carenv_policy_rollout_warp_pop).
static int policy_rollout_warp_launch(Handle *h, const ppo::Params &W, int n_members, int n_envs, int n_steps,
                                      int env_offset, unsigned long long seed, const unsigned long long *seeds,
                                      unsigned long long step0, double *pos, double *vel, int32_t *ints, float *cur_obs,
                                      float *cur_term, float *cur_trunc, double reward_scale, float *obs_buf,
                                      float *act_buf, float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                      float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    if (h->host.P.n_seg > 32)
        return fail(CARENV_E_TRACK, "the warp-per-environment rollout kernel supports tracks with at most 32 wall segments");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const int table_bytes = (int)((h->smem_bytes + 15) / 16 * 16);
    const size_t smem = (size_t)table_bytes + sizeof(float) * kWpFloats;
    if (smem > 227 * 1024) return fail(CARENV_E_TRACK, "track tables too large for the warp-per-environment rollout kernel");
    auto kern = n_members > 0 ? k_policy_rollout_warp<true> : k_policy_rollout_warp<false>;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 grid((n_envs + 3) / 4, n_members > 0 ? n_members : 1);
    kern<<<grid, 128, smem, static_cast<cudaStream_t>(stream)>>>(
        h->host.P, h->dev, W, n_envs, n_steps, env_offset, seed, step0, reinterpret_cast<double2 *>(pos),
        reinterpret_cast<double2 *>(vel), reinterpret_cast<int4 *>(ints), cur_obs, cur_term, cur_trunc, reward_scale, obs_buf,
        act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf, last_val, u_dbg, h->d_stats, table_bytes,
        h->pose_rows ? kObsPose : kObsFull, seeds, n_members * n_envs);
    CU(cudaGetLastError());
    return 0;
}

int carenv_policy_rollout_warp(void *handle, const float *w1a, const float *b1a, const float *w2a, const float *b2a,
                               const float *w1c, const float *b1c, const float *w2c, const float *b2c, int n_envs,
                               int n_steps, int env_offset, unsigned long long seed, unsigned long long step0,
                               double *pos, double *vel, int32_t *ints, float *cur_obs, float *cur_term,
                               float *cur_trunc, double reward_scale, float *obs_buf, float *act_buf, float *rew_buf,
                               float *val_buf, float *term_buf, float *trunc_buf, float *logp_buf, float *last_val,
                               float *u_dbg, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0 || n_steps < 0) return fail(CARENV_E_INVAL, "negative n_envs / n_steps");
    if (n_envs == 0) return 0;
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !pos || !vel || !ints || !cur_obs || !cur_term ||
        !cur_trunc || !obs_buf || !act_buf || !rew_buf || !val_buf || !term_buf || !trunc_buf || !logp_buf)
        return fail(CARENV_E_INVAL, "null pointer");
    return policy_rollout_warp_launch(h, ppo::Params{w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c}, 0, n_envs, n_steps,
                                      env_offset, seed, nullptr, step0, pos, vel, ints, cur_obs, cur_term, cur_trunc,
                                      reward_scale, obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf,
                                      last_val, u_dbg, stream);
}

/* Test hook: D[128,256] = A[128,24] * B[256,24]^T on the tensor cores (tcgen05, kind::tf32). */
int carenv_tc_gemm_test(const float *A, const float *B, float *D, void *stream) {
    if (!A || !B || !D) return fail(CARENV_E_INVAL, "null pointer");
    const size_t smem = tc::kABytes + tc::kBBytes + 128;
    CU(cudaFuncSetAttribute(k_tc_gemm_test, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_tc_gemm_test<<<1, 128, smem, static_cast<cudaStream_t>(stream)>>>(A, B, D);
    CU(cudaGetLastError());
    return 0;
}

int carenv_policy_weights_floats_tc(void) { return kTcWeightFloats; }

// k_policy_rollout_tc3 on a single-track handle.  n_members == 0: one policy; otherwise n_members packed policies
// [n_members][kTcWeightFloats] with n_envs environments each and seeds[p] (carenv_policy_rollout_tc_pop).
static int policy_rollout_tc_launch(Handle *h, const float *packed_weights, int n_members, int n_envs, int n_steps,
                                    int env_offset, unsigned long long seed, const unsigned long long *seeds,
                                    unsigned long long step0, double *pos, double *vel, int32_t *ints, float *cur_obs,
                                    float *cur_term, float *cur_trunc, double reward_scale, float *obs_buf,
                                    float *act_buf, float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                    float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    if (h->host.P.n_seg > kMaxSeg)
        return fail(CARENV_E_TRACK, "the fused rollout kernels support tracks with at most 128 wall segments");
    if (h->tc_tiles >= 2 && h->tc_tiles <= 4)
        return fail(CARENV_E_INVAL, "tc_tiles 2, 3 and 4 selected tensor-core rollout kernels that have been removed; "
                                    "use 0 or 5 (k_policy_rollout_tc3)");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    const int table_bytes = (int)h->smem_bytes;
    int U = h->force_generic ? 1 : h->host.P.unroll4;
    if (h->max_unroll > 0 && U > h->max_unroll) U = (U % h->max_unroll == 0) ? h->max_unroll : 1;
    const int n_pairs = h->host.n_pairs;
    const int row_f4 = ((n_pairs + 7) / 8 * 8) | 1;         // odd number of 16-byte units: rows skewed by one bank group
    const size_t smem_base = (size_t)table_bytes + 128 + (size_t)((kTcWeightFloats * 4 + 127) / 128 * 128) +
                             (size_t)2 * 2 * tc::kABytes + (size_t)2 * 128 * 12 * sizeof(float);
    const size_t tab_bytes = (size_t)kHeadings * row_f4 * 16;
    // denominators from a (row-skewed) table in shared memory where it fits (tracks of up to about 80 segments);
    // otherwise the arithmetic instantiation of the same U, which gives the same results
    const bool tab = U >= 2 && h->d_den4 && h->tab >= 0 && smem_base + tab_bytes <= 227 * 1024;
    const size_t smem = smem_base + (tab ? tab_bytes : 0);
    if (smem > 227 * 1024) return fail(CARENV_E_TRACK, "track tables too large for the tensor-core rollout kernel");
    const dim3 grid((n_envs + 255) / 256, n_members > 0 ? n_members : 1);
    auto launch = [&](auto kern) -> int {
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 256 + 128 + 32, smem, static_cast<cudaStream_t>(stream)>>>(
            h->host.P, h->dev, packed_weights, n_envs, n_steps, env_offset, seed, step0,
            reinterpret_cast<double2 *>(pos), reinterpret_cast<double2 *>(vel), reinterpret_cast<int4 *>(ints), cur_obs,
            cur_term, cur_trunc, reward_scale, obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf,
            last_val, u_dbg, h->d_stats, table_bytes, h->pose_rows ? kObsPose : kObsFull, h->d_den4, n_pairs, row_f4,
            nullptr, nullptr, 0, nullptr, seeds, n_members * n_envs);
        CU(cudaGetLastError());
        return 0;
    };
    if (n_members > 0) {
        if (U == 4) return tab ? launch(k_policy_rollout_tc3<4, true, true>) : launch(k_policy_rollout_tc3<4, false, true>);
        if (U == 2) return tab ? launch(k_policy_rollout_tc3<2, true, true>) : launch(k_policy_rollout_tc3<2, false, true>);
        return launch(k_policy_rollout_tc3<1, false, true>);
    }
    if (U == 4) return tab ? launch(k_policy_rollout_tc3<4, true>) : launch(k_policy_rollout_tc3<4, false>);
    if (U == 2) return tab ? launch(k_policy_rollout_tc3<2, true>) : launch(k_policy_rollout_tc3<2, false>);
    return launch(k_policy_rollout_tc3<1, false>);
}

/* Tensor-core variant of carenv_policy_rollout (same arguments; packed_weights in the layout of
 * ppo_car_b200/policy.py: pack_policy_weights_tc): k_policy_rollout_tc3. */
int carenv_policy_rollout_tc(void *handle, const float *packed_weights, int n_envs, int n_steps, int env_offset,
                             unsigned long long seed, unsigned long long step0, double *pos, double *vel,
                             int32_t *ints, float *cur_obs, float *cur_term, float *cur_trunc, double reward_scale,
                             float *obs_buf, float *act_buf, float *rew_buf, float *val_buf, float *term_buf,
                             float *trunc_buf, float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    Handle *h = static_cast<Handle *>(handle);
    if (!h) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0 || n_steps < 0) return fail(CARENV_E_INVAL, "negative n_envs / n_steps");
    if (n_envs == 0) return 0;
    if (!packed_weights || !pos || !vel || !ints || !cur_obs || !cur_term || !cur_trunc || !obs_buf || !act_buf ||
        !rew_buf || !val_buf || !term_buf || !trunc_buf || !logp_buf)
        return fail(CARENV_E_INVAL, "null pointer");
    return policy_rollout_tc_launch(h, packed_weights, 0, n_envs, n_steps, env_offset, seed, nullptr, step0, pos, vel,
                                    ints, cur_obs, cur_term, cur_trunc, reward_scale, obs_buf, act_buf, rew_buf, val_buf,
                                    term_buf, trunc_buf, logp_buf, last_val, u_dbg, stream);
}

/* Largest wall-segment count over the tracks of a multi-track handle: the handle keeps its TrackParams on the device
 * only, so this is one small strided copy, synchronous with `stream`. */
static int multi_max_seg(const MultiTrack *m, cudaStream_t stream, int *max_seg) {
    std::vector<int> n_seg((size_t)m->n_tracks);
    CU(cudaMemcpy2DAsync(n_seg.data(), sizeof(int), &m->d_params[0].n_seg, sizeof(TrackParams), sizeof(int),
                         (size_t)m->n_tracks, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    *max_seg = 0;
    for (int v : n_seg) *max_seg = v > *max_seg ? v : *max_seg;
    return 0;
}

/* carenv_policy_rollout_tc on several tracks (k_policy_rollout_tc3<0, false>): environment e runs on track
 * track_ids[e] of the multi-track handle (clamped to 0..n_tracks - 1 as carenv_multi_rollout does). */
int carenv_policy_rollout_tc_multi(void *multi, const int32_t *track_ids, const float *packed_weights, int n_envs,
                                   int n_steps, int env_offset, unsigned long long seed, unsigned long long step0,
                                   double *pos, double *vel, int32_t *ints, float *cur_obs, float *cur_term,
                                   float *cur_trunc, double reward_scale, float *obs_buf, float *act_buf,
                                   float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                   float *logp_buf, float *last_val, float *u_dbg, void *stream) {
    MultiTrack *m = static_cast<MultiTrack *>(multi);
    if (!m) return fail(CARENV_E_INVAL, "null handle");
    if (n_envs < 0 || n_steps < 0) return fail(CARENV_E_INVAL, "negative n_envs / n_steps");
    if (n_envs == 0) return 0;
    if (!track_ids || !packed_weights || !pos || !vel || !ints || !cur_obs || !cur_term || !cur_trunc || !obs_buf ||
        !act_buf || !rew_buf || !val_buf || !term_buf || !trunc_buf || !logp_buf)
        return fail(CARENV_E_INVAL, "null pointer");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(CARENV_E_NOGPU, "cannot select the handle's CUDA device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int max_seg = 0;
    if (const int rc = multi_max_seg(m, st, &max_seg)) return rc;
    if (max_seg > kMaxSeg)
        return fail(CARENV_E_TRACK, "the fused rollout kernels support tracks with at most 128 wall segments");
    // no staged tables: weights after a 128-byte alignment pad, A tiles, exchanged partial logits
    const size_t smem = 128 + (size_t)((kTcWeightFloats * 4 + 127) / 128 * 128) + (size_t)2 * 2 * tc::kABytes +
                        (size_t)2 * 128 * 12 * sizeof(float);
    static const TrackParams kNoTrack{};                     // P and G of the single-track instantiations: unused
    auto kern = k_policy_rollout_tc3<0, false>;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(n_envs + 255) / 256, 256 + 128 + 32, smem, st>>>(
        kNoTrack, Tables{}, packed_weights, n_envs, n_steps, env_offset, seed, step0, reinterpret_cast<double2 *>(pos),
        reinterpret_cast<double2 *>(vel), reinterpret_cast<int4 *>(ints), cur_obs, cur_term, cur_trunc, reward_scale,
        obs_buf, act_buf, rew_buf, val_buf, term_buf, trunc_buf, logp_buf, last_val, u_dbg, m->d_stats, 0, kObsFull,
        nullptr, 0, 0, m->d_params, m->d_tables, m->n_tracks, track_ids, nullptr, 0);
    CU(cudaGetLastError());
    return 0;
}

#include "policy_eval.cuh"      // carenv_policy_eval: k_policy_eval, whole episodes of one actor per launch
#include "population.cuh"       // carenv_*_pop: independent policies trained side by side (member-batched kernels)
