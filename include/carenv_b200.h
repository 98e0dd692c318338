/* carenv_b200.h — C ABI of libcarenv_b200.so (B200 / sm_100a).
 *
 * The drop-in boundary for the one hot path of ProfessorNova/PPO-Car that this repository
 * accelerates: the batched CarEnv step with same-step autoreset and the GAE reverse scan.
 * The reference has no FFI layer (it is pure Python); each entry point below names the
 * reference interface it stands in for (file:line in the reference tree).  INTEGRATION.md
 * shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success and a negative code on failure
 *     (CARENV_E_* below, or -1000 - cudaError_t for CUDA failures); no exception or abort
 *     crosses the boundary; carenv_last_error() returns a thread-local message.
 *   - all pointers except `handle` and the *_host arguments are DEVICE pointers owned by
 *     the caller (PyTorch tensors); they are borrowed for the duration of the enqueued
 *     kernel.  The library owns only the opaque handle and its small geometry tables.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *     all work is enqueued on it and the call returns without synchronising.
 *   - there is no CPU implementation behind this interface.
 *
 * Environment state (structure of arrays, one element per environment):
 *   pos  double[N][2]   x, y in pixels                     (Car.__pos,      lib/car_env.py:245)
 *   vel  double[N][2]   vx, vy in pixels/step              (Car.__velocity, lib/car_env.py:262)
 *   ints int32 [N][4]   heading index k (rotation = initial_angle + 5k degrees, k mod 72),
 *                       time_step, next_gate_index, passed_reward_gates
 *                                                          (lib/car_env.py:247, 490, 494-496)
 */
#ifndef CARENV_B200_H
#define CARENV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CARENV_ABI_VERSION 1
#define CARENV_OBS_DIM 18      /* 6 + num_rays, lib/car_env.py:513-519 */
#define CARENV_NUM_ACTIONS 9   /* spaces.Discrete(9), lib/car_env.py:525 */
#define CARENV_MAX_SEGMENTS 2048   /* up to 128: geometry as kernel constants (fast kernels); above: staged in shared memory */

#define CARENV_E_INVAL (-1)    /* bad argument (null pointer, size, dtype) */
#define CARENV_E_TRACK (-2)    /* track does not fit (too many segments) or is malformed */
#define CARENV_E_NOGPU (-3)    /* no usable CUDA device */

/* action element type of the `actions` argument */
#define CARENV_ACT_U8 0
#define CARENV_ACT_I32 1
#define CARENV_ACT_I64 2       /* what Categorical.sample() yields, lib/model.py:38 */

/* element type of the terminated / truncated outputs */
#define CARENV_FLAG_U8 0
#define CARENV_FLAG_F32 1      /* what lib/buffer.py:16-17 stores */

int carenv_abi_version(void);
const char *carenv_last_error(void);

/* Build the per-track tables on `device`.
 * Stands in for CarEnv.__init__ + CarEnv.load_track + the geometry rebuild in CarEnv.reset
 * (lib/car_env.py:475-533, 535-567, 638-676).  Coordinates are already in pixels (x*1280,
 * y*720); walls are [n_walls][4] = x1 y1 x2 y2, outer polyline first then inner, in the
 * reference's order; gates are [n_gates][4] from consecutive point pairs. */
int carenv_create(const double *walls_xyxy_host, int n_walls, const double *gates_xyxy_host, int n_gates,
                  double init_x, double init_y, double init_angle_deg, int device, void **handle);
int carenv_destroy(void *handle);

/* The observation CarEnv.reset returns (a constant of the track; lib/car_env.py:682-691). */
int carenv_reset_obs(void *handle, float *obs18_host);

/* CarEnv.reset for n_envs environments (lib/car_env.py:605-691): start pose, zero velocity,
 * counters cleared; obs_out [n_envs][18] float32 (may be NULL). */
int carenv_reset(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, float *obs_out, void *stream);

/* One CarEnv.step for every environment, with the same-step autoreset of
 * gymnasium.vector.AsyncVectorEnv (lib/car_env.py:693-760; train.py:138,185).
 *   actions     [n_envs] of action_dtype, values 0..8; any other value (in any dtype) does nothing, like 8
 *   reward_scale            TransformReward factor (train.py:65,68); reward_out = float32(r * scale)
 *   obs_out     [n_envs][18] float32; the RESET observation where the episode ended
 *   reward_out  [n_envs] float32
 *   term_out / trunc_out [n_envs] of flag_dtype
 *   info_out    [n_envs][4] int32 or NULL: gates_passed, time_passed (info dict of the finished
 *               step, lib/car_env.py:599-603), next_gate_index, bit0 = gate hit, bit1 = lap */
int carenv_step(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions,
                int action_dtype, double reward_scale, float *obs_out, float *reward_out, void *term_out,
                void *trunc_out, int flag_dtype, int32_t *info_out, void *stream);

/* carenv_step that also returns the observation of the state each step ENDED in, before the autoreset — gymnasium's
 * info["final_observation"] (AsyncVectorEnv worker, SURVEY 3.5; train.py:185 discards it, value-bootstrapping users need
 * it).  final_obs_out [n_envs][18] float32 equals obs_out wherever the episode did not end. */
int carenv_step_final(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions,
                      int action_dtype, double reward_scale, float *obs_out, float *final_obs_out, float *reward_out,
                      void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out, void *stream);

/* carenv_step with HOST buffers — what the reference's rollout loop does around envs.step (train.py:185-192:
 * numpy actions in, numpy observations / rewards / flags out).  actions_host [n_envs] of action_dtype and the
 * *_host outputs (layouts as in carenv_step; info_host may be NULL) are host pointers; pinned memory
 * (carenv_host_alloc, or any cudaHostAlloc / torch pin_memory buffer) makes the copies asynchronous — the batch
 * is cut into sub-ranges of 16,384 or more environments (at most 8) on internal streams so that the device->host copy of one
 * range overlaps the kernel and copies of the next.  The state arrays stay on the device.  The call is ordered
 * after earlier work on `stream`, later work on `stream` sees the new state, and it RETURNS WHEN THE RESULTS ARE
 * IN THE HOST BUFFERS.  The library owns the staging buffers (per handle, sized on first use). */
int carenv_step_host(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions_host,
                     int action_dtype, double reward_scale, float *obs_host, float *reward_host, void *term_host,
                     void *trunc_host, int flag_dtype, int32_t *info_host, void *stream);

/* The same step with ONE 16-byte record per environment instead of three arrays (reward, terminated, truncated)
 * plus the info array: what the reference returns besides the observation (lib/car_env.py:760 reward and flags,
 * 599-603 the info dict), already in the reference's dtypes and in the layout that costs the least PCIe traffic —
 * 72 + 16 = 88 bytes per environment and two device->host copies per sub-range, no conversion pass on the host.
 * numpy reads the fields as strided views of the record array.
 *   rec_host         [n_envs] records (pinned memory recommended)
 *   debug_info_host  [n_envs][4] int32 or NULL: gates_passed, time_passed, next_gate_index, events (as info_out of
 *                    carenv_step; 16 more bytes per environment over PCIe — for parity tests, off by default)
 * carenv_step_records is the device-buffer variant (rec_out / debug_info_out are device pointers). */
typedef struct carenv_step_record {
    double reward;           /* reward_f64 * reward_scale: the float64 TransformReward yields (train.py:65, 68) */
    int32_t gates_passed;    /* info["gates_passed"] of the finished step (pre-reset), lib/car_env.py:599-603 */
    uint16_t time_passed;    /* info["time_passed"], 1..1000 */
    uint8_t terminated;      /* lib/car_env.py:745-748 */
    uint8_t truncated;       /* lib/car_env.py:749-750 */
} carenv_step_record;
int carenv_step_host_records(void *handle, int n_envs, double *pos, double *vel, int32_t *ints,
                             const void *actions_host, int action_dtype, double reward_scale, float *obs_host,
                             carenv_step_record *rec_host, int32_t *debug_info_host, void *stream);
int carenv_step_records(void *handle, int n_envs, double *pos, double *vel, int32_t *ints, const void *actions,
                        int action_dtype, double reward_scale, float *obs_out, carenv_step_record *rec_out,
                        int32_t *debug_info_out, void *stream);
int carenv_host_alloc(size_t bytes, void **ptr);   /* pinned host memory for the calls above */
int carenv_host_free(void *ptr);

/* n_steps consecutive steps in ONE launch (the rollout loop of train.py:173-195 with the
 * actions given up front).  actions is [n_steps][n_envs]; every output is [n_steps][n_envs]...
 * with the same element layouts as carenv_step; obs_out, info_out may be NULL.  The state
 * arrays hold the final state on completion. */
int carenv_rollout(void *handle, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints,
                   const void *actions, int action_dtype, double reward_scale, float *obs_out, float *reward_out,
                   void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out, void *stream);

/* Compact rollout storage (the reference stores obs [T][N][18] float32, lib/buffer.py:12; SURVEY §8 f-3).
 * carenv_rollout_poses is carenv_rollout with a 32-byte pose record per env-step instead of the 72-byte
 * observation: { double x, y; float obs2, obs3; int32 heading_index; int32 reset } — `reset` = 1 where the
 * episode ended in that step (the row's observation is the reset observation).
 * carenv_observe recomputes observations from n records (records poses[index[i]] if index is not NULL, else
 * poses[i]) into obs_out [n][18]; the result is bit-identical to what carenv_rollout would have written. */
#define CARENV_POSE_BYTES 32
int carenv_rollout_poses(void *handle, int n_envs, int n_steps, double *pos, double *vel, int32_t *ints,
                         const void *actions, int action_dtype, double reward_scale, void *pose_out, float *reward_out,
                         void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out, void *stream);
int carenv_observe(void *handle, long long n, const void *poses, const long long *index, float *obs_out, void *stream);

/* Several tracks in ONE launch — CarEnv.reset(options={"track_path": ...}) per environment (lib/car_env.py:621-628):
 * `handles` are n_tracks handles from carenv_create (they own the per-track tables and must outlive `multi`);
 * track_ids [n_envs] int32 (device) selects every environment's track; carenv_multi_reset / carenv_multi_rollout are
 * carenv_reset / carenv_rollout with that extra argument (n_steps = 1 is a step).  Environments of different tracks
 * may be mixed freely; results are bit-identical to stepping each environment in a single-track handle. */
int carenv_multi_create(void *const *handles, int n_tracks, void **multi);
int carenv_multi_destroy(void *multi);
int carenv_multi_reset(void *multi, int n_envs, const int32_t *track_ids, double *pos, double *vel, int32_t *ints,
                       float *obs_out, void *stream);
int carenv_multi_rollout(void *multi, int n_envs, int n_steps, const int32_t *track_ids, double *pos, double *vel,
                         int32_t *ints, const void *actions, int action_dtype, double reward_scale, float *obs_out,
                         float *reward_out, void *term_out, void *trunc_out, int flag_dtype, int32_t *info_out,
                         void *stream);

/* Headless render_mode="rgb_array" frames (CarEnv.render / __render_frame, lib/car_env.py:762-812; consumer: the video
 * logger train.py:23-50) for n_frames environments env_index[f] (device int32): rgb_out [n_frames][height][width][3]
 * uint8 — background, corridor, walls, active gates (the next one yellow), rays and the car as a box (the reference
 * blits a sprite).  width x height = 1280 x 720 is the reference's canvas; n_outer_segments = how many of the
 * handle's wall segments belong to the outer polygon.  A diagnostic picture, not a pixel-exact copy of pygame. */
int carenv_render(void *handle, int n_outer_segments, int n_frames, const int32_t *env_index, const double *pos,
                  const int32_t *ints, const float *obs, int width, int height, unsigned char *rgb_out, void *stream);

/* Options.  "pose_rows" = 1: the fused rollout kernels below write 32-byte pose records (see
 * carenv_rollout_poses) through their obs_buf argument instead of observations.  Tuning / test hooks:
 * "force_generic" = 1 runs the generic segment loop even for tracks that have an unrolled kernel instantiation
 * (identical results); "warp_per_env" = 1 / -1 forces / forbids the warp-per-environment kernel that small
 * batches (at most 2,048 environments, at most 32 wall segments) run by default (identical results);
 * "tab" = 1 / -1 forces / forbids the table kernel (k_rollout_tab: denominators from a shared-memory table) that large
 * launches on tracks with at most 128 segments run by default (identical results);
 * "tc_tiles" = 0 (default) or 5 runs carenv_policy_rollout_tc on k_policy_rollout_tc3, its only kernel; 2, 3 and 4
 * selected kernels that have been removed, are still accepted here and make carenv_policy_rollout_tc fail with
 * CARENV_E_INVAL;
 * "tab_slice" = -1 keeps the block-round table kernel where the time-sliced one (k_rollout_tab_sliced) would run;
 * "max_unroll", "block", "smem_pad", "host_ranges" select kernel / pipeline variants for measurements;
 * "tc_stagger" is accepted and has no effect. */
int carenv_set_option(void *handle, const char *name, int value);

/* Slow-path counters since the last reset of the counters: [0] lines re-evaluated in float64
 * because an endpoint was within eps of a ray line, [1] rays re-evaluated because a cardinal
 * distance was within the band around 10 px, [2] gate tests re-evaluated, [3] distances below
 * the tiny threshold.  Synchronises the device. */
int carenv_stats(void *handle, unsigned long long out4_host[4], int reset_counters);

/* Buffer.calculate_advantages (lib/buffer.py:36-64): float32 GAE(lambda) reverse scan in the
 * reference's own operation order, every operation individually rounded.
 *   rew, val, term, trunc   [T][N] float32 (the Buffer layout, lib/buffer.py:14-17)
 *   last_val, last_term, last_trunc [N] float32
 *   adv, ret                [T][N] float32 outputs (ret = adv + val) */
int gae_reverse_scan(const float *rew, const float *val, const float *term, const float *trunc,
                     const float *last_val, const float *last_term, const float *last_trunc, float *adv, float *ret,
                     int T, int N, double gamma, double gae_lambda, void *stream);

/* Fused rollout (the loop of train.py:173-195 in one launch): for n_steps steps, per environment:
 * actor/critic forward (lib/model.py:10-40, float32), categorical sample by inverse CDF on a Philox4x32-10
 * uniform keyed by (seed; env_offset + env, step0 + t), Buffer row writes (lib/buffer.py:22-34: obs, action
 * as float32, reward, value, the flags that came WITH the observation, logprob), CarEnv.step with autoreset.
 *   packed_weights  device float[carenv_policy_weights_floats()] in the layout of ppo_car_b200/policy.py
 *   cur_obs [n][18], cur_term [n], cur_trunc [n]   in: observation/flags the rollout starts from; out: those it ends with
 *   *_buf           [n_steps][n_envs](,18) float32 Buffer tensors
 *   last_val [n] or NULL  critic value of the final observation (bootstrap for GAE, train.py:200)
 *   u_dbg [n_steps][n_envs] or NULL  the uniforms that were used (tests) */
int carenv_policy_weights_floats(void);
/* Pack the reference network's parameters (device pointers, nn.Linear layout weight[out][in], lib/model.py:10-26:
 * actor 18-256-9, critic 18-256-1) into packed_out: carenv_policy_weights_floats() floats for
 * carenv_policy_rollout (tensor_cores = 0) or carenv_policy_weights_floats_tc() for carenv_policy_rollout_tc. */
int carenv_pack_policy(int tensor_cores, const float *w1_actor, const float *b1_actor, const float *w2_actor,
                       const float *b2_actor, const float *w1_critic, const float *b1_critic, const float *w2_critic,
                       const float *b2_critic, float *packed_out, void *stream);
int carenv_policy_rollout(void *handle, const float *packed_weights, int n_envs, int n_steps, int env_offset,
                          unsigned long long seed, unsigned long long step0, double *pos, double *vel, int32_t *ints,
                          float *cur_obs, float *cur_term, float *cur_trunc, double reward_scale, float *obs_buf,
                          float *act_buf, float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                          float *logp_buf, float *last_val, float *u_dbg, void *stream);

/* Tensor-core variant of the fused rollout: the two 18->256 layers run as tcgen05.mma kind::tf32 (3xTF32
 * split, float32-level accuracy) with accumulators in tensor memory; same arguments and results (to float32
 * rounding of the network outputs) as carenv_policy_rollout.  packed_weights: device
 * float[carenv_policy_weights_floats_tc()] from ppo_car_b200.policy.pack_policy_weights_tc.  On tracks whose
 * denominator table does not fit next to the weights in 227 KB of shared memory (above about 80 wall segments) it
 * computes the denominators instead, so every track of up to 128 segments with few enough gates runs. */
int carenv_policy_weights_floats_tc(void);
int carenv_policy_rollout_tc(void *handle, const float *packed_weights, int n_envs, int n_steps, int env_offset,
                             unsigned long long seed, unsigned long long step0, double *pos, double *vel,
                             int32_t *ints, float *cur_obs, float *cur_term, float *cur_trunc, double reward_scale,
                             float *obs_buf, float *act_buf, float *rew_buf, float *val_buf, float *term_buf,
                             float *trunc_buf, float *logp_buf, float *last_val, float *u_dbg, void *stream);

/* One PPO minibatch update of the reference network (train.py:223-261: clipped surrogate, 0.5-weighted value
 * loss, entropy bonus, advantage normalised per minibatch with the unbiased std clamped at 1e-5,
 * clip_grad_norm_, Adam) in three launches instead of an autograd graph of ~60 kernels.  All pointers are
 * device pointers; parameters in nn.Linear layout (lib/model.py:10-26).
 *   carenv_ppo_grad   gradients of the minibatch `idx` [batch] (rows of obs [.][18] — or obs already gathered
 *                     [batch][18] if obs_is_gathered — and of the flat act / old_logp / adv / ret arrays) into
 *                     grads [carenv_ppo_num_params()] in the order W1a b1a W2a b2a W1c b1c W2c b2c; deterministic.
 *   carenv_ppo_adam   grads *= grad_scale (1 / world size after an all-reduce), global-norm clip, Adam step
 *                     (exp_avg / exp_avg_sq [num_params], *step incremented, learning rate read from *lr),
 *                     sums4 += (policy loss, value loss, entropy, total loss) of the minibatch.
 *   scratch           carenv_ppo_scratch_floats(batch) floats, written by _grad and read by _adam. */
int carenv_ppo_num_params(void);
int carenv_ppo_scratch_floats(int batch);
int carenv_ppo_grad(const float *w1_actor, const float *b1_actor, const float *w2_actor, const float *b2_actor,
                    const float *w1_critic, const float *b1_critic, const float *w2_critic, const float *b2_critic,
                    const float *obs, int obs_is_gathered, const long long *idx, const float *act,
                    const float *old_logp, const float *adv, const float *ret, int batch, double clip_ratio,
                    double vf_coef, double ent_coef, float *scratch, float *grads, void *stream);
int carenv_ppo_adam(float *w1_actor, float *b1_actor, float *w2_actor, float *b2_actor, float *w1_critic,
                    float *b1_critic, float *w2_critic, float *b2_critic, float *grads, double grad_scale,
                    float *exp_avg, float *exp_avg_sq, const float *lr, int *step, double beta1, double beta2,
                    double eps, double max_grad_norm, const float *scratch, int batch, double vf_coef,
                    double ent_coef, float *sums4, void *stream);

/* carenv_policy_rollout for SMALL batches (the reference's own training shape is 24 environments): one warp per
 * environment — lane = wall segment in the env step, lane = 16 hidden units in the policy — on tracks with at most 32
 * wall segments.  The network parameters are passed in nn.Linear layout (lib/model.py:10-26: weight [out][in], bias),
 * no packing; other arguments as carenv_policy_rollout.  Same random stream; float32 CUDA cores. */
int carenv_policy_rollout_warp(void *handle, const float *w1_actor, const float *b1_actor, const float *w2_actor,
                               const float *b2_actor, const float *w1_critic, const float *b1_critic,
                               const float *w2_critic, const float *b2_critic, int n_envs, int n_steps, int env_offset,
                               unsigned long long seed, unsigned long long step0, double *pos, double *vel,
                               int32_t *ints, float *cur_obs, float *cur_term, float *cur_trunc, double reward_scale,
                               float *obs_buf, float *act_buf, float *rew_buf, float *val_buf, float *term_buf,
                               float *trunc_buf, float *logp_buf, float *last_val, float *u_dbg, void *stream);

/* Policy evaluation: n_episodes whole episodes of the actor (nn.Linear layout, 18-256-9) on the handle's track in ONE
 * launch (k_policy_eval, csrc/policy_eval.cuh), one record per episode.  Episode i of the call has the global id
 * episode0 + i and starts from the start pose; its result depends only on (weights, seed, id, greedy), not on
 * n_episodes or on how the library schedules the episodes.  The environment state arrays are not touched.
 *   greedy          1: the argmax of the logits (lowest index on a tie); 0: a sample by inverse CDF on a
 *                   Philox4x32-10 uniform keyed by `seed`, counter (id low 32 bits, step within the episode,
 *                   id high 32 bits, 0x4556414C)
 *   records         [n_episodes], written when the episode ends (terminated or truncated at 1000 steps):
 *                     ret        float64 sum of the unscaled rewards, in step order
 *                     length     time_passed of the last step; gates: gates_passed of the last step
 *                     laps       completed laps; first_lap: time_passed at the first lap, or -1
 *                     outcome    1 = crash (terminated), 2 = time limit (truncated)
 *   n_trace         episodes i < n_trace also write their actions to trace_actions [n_trace][1000] and, when
 *                   trace_u is not NULL and greedy == 0, the uniforms to trace_u [n_trace][1000]; entries past an
 *                   episode's end are not written.  The environment is deterministic: the actions replay the episode.
 * Tracks with at most 128 wall segments (CARENV_E_TRACK otherwise).  Float32 CUDA cores; the logits equal those of
 * carenv_policy_rollout for the same weights and observation. */
typedef struct {
    double ret;
    int32_t length, gates, laps, first_lap, outcome, pad;
} carenv_eval_record;
int carenv_policy_eval(void *handle, const float *w1_actor, const float *b1_actor, const float *w2_actor,
                       const float *b2_actor, long long n_episodes, unsigned long long episode0, int greedy,
                       unsigned long long seed, carenv_eval_record *records, int n_trace, unsigned char *trace_actions,
                       float *trace_u, void *stream);

/* Several tracks in the fused rollout and in policy evaluation, one launch each.  `multi` is a multi-track handle
 * (carenv_multi_create); every track of it must have at most 128 wall segments (CARENV_E_TRACK otherwise).  Track ids
 * outside 0..n_tracks - 1 are clamped as in carenv_multi_rollout.  Each call reads the tracks' segment counts from the
 * handle with one small copy that synchronises with `stream`.
 *   carenv_policy_rollout_tc_multi   carenv_policy_rollout_tc with environment e on track track_ids[e] (device int32
 *       [n_envs]); the random stream is keyed by the global env id as before, so every environment's rows are
 *       bit-identical to carenv_policy_rollout_tc on its track alone.  obs_buf always holds [n_steps][n_envs][18]
 *       observations: pose records do not carry a track.
 *   carenv_policy_eval_multi   carenv_policy_eval with episode i of the call on track episode_tracks[i] (device int32
 *       [n_episodes]); each episode starts from its track's start pose, and its record equals the one
 *       carenv_policy_eval gives for the same id on that track alone. */
int carenv_policy_rollout_tc_multi(void *multi, const int32_t *track_ids, const float *packed_weights, int n_envs,
                                   int n_steps, int env_offset, unsigned long long seed, unsigned long long step0,
                                   double *pos, double *vel, int32_t *ints, float *cur_obs, float *cur_term,
                                   float *cur_trunc, double reward_scale, float *obs_buf, float *act_buf,
                                   float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf, float *logp_buf,
                                   float *last_val, float *u_dbg, void *stream);
int carenv_policy_eval_multi(void *multi, const int32_t *episode_tracks, const float *w1_actor, const float *b1_actor,
                             const float *w2_actor, const float *b2_actor, long long n_episodes,
                             unsigned long long episode0, int greedy, unsigned long long seed,
                             carenv_eval_record *records, int n_trace, unsigned char *trace_actions, float *trace_u,
                             void *stream);

/* All minibatch updates of one PPO epoch in ONE persistent cooperative launch (csrc/ppo_epoch.cuh; replaces the
 * loops of train.py:223-261 — `for _ in range(train_iters): for start in range(0, n_steps, batch_size): ...` — and,
 * with several GPUs, the gradient all-reduce between backward and optimizer.step()).
 *   idx          device int64 [n_updates][batch]: the sample rows of every minibatch, in order
 *   workspace    device float[carenv_ppo_epoch_workspace_floats()]
 *   sync_words   device int[2]: grid-barrier counter (cleared by the call) and an error word that stays 0 unless a
 *                wait inside the kernel ran out of time (a peer rank that never launched)
 *   comm         NULL on one GPU; otherwise a communicator from carenv_ppo_comm_create + _connect.  The gradient
 *                elements are pushed into IPC-mapped peer buffers over NVLink inside the kernel and summed in rank
 *                order, so every rank applies bit-identical updates; every rank must make the same sequence of calls.
 *   n_ctas       0 = default (64, or ceil(batch / 8) if larger); must be the same on every rank
 *   prof         NULL, or device int64 [n_updates][4]: nanosecond stamps of update start and of the three grid barriers
 * Other arguments as carenv_ppo_grad / carenv_ppo_adam.
 *
 * carenv_ppo_epoch_kl: carenv_ppo_epoch with PPO's divergence statistics and an early stop.  Update u's statistics are
 * taken over its minibatch (all ranks' samples) at the parameters before its step, log ratio = new_logp - old_logp:
 *   kl_out      device float [n_updates][2]: approx KL mean((ratio - 1) - log ratio) and clip fraction
 *               mean(|ratio - 1| > clip_ratio); rows after the stopping update are NaN
 *   n_done      device int: the updates that applied a step; step advances by n_done
 *   target_kl   update u applies no step, and the launch ends, when its approx KL > target_kl (compared in double; no
 *               1.5 factor); +inf gives the statistics with every step applied, bit-identical to carenv_ppo_epoch
 * CARENV_E_INVAL for a null kl_out or n_done and for a target_kl that is NaN or <= 0.  Every rank reaches the same
 * decision from the same bits.  With a communicator the exchange count is kept on the device across these calls; a
 * carenv_ppo_epoch call after one reads it back (one synchronising copy). */
#define CARENV_IPC_HANDLE_BYTES 64
int carenv_ppo_comm_create(int world, int rank, void **comm, unsigned char *ipc_handle_out /* [64] */);
int carenv_ppo_comm_connect(void *comm, const unsigned char *all_handles /* [world][64], rank order */);
int carenv_ppo_comm_destroy(void *comm);
int carenv_ppo_epoch_workspace_floats(void);
int carenv_ppo_epoch(float *w1_actor, float *b1_actor, float *w2_actor, float *b2_actor, float *w1_critic,
                     float *b1_critic, float *w2_critic, float *b2_critic, const float *obs, const long long *idx,
                     const float *act, const float *old_logp, const float *adv, const float *ret, int batch,
                     int n_updates, double clip_ratio, double vf_coef, double ent_coef, float *exp_avg,
                     float *exp_avg_sq, const float *lr, int *step, double beta1, double beta2, double eps,
                     double max_grad_norm, float *sums4, float *workspace, int *sync_words, void *comm, int n_ctas,
                     long long *prof, void *stream);
int carenv_ppo_epoch_kl(float *w1_actor, float *b1_actor, float *w2_actor, float *b2_actor, float *w1_critic,
                        float *b1_critic, float *w2_critic, float *b2_critic, const float *obs, const long long *idx,
                        const float *act, const float *old_logp, const float *adv, const float *ret, int batch,
                        int n_updates, double clip_ratio, double vf_coef, double ent_coef, float *exp_avg,
                        float *exp_avg_sq, const float *lr, int *step, double beta1, double beta2, double eps,
                        double max_grad_norm, float *sums4, float *workspace, int *sync_words, void *comm, int n_ctas,
                        long long *prof, void *stream, double target_kl, float *kl_out, int *n_done);

/* Populations: P independent policies ("members") trained side by side in one process, one launch per stage for all
 * of them (csrc/population.cuh).  Member p owns its parameters, Adam state, hyperparameters, seed and n environments,
 * which are columns p*n .. p*n + n - 1 of every [N] / [T][N] array (N = P*n); members never exchange data.
 * Parameters are stacked nn.Linear tensors: w1 [P][256][18], b1 [P][256], w2_actor [P][9][256], b2_actor [P][9],
 * w2_critic [P][1][256], b2_critic [P][1].  Every call refuses n_members or n_envs_per_member <= 0, a negative n_steps
 * and null pointers (CARENV_E_INVAL).
 *   carenv_pack_policy_pop   carenv_pack_policy for every member in one launch: packed_out [P][floats], block p
 *       bit-identical to carenv_pack_policy of member p.
 *   carenv_policy_rollout_warp_pop / carenv_policy_rollout_tc_pop   one launch plays all members' rollouts (replaces,
 *       per member, the loop of train.py:173-195 as carenv_policy_rollout_warp / _tc do).  Member p keys its random
 *       stream with seeds[p] (device uint64 [P]) and its member-local env index, so its rows are bit-identical to
 *       carenv_policy_rollout_warp / _tc run alone on member p with env_offset 0 and n environments.  The warp kernel
 *       takes tracks of at most 32 wall segments, the tensor-core kernel tracks of at most 128 (CARENV_E_TRACK
 *       otherwise).  obs_buf holds full [T][N][18] rows: the handle's pose_rows option must be 0.
 *   carenv_ppo_epoch_pop   all n_updates minibatch updates of an epoch for every member in ONE cluster launch
 *       (replaces, per member, train.py:223-261 as carenv_ppo_epoch does): one thread-block cluster of
 *       carenv_ppo_epoch_pop_cluster_size() CTAs per member, gradients reduced through distributed shared memory.
 *         idx                  device int64 [P][n_updates][batch]: global rows of obs / act / ... (member p's own)
 *         lr, clip_ratio, vf_coef, ent_coef, max_grad_norm   device float [P]
 *         exp_avg, exp_avg_sq  device float [P][12,298] (flat parameter layout); step device int [P];
 *         sums4                device float [P][4]: policy loss, value loss, entropy, total loss, accumulated
 *       Deterministic, and member p's results do not depend on the other members; not bit-identical to
 *       carenv_ppo_epoch (another reduction order).  Needs no workspace.
 *   carenv_ppo_epoch_pop_kl   carenv_ppo_epoch_pop with carenv_ppo_epoch_kl's statistics and stop rule, per member:
 *       kl_out device float [P][n_updates][2], n_done device int [P]; one target_kl for every member, each member stops
 *       on its own and its bits do not depend on the other members.  Same refusals as carenv_ppo_epoch_kl.
 *   carenv_ppo_epoch_pop_resident_clusters   how many clusters of the update kernel the current device keeps resident
 *       at once (cudaOccupancyMaxActiveClusters).
 *   carenv_policy_eval_pop   carenv_policy_eval of every member in ONE launch: n_episodes_per_member episodes (global
 *       ids episode0 .. episode0 + n - 1) of each member's actor (w1_actor .. b2_actor as above) on the handle's track.
 *       Member p samples with seeds[p] (device uint64 [P]) and writes records [P][n] (block p) and, for its first
 *       n_trace episodes, trace_actions / trace_u [P][n_trace][1000] (block p), so member p's records and traces
 *       equal carenv_policy_eval of member p with seed seeds[p].  Refuses n_members outside 1..65535, a negative
 *       n_episodes_per_member or n_trace, n_trace > 0 without trace_actions and null pointers (CARENV_E_INVAL) and
 *       tracks over 128 wall segments (CARENV_E_TRACK); 0 episodes launch nothing. */
int carenv_pack_policy_pop(int tensor_cores, int n_members, const float *w1_actor, const float *b1_actor,
                           const float *w2_actor, const float *b2_actor, const float *w1_critic, const float *b1_critic,
                           const float *w2_critic, const float *b2_critic, float *packed_out, void *stream);
int carenv_policy_rollout_warp_pop(void *handle, int n_members, const float *w1_actor, const float *b1_actor,
                                   const float *w2_actor, const float *b2_actor, const float *w1_critic,
                                   const float *b1_critic, const float *w2_critic, const float *b2_critic,
                                   int n_envs_per_member, int n_steps, const unsigned long long *seeds,
                                   unsigned long long step0, double *pos, double *vel, int32_t *ints, float *cur_obs,
                                   float *cur_term, float *cur_trunc, double reward_scale, float *obs_buf,
                                   float *act_buf, float *rew_buf, float *val_buf, float *term_buf, float *trunc_buf,
                                   float *logp_buf, float *last_val, float *u_dbg, void *stream);
int carenv_policy_rollout_tc_pop(void *handle, int n_members, const float *packed_weights, int n_envs_per_member,
                                 int n_steps, const unsigned long long *seeds, unsigned long long step0, double *pos,
                                 double *vel, int32_t *ints, float *cur_obs, float *cur_term, float *cur_trunc,
                                 double reward_scale, float *obs_buf, float *act_buf, float *rew_buf, float *val_buf,
                                 float *term_buf, float *trunc_buf, float *logp_buf, float *last_val, float *u_dbg,
                                 void *stream);
int carenv_ppo_epoch_pop_cluster_size(void);
int carenv_ppo_epoch_pop_resident_clusters(int *n_clusters);
int carenv_ppo_epoch_pop(int n_members, float *w1_actor, float *b1_actor, float *w2_actor, float *b2_actor,
                         float *w1_critic, float *b1_critic, float *w2_critic, float *b2_critic, const float *obs,
                         const long long *idx, const float *act, const float *old_logp, const float *adv,
                         const float *ret, int batch, int n_updates, const float *lr, const float *clip_ratio,
                         const float *vf_coef, const float *ent_coef, const float *max_grad_norm, double beta1,
                         double beta2, double eps, float *exp_avg, float *exp_avg_sq, int *step, float *sums4,
                         void *stream);
int carenv_ppo_epoch_pop_kl(int n_members, float *w1_actor, float *b1_actor, float *w2_actor, float *b2_actor,
                            float *w1_critic, float *b1_critic, float *w2_critic, float *b2_critic, const float *obs,
                            const long long *idx, const float *act, const float *old_logp, const float *adv,
                            const float *ret, int batch, int n_updates, const float *lr, const float *clip_ratio,
                            const float *vf_coef, const float *ent_coef, const float *max_grad_norm, double beta1,
                            double beta2, double eps, float *exp_avg, float *exp_avg_sq, int *step, float *sums4,
                            void *stream, double target_kl, float *kl_out, int *n_done);
int carenv_policy_eval_pop(void *handle, int n_members, const float *w1_actor, const float *b1_actor,
                           const float *w2_actor, const float *b2_actor, long long n_episodes_per_member,
                           unsigned long long episode0, int greedy, const unsigned long long *seeds,
                           carenv_eval_record *records, int n_trace, unsigned char *trace_actions, float *trace_u,
                           void *stream);

/* Test hook for the tensor-core building blocks (csrc/tc_mlp.cuh): D[128][256] = A[128][24] * B[256][24]^T,
 * tcgen05.mma kind::tf32 with the accumulator in tensor memory; device pointers, row-major float32. */
int carenv_tc_gemm_test(const float *A, const float *B, float *D, void *stream);

/* Measurement helper (no reference counterpart): an FFMA-only kernel, blocks x 256 threads x
 * iters x 64 FFMA, used by bench.py to measure the FP32-pipe peak the step kernel is compared with. */
int carenv_bench_ffma(int blocks, int iters, float *scratch, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CARENV_B200_H */
