"""The three fused rollout kernels against float64 and Philox references, on every instantiation the C ABI can launch.

``carenv_policy_rollout_tc`` launches ``k_policy_rollout_tc3<U, TAB>`` (U = 4, 2 with and without the denominator
table, U = 1 without), ``carenv_policy_rollout`` launches ``k_policy_rollout<U>`` (U = 4, 2, 1) and
``carenv_policy_rollout_warp`` launches ``k_policy_rollout_warp``.  Which one runs depends on the track (its
``unroll4`` and pair count, carenv_tables.h, restated in :func:`track_layout`) and on the options ``tab``,
``max_unroll`` and ``force_generic``.  Every row of the track matrix below checks, for one kernel:

* the uniforms (``u_dbg``) bit for bit against :func:`philox4x32_10`, a NumPy Philox4x32-10 pinned by the Random123
  known-answer vectors, with a seed whose high word is not zero, an ``env_offset`` and a ``step0`` that crosses 2^32;
* the values, log-probabilities, bootstrap values and sampled actions against a float64 evaluation of the same weights
  (``tests.ppo_reference.net_f64``), within bounds propagated from the kernels' operation counts (below);
* every environment row, ``pos`` and ``ints`` bit for bit against a replay of the sampled actions through
  ``VecCarEnv.rollout``.

Error bounds (u = 2^-24, the float32 unit roundoff; x the observation row, exact in float32 as stored):

* First layer: |dz_j| <= c1 u (|b1_j| + sum_k |W1_jk x_k|).  A chain of n rounded FMAs that starts from one of its
  terms errs by at most gamma_n = n u / (1 - n u) times the sum of the terms' magnitudes.

  - ``k_policy_rollout`` (policy_forward): the bias, then 18 FMAs in one chain: gamma_18 < 19 u, c1 = 19.
  - ``k_policy_rollout_warp``: three chains of 6 FMAs (one starts from the bias), summed as (a + b) + c: every term
    passes at most 8 roundings, c1 = 9.
  - ``k_policy_rollout_tc3`` (3xTF32): x = x_hi + x_lo + dx with |x_lo| <= 2^-11 |x| and |dx| <= 2^-22 |x| = 4u |x|
    (x_lo is x - x_hi rounded to 11 bits), the same for the weights and the bias (column 18, times an exact 1).  The
    dropped x_lo w_lo term and the two split residues give 12 u per product.  Products of TF32 operands are exact in
    float32; the tensor core adds them to the float32 accumulator in 9 MMAs (3 passes x K 24 / 8), each allowed 4 u
    of the magnitudes involved (2 ulp: alignment and a normalisation that may truncate).  c1 = 12 + 9 x 4 = 48.

* ReLU is 1-Lipschitz: |dh_j| <= |dz_j|.
* Second layer: |dy_q| <= sum_j |W2_qj| |dz_j| + c2 u S_q + 2 u (S_q + |b2_q|), S_q = sum_j |W2_qj| (h_j + |dz_j|)
  (a bound on the magnitudes of the terms the kernel actually sums).  The bias is added last, by one rounding in
  every kernel, hence its own 2 u term instead of c2 u.

  - ``k_policy_rollout``: each logit is one FFMA2 lane over all 256 units: c2 = 257; the value sums even and odd units
    in two lanes of 128 and adds them: c2 = 130.
  - ``k_policy_rollout_tc3``: 128 units per thread in one chain, then (units 0..127) + (units 128..255): c2 = 130;
    the critic as ``k_policy_rollout``'s: 130.
  - ``k_policy_rollout_warp``: 8 FMAs per lane and a 5-level butterfly: c2 = 14 for both nets.

* Log-probability: log_softmax moves by at most 2 max_q |dy_q| under logit errors dy; the float32 evaluation
  ((l_a - m) - logf(sum expf(l_q - m)), expf within 2 ulp, logf within 1 ulp) adds (20 + 2 L + 2 |logp|) u,
  L = max_q |l_q - m|.
* Sampling: the kernel takes the first action q with u * s < c_q (s the sum of the exponentials, c_q their running
  sums), i.e. u < CDF_q.  Logit errors dy move every CDF value by at most e^(2 max|dy|) - 1 <= 2.01 max|dy|, the
  float32 arithmetic by (32 + 2 L) u more.  The sampled action must be the float64 inverse CDF of its uniform unless
  the uniform lies within that margin of a CDF value, and fewer than 1e-3 of the rows (or a single row) may be so
  close.

Tests print the worst error they saw as a fraction of its bound (run pytest with -s), and the worst per kernel over
the module when it ends.
"""
import collections
import functools
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import ppo_car_b200
from ppo_car_b200.track import builtin_track, load_track
from ppo_car_b200.train_ppo import ActorCritic
from tests.ppo_reference import net_f64
from tests.synth_tracks import near_wall_track, ring_track

needs_gpu = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")

U32 = 2.0 ** -24                       # float32 unit roundoff
MASK32 = 0xFFFFFFFF
SEED = (0x5EED << 32) | 11             # a non-zero high key word
ENV_OFFSET = 70001
STEP0 = 2 ** 32 - 17                   # the 64-bit step counter crosses 2^32 inside a 40-step rollout
ROLLOUT_STREAM, EVAL_STREAM = 0x43415245, 0x4556414C     # Philox counter word 3: "CARE" (rollouts), "EVAL"
SMEM_LIMIT = 227 * 1024
MAX_SEG, WARP_MAX_SEG = 128, 32

# ---- Philox4x32-10 ---------------------------------------------------------------------------------------------------
PHILOX_M0, PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
PHILOX_W0, PHILOX_W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al. 2011) on NumPy integers.  ``ctr``: four arrays (or ints) of 32-bit words that
    broadcast against each other; ``key``: two ints.  Returns the four output words as uint32 arrays."""
    m = np.uint64(MASK32)
    c = [np.asarray(w, dtype=np.uint64) & m for w in ctr]
    k0, k1 = np.uint64(int(key[0]) & MASK32), np.uint64(int(key[1]) & MASK32)
    for _ in range(10):
        p0, p1 = PHILOX_M0 * c[0], PHILOX_M1 * c[2]        # < 2^64: exact
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m]
        k0, k1 = (k0 + PHILOX_W0) & m, (k1 + PHILOX_W1) & m
    return [w.astype(np.uint32) for w in c]


def uniform_from_bits(c0):
    """The kernels' uniform: the top 24 bits of counter word 0 times 2^-24 (exact in float32)."""
    return ((np.asarray(c0, np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24).astype(np.float32)


def rollout_uniforms(seed, env_offset, n, step0, T):
    """[T, n] uniforms of a fused rollout: key (seed lo, seed hi), counter (env_offset + e, step lo, step hi, "CARE")."""
    gid = (np.arange(n, dtype=np.int64) + env_offset).astype(np.uint64)[None, :]
    gs = np.uint64(step0) + np.arange(T, dtype=np.uint64)[:, None]
    c0 = philox4x32_10((gid, gs & np.uint64(MASK32), gs >> np.uint64(32), ROLLOUT_STREAM), (seed & MASK32, seed >> 32))[0]
    return uniform_from_bits(c0)


def eval_uniforms(seed, episode0, n, steps):
    """[n, steps] uniforms of evaluate_policy: counter (episode id lo, step in the episode, id hi, "EVAL")."""
    ids = np.uint64(episode0) + np.arange(n, dtype=np.uint64)[:, None]
    step = np.arange(steps, dtype=np.uint64)[None, :]
    c0 = philox4x32_10((ids & np.uint64(MASK32), step, ids >> np.uint64(32), EVAL_STREAM), (seed & MASK32, seed >> 32))[0]
    return uniform_from_bits(c0)


def test_philox_known_answer_vectors():
    """Random123's known-answer vectors for philox4x32 with 10 rounds."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((MASK32,) * 4, (MASK32, MASK32), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert [int(w) for w in philox4x32_10(ctr, key)] == list(want), (ctr, key)
    # vectorised counters give the scalar results
    got = philox4x32_10((np.array([0, 0x243F6A88]), np.array([0, 0x85A308D3]), np.array([0, 0x13198A2E]),
                         np.array([0, 0x03707344])), (0, 0))[0]
    assert int(got[0]) == 0x6627E8D5 and int(got[1]) == int(philox4x32_10((0x243F6A88, 0x85A308D3, 0x13198A2E,
                                                                            0x03707344), (0, 0))[0])


def test_uniform_stream_layout():
    """The key and counter words the rollout stream uses are all significant: the high words of the seed and of the
    64-bit step move the stream, and a uniform is (c0 >> 8) 2^-24 in [0, 1)."""
    u = rollout_uniforms(SEED, ENV_OFFSET, 5, 2 ** 32 - 2, 4)
    assert u.dtype == np.float32 and u.shape == (4, 5) and (u >= 0).all() and (u < 1).all()
    assert not np.array_equal(u, rollout_uniforms(SEED & MASK32, ENV_OFFSET, 5, 2 ** 32 - 2, 4))
    low_only = philox4x32_10((ENV_OFFSET, 0, 0, ROLLOUT_STREAM), (SEED & MASK32, SEED >> 32))[0]
    assert u[2, 0] != uniform_from_bits(low_only)                # step 2^32 is not step 0
    assert np.array_equal((u * 2.0 ** 24).astype(np.float64) % 1.0, np.zeros_like(u, np.float64))


# ---- the track rule of carenv_tables.h and the launch choice of policy_abi.cuh ------------------------------------------
RINGS = {"ring10_6": (10, 6), "ring7_5": (7, 5), "ring18_12": (18, 12), "ring16_16": (16, 16), "ring42_42": (42, 42),
         "ring64_64": (64, 64)}
K_HEADINGS = 72
TC3_FIXED_SMEM = 128 + (27404 * 4 + 127) // 128 * 128 + 2 * 2 * 128 * 24 * 4 + 2 * 128 * 12 * 4   # pad, weights, A, xchg
CUDA_WEIGHT_BYTES = 13324 * 4
REQUIRED = {("tc3", 4, True), ("tc3", 4, False), ("tc3", 2, True), ("tc3", 2, False), ("tc3", 1, False),
            ("cuda", 4), ("cuda", 2), ("cuda", 1), ("warp",)}


def track_path(name, directory):
    if name in ("big_track", "track"):
        return builtin_track(name)
    if name == "near_wall":
        return near_wall_track(os.path.join(directory, "near_wall.json"))
    n_outer, n_inner = RINGS[name]
    return ring_track(os.path.join(directory, name + ".json"), n_outer, n_inner,
                      wobble=0.03 if n_outer + n_inner > 64 else 0.08)


def track_layout(path):
    """What build_host_track (carenv_tables.h) derives from a track: segment count, ``unroll`` (the first of 6, 4, 2
    that divides the segment count and every polyline start, else 1), ``unroll4`` (the same over 4, 2), the pair
    count of the denominator table (segments / 2 when unroll >= 2) and the staged table bytes."""
    t = load_track(path)
    w = t.walls
    n = len(w)
    starts = [j for j in range(n) if j == 0 or w[j - 1, 2] != w[j, 0] or w[j - 1, 3] != w[j, 1]]
    fits = lambda U: n % U == 0 and all(j % U == 0 for j in starts)
    unroll = next((U for U in (6, 4, 2) if fits(U)), 1) if n <= MAX_SEG else 0
    unroll4 = next((U for U in (4, 2) if fits(U)), 1) if n <= MAX_SEG else 1
    n_pairs = n // 2 if unroll >= 2 else 0
    return SimpleNamespace(n_seg=n, n_gates=len(t.gates), unroll=unroll, unroll4=unroll4, n_pairs=n_pairs,
                           table_bytes=3456 + 48 * len(t.gates) + 32 * n)


def instantiation(kernel, layout, opts):
    """The kernel instantiation the C ABI launches for this track and these options (policy_abi.cuh)."""
    if kernel == "warp":
        return ("warp",)
    U = 1 if opts.get("force_generic") else layout.unroll4
    cap = opts.get("max_unroll", 0)
    if cap > 0 and U > cap:
        U = cap if U % cap == 0 else 1
    if kernel == "cuda":
        return ("cuda", U)
    row_f4 = ((layout.n_pairs + 7) // 8 * 8) | 1
    fits = layout.table_bytes + TC3_FIXED_SMEM + K_HEADINGS * row_f4 * 16 <= SMEM_LIMIT
    return ("tc3", U, bool(U >= 2 and layout.n_pairs > 0 and opts.get("tab", 0) >= 0 and fits))


MATRIX = [
    ("big_track", {}, "tc3"), ("big_track", {}, "cuda"), ("big_track", {}, "warp"),
    ("big_track", {"tab": -1}, "tc3"),
    ("big_track", {"max_unroll": 2}, "tc3"), ("big_track", {"max_unroll": 2}, "cuda"),
    ("big_track", {"force_generic": 1}, "tc3"), ("big_track", {"force_generic": 1}, "cuda"),
    ("track", {}, "tc3"), ("track", {}, "cuda"), ("track", {}, "warp"),
    ("ring10_6", {}, "tc3"), ("ring10_6", {}, "cuda"), ("ring10_6", {"tab": -1}, "tc3"),
    ("ring7_5", {}, "tc3"), ("ring7_5", {}, "cuda"), ("ring7_5", {}, "warp"),
    ("ring18_12", {}, "tc3"), ("ring18_12", {}, "cuda"), ("ring18_12", {}, "warp"),
    ("ring16_16", {}, "tc3"), ("ring16_16", {}, "warp"),
    ("ring42_42", {}, "tc3"), ("ring42_42", {}, "cuda"),
    ("ring64_64", {}, "tc3"), ("ring64_64", {}, "cuda"),
    ("near_wall", {}, "tc3"), ("near_wall", {}, "cuda"), ("near_wall", {}, "warp"),
]
MATRIX_IDS = ["-".join([t] + [f"{k}{v}" for k, v in o.items()] + [k]) for t, o, k in MATRIX]


@pytest.fixture(scope="module")
def tracks(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("tracks"))
    return functools.lru_cache(maxsize=None)(lambda name: track_path(name, d))


def test_track_rule_and_matrix_reach_every_instantiation(tracks):
    """The track properties each matrix row is there for, and together the rows launch every instantiation."""
    L = {name: track_layout(tracks(name)) for name in {t for t, _, _ in MATRIX}}
    big, trk = L["big_track"], L["track"]
    assert (big.n_seg, big.unroll, big.unroll4, big.n_pairs) == (24, 6, 4, 12)
    assert (trk.n_seg, trk.unroll4, trk.n_pairs) == (16, 4, 8)                         # another n_pairs and row_f4
    assert (L["ring10_6"].unroll4, L["ring10_6"].n_pairs) == (2, 8)
    assert (L["ring7_5"].unroll, L["ring7_5"].unroll4, L["ring7_5"].n_pairs) == (1, 1, 0)
    assert (L["ring18_12"].unroll, L["ring18_12"].unroll4, L["ring18_12"].n_pairs) == (6, 2, 15)
    assert L["ring16_16"].n_seg == WARP_MAX_SEG
    assert (L["ring42_42"].n_seg, L["ring42_42"].unroll4, L["ring64_64"].n_seg, L["ring64_64"].unroll4) == (84, 2, 128, 4)
    assert L["near_wall"].n_seg == 16
    reached = {}
    for (t, opts, kernel), name in zip(MATRIX, MATRIX_IDS):
        if kernel == "warp":
            assert L[t].n_seg <= WARP_MAX_SEG, name
        reached.setdefault(instantiation(kernel, L[t], opts), []).append(name)
    assert REQUIRED <= set(reached), REQUIRED - set(reached)
    # 84 and 128 segments: the table does not fit next to tc3's weights, the table-free instantiation does
    for t in ("ring42_42", "ring64_64"):
        assert instantiation("tc3", L[t], {}) == ("tc3", L[t].unroll4, False)
        assert L[t].table_bytes + TC3_FIXED_SMEM <= SMEM_LIMIT
        assert L[t].table_bytes + CUDA_WEIGHT_BYTES <= SMEM_LIMIT
    assert instantiation("tc3", L["ring18_12"], {}) == ("tc3", 2, True)
    assert instantiation("tc3", big, {"max_unroll": 2}) == ("tc3", 2, True)


# ---- float64 network reference ---------------------------------------------------------------------------------------
C1 = {"cuda": 19, "warp": 9, "tc3": 48}
C2 = {"cuda": (257, 130), "warp": (14, 14), "tc3": (130, 130)}     # (actor logits, critic value)
WORST = collections.defaultdict(float)                               # (kernel, quantity) -> worst error / bound
MAX_REF_ROWS = 20000


def _layer_bounds(seq, x, c1, c2):
    """float64 outputs of nn.Sequential(Linear, ReLU, Linear) ``seq`` at ``x`` and the bound on a kernel's error."""
    W1, b1, W2, b2 = (p.detach() for p in (seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias))
    z = x @ W1.T + b1
    dz = c1 * U32 * (x.abs() @ W1.abs().T + b1.abs())
    h = z.clamp(min=0.0)
    y = h @ W2.T + b2
    s = (h + dz) @ W2.abs().T
    dy = dz @ W2.abs().T + c2 * U32 * s + 2 * U32 * (s + b2.abs())
    return y, dy


def reference(net, obs, kernel):
    """float64 logits, their error bounds, values and their bounds for float32 observation rows [M, 18]."""
    ref = net_f64([net.actor[0].weight, net.actor[0].bias, net.actor[2].weight, net.actor[2].bias,
                   net.critic[0].weight, net.critic[0].bias, net.critic[2].weight, net.critic[2].bias])
    x = torch.as_tensor(np.asarray(obs, np.float32)).double()
    with torch.no_grad():
        logits, dlogits = _layer_bounds(ref.actor, x, C1[kernel], C2[kernel][0])
        value, dvalue = _layer_bounds(ref.critic, x, C1[kernel], C2[kernel][1])
    return logits, dlogits, value[:, 0], dvalue[:, 0]


def _record(kernel, what, frac, tag):
    WORST[(kernel, what)] = max(WORST[(kernel, what)], frac)
    print(f"{tag}: {what} worst error {frac:.3g} of its bound")


def check_network(kernel, net, r, final_obs=None, tag="", near_limit=1e-3, rows=None):
    """Values, log-probabilities, sampled actions (and last_val against ``final_obs``) of the run ``r`` against the
    float64 reference.  ``rows``: the flat row indices to check (default: all, or MAX_REF_ROWS of them)."""
    obs = r.obs.reshape(-1, 18).cpu().numpy()
    M = obs.shape[0]
    if rows is None:
        rows = np.arange(M) if M <= MAX_REF_ROWS else np.sort(np.random.default_rng(M).choice(M, MAX_REF_ROWS, False))
    take = lambda t: torch.from_numpy(t.reshape(-1).cpu().numpy()[rows]).double()
    act, logp, val, u = take(r.act).long(), take(r.logp), take(r.val), take(r.u)
    logits, dl, value, dv = reference(net, obs[rows], kernel)
    assert torch.isfinite(logp).all() and torch.isfinite(val).all()
    assert ((act >= 0) & (act <= 8)).all()
    dmax = dl.max(-1).values
    spread = (logits - logits.max(-1, keepdim=True).values).abs().max(-1).values
    logp64 = torch.log_softmax(logits, -1).gather(-1, act[:, None])[:, 0]
    tol_logp = 2.0 * dmax + (20.0 + 2.0 * spread + 2.0 * logp64.abs()) * U32
    f_logp = ((logp - logp64).abs() / tol_logp).max().item()
    f_val = ((val - value).abs() / dv).max().item()
    _record(kernel, "logp", f_logp, tag)
    _record(kernel, "value", f_val, tag)
    assert f_logp <= 1.0 and f_val <= 1.0, (f_logp, f_val)
    cdf = torch.softmax(logits, -1).cumsum(-1)[:, :-1]
    margin = 2.01 * dmax + (32.0 + 2.0 * spread) * U32
    expect = (cdf <= u[:, None]).sum(-1)
    near = ((cdf - u[:, None]).abs() < margin[:, None]).any(-1)
    bad = (expect != act) & ~near
    assert not bad.any(), (int(bad.sum()), rows[bad.numpy()][:5])
    assert near.double().mean().item() < near_limit or near.sum().item() <= 1, near.double().mean().item()
    if final_obs is not None and r.last_val is not None:
        _, _, v_last, dv_last = reference(net, final_obs.cpu().numpy(), kernel)
        f_last = ((r.last_val.cpu().double() - v_last).abs() / dv_last).max().item()
        _record(kernel, "last_val", f_last, tag)
        assert f_last <= 1.0, f_last


def check_uniforms(r, n, T, step0, env_offset=ENV_OFFSET, seed=SEED):
    want = rollout_uniforms(seed, env_offset, n, step0, T)
    got = r.u.cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), int((got != want).sum())


# ---- running the kernels -----------------------------------------------------------------------------------------------
def make_policy(seed=3, actor_scale=4.0, bias=None):
    """ActorCritic with a non-uniform actor (second layer x actor_scale, biases ``bias`` or -1..1) on the GPU."""
    torch.manual_seed(seed)
    net = ActorCritic(18, 9).cuda()
    with torch.no_grad():
        net.actor[2].weight.mul_(actor_scale)
        net.actor[2].bias.copy_(torch.linspace(-1, 1, 9) if bias is None else torch.as_tensor(bias, dtype=torch.float32))
        net.critic[2].bias.fill_(0.3)
    return net


def make_env(path, n, opts=None):
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    for k, v in (opts or {}).items():
        env.set_option(k, v)
    return env


def start_state(env):
    n = env.num_envs
    return [env.reset()[0].clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")]


def fused(kernel, env, net, T, step0, state, last_val=True, env_offset=ENV_OFFSET, seed=SEED):
    """One launch of ``kernel`` ("tc3", "cuda" or "warp") for T steps from ``state`` = [cur_obs, cur_term, cur_trunc]
    (updated in place).  Returns the Buffer rows, the uniforms and the bootstrap values."""
    n = env.num_envs
    buf = ppo_car_b200.Buffer((18,), T, n, torch.device("cuda"))
    lv = torch.full((n,), float("nan"), device="cuda") if last_val else None
    u = torch.full((T, n), float("nan"), device="cuda")
    if kernel == "warp":
        ppo_car_b200.fused_rollout_warp(env, net.actor, net.critic, buf, *state, seed=seed, step0=step0,
                                        env_offset=env_offset, last_val=lv, u_dbg=u)
    else:
        tc = kernel == "tc3"
        pack = ppo_car_b200.pack_policy_weights_tc if tc else ppo_car_b200.pack_policy_weights
        ppo_car_b200.fused_rollout(env, pack(net.actor, net.critic), buf, *state, seed=seed, step0=step0,
                                   env_offset=env_offset, last_val=lv, u_dbg=u, tensor_cores=tc)
    torch.cuda.synchronize()
    return SimpleNamespace(obs=buf.obs_buf, act=buf.act_buf, rew=buf.rew_buf, val=buf.val_buf, term=buf.term_buf,
                           trunc=buf.trunc_buf, logp=buf.logprob_buf, u=u, last_val=lv)


def check_replay(path, env, runs, state, store_info=False):
    """The rows of consecutive launches ``runs`` (from reset) against VecCarEnv.rollout of their actions, bit for bit:
    observations, rewards, the flags that came with each observation, the final state, pos and ints."""
    cat = lambda k: torch.cat([getattr(r, k) for r in runs])
    act, obs, rew, term, trunc = cat("act"), cat("obs"), cat("rew"), cat("term"), cat("trunc")
    env2 = make_env(path, env.num_envs)
    obs0 = env2.reset()[0].clone()
    out = env2.rollout(act.to(torch.uint8), store_info=store_info)
    assert torch.equal(obs[0], obs0) and torch.equal(obs[1:], out["obs"][:-1])
    assert torch.equal(rew, out["reward"])
    assert not term[0].any() and not trunc[0].any()
    assert torch.equal(term[1:], out["terminated"][:-1]) and torch.equal(trunc[1:], out["truncated"][:-1])
    cur_obs, cur_term, cur_trunc = state
    assert torch.equal(cur_obs, out["obs"][-1]) and torch.equal(cur_term, out["terminated"][-1])
    assert torch.equal(cur_trunc, out["truncated"][-1])
    assert torch.equal(env.pos, env2.pos) and torch.equal(env.vel, env2.vel) and torch.equal(env.ints, env2.ints)
    return out


def full_check(kernel, path, n, T, net=None, opts=None, step0=STEP0, last_val=True, tag="", ref_rows=None):
    net = net if net is not None else make_policy()
    env = make_env(path, n, opts)
    state = start_state(env)
    r = fused(kernel, env, net, T, step0, state, last_val=last_val)
    check_uniforms(r, n, T, step0)
    check_network(kernel, net, r, state[0] if last_val else None, tag=tag, rows=ref_rows)
    check_replay(path, env, [r], state)
    return r


# ---- c. every instantiation on tracks of 16 to 128 segments ------------------------------------------------------------
@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("track,opts,kernel", MATRIX, ids=MATRIX_IDS)
def test_variant_track_matrix(tracks, track, opts, kernel):
    path = tracks(track)
    r = full_check(kernel, path, 300, 40, opts=opts, tag=f"{track} {opts} {kernel}")
    if track == "near_wall":                                         # the start pose is inside the wall
        assert r.term[1:].all() and r.rew.lt(0).all()
    else:
        assert len(torch.unique(r.act)) == 9


# ---- a. the evaluation kernel's random stream -------------------------------------------------------------------------
@pytest.mark.gpu
@needs_gpu
def test_policy_eval_trace_uniforms_are_philox(tracks):
    from ppo_car_b200 import evaluate_policy

    env = ppo_car_b200.VecCarEnv(1, tracks("track"), device="cuda:0")
    n, episode0 = 48, 2 ** 32 - 20                                   # episode ids cross 2^32
    res = evaluate_policy(env, make_policy(5).actor, n, greedy=False, seed=SEED, episode0=episode0, trace=n)
    torch.cuda.synchronize()
    got = res.trace_u.cpu().numpy()
    want = eval_uniforms(SEED, episode0, n, got.shape[1])
    live = ~np.isnan(got)
    assert live.sum() >= n and live[:, 0].all()
    assert np.array_equal(got[live].view(np.uint32), want[live].view(np.uint32))


# ---- d. episode boundaries ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("kernel", ["tc3", "cuda", "warp"])
def test_standing_still_truncates_and_resets(tracks, kernel):
    """An actor that almost always picks action 8 (no thrust, no turn) never crashes, so every episode runs into the
    1000-step limit.  The first launch ends on the truncating step: cur_trunc is set everywhere and last_val is the
    value of the reset observation; the second launch starts from it (trunc_buf row 0 set, the reset observation)."""
    path = tracks("big_track")
    n = 64
    net = make_policy(7, actor_scale=0.1, bias=[0.0] * 8 + [20.0])
    env = make_env(path, n)
    state = start_state(env)
    obs0 = state[0].clone()
    a = fused(kernel, env, net, 1000, STEP0, state)
    assert state[2].eq(1).all() and not state[1].any() and torch.equal(state[0], obs0)
    check_network(kernel, net, a, state[0], tag=f"stand still {kernel}, launch 1")
    b = fused(kernel, env, net, 100, STEP0 + 1000, state)
    assert b.trunc[0].eq(1).all() and not b.trunc[1:].any() and torch.equal(b.obs[0], obs0)
    assert a.act.eq(8).float().mean() > 0.999
    check_network(kernel, net, b, state[0], tag=f"stand still {kernel}, launch 2")
    check_uniforms(a, n, 1000, STEP0)
    check_uniforms(b, n, 100, STEP0 + 1000)
    out = check_replay(path, env, [a, b], state)
    assert out["truncated"][999].eq(1).all() and not out["terminated"].any()


@pytest.fixture(scope="module")
def trained_net(tmp_path_factory):
    """The README run's shape (24 envs x 1024 steps x 200 epochs on big_track, fused rollout and update), read back
    from its model.dat."""
    from ppo_car_b200.evaluate import load_checkpoint
    from ppo_car_b200.train_ppo import parse_args, train

    d = tmp_path_factory.mktemp("ckpt")
    train(parse_args(["--track", "big_track", "--n-envs", "24", "--fused-rollout", "--fused-update",
                      "--checkpoint-dir", str(d), "--run-name", "readme"]))
    return load_checkpoint(str(d / "readme" / "model.dat")).cuda()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("kernel", ["tc3", "cuda", "warp"])
def test_trained_policy_laps(tracks, trained_net, kernel):
    """A trained policy completes laps (+10) inside the fused rollout; the replay's lap events and rewards agree bit for
    bit, and the trained network's outputs stay within the float64 bounds."""
    path = tracks("big_track")
    n, T = 1024, 1000
    env = make_env(path, n)
    state = start_state(env)
    r = fused(kernel, env, trained_net, T, 0, state)
    out = check_replay(path, env, [r], state, store_info=True)
    laps = (out["info"]["events"] & 2) != 0
    assert laps.sum().item() > 0
    check_uniforms(r, n, T, 0)
    # a trained actor is sharper: more rows sit near a CDF value at the same relative precision
    check_network(kernel, trained_net, r, state[0], tag=f"trained {kernel}", near_limit=0.05)


# ---- e. launch shapes -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, 255, 257])
@pytest.mark.parametrize("kernel", ["tc3", "cuda", "warp"])
def test_environment_counts(tracks, kernel, n):
    full_check(kernel, tracks("big_track"), n, 24, tag=f"n={n} {kernel}")


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("kernel", ["tc3", "cuda"])
def test_more_ctas_than_sms(tracks, kernel):
    """40,003 environments: 157 tc3 CTAs / 313 CUDA-core CTAs, more than the 148 SMs of a B200."""
    n, T = 40003, 8
    rows = np.sort(np.random.default_rng(1).choice(n * T, 4000, replace=False))
    full_check(kernel, tracks("big_track"), n, T, tag=f"n={n} {kernel}", ref_rows=rows)


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("last_val", [False, True])
@pytest.mark.parametrize("T", [1, 2, 3, 7])
@pytest.mark.parametrize("kernel", ["tc3", "cuda", "warp"])
def test_step_counts(tracks, kernel, T, last_val):
    """tc3's bootstrap pass uses the mbarrier parity of pass T: odd and even T, with and without it."""
    r = full_check(kernel, tracks("big_track"), 300, T, last_val=last_val, tag=f"T={T} last_val={last_val} {kernel}")
    assert r.last_val is None or torch.isfinite(r.last_val).all()


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("kernel", ["tc3", "cuda", "warp"])
def test_two_launches_equal_one(tracks, kernel):
    """A rollout split into two launches (the second from the first's cur_obs / cur_term / cur_trunc, step0 + T), as
    training does every epoch, is bit-identical to one launch of 2T."""
    path = tracks("big_track")
    n, T = 300, 37
    net = make_policy(11)
    env1, env2 = make_env(path, n), make_env(path, n)
    s1, s2 = start_state(env1), start_state(env2)
    one = fused(kernel, env1, net, 2 * T, STEP0, s1)
    a = fused(kernel, env2, net, T, STEP0, s2, last_val=False)
    b = fused(kernel, env2, net, T, STEP0 + T, s2)
    for k in ("obs", "act", "rew", "val", "term", "trunc", "logp", "u"):
        assert torch.equal(getattr(one, k), torch.cat([getattr(a, k), getattr(b, k)])), k
    assert torch.equal(one.last_val, b.last_val)
    for x, y in zip(s1, s2):
        assert torch.equal(x, y)
    assert torch.equal(env1.pos, env2.pos) and torch.equal(env1.vel, env2.vel) and torch.equal(env1.ints, env2.ints)


# ---- f. errors -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@needs_gpu
def test_tracks_the_kernels_refuse(tmp_path):
    """Refusals are CARENV_E_TRACK (code -2) errors raised before anything is launched or configured, not CUDA
    errors (code -1000 - cudaError_t)."""
    net = make_policy()

    def attempt(kernel, path):
        env = make_env(path, 8)
        return fused(kernel, env, net, 4, 0, start_state(env))

    too_many = ring_track(str(tmp_path / "ring_140.json"), 100, 40, wobble=0.03)
    for kernel in ("tc3", "cuda"):
        with pytest.raises(ppo_car_b200.CarEnvError, match=r"\(code -2\).*at most 128 wall segments"):
            attempt(kernel, too_many)
    ring33 = ring_track(str(tmp_path / "ring_33.json"), 17, 16)
    with pytest.raises(ppo_car_b200.CarEnvError, match=r"\(code -2\).*at most 32 wall segments"):
        attempt("warp", ring33)
    attempt("tc3", ring33)                                           # the packed kernels take it
    # 4,000 gates: 196 KB of track tables, no room for any kernel's weights
    gates = ring_track(str(tmp_path / "gates_4000.json"), 10, 6, n_gates=4000)
    for kernel in ("tc3", "cuda", "warp"):
        with pytest.raises(ppo_car_b200.CarEnvError, match=r"\(code -2\).*too large"):
            attempt(kernel, gates)
    full_check("cuda", ring_track(str(tmp_path / "ring_ok.json"), 10, 6), 8, 4)    # the device is still usable


# ---- report -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", autouse=True)
def report_worst_errors():
    """After the module: the worst error per kernel and quantity over the tests that ran (pytest -s)."""
    yield
    for (kernel, what), frac in sorted(WORST.items()):
        print(f"worst {kernel:5s} {what:9s} {frac:.3g} of its bound")
