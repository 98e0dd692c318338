"""The environment step kernels against the float64 C oracle, on every instantiation the C ABI can launch.

``carenv_rollout`` (``launch_rollout`` / ``launch_rollout_tab`` in csrc/carenv_kernels.cu) runs one of four kernels:

* ``k_rollout_warp``: one warp per environment, for at most 32 segments and small batches (or ``warp_per_env=1``);
* ``k_rollout<U>``, U = 6, 4, 2, 1, 0: the segment loop unrolled U times (0: more than 128 segments, geometry in shared
  memory), from the track's ``unroll``, ``max_unroll`` and ``force_generic``;
* ``k_rollout_tab<U>``, U = 6, 4, 2: the denominators from a shared-memory table kept in 8, 4, 2 or 1 skewed copies,
  for launches of 4,096 environments or more (or ``tab=1``) when at least one copy fits;
* ``k_rollout_tab_sliced<U>``: the table kernel with an SM's env-steps cut into one equal interval per warp, when every
  SM gets at least one 32-environment job per warp and a launch has at least 4 steps.

:func:`step_instantiation` restates that choice, with the constants read from the sources, and
:func:`test_launch_rule_and_matrix_reach_every_instantiation` proves that the matrix below reaches every
instantiation.  On the GPU each row is checked three ways:

* the profiler names the kernel that ran, its template arguments and its shared memory (the table's copy count), and
  they must be what :func:`step_instantiation` says;
* integers bit for bit, rewards as float32 of the float64 reward and observations to 1e-5 relative against
  ``oracle.c_oracle.COracleVecEnv``, from a forward-biased random rollout;
* every output, ``pos``, ``vel``, ``ints`` and ``slow_path_counts()`` bit for bit against the same rollout forced onto
  ``k_rollout`` (``tab=-1``, ``tab_slice=-1``, ``warp_per_env=-1``).

Launches of the time-sliced kernel are about 75 k environments or more.  There the oracle runs on the environments of
every job that is cut between two warps (from ``slice_items``, emulated on the host), the grid's first and last jobs
and a random sample; the bit-for-bit comparison with ``k_rollout`` covers the rest of the grid.

The sliced kernel's condition depends on the SM count, so every GPU test fails on a device whose SM count differs
from the one the matrix assumes.
"""
import functools
import json
import os
import re
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import ppo_car_b200
from tests.parity import RTOL, RTOL_SYNTHETIC, assert_trajectory_matches
from tests.synth_tracks import ring_track
from tests.test_fused_rollout_reference import RINGS, track_layout, track_path

needs_gpu = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")

SMS = 148                                         # a B200
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ppo_car_b200", "csrc")


# ---- the launch rule of launch_rollout / launch_rollout_tab, with its constants read from the sources ------------------
def _read(name):
    with open(os.path.join(CSRC, name)) as fh:
        return fh.read()


def _int(pattern, text):
    m = re.search(pattern, text)
    assert m, f"launch rule changed: {pattern!r} not found; restate step_instantiation"
    return int(m.group(1))


@functools.lru_cache(maxsize=None)
def launch_constants():
    k, core = _read("carenv_kernels.cu"), _read("carenv_core.cuh")
    assert "const int row_f4 = (n_pairs + 7) / 8 * 8;" in k, "table row rule changed; restate table_copies"
    assert "if (h->host.P.n_seg > kMaxSeg) U = 0;" in k and "copies >>= 1;" in k
    return SimpleNamespace(
        headings=_int(r"constexpr int kHeadings = (\d+);", core),
        max_seg=_int(r"constexpr int kMaxSeg = (\d+);", core),
        warp_max_seg=_int(r"const bool warp_ok = h->host\.P\.n_seg <= (\d+) && !h->force_generic;", k),
        warp_per_env_max=_int(r"constexpr int kWarpPerEnvMax = (\d+);", k),
        tab_min_envs=_int(r"\(h->tab == 1 \|\| n_envs >= (\d+)\)\)", k),
        tab_threads=_int(r"#define CARENV_TAB_THREADS (\d+)", k),
        copies=_int(r"int copies = (\d+);", k),
        pad=_int(r"\(size_t\)table_bytes \+ (\d+) \+ \(size_t\)c \* \(kHeadings \* row_f4 \+ 1\) \* 16", k),
        smem_limit=_int(r"while \(copies > 1 && total\(copies\) > (\d+) \* 1024\)", k) * 1024,
        job=_int(r"const long long jobs = \(n_envs \+ \d+\) / (\d+);", k),
        slice_min_steps=_int(r"jobs / sms >= block / 32 && block == kTabThreads && n_steps >= (\d+);", k),
    )


def table_bytes(layout, copies):
    """Dynamic shared memory of a table-kernel launch with ``copies`` copies: the staged track tables (rounded to 16
    bytes), a 128-byte alignment pad, then per copy 72 rows of ``row_f4`` float4 plus one float4 of skew."""
    c = launch_constants()
    row_f4 = (layout.n_pairs + 7) // 8 * 8
    return (layout.table_bytes + 15) // 16 * 16 + c.pad + copies * (c.headings * row_f4 + 1) * 16


def table_copies(layout):
    """Copies of the denominator table launch_rollout_tab keeps: halved from 8 until the table fits, 0 when even one
    copy does not fit (the launch then falls through to k_rollout)."""
    c = launch_constants()
    copies = c.copies
    while copies > 1 and table_bytes(layout, copies) > c.smem_limit:
        copies //= 2
    return copies if table_bytes(layout, copies) <= c.smem_limit else 0


def step_instantiation(layout, n_envs, n_steps, opts, sms=SMS):
    """The kernel carenv_rollout launches: ``("warp",)``, ``("arith", U)`` (k_rollout<U>), ``("tab", U, copies)`` or
    ``("sliced", U, copies)``.  ``opts``: the handle options ``tab``, ``tab_slice``, ``warp_per_env``, ``max_unroll``,
    ``force_generic``, and ``capture=True`` for a launch inside a CUDA graph capture on a handle that has not allocated
    the sliced kernel's flags yet (no allocation is allowed there: the block scheme runs)."""
    c = launch_constants()
    assert not set(opts) - {"tab", "tab_slice", "warp_per_env", "max_unroll", "force_generic", "capture"}, opts
    sign = lambda v: (v > 0) - (v < 0)
    wpe = sign(opts.get("warp_per_env", 0))
    if layout.n_seg <= c.warp_max_seg and not opts.get("force_generic") and (
            wpe == 1 or (wpe == 0 and n_envs <= c.warp_per_env_max)):
        return ("warp",)
    U = 1 if opts.get("force_generic") else layout.unroll
    cap = opts.get("max_unroll", 0)
    if cap > 0 and U > cap:
        U = cap if U % cap == 0 else 1
    if layout.n_seg > c.max_seg:
        U = 0
    tab = sign(opts.get("tab", 0))
    if U >= 2 and layout.n_pairs > 0 and tab >= 0 and (tab == 1 or n_envs >= c.tab_min_envs):
        copies = table_copies(layout)
        if copies:
            jobs = -(-n_envs // c.job)
            sliced = (opts.get("tab_slice", 0) >= 0 and jobs // sms >= c.tab_threads // 32
                      and n_steps >= c.slice_min_steps and not opts.get("capture"))
            return ("sliced" if sliced else "tab", U, copies)
    return ("arith", U)


def reference_opts(layout, n_envs, n_steps, opts):
    """Options that run the same rollout on k_rollout: the table and warp kernels switched off, and for a row that
    already runs k_rollout<U> the generic loop (None when that is the same kernel again)."""
    base = {k: v for k, v in opts.items() if k != "capture"}
    base.update(tab=-1, tab_slice=-1, warp_per_env=-1)
    if step_instantiation(layout, n_envs, n_steps, base) == step_instantiation(layout, n_envs, n_steps, opts):
        base["force_generic"] = 1
        if step_instantiation(layout, n_envs, n_steps, base) == step_instantiation(layout, n_envs, n_steps, opts):
            return None
    return base


# ---- tracks and the matrix ---------------------------------------------------------------------------------------------
# Tracks the fused-rollout module does not need: 48 segments (4 table copies), 3,900 gates (1 copy), 4,000 gates (no
# copy fits), 140 segments (U = 0).  (outer, inner, gates)
EXTRA = {"ring24_24": (24, 24, 12), "gates3900": (10, 6, 3900), "gates4000": (10, 6, 4000), "ring100_40": (100, 40, 12)}
SLICED_N = 100_003                 # 3,126 jobs, 21 or 22 per SM; the last job has 3 environments

MATRIX = [
    # track, n_envs, n_steps, opts, the instantiation the row is there for
    ("big_track", 1000, 200, {}, ("warp",)),
    ("big_track", 3000, 200, {}, ("arith", 6)),
    ("big_track", 3000, 200, {"max_unroll": 4}, ("arith", 1)),          # 4 does not divide 6: the generic loop
    ("big_track", 5000, 100, {"force_generic": 1}, ("arith", 1)),
    ("big_track", 4095, 100, {}, ("arith", 6)),
    ("big_track", 4096, 100, {}, ("tab", 6, 8)),
    ("big_track", 3000, 100, {"tab": 1}, ("tab", 6, 8)),
    ("big_track", 5000, 200, {}, ("tab", 6, 8)),
    ("big_track", SLICED_N, 40, {}, ("sliced", 6, 8)),
    ("big_track", 5000, 200, {"max_unroll": 2}, ("tab", 2, 8)),
    ("big_track", SLICED_N, 40, {"max_unroll": 2}, ("sliced", 2, 8)),
    ("track", 3000, 200, {}, ("arith", 4)),
    ("track", 5000, 200, {}, ("tab", 4, 8)),
    ("track", SLICED_N, 40, {}, ("sliced", 4, 8)),
    ("ring10_6", 3000, 200, {}, ("arith", 2)),
    ("ring10_6", 5000, 200, {}, ("tab", 2, 8)),
    ("ring10_6", SLICED_N, 40, {}, ("sliced", 2, 8)),
    ("ring18_12", 1000, 200, {}, ("warp",)),
    ("ring18_12", 5000, 200, {}, ("tab", 6, 8)),
    ("ring24_24", 5000, 200, {}, ("tab", 6, 4)),
    ("ring24_24", SLICED_N, 40, {}, ("sliced", 6, 4)),
    ("ring42_42", 1000, 200, {}, ("arith", 6)),
    ("ring42_42", 5000, 200, {}, ("tab", 6, 2)),
    ("ring64_64", 5000, 200, {}, ("tab", 4, 2)),
    ("ring64_64", SLICED_N, 40, {}, ("sliced", 4, 2)),
    ("near_wall", 1000, 40, {}, ("warp",)),
    ("near_wall", 5000, 40, {}, ("tab", 2, 8)),
    ("near_wall", SLICED_N, 8, {}, ("sliced", 2, 8)),
    ("gates3900", 5000, 200, {}, ("tab", 2, 1)),
    ("gates3900", SLICED_N, 40, {}, ("sliced", 2, 1)),
    ("gates4000", 5000, 200, {}, ("arith", 2)),                         # not even one table copy fits
    ("ring100_40", 1000, 100, {}, ("arith", 0)),
]
MATRIX_IDS = ["-".join([t, f"{n}x{T}"] + [f"{k}{v}" for k, v in o.items()]) for t, n, T, o, _ in MATRIX]
REQUIRED = ({("warp",)} | {("arith", U) for U in (6, 4, 2, 1, 0)}
            | {(k, U) for k in ("tab", "sliced") for U in (6, 4, 2)})

# The table and time-sliced kernels at U = 6 and U = 2, for the dtype, observation-mode and launch-sequence tests.
CASES = {"tab6": ("big_track", 5000, {}), "sliced6": ("big_track", SLICED_N, {}),
         "tab2": ("ring10_6", 5000, {}), "sliced2": ("ring10_6", SLICED_N, {})}
# Sizes around the sliced kernel's condition jobs / SMs >= 16: 2,368 jobs of 32 environments are 75,745 .. 75,776
# environments (exactly 16 jobs per SM at 75,776), one environment fewer than 75,745 is 2,367 jobs.
THRESHOLD_N = (SMS * 16 * 32, SMS * 16 * 32 - 1, SMS * 16 * 32 - 31, SMS * 16 * 32 - 32)
THRESHOLD_T = (3, 4, 5)


def make_track(name, directory):
    if name in EXTRA:
        n_outer, n_inner, n_gates = EXTRA[name]
        return ring_track(os.path.join(directory, name + ".json"), n_outer, n_inner, n_gates=n_gates,
                          wobble=0.03 if n_outer + n_inner > 64 else 0.08)
    return track_path(name, directory)


@pytest.fixture(scope="module")
def tracks(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("step_tracks"))
    return functools.lru_cache(maxsize=None)(lambda name: make_track(name, d))


def test_launch_constants_read_from_the_sources():
    c = launch_constants()
    assert c.tab_threads % 32 == 0 and c.copies in (1, 2, 4, 8) and c.job == 32
    assert c.warp_max_seg == 32 and c.max_seg == 128 and c.headings == 72
    # the smallest sliced launch on a B200: every SM holds tab_threads / 32 jobs, the last one may hold 1 environment
    lo = (SMS * (c.tab_threads // 32) - 1) * c.job + 1
    layout = SimpleNamespace(n_seg=24, unroll=6, n_pairs=12, table_bytes=6000)
    assert step_instantiation(layout, lo, c.slice_min_steps, {})[0] == "sliced"
    assert step_instantiation(layout, lo - 1, c.slice_min_steps, {})[0] == "tab"
    assert step_instantiation(layout, lo, c.slice_min_steps - 1, {})[0] == "tab"


def test_launch_rule_and_matrix_reach_every_instantiation(tracks):
    """The track properties each matrix row is there for, and together the rows launch every instantiation: warp,
    k_rollout<6, 4, 2, 1, 0>, both table kernels at U = 6, 4, 2, every copy count, and the fall-through to k_rollout."""
    c = launch_constants()
    L = {name: track_layout(tracks(name)) for name in {t for t, *_ in MATRIX}}
    prop = lambda t: (L[t].n_seg, L[t].unroll, L[t].n_pairs, table_copies(L[t]))
    assert prop("big_track") == (24, 6, 12, 8)
    assert prop("track") == (16, 4, 8, 8)
    assert prop("ring10_6") == (16, 2, 8, 8)
    assert prop("ring18_12") == (30, 6, 15, 8) and L["ring18_12"].n_seg <= c.warp_max_seg   # odd pair count
    assert prop("ring24_24") == (48, 6, 24, 4)
    assert prop("ring42_42") == (84, 6, 42, 2)
    assert prop("ring64_64") == (128, 4, 64, 2) and L["ring64_64"].n_seg == c.max_seg
    assert prop("near_wall") == (16, 2, 8, 8)
    assert prop("gates3900") == (16, 2, 8, 1) and L["gates3900"].n_gates == 3900
    assert prop("gates4000") == (16, 2, 8, 0) and L["gates4000"].n_gates == 4000
    assert L["ring100_40"].n_seg == 140 and L["ring100_40"].unroll == 0
    # a copy count one step up does not fit: the rows really sit at the copy counts they are there for
    for t, copies in (("ring24_24", 4), ("ring42_42", 2), ("ring64_64", 2), ("gates3900", 1)):
        assert table_bytes(L[t], 2 * copies) > c.smem_limit >= table_bytes(L[t], copies), t
    assert table_bytes(L["gates4000"], 1) > c.smem_limit
    reached, copies = {}, set()
    for (t, n, T, opts, want), name in zip(MATRIX, MATRIX_IDS):
        got = step_instantiation(L[t], n, T, opts)
        assert got == want, (name, got)
        reached.setdefault(got[:2], []).append(name)
        if got[0] in ("tab", "sliced"):
            copies.add(got[2])
    assert REQUIRED <= set(reached), REQUIRED - set(reached)
    assert {8, 4, 2, 1} <= copies
    fall_through = [r for r in MATRIX if r[0] == "gates4000"]
    assert fall_through and all(r[1] >= c.tab_min_envs and L["gates4000"].unroll >= 2 for r in fall_through)
    for t, n, _ in CASES.values():
        assert L[t].unroll in (6, 2)


def test_threshold_and_capture_rows_take_the_kernels_they_test(tracks):
    """75,776 and 75,775 environments are both 2,368 jobs: time-sliced from 4 steps on.  The boundary is one
    environment above 2,367 full jobs (75,745 sliced, 75,744 block rounds).  A fresh handle inside a graph capture
    takes the block scheme."""
    for name in ("big_track", "ring10_6"):
        L = track_layout(tracks(name))
        U = L.unroll
        for n in THRESHOLD_N:
            for T in THRESHOLD_T:
                want = ("sliced" if n > THRESHOLD_N[-1] and T >= 4 else "tab", U, 8)
                assert step_instantiation(L, n, T, {}) == want, (name, n, T)
        assert step_instantiation(L, SLICED_N, 24, {"capture": True}) == ("tab", U, 8)
        assert step_instantiation(L, SLICED_N, 24, {"tab_slice": -1}) == ("tab", U, 8)
        assert step_instantiation(L, SLICED_N, 24, {}) == ("sliced", U, 8)
    # the same launch on a GPU with 8 more SMs would take the other kernel
    assert step_instantiation(track_layout(tracks("big_track")), THRESHOLD_N[0], 24, {}, sms=SMS + 8)[0] == "tab"


def straddling_jobs(n_envs, n_steps, sms=SMS):
    """Jobs (32-environment blocks) that k_rollout_tab_sliced splits between two warps: CTA b owns jobs
    [b J / sms, (b + 1) J / sms), and a job is cut where a warp's work list (slice_items) starts with a head part."""
    import ctypes as C

    from tests.emul_util import lib

    c = launch_constants()
    L = lib()
    out = (C.c_int * 4)()
    jobs, n_slots = -(-n_envs // c.job), c.tab_threads // 32
    cut = []
    for b in range(sms):
        lo, hi = b * jobs // sms, (b + 1) * jobs // sms
        for slot in range(n_slots):
            L.emul_slice_items(hi - lo, n_steps, slot, n_slots, out)
            if out[1] > 0:
                cut.append(lo + out[0])
    return np.array(sorted(set(cut)), np.int64)


def test_straddling_jobs_of_the_sliced_sizes():
    """The cuts the oracle slices are chosen from: at 21 or 22 jobs per SM nearly every warp boundary cuts a job; at
    exactly 16 jobs per SM and any step count no job is cut."""
    cut = straddling_jobs(SLICED_N, 40)
    assert 0.9 * SMS * 15 <= len(cut) <= SMS * 15 and cut.max() < -(-SLICED_N // 32)
    assert len(straddling_jobs(THRESHOLD_N[0], 4)) == 0 and len(straddling_jobs(THRESHOLD_N[0], 5)) == 0
    assert len(straddling_jobs(THRESHOLD_N[2], 5)) == 0


def oracle_columns(inst, n_envs, n_steps, seed, sample=1024):
    """Environments the oracle replays: all of them for launches below the sliced sizes; otherwise every environment
    of a straddling job, the first and last jobs and a random sample."""
    if n_envs <= 20_000:
        return None
    cols = [np.arange(32), np.arange((n_envs - 1) // 32 * 32, n_envs),
            np.random.default_rng(seed).choice(n_envs, sample, replace=False)]
    if inst[0] == "sliced":
        jobs = straddling_jobs(n_envs, n_steps)
        cols.append((jobs[:, None] * 32 + np.arange(32)[None, :]).reshape(-1))
    cols = np.unique(np.concatenate(cols))
    return cols[cols < n_envs]


# ---- running the kernels ---------------------------------------------------------------------------------------------------
ACTION_P = [.3, .02, .1, .1, .2, .2, .02, .02, .04]      # forward-biased: gates, crashes and resets in every launch
WANT = ("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index")
KERNEL_RE = re.compile(r"k_rollout(_tab_sliced|_tab|_warp)?<([^>]*)>")
KIND = {None: "arith", "_tab": "tab", "_tab_sliced": "sliced", "_warp": "warp"}
CXX_TYPES = {"unsigned char": "u8", "int": "i32", "long": "i64", "long long": "i64", "float": "f32"}


def forward_actions(T, n, seed):
    return np.random.default_rng(seed).choice(9, size=(T, n), p=ACTION_P).astype(np.uint8)


@pytest.fixture(scope="module")
def sms():
    n = torch.cuda.get_device_properties(0).multi_processor_count
    assert n == SMS, f"the matrix assumes {SMS} SMs; this device has {n}, which moves the sliced kernel's boundary"
    return n


def launched(fn):
    """Run ``fn`` under the profiler; returns its result and the step kernels it launched as
    (instantiation without copies, action type, flag type, shared memory bytes, grid, block)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    kernels = []
    for e in events:
        m = KERNEL_RE.search(e.get("name", "")) if e.get("cat") == "kernel" else None
        if m:
            targs = [a.strip() for a in m.group(2).split(",")]
            kind = KIND[m.group(1)]
            inst = ("warp",) if kind == "warp" else (kind, int(targs[2]))
            a = e.get("args", {})
            kernels.append(SimpleNamespace(inst=inst, act=CXX_TYPES[targs[0]], flag=CXX_TYPES[targs[1]],
                                           smem=a.get("shared memory"), grid=a.get("grid"), block=a.get("block")))
    return res, kernels


def assert_ran(kernels, layout, want, act="u8", flag="u8"):
    """One step-kernel launch, of the instantiation ``want``; the table kernels' shared memory is the copy count's."""
    assert len(kernels) == 1, [k.inst for k in kernels]
    k = kernels[0]
    assert k.inst == want[:2] and (k.act, k.flag) == (act, flag), (k.inst, k.act, k.flag, want)
    if want[0] in ("tab", "sliced"):
        # dynamic shared memory plus the static part, which may count the 1 KB the system reserves per CTA; one copy
        # of the table is at least 9 KB, so the copy count is still unambiguous
        assert k.smem is not None and 0 <= k.smem - table_bytes(layout, want[2]) <= 1024, (k.smem, want)
        assert k.block[0] == launch_constants().tab_threads
    if want[0] == "sliced":
        assert k.grid[0] == SMS


def make_env(path, n, opts, float_flags=False):
    env = ppo_car_b200.VecCarEnv(n, path, float_flags=float_flags)
    for k, v in opts.items():
        if k != "capture":
            env.set_option(k, v)
    env.reset()
    return env


def run(path, acts, opts, float_flags=False, mode="full", profile=True, env=None):
    """One carenv_rollout launch (store_info) from reset or from ``env``'s state.  ``mode``: "full" observations,
    "pose" records or "none"."""
    env = env if env is not None else make_env(path, acts.shape[1], opts, float_flags)
    go = lambda: env.rollout(acts, store_info=True, store_obs=mode == "full", store_poses=mode == "pose")
    out, kernels = launched(go) if profile else (go(), None)
    torch.cuda.synchronize()
    return SimpleNamespace(env=env, out=out, kernels=kernels, pos=env.pos.clone(), vel=env.vel.clone(),
                           ints=env.ints.clone(), counts=env.slow_path_counts())


def assert_same(a, b, what, counts=True):
    """Every output and the final state bit for bit (flags compared as values: u8 and f32 flags are the same flags)."""
    for k in ("obs", "reward", "terminated", "truncated", "poses"):
        x, y = a.out.get(k), b.out.get(k)
        if x is not None and y is not None:
            assert torch.equal(x.float() if k in ("terminated", "truncated") else x,
                               y.float() if k in ("terminated", "truncated") else y), (what, k)
    for k in a.out["info"]:
        assert torch.equal(a.out["info"][k], b.out["info"][k]), (what, k)
    assert torch.equal(a.pos, b.pos) and torch.equal(a.vel, b.vel) and torch.equal(a.ints, b.ints), what
    if counts:
        assert a.counts == b.counts, (what, a.counts, b.counts)


def trajectory(r, cols=None, T=None):
    t = torch.as_tensor(cols, device="cuda") if cols is not None else None
    take = lambda x: (x if t is None else x.index_select(1, t))[:T].cpu().numpy()
    info = r.out["info"]
    return dict(obs=take(r.out["obs"]), rew=take(r.out["reward"]), term=take(r.out["terminated"]),
                trunc=take(r.out["truncated"]), gates_passed=take(info["gates_passed"]),
                time_passed=take(info["time_passed"]), next_gate_index=take(info["next_gate_index"]))


def oracle(path, acts, cols=None):
    from oracle.c_oracle import COracleVecEnv

    a = acts if cols is None else acts[:, cols]
    ora = COracleVecEnv(a.shape[1], path, scan_all_gates=False)
    ora.reset()
    return ora.rollout(a, want=WANT)


def check_oracle(name, path, acts, runs, cols, what):
    """The rows of consecutive launches ``runs`` (from reset) against the oracle on the columns ``cols``."""
    ref = oracle(path, acts, cols)
    got = [trajectory(r, cols) for r in runs]
    got = {k: np.concatenate([g[k] for g in got]) for k in got[0]}
    rtol = RTOL if name in ("big_track", "track") else RTOL_SYNTHETIC
    assert_trajectory_matches(got, ref, what=what, rtol=rtol)
    return ref


# ---- every matrix row against the oracle and against k_rollout ---------------------------------------------------------
@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("track,n,T,opts,want", MATRIX, ids=MATRIX_IDS)
def test_step_kernel_matrix(tracks, sms, track, n, T, opts, want):
    path = tracks(track)
    layout = track_layout(path)
    assert step_instantiation(layout, n, T, opts, sms) == want
    acts_np = forward_actions(T, n, seed=n + T)
    acts = torch.from_numpy(acts_np).cuda()
    r = run(path, acts, opts)
    assert_ran(r.kernels, layout, want)
    ref = check_oracle(track, path, acts_np, [r], oracle_columns(want, n, T, seed=n), f"{track} {n}x{T} {opts} {want}")
    if track == "near_wall":                                         # the start pose is inside the wall
        assert ref["term"].all()
    else:
        assert ref["term"].sum() > 0 and (T < 100 or ref["gates_passed"].max() > 0)
    base = reference_opts(layout, n, T, opts)
    if base is not None:
        b = run(path, acts, base)
        other = step_instantiation(layout, n, T, base)
        assert_ran(b.kernels, layout, other)
        # the table and warp kernels make the same float64 fallback decisions as k_rollout<U> of the same U
        assert_same(r, b, f"{want} vs {other}", counts=other[1] == (want[1] if len(want) > 1 else layout.unroll))


# ---- the table kernels at U = 6 and U = 2: dtypes, observation modes, launch sequences -------------------------------------
OUT_OF_RANGE = {torch.uint8: [9, 17, 255], torch.int32: [-1, 9, 2 ** 31 - 1, -2 ** 31],
                torch.int64: [-1, 9, 2 ** 32, 2 ** 32 + 1, 2 ** 32 + 4, 2 ** 63 - 1, -2 ** 63]}


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_action_and_flag_dtypes(tracks, sms, case):
    """All six (action, flag) dtype pairs of carenv_rollout (uint8 / int32 / int64 actions from the tensor's dtype,
    uint8 / float32 flags from ``float_flags``) give the same bits and match the oracle.  3 % of the actions are
    outside 0..8 in each dtype's own way; every such action does nothing, as 8 does (a 64-bit 2^32 + 1 is not 1)."""
    track, n, opts = CASES[case]
    T = 24
    path = tracks(track)
    layout = track_layout(path)
    want = step_instantiation(layout, n, T, opts, sms)
    eff = forward_actions(T, n, seed=7 + n)
    odd = np.random.default_rng(8).random((T, n)) < 0.03
    eff[odd] = 8
    cols = oracle_columns(want, n, T, seed=9)
    ref = oracle(path, eff, cols)
    assert ref["term"].sum() > 0
    first = None
    for dt, act in ((torch.uint8, "u8"), (torch.int32, "i32"), (torch.int64, "i64")):
        a = torch.from_numpy(eff.astype(np.int64))
        pick = np.random.default_rng(10).integers(0, len(OUT_OF_RANGE[dt]), size=int(odd.sum()))
        a[torch.from_numpy(odd)] = torch.tensor(OUT_OF_RANGE[dt], dtype=torch.int64)[torch.from_numpy(pick)]
        a = a.to(dt).cuda()
        for float_flags, flag in ((False, "u8"), (True, "f32")):
            r = run(path, a, opts, float_flags=float_flags)
            assert_ran(r.kernels, layout, want, act, flag)
            got = trajectory(r, cols)
            assert_trajectory_matches(got, ref, what=f"{case} {act}/{flag}",
                                      rtol=RTOL if track == "big_track" else RTOL_SYNTHETIC)
            if first is None:
                first = r
            else:
                assert_same(r, first, f"{case} {act}/{flag} vs u8/u8")


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_observation_modes(tracks, sms, case):
    """Full observations, 32-byte pose records (turned back into observations by carenv_observe) and no observations:
    the same kernel runs, the records give the full observations bit for bit, and nothing else changes."""
    track, n, opts = CASES[case]
    T = 24
    path = tracks(track)
    layout = track_layout(path)
    want = step_instantiation(layout, n, T, opts, sms)
    acts = torch.from_numpy(forward_actions(T, n, seed=11 + n)).cuda()
    full = run(path, acts, opts, mode="full")
    pose = run(path, acts, opts, mode="pose")
    none = run(path, acts, opts, mode="none")
    for r in (full, pose, none):
        assert_ran(r.kernels, layout, want)
    assert pose.out["obs"] is None and none.out["obs"] is None and none.out.get("poses") is None
    obs = pose.env.observe(pose.out["poses"]).view(T, n, 18)
    assert torch.equal(obs, full.out["obs"]), case
    assert_same(pose, full, f"{case} pose records")
    assert_same(none, full, f"{case} no observations")
    done = (full.out["terminated"] | full.out["truncated"]).bool()
    assert int(done.sum()) > 0


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_two_launches_equal_one_of_twice_the_length(tracks, sms, case):
    """A rollout of 2T steps in one launch and in two launches of T (the second from the state the first handed
    over): the same bits, with episodes ending inside both halves, and the oracle agrees with the two-launch rows."""
    track, n, opts = CASES[case]
    T = 48 if n > 20_000 else 150
    path = tracks(track)
    layout = track_layout(path)
    acts_np = forward_actions(2 * T, n, seed=13 + n)
    acts = torch.from_numpy(acts_np).cuda()
    one = run(path, acts, opts)
    assert_ran(one.kernels, layout, step_instantiation(layout, n, 2 * T, opts, sms))
    a = run(path, acts[:T], opts)
    b = run(path, acts[T:], opts, env=a.env)
    for r in (a, b):
        assert_ran(r.kernels, layout, step_instantiation(layout, n, T, opts, sms))
    for k in ("obs", "reward", "terminated", "truncated"):
        assert torch.equal(one.out[k], torch.cat([a.out[k], b.out[k]])), k
    for k in one.out["info"]:
        assert torch.equal(one.out["info"][k], torch.cat([a.out["info"][k], b.out["info"][k]])), k
    assert torch.equal(one.pos, b.pos) and torch.equal(one.vel, b.vel) and torch.equal(one.ints, b.ints)
    want = step_instantiation(layout, n, T, opts, sms)
    ref = check_oracle(track, path, acts_np, [a, b], oracle_columns(want, n, T, seed=14), f"{case} two launches")
    assert ref["term"][:T].sum() > 0 and ref["term"][T:].sum() > 0


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("track", ["big_track", "ring10_6"])
@pytest.mark.parametrize("n", THRESHOLD_N)
def test_sliced_threshold(tracks, sms, track, n):
    """On both sides of the sliced kernel's condition (16 jobs per SM, 4 steps) the launch takes the kernel
    step_instantiation names, and the results do not depend on which one it is: the oracle, and k_rollout bit for
    bit."""
    path = tracks(track)
    layout = track_layout(path)
    for T in THRESHOLD_T:
        want = step_instantiation(layout, n, T, {}, sms)
        acts_np = forward_actions(T, n, seed=n * 7 + T)
        acts = torch.from_numpy(acts_np).cuda()
        r = run(path, acts, {})
        assert_ran(r.kernels, layout, want)
        check_oracle(track, path, acts_np, [r], oracle_columns(want, n, T, seed=T, sample=512), f"{track} {n}x{T}")
        b = run(path, acts, reference_opts(layout, n, T, {}), profile=False)
        assert_same(r, b, f"{track} {n}x{T} {want} vs k_rollout")


@pytest.mark.gpu
@needs_gpu
@pytest.mark.parametrize("track", ["big_track", "ring10_6"])
def test_graph_capture(tracks, sms, track):
    """carenv_rollout captured in a CUDA graph and replayed twice equals two eager launches.  On a fresh handle the
    capture cannot allocate the sliced kernel's flags and records the block-round table kernel; on a handle that has
    run a sliced launch before it records the sliced kernel (with the flags' memset)."""
    n, T = SLICED_N, 24
    path = tracks(track)
    layout = track_layout(path)
    a1 = torch.from_numpy(forward_actions(T, n, seed=21)).cuda()
    a2 = torch.from_numpy(forward_actions(T, n, seed=22)).cuda()
    eager = make_env(path, n, {})
    e1, e2 = run(path, a1, {}, env=eager), run(path, a2, {}, env=eager)
    block = make_env(path, n, {"tab_slice": -1})                    # loads the block-round kernel before any capture
    run(path, a1, {}, env=block, profile=False)
    for warm in (False, True):
        env = make_env(path, n, {})
        if warm:
            env.rollout(a1)
            env.reset()
        act = a1.clone()
        outs = dict(obs_out=torch.empty((T, n, 18), device="cuda"), reward_out=torch.empty((T, n), device="cuda"),
                    term_out=torch.empty((T, n), dtype=torch.uint8, device="cuda"),
                    trunc_out=torch.empty((T, n), dtype=torch.uint8, device="cuda"),
                    info_out=torch.empty((T, n, 4), dtype=torch.int32, device="cuda"))
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            env.rollout(act, **outs)
        want = step_instantiation(layout, n, T, {} if warm else {"capture": True}, sms)
        assert want[0] == ("sliced" if warm else "tab")
        for ref, a in ((e1, a1), (e2, a2)):
            act.copy_(a)
            _, kernels = launched(graph.replay)
            assert_ran(kernels, layout, want)
            got = SimpleNamespace(out=dict(obs=outs["obs_out"], reward=outs["reward_out"], terminated=outs["term_out"],
                                           truncated=outs["trunc_out"], info=env._info_dict(outs["info_out"])),
                                  pos=env.pos, vel=env.vel, ints=env.ints)
            assert_same(got, ref, f"{track} graph replay (warm={warm})", counts=False)
        del graph
