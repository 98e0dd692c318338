"""The candidate table of the culled table kernels (build_cull_table, carenv_tables.h).

* Host, property: from random points in every cell, cell corners and edges, points outside the corridor and off the grid,
  for every heading, the float64 literal nearest hit (exact_cast) of every ray has its pair bit in the entry the kernel
  reads.  A mutation check shows that clearing a needed bit is caught.
* Host, replay: the culled step (each environment with its own entry: stricter than the kernel's OR over a warp) is
  bit-identical to the full one — outputs, state and slow-path counters — from random states over the whole bounding
  box and beyond, all 72 headings.
* GPU: the culled table kernels against k_rollout, bit for bit, from such states, at a time-sliced kernel size.
"""
import ctypes as C
import os
import subprocess
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import ppo_car_b200
from ppo_car_b200.track import load_track
from tests.synth_tracks import ring_track

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_cull", "cull.cpp")
TRACKS = os.path.join(os.path.dirname(HERE), "ppo_car_b200", "tracks")


@pytest.fixture(scope="module")
def L():
    d = tempfile.mkdtemp(prefix="cull_harness_")
    so = os.path.join(d, "libcull.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-x", "c++",
                           "-o", so, SRC, "-lm", "-pthread"])
    lib = C.CDLL(so)
    lib.cull_table.restype = C.c_longlong
    lib.cull_check.restype = C.c_longlong
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _geom(path):
    tr = load_track(path)
    w, g = np.ascontiguousarray(tr.walls, np.float64), np.ascontiguousarray(tr.gates, np.float64)
    return (_p(w), len(w), _p(g), len(g), C.c_double(tr.start[0]), C.c_double(tr.start[1]), C.c_double(tr.angle)), (w, g)


def table(L, path):
    args, keep = _geom(path)
    grid = np.zeros(5)
    n = L.cull_table(*args, None, C.c_longlong(0), _p(grid), None)
    assert n > 0, n
    t = np.zeros(n, np.uint16)
    assert L.cull_table(*args, _p(t), C.c_longlong(n), _p(grid), None) == n
    x0, y0, inv, nx, ny = grid
    return t, dict(x0=x0, y0=y0, cell=1.0 / inv, nx=int(nx), ny=int(ny))


def check(L, path, px, py, tab=None, threads=8):
    """(rays whose nearest hit is culled, rays with a hit) over all points and headings."""
    args, keep = _geom(path)
    px, py = np.ascontiguousarray(px, np.float64), np.ascontiguousarray(py, np.float64)
    edges = np.linspace(0, len(px), threads + 1).astype(int)

    def part(i):
        a, b = int(edges[i]), int(edges[i + 1])
        hits = C.c_longlong()
        bad = L.cull_check(*args, _p(tab), C.c_longlong(b - a), C.c_void_p(px.ctypes.data + 8 * a),
                           C.c_void_p(py.ctypes.data + 8 * a), C.byref(hits))
        assert bad >= 0
        return bad, hits.value

    with ThreadPoolExecutor(threads) as ex:
        res = list(ex.map(part, range(threads)))
    return sum(r[0] for r in res), sum(r[1] for r in res)


def points(g, rng):
    """One random point per cell, every cell corner, points on the cell edges, and a band off the grid."""
    cell, nx, ny = g["cell"], g["nx"], g["ny"]
    cx, cy = np.meshgrid(np.arange(nx), np.arange(ny))
    cx, cy = cx.ravel(), cy.ravel()
    rx = g["x0"] + (cx + rng.random(cx.size)) * cell
    ry = g["y0"] + (cy + rng.random(cy.size)) * cell
    kx, ky = np.meshgrid(np.arange(0, nx + 1, 3), np.arange(0, ny + 1, 3))      # corners (every third grid line)
    corners_x, corners_y = g["x0"] + kx.ravel() * cell, g["y0"] + ky.ravel() * cell
    ex_ = g["x0"] + (cx[::5] + rng.random(cx[::5].size)) * cell                  # on horizontal / vertical edges
    ey_ = g["y0"] + cy[::5] * cell
    fx = g["x0"] + cx[::7] * cell
    fy = g["y0"] + (cy[::7] + rng.random(cy[::7].size)) * cell
    w, h = nx * cell, ny * cell                                                   # off the grid, up to 200 px out
    ox = g["x0"] - 200 + rng.random(400) * (w + 400)
    oy = np.where(rng.random(400) < 0.5, g["y0"] - 1 - rng.random(400) * 200, g["y0"] + h + rng.random(400) * 200)
    px = np.concatenate([rx, corners_x, ex_, fx, ox])
    py = np.concatenate([ry, corners_y, ey_, fy, oy])
    return px, py


def track_paths(tmp):
    return {"big_track": os.path.join(TRACKS, "big_track.json"), "track": os.path.join(TRACKS, "track.json"),
            "ring12_12": ring_track(os.path.join(tmp, "ring12_12.json"), 12, 12),
            "ring14_10": ring_track(os.path.join(tmp, "ring14_10.json"), 14, 10, seed_phase=1.1)}


@pytest.fixture(scope="module")
def paths():
    return track_paths(tempfile.mkdtemp(prefix="cull_tracks_"))


@pytest.mark.parametrize("name", ["big_track", "track", "ring12_12", "ring14_10"])
def test_table_keeps_every_nearest_hit(L, paths, name):
    t, g = table(L, paths[name])
    px, py = points(g, np.random.default_rng(7))
    bad, hits = check(L, paths[name], px, py)
    assert hits > 0
    assert bad == 0, f"{bad} of {hits} rays have their nearest hit culled"
    assert (t[-6:] == 0xFFFF).all()                          # off the grid: every pair


@pytest.mark.parametrize("name", ["big_track", "track"])
def test_clearing_a_needed_bit_is_caught(L, paths, name):
    """Mutation check of the property test: clear, one at a time, each set bit of the entries of a sample of cells on
    the track, and re-run the check on that cell's points.  A bit that one of the points needs must be caught; report
    how many of the set bits the points witness (the rest are kept by the proof's conservatism)."""
    t, g = table(L, paths[name])
    rng = np.random.default_rng(3)
    n_cells = g["nx"] * g["ny"]
    cells = rng.choice(np.flatnonzero(t[:6 * n_cells].reshape(n_cells, 6).any(1)), 12, replace=False)
    caught = total = 0
    for c in cells:
        cx, cy = c % g["nx"], c // g["nx"]
        px = g["x0"] + (cx + np.concatenate([rng.random(24), [0.0, 1.0 - 1e-9, 0.5]])) * g["cell"]
        py = g["y0"] + (cy + np.concatenate([rng.random(24), [0.0, 1.0 - 1e-9, 0.5]])) * g["cell"]
        base, _ = check(L, paths[name], px, py, t, threads=1)
        assert base == 0
        for m in range(6):
            e = 6 * c + m
            for bit in range(16):
                if not (t[e] >> bit) & 1:
                    continue
                mut = t.copy()
                mut[e] &= ~np.uint16(1 << bit)
                bad, _ = check(L, paths[name], px, py, mut, threads=1)
                caught += bad > 0
                total += 1
    print(f"{name}: {caught} of {total} set bits of {len(cells)} cells are needed by the cells' points")
    assert total > 0 and caught > 0.5 * total, (caught, total)


def random_states(path, n, rng, margin=60.0):
    """Positions uniform over the walls' bounding box plus `margin` px (on the track, inside walls, outside it), every
    heading, random velocities, time steps and gate counters."""
    tr = load_track(path)
    w = np.asarray(tr.walls)
    xs, ys = np.concatenate([w[:, 0], w[:, 2]]), np.concatenate([w[:, 1], w[:, 3]])
    pv = np.zeros((n, 4))
    pv[:, 0] = rng.uniform(xs.min() - margin, xs.max() + margin, n)
    pv[:, 1] = rng.uniform(ys.min() - margin, ys.max() + margin, n)
    pv[:, 2:] = rng.uniform(-10, 10, (n, 2))
    si = np.zeros((n, 4), np.int32)
    si[:, 0] = np.arange(n) % 72
    si[:, 1] = rng.integers(0, 1000, n)
    si[:, 2] = rng.integers(0, len(tr.gates), n)
    si[:, 3] = rng.integers(0, 50, n)
    return pv, si


@pytest.mark.parametrize("name", ["big_track", "track"])
def test_culled_step_replay_is_bit_identical(L, paths, name):
    args, keep = _geom(paths[name])
    rng = np.random.default_rng(11)
    n = 20_000
    pv0, si0 = random_states(paths[name], n, rng)
    res = {}
    for cull in (0, 1):
        pv, si = pv0.copy(), si0.copy()
        steps = []
        stats = np.zeros(4, np.uint64)
        for t in range(4):
            a = np.random.default_rng(100 + t).integers(0, 9, n).astype(np.uint8)
            o = dict(obs=np.zeros((n, 18), np.float32), rew=np.zeros(n, np.float32), term=np.zeros(n, np.uint8),
                     trunc=np.zeros(n, np.uint8), info=np.zeros((n, 4), np.int32))
            assert L.cull_step(*args, n, _p(a), cull, _p(pv), _p(si), _p(o["obs"]), _p(o["rew"]), _p(o["term"]),
                               _p(o["trunc"]), _p(o["info"]), _p(stats)) == 0
            steps.append(o)
        res[cull] = (steps, pv, si, stats)
    (s0, pv0_, si0_, st0), (s1, pv1, si1, st1) = res[0], res[1]
    for t, (a, b) in enumerate(zip(s0, s1)):
        for k in a:
            assert a[k].tobytes() == b[k].tobytes(), (t, k)
    assert pv0_.tobytes() == pv1.tobytes() and (si0_ == si1).all()
    assert (st0 == st1).all(), (st0, st1)
    assert st0.sum() > 0                                     # the states reach the slow paths too


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["big_track", "track"])
def test_culled_table_kernel_matches_k_rollout(paths, name):
    import torch

    n, T = 151_552, 24                                       # 32 jobs per SM on 148 SMs: the time-sliced kernel
    pv, si = random_states(paths[name], n, np.random.default_rng(5))
    acts = torch.from_numpy(np.random.default_rng(6).integers(0, 9, (T, n)).astype(np.uint8)).cuda()
    runs = []
    for opts in ({}, {"tab": -1, "tab_slice": -1, "warp_per_env": -1}, {"tab_slice": -1}):
        env = ppo_car_b200.VecCarEnv(n, paths[name])
        for k, v in opts.items():
            env.set_option(k, v)
        env.reset()
        env.pos.copy_(torch.from_numpy(pv[:, :2]))
        env.vel.copy_(torch.from_numpy(pv[:, 2:]))
        env.ints.copy_(torch.from_numpy(si))
        env.slow_path_counts()
        out = env.rollout(acts, store_info=True)
        torch.cuda.synchronize()
        runs.append((out, env.pos.clone(), env.vel.clone(), env.ints.clone(), env.slow_path_counts()))
    ref = runs[1]
    for got, what in ((runs[0], "sliced"), (runs[2], "block")):
        out, pos, vel, ints, counts = got
        for k in ("obs", "reward", "terminated", "truncated"):
            assert torch.equal(out[k], ref[0][k]), (what, k)
        for k in out["info"]:
            assert torch.equal(out["info"][k], ref[0]["info"][k]), (what, k)
        assert torch.equal(pos, ref[1]) and torch.equal(vel, ref[2]) and torch.equal(ints, ref[3]), what
        assert counts == ref[4], (what, counts, ref[4])
    assert sum(ref[4].values()) > 0
