// TEST HARNESS — the candidate table of the culled table kernels (build_cull_table, ppo_car_b200/csrc/carenv_tables.h)
// and the culled per-environment step (env_step<U, true, NS, true>, carenv_core.cuh) compiled for the HOST.  Not part
// of the product.  On the host cull_keep reads the environment's own entry (a "warp of one"): stricter than the
// kernel's OR over the warp.
#include <stdint.h>

#include <chrono>

#include "../../ppo_car_b200/csrc/carenv_tables.h"

using namespace carenv;

namespace {
int build(const double *walls, int n_walls, const double *gates, int n_gates, double sx, double sy, double angle,
          HostTrack &H) {
    if (build_host_track(walls, n_walls, gates, n_gates, sx, sy, angle, H) != 0) return -1;
    H.cull_grid.mask = H.cull.data();
    return H.cull.empty() ? -2 : 0;
}
}  // namespace

// The table and its grid: grid_out = {x0, y0, inv_cell, nx, ny}; returns the number of uint16 entries (copied into
// `out` when cap allows), < 0 if the track gets no table.  build_ms_out: time of build_host_track.
extern "C" long long cull_table(const double *walls, int n_walls, const double *gates, int n_gates, double sx, double sy,
                                double angle, uint16_t *out, long long cap, double *grid_out, double *build_ms_out) {
    HostTrack H;
    const auto t0 = std::chrono::steady_clock::now();
    const int rc = build(walls, n_walls, gates, n_gates, sx, sy, angle, H);
    const auto t1 = std::chrono::steady_clock::now();
    if (build_ms_out) *build_ms_out = std::chrono::duration<double, std::milli>(t1 - t0).count();
    if (rc != 0) return rc;
    const long long n = (long long)H.cull.size();
    if (out && cap >= n) memcpy(out, H.cull.data(), sizeof(uint16_t) * n);
    grid_out[0] = H.cull_grid.x0; grid_out[1] = H.cull_grid.y0; grid_out[2] = H.cull_grid.inv_cell;
    grid_out[3] = H.cull_grid.nx; grid_out[4] = H.cull_grid.ny;
    return n;
}

// For every point and every heading k: the literal float64 nearest hit (exact_cast) of each of the 12 rays must have its
// pair bit in the entry cull_keep picks.  `table` (optional) replaces the built table (mutation checks).  Returns the
// number of rays whose nearest hit is culled; *n_hits_out = rays with a hit that were checked.
extern "C" long long cull_check(const double *walls, int n_walls, const double *gates, int n_gates, double sx, double sy,
                                double angle, const uint16_t *table, long long n_pts, const double *px, const double *py,
                                long long *n_hits_out) {
    HostTrack H;
    if (build(walls, n_walls, gates, n_gates, sx, sy, angle, H) != 0) return -1;
    CullGrid g = H.cull_grid;
    if (table) g.mask = table;
    long long bad = 0, hits = 0;
    for (long long p = 0; p < n_pts; ++p)
        for (int k = 0; k < kHeadings; ++k) {
            const unsigned keep = cull_keep(g, px[p], py[p], k);
            for (int i = 0; i < kNumRays; ++i) {
                const D2 d = H.trig64[wrap72(k + 6 * i)];
                double best = INFINITY;
                int jb = -1;
                for (int j = 0; j < n_walls; ++j) {
                    double dist;
                    if (exact_cast(px[p], py[p], d.x, d.y, H.walls64.data() + 4 * j, dist) && dist < best) {
                        best = dist; jb = j;
                    }
                }
                if (jb < 0) continue;
                ++hits;
                if (!((keep >> (jb >> 1)) & 1u)) ++bad;
            }
        }
    if (n_hits_out) *n_hits_out = hits;
    return bad;
}

// One step from each given state, with the culled (cull = 1) or the full (cull = 0) pair path of the table kernel's
// full unroll (big_track: U = 6, NS = 24; track.json: U = 4, NS = 16).  State is updated in place.
extern "C" int cull_step(const double *walls, int n_walls, const double *gates, int n_gates, double sx, double sy,
                         double angle, int n_envs, const uint8_t *actions, int cull, double *state_pv, int32_t *state_i,
                         float *obs, float *rew, uint8_t *term, uint8_t *trunc, int32_t *info, unsigned long long *stats) {
    HostTrack H;
    if (build(walls, n_walls, gates, n_gates, sx, sy, angle, H) != 0) return -1;
    const Tables Tb = H.tables();
    TabView tv{reinterpret_cast<const float4 *>(H.den4.data()), H.n_pairs, H.cull_grid};
    const int U = H.P.unroll;
    if (!((U == 6 && n_walls == 24) || (U == 4 && n_walls == 16))) return -3;
    for (int e = 0; e < n_envs; ++e) {
        EnvState s{state_pv[4 * e], state_pv[4 * e + 1], state_pv[4 * e + 2], state_pv[4 * e + 3],
                   state_i[4 * e], state_i[4 * e + 1], state_i[4 * e + 2], state_i[4 * e + 3]};
        StepResult o;
        if (U == 6 && cull) env_step<6, true, 24, true>(s, actions[e], 1.0, H.P, Tb, o, stats, nullptr, &tv);
        else if (U == 6) env_step<6, true, 24, false>(s, actions[e], 1.0, H.P, Tb, o, stats, nullptr, &tv);
        else if (cull) env_step<4, true, 16, true>(s, actions[e], 1.0, H.P, Tb, o, stats, nullptr, &tv);
        else env_step<4, true, 16, false>(s, actions[e], 1.0, H.P, Tb, o, stats, nullptr, &tv);
        for (int i = 0; i < kObsDim; ++i) obs[(size_t)e * kObsDim + i] = o.obs[i];
        rew[e] = o.reward; term[e] = (uint8_t)o.terminated; trunc[e] = (uint8_t)o.truncated;
        info[4 * e] = o.gates_passed; info[4 * e + 1] = o.time_passed; info[4 * e + 2] = o.next_gate;
        info[4 * e + 3] = o.gate_hit | (o.lap << 1);
        state_pv[4 * e] = s.px; state_pv[4 * e + 1] = s.py; state_pv[4 * e + 2] = s.vx; state_pv[4 * e + 3] = s.vy;
        state_i[4 * e] = s.k; state_i[4 * e + 1] = s.t; state_i[4 * e + 2] = s.next_gate; state_i[4 * e + 3] = s.passed;
    }
    return 0;
}

// Pairs the kernel evaluates per warp-step for the given states (consecutive groups of 32 = warps): the OR of the
// entries over each warp, as cull_keep forms it on the GPU.  kept_out[w] = set bits of warp w's mask.
extern "C" int cull_warp_pairs(const double *walls, int n_walls, const double *gates, int n_gates, double sx, double sy,
                               double angle, long long n_envs, const double *px, const double *py, const int32_t *k,
                               int32_t *kept_out) {
    HostTrack H;
    if (build(walls, n_walls, gates, n_gates, sx, sy, angle, H) != 0) return -1;
    for (long long w = 0; w * 32 < n_envs; ++w) {
        unsigned m = 0;
        for (long long e = w * 32; e < n_envs && e < w * 32 + 32; ++e) m |= cull_keep(H.cull_grid, px[e], py[e], k[e]);
        kept_out[w] = __builtin_popcount(m);
    }
    return 0;
}
