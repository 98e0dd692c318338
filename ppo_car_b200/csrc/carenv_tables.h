// carenv_tables.h — host-side preparation of the per-track constants (runs once per handle).
//
// Input is the track exactly as the reference builds it in CarEnv.reset
// (lib/car_env.py:651-676): wall segments in pixel coordinates, outer polyline first then
// inner, gates from consecutive point pairs, the start pose in pixels / degrees.
#pragma once
#include <math.h>
#include <string.h>

#include <thread>
#include <vector>

#include "carenv_core.cuh"

namespace carenv {

struct HostTrack {
    TrackParams P;
    std::vector<F2> trig32, trig32s;
    std::vector<float> den4;     // [72][n_pairs][4]: seg_den of both segments of a pair (tracks the pair kernels take)
    int n_pairs = 0;
    std::vector<uint16_t> cull;  // candidate table of the culled pair kernels (build_cull_table; empty: none)
    CullGrid cull_grid{};        // its grid (mask pointer null: set to wherever the table is uploaded)
    std::vector<D2> trig64, acc64;
    std::vector<GateRec> gates;
    std::vector<double> walls64;
    std::vector<SegF> segf;      // every segment (TrackParams only holds them up to kMaxSeg)
    std::vector<SegD> segd;
    Tables tables() const {
        return Tables{trig32.data(), trig32s.data(), trig64.data(), acc64.data(), gates.data(), walls64.data(),
                      segf.data(), segd.data()};
    }
};

// ---- candidate table (CullGrid, carenv_core.cuh) ------------------------------------------------------------------
// Bit jp of entry [cell][m] is cleared only when each segment S of pair jp is proven irrelevant, for every point P of
// the cell dilated by kCullDilate and every ray direction d = heading m + 6i (i = 0..11), by one of:
//   (a) no ray from P in direction d meets S with u >= 0: a separating axis between the dilated cell and the region
//       S - t d (t >= 0) of origins whose ray can reach S — d's normal (S beside the strip the cell sweeps), S's
//       normal (S behind the cell), x or y (S behind the cell along that axis);
//   (b) a segment B blocks it: every such ray crosses B (B's end points strictly on opposite sides of the swept
//       strip), 0 < u_B throughout, and max u_B < (least possible u of a hit of S) - kCullMargin.
// u and the offsets of points from the ray line are affine in P, so their extremes over the square are the value at
// its centre plus or minus the half-width times the L1 norm of the gradient.
// Why skipping such a pair leaves the kernel's results unchanged: the nearest hit of a ray is never skippable (it is
// not separated, and nothing hits before it), and a skipped segment is either missed or more than kCullMargin farther
// than that hit.  kCullMargin = 1 px is >= 1/2000 of any distance on the grid, 300x the float32 error of r = 1/u.
// kCullDilate covers the float32 rounding of the position and of the cell arithmetic in cull_keep (< 1e-3 px).
constexpr double kCullCell = 8.0;       // px (DESIGN.md §3: cell sizes)
constexpr double kCullDilate = 0.5;     // px
constexpr double kCullMargin = 1.0;     // px
constexpr double kCullPad = 16.0;       // grid margin around the walls' bounding box, px

inline void build_cull_table(HostTrack &H) {
    H.cull.clear();
    H.cull_grid = CullGrid{};
    const int n = H.P.n_seg, np = n / 2;
    if (n % 2 != 0 || np < 1 || np > 16) return;
    const double *W = H.walls64.data();
    double xmin = W[0], xmax = W[0], ymin = W[1], ymax = W[1];
    for (int j = 0; j < 2 * n; ++j) {
        xmin = fmin(xmin, W[2 * j]); xmax = fmax(xmax, W[2 * j]);
        ymin = fmin(ymin, W[2 * j + 1]); ymax = fmax(ymax, W[2 * j + 1]);
    }
    const double x0 = floor(xmin - kCullPad), y0 = floor(ymin - kCullPad);
    const bool sized = xmax - xmin < 1e4 && ymax - ymin < 1e4;    // else an empty grid: every position is off it
    const int nx = sized ? (int)ceil((xmax + kCullPad - x0) / kCullCell) : 0;
    const int ny = sized ? (int)ceil((ymax + kCullPad - y0) / kCullCell) : 0;
    const size_t n_cells = (size_t)nx * ny;
    H.cull.assign((n_cells + 1) * kCullClasses, 0);
    for (int m = 0; m < kCullClasses; ++m) H.cull[n_cells * kCullClasses + m] = 0xffffu;
    const double h = 0.5 * kCullCell + kCullDilate, eps = 1e-6;
    // Per heading and segment, everything as an affine function of the cell centre P = (px, py):
    //   q_A(P) = cross(A - P, d) = qa - cr(P),  cr(P) = cross(P, d) (the same for every segment), q_B alike
    //   u(P)   = cross(e, A - P) / cross(e, d) = u0 + ux px + uy py    (distance along d to S's line; ur: its half-range)
    //   "behind along x / y": px outside [xlo, xhi] or py outside [ylo, yhi]
    //   lo     = least dot(X, d) over S: a hit of S from P has u >= lo - dot(P, d)
    // One thread per heading class, each on a plane of its own (interleaved below).
    const unsigned all = (1u << np) - 1u;
    std::vector<std::vector<uint16_t>> plane(kCullClasses, std::vector<uint16_t>(n_cells, 0));
    auto heading_class = [&](int m) {
        double qa[32], qb[32], u0[32], ux[32], uy[32], ur[32], lo[32], xlo[32], xhi[32], ylo[32], yhi[32];
        double qac[32], qbc[32], uc[32];
        for (int k = m; k < kHeadings; k += kCullClasses) {
            const double dx = H.trig64[k].x, dy = H.trig64[k].y;
            const double w = h * (fabs(dx) + fabs(dy)) + eps;     // half-range of cr(P) and dot(P, d), plus eps
            for (int j = 0; j < n; ++j) {
                const double ax = W[4 * j], ay = W[4 * j + 1], bx = W[4 * j + 2], by = W[4 * j + 3];
                const double ex = bx - ax, ey = by - ay, den = ex * dy - ey * dx;
                qa[j] = ax * dy - ay * dx;
                qb[j] = bx * dy - by * dx;
                if (den != 0.0) {
                    u0[j] = (ex * ay - ey * ax) / den; ux[j] = ey / den; uy[j] = -ex / den;
                    ur[j] = h * (fabs(ex) + fabs(ey)) / fabs(den);
                } else {                                           // parallel: never crossed, never behind its line
                    u0[j] = 0.0; ux[j] = 0.0; uy[j] = 0.0; ur[j] = INFINITY;
                }
                lo[j] = fmin(ax * dx + ay * dy, bx * dx + by * dy);
                xlo[j] = dx < 0.0 ? fmin(ax, bx) - h - eps : -INFINITY; xhi[j] = dx > 0.0 ? fmax(ax, bx) + h + eps : INFINITY;
                ylo[j] = dy < 0.0 ? fmin(ay, by) - h - eps : -INFINITY; yhi[j] = dy > 0.0 ? fmax(ay, by) + h + eps : INFINITY;
            }
            for (int cy = 0; cy < ny; ++cy)
                for (int cx = 0; cx < nx; ++cx) {
                    uint16_t &entry = plane[m][(size_t)cy * nx + cx];
                    const unsigned todo = all & ~(unsigned)entry;  // pairs no earlier direction of the class kept
                    if (!todo) continue;
                    const double px = x0 + (cx + 0.5) * kCullCell, py = y0 + (cy + 0.5) * kCullCell;
                    const double cr = px * dy - py * dx, dt = px * dx + py * dy;
                    unsigned cand = 0;                             // segments of `todo` pairs that (a) does not rule out
                    for (int j = 0; j < n; ++j) {
                        qac[j] = qa[j] - cr; qbc[j] = qb[j] - cr;
                        uc[j] = u0[j] + ux[j] * px + uy[j] * py;
                        const bool beside = qac[j] * qbc[j] > 0.0 && fmin(fabs(qac[j]), fabs(qbc[j])) > w;
                        const bool behind = uc[j] + ur[j] < -eps || px < xlo[j] || px > xhi[j] || py < ylo[j] || py > yhi[j];
                        cand |= (unsigned)(!(beside | behind) && ((todo >> (j >> 1)) & 1u)) << j;
                    }
                    if (!cand) continue;
                    double ublock = INFINITY;                      // least max u of a blocker
                    for (int j = 0; j < n; ++j) {
                        const bool crosses = qac[j] * qbc[j] < 0.0 && fmin(fabs(qac[j]), fabs(qbc[j])) > w;
                        const bool ahead = uc[j] - ur[j] > eps;
                        ublock = fmin(ublock, crosses && ahead ? uc[j] + ur[j] : INFINITY);
                    }
                    unsigned keep = 0;
                    for (; cand; cand &= cand - 1) {
                        const int j = __builtin_ctz(cand);
                        if (!(ublock < fmax(lo[j] - dt - w, uc[j] - ur[j]) - kCullMargin)) keep |= 1u << (j >> 1);
                    }
                    entry = (uint16_t)(entry | keep);
                }
        }
    };
    std::vector<std::thread> pool;
    for (int m = 1; m < kCullClasses; ++m) pool.emplace_back(heading_class, m);
    heading_class(0);
    for (auto &t : pool) t.join();
    for (size_t c = 0; c < n_cells; ++c)
        for (int m = 0; m < kCullClasses; ++m) H.cull[c * kCullClasses + m] = plane[m][c];
    H.cull_grid.x0 = (float)x0; H.cull_grid.y0 = (float)y0;
    H.cull_grid.inv_cell = (float)(1.0 / kCullCell);               // 1/8: exact
    H.cull_grid.nx = nx; H.cull_grid.ny = ny;
}

// returns 0 on success, <0 on invalid input
inline int build_host_track(const double *walls, int n_walls, const double *gates, int n_gates,
                            double sx, double sy, double angle_deg, HostTrack &H) {
    if (n_walls < 1 || n_walls > kMaxBigSeg || n_gates < 1 || !walls || !gates) return -1;
    memset(&H.P, 0, sizeof(H.P));
    TrackParams &P = H.P;
    P.n_seg = n_walls; P.n_gates = n_gates;
    P.start_x = sx; P.start_y = sy;

    const double DEG = M_PI / 180.0;   // np.radians
    H.trig32.resize(kHeadings); H.trig32s.resize(kHeadings); H.trig64.resize(kHeadings); H.acc64.resize(kHeadings);
    for (int k = 0; k < kHeadings; ++k) {
        const double ang = angle_deg + 5.0 * k;
        const double c = cos(ang * DEG), s = sin(ang * DEG);
        H.trig64[k] = D2{c, s};
        H.trig32[k] = F2{(float)c, (float)s};
        H.trig32s[k] = F2{(float)c * kQScale, (float)s * kQScale};      // exact: a power of two
        H.acc64[k] = D2{c * 0.8, s * 0.8};
    }

    H.walls64.assign(walls, walls + 4 * (size_t)n_walls);
    H.segf.resize(n_walls);
    H.segd.resize(n_walls);
    double min_sin = 1.0;
    for (int j = 0; j < n_walls; ++j) {
        const double ax = walls[4 * j], ay = walls[4 * j + 1], bx = walls[4 * j + 2], by = walls[4 * j + 3];
        SegF &f = H.segf[j];
        memset(&f, 0, sizeof(f));
        f.ahx = (float)ax; f.ahy = (float)ay; f.nahy = -f.ahy;
        f.bhx = (float)bx; f.bhy = (float)by; f.nbhy = -f.bhy;
        const double ex = bx - ax, ey = by - ay;
        f.ex = (float)ex; f.ey = (float)ey; f.ney = -f.ey;
        f.chain_start = (j == 0 || walls[4 * j - 2] != ax || walls[4 * j - 1] != ay) ? 1 : 0;
        H.segd[j] = SegD{fma(ex, ay, -(ey * ax)) * kQScaleD, ex * kQScaleD, ey * kQScaleD};   // exact scalings
        if (n_walls <= kMaxSeg) { P.segf[j] = H.segf[j]; P.segd[j] = H.segd[j]; }
        const double len = hypot(ex, ey);
        if (len > 0)
            for (int k = 0; k < kHeadings; ++k) {
                const double sn = fabs(ex * H.trig64[k].y - ey * H.trig64[k].x) / len;
                if (sn > 1e-7 && sn < min_sin) min_sin = sn;   // exactly parallel pairs cannot be hit
            }
    }

    H.gates.resize(n_gates);
    for (int g = 0; g < n_gates; ++g) {
        GateRec &r = H.gates[g];
        r.x1 = gates[4 * g]; r.y1 = gates[4 * g + 1]; r.x2 = gates[4 * g + 2]; r.y2 = gates[4 * g + 3];
        const double ex = r.x2 - r.x1, ey = r.y2 - r.y1;
        r.ex = (float)ex; r.ey = (float)ey; r.len = (float)hypot(ex, ey); r.pad = 0.0f;
    }

    // guard bands (DESIGN.md §3): bounds on the float32 error of q, r and the gate margin
    P.eps_q = 1.5e-3f;      // |dq| <= 5.7e-4 px for coordinates within 1280 x 720 (see wall_point)
    P.eps_qs = P.eps_q * kQScale;
    (void)min_sin;
    const double rel_r = 5.0e-7;   // relative error of r = cross(e,d) / cross(e,A'): both from float64, rounded once, one
                                   // approximate reciprocal, one multiply
    P.coll_band = (float)fmax(2.0e-4, 4.0 * rel_r);
    P.tiny_d = 1.0e-2f;
    P.gate_band = 2.0e-3f;
    P.tiny_un = 1.0e-3f * kQScale;   // float64 error of cross(e, A - pos) is ~1e-10: relative error < 1e-7 above 1e-3
    // loop unrolling the track allows (see cast_walls)
    P.unroll = (n_walls <= kMaxSeg) ? 1 : 0;
    P.unroll4 = 1;
    const int candidates[3] = {6, 4, 2};                     // measured on big_track: U = 6 2.31 ms, 4 2.36, 12 2.39, 2 2.53
    for (int ci = 0; ci < 3 && n_walls <= kMaxSeg; ++ci) {
        const int U = candidates[ci];
        bool ok = (n_walls % U == 0);
        for (int j = 0; j < n_walls && ok; ++j)
            if (H.segf[j].chain_start && j % U != 0) ok = false;
        if (ok && P.unroll <= 1) P.unroll = U;
        if (ok && U <= 4 && P.unroll4 <= 1) P.unroll4 = U;
    }

    // denominators of the pair kernels, tabulated per heading (k_rollout_tab): exactly what wall_pair computes
    H.n_pairs = 0;
    H.den4.clear();
    if (P.unroll >= 2) {
        H.n_pairs = n_walls / 2;
        H.den4.resize((size_t)kHeadings * H.n_pairs * 4);
        for (int k = 0; k < kHeadings; ++k)
            for (int jp = 0; jp < H.n_pairs; ++jp) {
                float *d = &H.den4[((size_t)k * H.n_pairs + jp) * 4];
                const D2 t = H.trig64[k];
                seg_den(H.segd[2 * jp].ex, H.segd[2 * jp].ey, t.y, t.x, d[0], d[1]);
                seg_den(H.segd[2 * jp + 1].ex, H.segd[2 * jp + 1].ey, t.y, t.x, d[2], d[3]);
            }
        build_cull_table(H);
    }

    const Tables T = H.tables();
    P.start_destroyed = reset_observation(P, T, P.reset_obs) ? 1 : 0;
    return 0;
}

}  // namespace carenv
