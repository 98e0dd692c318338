// carenv_core.cuh — per-environment arithmetic of the batched CarEnv step (sm_100a).
//
// One thread owns one environment.  Everything here is __host__ __device__ so that the
// very same arithmetic can be compiled for the host by tests/host_emul (a TEST harness
// that replays the kernel's decisions on the CPU against the float64 oracle); the product
// library only ever runs it on the GPU.
//
// What it computes (reference: /root/reference/lib/car_env.py):
//   decode_action      698-722   Discrete(9) -> thrust sign, turn sign, +0.01 bonus
//   gate_touched       394-408, 376-392, 725-726  test of the NEXT gate with the cardinal
//                                rays of the pose left by the previous update
//   integrate          444-461   vel += acc; friction iff no thrust; per-axis clip; pos += vel
//   cast_walls         155-213, 360-392, 463-469  12 ray distances + wall collision
//   step               693-760   reward schedule, flags, truncation, observation, autoreset
//
// Numerical design (DESIGN.md §3):
//   * pos/vel are float64 and integrated with the reference's operations in the
//     reference's order (no FMA contraction), so trajectories follow the float64 oracle.
//   * heading = initial_angle + 5*k degrees; all trigonometry is a 72-entry table.
//   * ray casting is float32 on the FMA pipe.  The 12 rays lie on 6 lines through the car
//     (ray i and ray i+6 are opposite), so each wall segment is tested once per LINE:
//       q(P)   = cross(P - pos, d)            signed offset of an endpoint from the line
//       hit   <=> q(A), q(B) have opposite signs            (== 0 < t < 1 of Ray.cast)
//       u      = cross(e, A - pos) / cross(e, d)            (== u of Ray.cast, = distance)
//     and the per-ray minimum distance is kept as the maximum of r = 1/u per sign.
//   * every decision that feeds an integer output (hit/miss, d < 10) is taken in float32
//     only when it is outside a guard band that bounds the float32 error; inside the band
//     the ray is re-evaluated with the reference's literal float64 formulas
//     (exact_ray_distance).  Integer outputs therefore follow the float64 oracle.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define CE_HD __host__ __device__ __forceinline__
#define CE_HD_NOINLINE __host__ __device__ __noinline__
#else
#define CE_HD inline
#define CE_HD_NOINLINE
#endif

namespace carenv {

constexpr int kNumRays = 12;
constexpr int kObsDim = 18;
constexpr int kHeadings = 72;      // 360 / 5 degrees
constexpr int kMaxSeg = 128;       // wall segments carried in kernel-parameter space (fast kernels)
constexpr int kMaxBigSeg = 2048;   // larger tracks: geometry staged in shared memory, generic loop (U = 0)
constexpr int kTimeLimit = 1000;   // lib/car_env.py:491
// The signed line offsets q are carried scaled by 2^50 (an exact scaling): the hit test "q(A) and q(B) have
// opposite signs" then is ONE saturating multiply, mask = sat(q'(A) * -q'(B)) in {0, 1}  (|q'(A) q'(B)| >= 1
// unless some |q| < 2^-50, far inside the eps_q guard band), instead of a multiply and a compare.  The
// denominators cross(e, d) and the ray-independent numerators cross(e, A - pos) are scaled alike, so that
// r = den' / un' is unchanged bit for bit.
constexpr float kQScale = 1125899906842624.0f;      // 2^50
// r = 1/u of "no hit yet": its reciprocal is far above the 1000 px the reference starts its running minimum from
// (lib/car_env.py:198), so min(1/r, 1000) is the reference's "if d < best".
constexpr float kNoHitR = 1.0e-30f;
constexpr double kQScaleD = 1125899906842624.0;

struct F2 { float x, y; };
struct D2 { double x, y; };

// One wall segment A->B in float32 (endpoints rounded from float64; they only feed sign tests).  The layout puts
// what a packed FFMA2 takes as ONE uniform operand next to each other: a scalar that is broadcast (bhx, ex, ahx)
// and 8-byte aligned pairs (-y, y).  The first 16 bytes are all the table kernel needs per segment.
struct alignas(16) SegF {
    float bhx, ex, nbhy, bhy;      // end point B: x (broadcast operand), (-y, y) (packed operand); ex = (B - A).x
    float ney, ey, ahx;            // (-ey, ey): packed operand of the denominators; ahx: only read at a polyline start
    int chain_start;               // 1: A is not the previous segment's B
    float nahy, ahy, pad0, pad1;   // (-ahy, ahy)
};
struct SegHead { float bhx, ex, nbhy, bhy; };
#if defined(__CUDA_ARCH__)
CE_HD SegHead seg_head(const SegF &f) {
    const float4 v = *reinterpret_cast<const float4 *>(&f);
    return SegHead{v.x, v.y, v.z, v.w};
}
#else
CE_HD SegHead seg_head(const SegF &f) { return SegHead{f.bhx, f.ex, f.nbhy, f.bhy}; }
#endif
struct SegD { double K, ex, ey; };   // 2^50 * (cross(e, A), ex, ey):  un' = 2^50 * cross(e, A - pos) = K - (ex*py - ey*px)

struct GateRec { double x1, y1, x2, y2; float ex, ey, len, pad; };

struct TrackParams {
    int n_seg, n_gates, start_destroyed, pad0;
    float eps_q;        // |q| below this: hit/miss undecidable in float32
    float coll_band;    // relative half-width of the band around d == 10
    float tiny_d;       // distances below this are re-evaluated (sign of u uncertain)
    float gate_band;    // gate margin band, in units of the gate length
    float tiny_un;      // |2^50 cross(e, A')| below this: every line is re-evaluated
    int unroll;         // first U of {6, 4, 2, 1} such that n_seg and every polyline start are multiples of U;
                        // 0 for tracks with more than kMaxSeg segments (geometry from Tables::segf/segd)
    int unroll4;        // same, restricted to {4, 2, 1} (the fused rollout kernels)
    int pad2;
    double start_x, start_y;
    float reset_obs[kObsDim];
    float eps_qs;       // 2^50 * eps_q: the guard on the scaled offsets q' of the wall tests
    float pad1;
    SegF segf[kMaxSeg];
    SegD segd[kMaxSeg];
};

// Small tables that are indexed per thread (heading, gate index): global memory on the
// host side of the handle, staged to shared memory by the kernels.
struct Tables {
    const F2 *trig32;        // [72] (cos, sin) of radians(initial_angle + 5k), float32
    const F2 *trig32s;       // [72] the same scaled by 2^50 (directions of the wall tests, see kQScale)
    const D2 *trig64;        // [72] same, float64
    const D2 *acc64;         // [72] (cos*0.8, sin*0.8), float64  (lib/car_env.py:430)
    const GateRec *gates;    // [n_gates]
    const double *walls64;   // [n_seg][4] x1 y1 x2 y2 — only read on the exact path
    const SegF *segf;        // [n_seg] only for tracks with more than kMaxSeg segments (else null: the
    const SegD *segd;        //         geometry is in TrackParams, i.e. constant-bank operands)
};

struct EnvState {
    double px, py, vx, vy;
    int k;          // heading index, rotation = initial_angle + 5k (mod 72)
    int t;          // time_step
    int next_gate;  // next_gate_index
    int passed;     // passed_reward_gates (cumulative over laps)
};

struct StepResult {
    float obs[kObsDim];
    float reward;       // float32(reward_f64 * reward_scale)
    double reward64;    // reward_f64 * reward_scale: what TransformReward hands to the reference's numpy boundary
    int terminated, truncated;
    int gates_passed, time_passed, next_gate;   // info of the finished step (pre-reset)
    int gate_hit, lap;
};

// Compact rollout row (SURVEY §8 f-3): what is needed to recompute the 72-byte observation bit for bit.
struct alignas(16) PoseRec {
    double px, py;      // position after the step (float64: the ray casting starts from it)
    float vx10, vy10;   // obs[2], obs[3] as the step computed them
    int k;              // heading index
    int reset;          // 1: the row's observation is the reset observation (episode ended in this step)
};

// slow-path counters (optional)
enum { kStatLine = 0, kStatBand = 1, kStatGate = 2, kStatTiny = 3, kNumStats = 4 };

// ---- individually rounded arithmetic (never contracted, identical on host and device) ----
#if defined(__CUDA_ARCH__)
CE_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
CE_HD double dsub(double a, double b) { return __dadd_rn(a, -b); }
CE_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
CE_HD double dfma(double a, double b, double c) { return __fma_rn(a, b, c); }
CE_HD float fadd(float a, float b) { return __fadd_rn(a, b); }
CE_HD float fsub(float a, float b) { return __fadd_rn(a, -b); }
CE_HD float fmul(float a, float b) { return __fmul_rn(a, b); }
CE_HD float ffma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
#if defined(CARENV_IEEE_RCP)
CE_HD float frcp(float x) { return __frcp_rn(x); }
#else
CE_HD float frcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
#endif
CE_HD void stat_add(unsigned long long *s, int i) { if (s) atomicAdd(s + i, 1ULL); }
#else
CE_HD double dadd(double a, double b) { return a + b; }   // host build: -ffp-contract=off
CE_HD double dsub(double a, double b) { return a - b; }
CE_HD double dmul(double a, double b) { return a * b; }
CE_HD double dfma(double a, double b, double c) { return fma(a, b, c); }
CE_HD float fadd(float a, float b) { return a + b; }
CE_HD float fsub(float a, float b) { return a - b; }
CE_HD float fmul(float a, float b) { return a * b; }
CE_HD float ffma(float a, float b, float c) { return fmaf(a, b, c); }
CE_HD float frcp(float x) { return 1.0f / x; }
CE_HD void stat_add(unsigned long long *s, int i) { if (s) __atomic_fetch_add(s + i, 1ULL, __ATOMIC_RELAXED); }
#endif

// ---- packed pairs of float32 (sm_100a FFMA2 / FMUL2 / FADD2: two IEEE operations per issue slot) ----
#if defined(__CUDA_ARCH__)
typedef float2 P2;
CE_HD P2 p2(float x, float y) { return make_float2(x, y); }
CE_HD P2 pfma(P2 a, P2 b, P2 c) { return __ffma2_rn(a, b, c); }
CE_HD P2 pmul(P2 a, P2 b) { return __fmul2_rn(a, b); }
CE_HD P2 padd(P2 a, P2 b) { return __fadd2_rn(a, b); }
CE_HD float fmin3(float a, float b, float c) { return fminf(fminf(a, b), c); }
CE_HD float fmax3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }
#else
struct P2 { float x, y; };
CE_HD P2 p2(float x, float y) { P2 r; r.x = x; r.y = y; return r; }
CE_HD P2 pfma(P2 a, P2 b, P2 c) { return p2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
CE_HD P2 pmul(P2 a, P2 b) { return p2(a.x * b.x, a.y * b.y); }
CE_HD P2 padd(P2 a, P2 b) { return p2(a.x + b.x, a.y + b.y); }
CE_HD float fmin3(float a, float b, float c) { return fminf(fminf(a, b), c); }
CE_HD float fmax3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }
#endif
// mask = clamp(a * b, 0, 1): FMUL.SAT, one FMA-pipe instruction (a NaN product cannot occur: q is finite)
#if defined(__CUDA_ARCH__)
CE_HD float sat_mul(float a, float b) { float r; asm("mul.rn.sat.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
#else
CE_HD float sat_mul(float a, float b) { const float p = a * b; return p > 1.0f ? 1.0f : (p > 0.0f ? p : 0.0f); }
#endif

CE_HD int wrap72(int k) { return k >= kHeadings ? k - kHeadings : (k < 0 ? k + kHeadings : k); }

// ---- literal float64 evaluation (the reference's formulas, lib/car_env.py:155-213) ----------
// The hit test is evaluated without dividing: for correctly rounded division fl(a/b) > 0 <=> a/b > 0 and
// fl(a/b) < 1 <=> |a| < |b|, so "0 < t < 1 and u > 0" on the reference's rounded quotients is decided by
// the signs and magnitudes of the very same numerators and denominator.  t itself (one division) is only
// formed for an actual hit, where the reference needs it for the hit point.
CE_HD bool exact_cast(double ox, double oy, double dx, double dy, const double *seg, double &dist) {
    const double x1 = seg[0], y1 = seg[1], x2 = seg[2], y2 = seg[3];
    const double x3 = ox, y3 = oy, x4 = dadd(ox, dx), y4 = dadd(oy, dy);
    const double den = dsub(dmul(dsub(x1, x2), dsub(y3, y4)), dmul(dsub(y1, y2), dsub(x3, x4)));
    if (den == 0) return false;
    const double tn = dsub(dmul(dsub(x1, x3), dsub(y3, y4)), dmul(dsub(y1, y3), dsub(x3, x4)));
    const double un = -dsub(dmul(dsub(x1, x2), dsub(y1, y3)), dmul(dsub(y1, y2), dsub(x1, x3)));
    const bool dpos = den > 0;
    const bool t_pos = dpos ? (tn > 0) : (tn < 0);
    const bool t_lt1 = fabs(tn) < fabs(den);
    const bool u_pos = dpos ? (un > 0) : (un < 0);
    if (t_pos && t_lt1 && u_pos) {
        const double t = tn / den;
        const double hx = dadd(x1, dmul(t, dsub(x2, x1))), hy = dadd(y1, dmul(t, dsub(y2, y1)));
        const double gx = dsub(ox, hx), gy = dsub(oy, hy);
        dist = sqrt(dadd(dmul(gx, gx), dmul(gy, gy)));
        return true;
    }
    return false;
}

CE_HD_NOINLINE double exact_ray_distance(double ox, double oy, double dx, double dy, const double *segs, int n) {
    double best = 1000.0;
    for (int j = 0; j < n; ++j) {
        double d;
        if (exact_cast(ox, oy, dx, dy, segs + 4 * j, d) && d < best) best = d;
    }
    return best;
}

// ---- action decode (lib/car_env.py:698-722) -------------------------------------------------
CE_HD void decode_action(int a, int &thrust, int &turn) {
    // two bits per action: value + 1.  thrust: 0,4,5 -> +1; 1,6,7 -> -1.  turn: 3,5,7 -> +1 (right,
    // rotation += 5); 2,4,6 -> -1 (left).  Anything else (8, or out of range) does nothing.
    const unsigned kThrust = 2u | (0u << 2) | (1u << 4) | (1u << 6) | (2u << 8) | (2u << 10) | (0u << 12) | (0u << 14) | (1u << 16);
    const unsigned kTurn = 1u | (1u << 2) | (0u << 4) | (2u << 6) | (0u << 8) | (2u << 10) | (0u << 12) | (2u << 14) | (1u << 16);
    const unsigned sh = 2u * ((unsigned)a < 8u ? (unsigned)a : 8u);
    thrust = (int)((kThrust >> sh) & 3u) - 1;
    turn = (int)((kTurn >> sh) & 3u) - 1;
}

// ---- gate test with the pose left by the previous update (lib/car_env.py:725, 394-408) ------
// Tests gate `next_gate` only: gates below it are exactly the inactive ones, so the first
// active gate the reference's ordered scan can return with index == next_gate is this one.
CE_HD bool gate_touched(const EnvState &s, const TrackParams &P, const Tables &T, unsigned long long *stats) {
    const GateRec g = T.gates[s.next_gate];
    const float x1 = (float)dsub(g.x1, s.px), y1 = (float)dsub(g.y1, s.py);
    const float x2 = (float)dsub(g.x2, s.px), y2 = (float)dsub(g.y2, s.py);
    const F2 d = T.trig32[s.k];
    const float un = ffma(g.ex, y1, -fmul(g.ey, x1));            // cross(e, A')
    const float q1 = ffma(x1, d.y, -fmul(y1, d.x)), q2 = ffma(x2, d.y, -fmul(y2, d.x));   // line of rays 0/6
    const float p1 = ffma(x1, d.x, fmul(y1, d.y)), p2 = ffma(x2, d.x, fmul(y2, d.y));     // line of rays 3/9
    const float den0 = ffma(g.ex, d.y, -fmul(g.ey, d.x));
    const float den3 = ffma(g.ex, d.x, fmul(g.ey, d.y));
    const float m0 = fsub(fabsf(un), fmul(10.0f, fabsf(den0)));  // < 0  <=>  |u| < 10 on that line
    const float m3 = fsub(fabsf(un), fmul(10.0f, fabsf(den3)));
    const bool c0 = fmul(q1, q2) < 0.0f, c3 = fmul(p1, p2) < 0.0f;
    const float qmin = fminf(fminf(fabsf(q1), fabsf(q2)), fminf(fabsf(p1), fabsf(p2)));
    const float band = fmul(P.gate_band, g.len);
    // a line only matters if it is (possibly) crossed; its margin only if it is close to 0
    const bool unsure = (qmin < P.eps_q) || (c0 && fabsf(m0) < band) || (c3 && fabsf(m3) < band);
    if (!unsure) return (c0 && m0 < 0.0f) || (c3 && m3 < 0.0f);
    stat_add(stats, kStatGate);
    const double seg[4] = {g.x1, g.y1, g.x2, g.y2};
    for (int r = 0; r < 4; ++r) {
        const D2 dd = T.trig64[wrap72(s.k + 18 * r)];
        double dist;
        if (exact_cast(s.px, s.py, dd.x, dd.y, seg, dist) && dist < 10.0) return true;
    }
    return false;
}

// ---- Car.update without the rays (lib/car_env.py:452-461) -----------------------------------
CE_HD void integrate(EnvState &s, int thrust, int k_pre, const Tables &T) {
    if (thrust != 0) {
        const D2 a = T.acc64[k_pre];
        s.vx = dadd(s.vx, thrust > 0 ? a.x : -a.x);
        s.vy = dadd(s.vy, thrust > 0 ? a.y : -a.y);
    } else {
        s.vx = dmul(s.vx, 0.8);      // vel + 0 == vel; friction only without thrust (1 - 0.2 == 0.8 in double)
        s.vy = dmul(s.vy, 0.8);
    }
    s.vx = fmin(fmax(s.vx, -10.0), 10.0);
    s.vy = fmin(fmax(s.vy, -10.0), 10.0);
    s.px = dadd(s.px, s.vx);
    s.py = dadd(s.py, s.vy);
}

// ---- the 12 ray distances and the wall-collision decision -------------------------------------
struct WallAcc {
    float c[3], sn[3];      // 2^50 * directions of lines 0..2 (heading + 0/30/60 deg); lines 3..5 are these rotated by 90 deg
    double cd[3], sd[3];    // the same directions in float64, unscaled (denominators, seg_den)
    float cp[6];            // q' of the car's own position: q'(P) = cross(P, d') - cp  (see line_origin)
    float Rp[6], Rm[6];     // max of r = 1/u over hits with u > 0 (ray l) / min over hits with u < 0 (ray l+6)
    float gq[6];            // min |q'| per line  -> hit/miss guard
    float gu;               // min |un'| -> sign-of-u guard
    float qa[6];            // q' of the previous endpoint on each line
};

// q'(P) = 2^50 cross(P - pos, d) is evaluated as cross(P, d') - cross(pos, d'): the wall points P are per-track
// constants (uniform operands of the FMA), so an endpoint costs two FMAs per line and nothing else.  Only the SIGN
// of q is used (and |q| for the guard).  Error bound for coordinates <= 1280 x 720 and |P - pos| <= 1469 px:
// float32(P) 6.1e-5 + 3.1e-5, float32(pos) the same, direction 1.2e-4, the product and the two sums of cp and of
// the inner FMA 3.1e-5 + 6.1e-5 + 1.2e-4, the final rounding 6.1e-5: |dq| <= 5.7e-4 px < eps_q = 1.5e-3.
CE_HD void line_origin(WallAcc &w, double px, double py) {
    const float phx = (float)px, phy = (float)py;
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        w.cp[l] = ffma(phx, w.sn[l], -fmul(phy, w.c[l]));
        w.cp[l + 3] = ffma(phx, w.c[l], fmul(phy, w.sn[l]));
    }
}
CE_HD void wall_point(const WallAcc &w, float hx, float hy, float q[6]) {
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        q[l] = ffma(hx, w.sn[l], ffma(-hy, w.c[l], -w.cp[l]));          // cross(P', d_l)
        q[l + 3] = ffma(hx, w.c[l], ffma(hy, w.sn[l], -w.cp[l + 3]));   // cross(P', rot90 d_l) = dot(P', d_l)
    }
}

// Start of a polyline: q of its first point (the previous segment's end point does not carry over).
CE_HD void wall_chain_start(WallAcc &w, const SegF &f) {
    wall_point(w, f.ahx, f.ahy, w.qa);
#pragma unroll
    for (int l = 0; l < 6; ++l) w.gq[l] = fminf(w.gq[l], fabsf(w.qa[l]));
}

// The denominators 2^50 cross(e, d) of one segment for one heading, (line l, line l + 3): evaluated in FLOAT64 from the
// float64 segment vector and heading table and rounded once.  (In float32 the rounding of the heading's cos / sin
// alone costs 6e-8 / sin(incidence) relative: 4e-5 for a ray that grazes a wall at 0.05 degrees — measured on
// big_track, twice in 2e8 ray distances.)  This is THE definition: the table kernel reads values computed by this
// very function on the host, the other kernels evaluate it on the FP64 pipe — same bits everywhere.
CE_HD void seg_den(double exs, double eys, double sn, double c, float &den0, float &den3) {
    den0 = (float)dfma(exs, sn, -dmul(eys, c));
    den3 = (float)dfma(exs, c, dmul(eys, sn));
}

// One wall segment against the six lines.
// GUARD: 1 = fold |q| of this segment's end point into the guard, 2 = fold |q| of BOTH end points
// (one 3-input min per line covers two polyline points), 0 = leave it to the next segment's GUARD 2.
template <int GUARD>
CE_HD void wall_segment(WallAcc &w, const SegF &f, const SegD &g, double px, double py) {
    float qb[6];
    wall_point(w, f.bhx, f.bhy, qb);
    // 2^50 cross(e, A - pos) in float64 (two FMAs on the FP64 pipe), rounded once, one float32 reciprocal
    const float un = (float)dfma(g.ey, px, dfma(-g.ex, py, g.K));
    const float inv = frcp(un);
    w.gu = fminf(w.gu, fabsf(un));
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        // cross(e, d_l) / cross(e, A') = 1/u
        float den0, den3;
        seg_den(g.ex, g.ey, w.sd[l], w.cd[l], den0, den3);
        const float h0 = fmul(fmul(den0, inv), sat_mul(w.qa[l], -qb[l]));            // r * (hit ? 1 : 0)
        const float h3 = fmul(fmul(den3, inv), sat_mul(w.qa[l + 3], -qb[l + 3]));
        w.Rp[l] = fmaxf(w.Rp[l], h0); w.Rm[l] = fminf(w.Rm[l], h0);
        w.Rp[l + 3] = fmaxf(w.Rp[l + 3], h3); w.Rm[l + 3] = fminf(w.Rm[l + 3], h3);
    }
#pragma unroll
    for (int l = 0; l < 6; ++l) {
        if (GUARD == 1) w.gq[l] = fminf(w.gq[l], fabsf(qb[l]));
        if (GUARD == 2) w.gq[l] = fminf(fminf(w.gq[l], fabsf(w.qa[l])), fabsf(qb[l]));
        w.qa[l] = qb[l];
    }
}

// Two consecutive segments j, j+1 of one polyline, packed: the lines l and l+3 (perpendicular) share
// one FFMA2/FMUL2 each because q_l = x*s_l - y*c_l and q_{l+3} = x*c_l + y*s_l are the two components of
// x*(s_l, c_l) + y*(-c_l, s_l).  Hits are selected arithmetically (r * mask, mask in {0,1} from FMUL.SAT) so
// that one 3-input max/min per ray folds both segments.  Every component is the same IEEE operation as
// in wall_segment, so both paths give bit-identical results.
struct WallAcc2 {
    P2 S[3];                // S_l = 2^50 (s_l, c_l); its half-swap (c_l, s_l) is a free operand modifier
    P2 CP[3];               // (cp_l, cp_{l+3}): q' of the car's own position (line_origin2)
    D2 T64[3];              // (cos, sin) of the three lines in float64 (denominators of the arithmetic path; unused with TAB)
    float Rp[6], Rm[6], gq[6], gu;
    P2 QA[3];               // (q'_l, q'_{l+3}) of the previous endpoint
};

// Per-track table of the denominators for the thread-per-environment kernel (k_rollout_tab): row k (heading
// index), entry jp (segment pair) = (den_l(2jp), den_{l+3}(2jp), den_l(2jp+1), den_{l+3}(2jp+1)) as seg_den computes
// them.  The kernel keeps `copies` skewed copies in shared memory (copy c starts one 16-byte bank group after
// copy c - 1, rows are multiples of 128 bytes) and thread t reads copy t % 8: the eight threads of a quarter warp
// then hit eight different bank groups whatever their headings are — a conflict-free LDS.128 per pair and line.
#if !defined(__CUDACC__)
struct float4 { float x, y, z, w; };
#endif
// Candidate table of the culled pair kernels (build_cull_table, carenv_tables.h): a square grid of kCullCell px cells
// over the track; entry [cell][k mod 6] has bit jp set unless segment pair jp provably cannot be the nearest hit of any
// of the 12 rays of a heading k from anywhere in the cell.  Row nx * ny (positions off the grid) has every bit set.
constexpr int kCullClasses = 6;     // the 12 ray directions of heading k are k + 6i: they depend on k mod 6 only
struct CullGrid {
    const uint16_t *mask;   // [nx * ny + 1][kCullClasses]
    float x0, y0, inv_cell;
    int nx, ny;
};
struct TabView {
    const float4 *base;     // this thread's copy
    int row_f4;             // float4 per row
    CullGrid cull;          // read by the CULL instantiations only
};

// Pairs that may hold a nearest hit for the position (px, py) and heading k.  The cell is found in float32 from the
// float32 position: far less than the table's dilation of the cells (kCullDilate) away from the float64 one.  On the
// GPU the entry is OR-ed over the lanes that run together, so the mask is warp-uniform and every lane keeps a superset
// of its own candidates.
CE_HD unsigned cull_keep(const CullGrid &g, double px, double py, int k) {
    const float fx = fmul(fsub((float)px, g.x0), g.inv_cell), fy = fmul(fsub((float)py, g.y0), g.inv_cell);
    const bool on = fx >= 0.0f && fx < (float)g.nx && fy >= 0.0f && fy < (float)g.ny;   // false for NaN too
    const int cell = on ? (int)fx + g.nx * (int)fy : g.nx * g.ny;
#if defined(__CUDA_ARCH__)
    const unsigned m = __ldg(g.mask + cell * kCullClasses + k % kCullClasses);
    return __reduce_or_sync(__activemask(), m);
#else
    return g.mask[cell * kCullClasses + k % kCullClasses];
#endif
}

// (q_l, q_{l+3}) = hx*(s_l, c_l) + ((-hy, hy)*(c_l, s_l) - (cp_l, cp_{l+3})): two FFMA2 whose wall-point operands
// come straight from uniform registers — the same IEEE operations per component as wall_point.
CE_HD void line_origin2(WallAcc2 &w, double px, double py) {
    const float phx = (float)px, phy = (float)py, nphy = -phy;
#pragma unroll
    for (int l = 0; l < 3; ++l)
        w.CP[l] = pfma(p2(phx, phx), w.S[l], pmul(p2(nphy, phy), p2(w.S[l].y, w.S[l].x)));
}
CE_HD void wall_point2(const WallAcc2 &w, float hx, float nhy, float hy, P2 Q[3]) {
#pragma unroll
    for (int l = 0; l < 3; ++l)
        Q[l] = pfma(p2(hx, hx), w.S[l], pfma(p2(nhy, hy), p2(w.S[l].y, w.S[l].x), p2(-w.CP[l].x, -w.CP[l].y)));
}

CE_HD void wall_chain_start2(WallAcc2 &w, const SegF &f) {
    wall_point2(w, f.ahx, f.nahy, f.ahy, w.QA);
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        w.gq[l] = fminf(w.gq[l], fabsf(w.QA[l].x));
        w.gq[l + 3] = fminf(w.gq[l + 3], fabsf(w.QA[l].y));
    }
}

// TAB: the denominators come from the table rows tb[l] (entry jp) instead of two DMUL + two DFMA + two F2F per segment
// and line pair — same values (seg_den).
// hits = false (culled pairs, see cull_keep): only the end points' offsets, the guards and un; the reciprocals, the
// denominators and the folds into Rp / Rm are skipped.  The guards gq / gu are then what the full pair gives, so every
// slow-path decision is unchanged; a line whose guard did not trip has exact hit masks, and on it a culled pair is
// missed or strictly farther than a kept hit, so Rp and Rm are unchanged too (DESIGN.md §3).
template <bool TAB>
CE_HD void wall_pair(WallAcc2 &w, const SegF &f0, const SegD &g0, const SegF &f1, const SegD &g1, double px,
                     double py, const float4 *const *tb = nullptr, int jp = 0, bool hits = true) {
    P2 QB0[3], QB1[3];
    const SegHead h0 = seg_head(f0), h1 = seg_head(f1);     // bhx, ex, -bhy, bhy: one 128-bit uniform load each
    wall_point2(w, h0.bhx, h0.nbhy, h0.bhy, QB0);
    wall_point2(w, h1.bhx, h1.nbhy, h1.bhy, QB1);
    const float un0 = (float)dfma(g0.ey, px, dfma(-g0.ex, py, g0.K));
    const float un1 = (float)dfma(g1.ey, px, dfma(-g1.ex, py, g1.K));
    w.gu = fmin3(w.gu, fabsf(un0), fabsf(un1));
    if (hits) {
        const float inv0 = frcp(un0), inv1 = frcp(un1);
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            P2 D0, D1;
            if (TAB) {
                const float4 t = tb[l][jp];
                D0 = p2(t.x, t.y); D1 = p2(t.z, t.w);
            } else {
                float a0, a3, b0, b3;
                seg_den(g0.ex, g0.ey, w.T64[l].y, w.T64[l].x, a0, a3);
                seg_den(g1.ex, g1.ey, w.T64[l].y, w.T64[l].x, b0, b3);
                D0 = p2(a0, a3); D1 = p2(b0, b3);
            }
            const P2 R0 = pmul(D0, p2(inv0, inv0)), R1 = pmul(D1, p2(inv1, inv1));
            const P2 H0 = pmul(R0, p2(sat_mul(w.QA[l].x, -QB0[l].x), sat_mul(w.QA[l].y, -QB0[l].y)));
            const P2 H1 = pmul(R1, p2(sat_mul(QB0[l].x, -QB1[l].x), sat_mul(QB0[l].y, -QB1[l].y)));
            w.Rp[l] = fmax3(w.Rp[l], H0.x, H1.x); w.Rm[l] = fmin3(w.Rm[l], H0.x, H1.x);
            w.Rp[l + 3] = fmax3(w.Rp[l + 3], H0.y, H1.y); w.Rm[l + 3] = fmin3(w.Rm[l + 3], H0.y, H1.y);
        }
    }
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        w.gq[l] = fmin3(w.gq[l], fabsf(QB0[l].x), fabsf(QB1[l].x));
        w.gq[l + 3] = fmin3(w.gq[l + 3], fabsf(QB0[l].y), fabsf(QB1[l].y));
        w.QA[l] = QB1[l];
    }
}

// Warp-per-environment variant (small batches, U = kWarpPerEnv): lane j owns wall segment j — its records live in
// registers for the whole launch — and evaluates it against the six lines with the arithmetic of wall_point /
// wall_segment; the per-ray extrema and the guards are then folded over the warp with integer REDUX on the
// float bit patterns (all positive after a sign flip), which is exact, so the result is bit-identical to the
// sequential fold of the thread-per-environment kernels.
constexpr int kWarpPerEnv = -1;
struct WarpSeg { SegF f; SegD g; int active; };

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ float warp_max_pos(float v) {     // v >= 0 in every lane
    return __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(v)));
}
__device__ __forceinline__ float warp_min_pos(float v) {
    return __uint_as_float(__reduce_min_sync(0xffffffffu, __float_as_uint(v)));
}
__device__ __forceinline__ void cast_walls_warp(const EnvState &s, const Tables &T, const WarpSeg &ws, float Rp[6],
                                                float Rm[6], float gq[6], float &gu) {
    const float R0 = kNoHitR;
    WallAcc w;
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        const int kl = wrap72(s.k + 6 * l);
        const F2 d = T.trig32s[kl];
        const D2 dd = T.trig64[kl];
        w.c[l] = d.x; w.sn[l] = d.y; w.cd[l] = dd.x; w.sd[l] = dd.y;
    }
    line_origin(w, s.px, s.py);
    float qa[6], qb[6];
    wall_point(w, ws.f.ahx, ws.f.ahy, qa);
    wall_point(w, ws.f.bhx, ws.f.bhy, qb);
    const float un = (float)dfma(ws.g.ey, s.px, dfma(-ws.g.ex, s.py, ws.g.K));
    const float inv = frcp(un);
    const bool on = ws.active != 0;
    float rp[6], rm[6], g[6];
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        float den0, den3;
        seg_den(ws.g.ex, ws.g.ey, w.sd[l], w.cd[l], den0, den3);
        const float h0 = on ? fmul(fmul(den0, inv), sat_mul(qa[l], -qb[l])) : 0.0f;
        const float h3 = on ? fmul(fmul(den3, inv), sat_mul(qa[l + 3], -qb[l + 3])) : 0.0f;
        rp[l] = fmaxf(R0, h0);          rm[l] = fminf(-R0, h0);
        rp[l + 3] = fmaxf(R0, h3);      rm[l + 3] = fminf(-R0, h3);
    }
#pragma unroll
    for (int l = 0; l < 6; ++l) g[l] = on ? fminf(fabsf(qa[l]), fabsf(qb[l])) : 1.0e30f;
#pragma unroll
    for (int l = 0; l < 6; ++l) {
        Rp[l] = warp_max_pos(rp[l]);
        Rm[l] = -warp_max_pos(-rm[l]);
        gq[l] = warp_min_pos(g[l]);
    }
    gu = warp_min_pos(on ? fabsf(un) : 1.0e30f);
}
#endif

// dist[i] (pixels, float32) for ray i = heading + 30*i degrees; returns destroyed.
// U = segments per loop iteration.  U > 1 requires (checked on the host, TrackParams::unroll) that
// n_seg and every polyline start are multiples of U; the body is then U segments of straight-line
// code (about 1.5 KB each).
// NS > 0 (U > 1 only): the track has exactly NS segments (and its unroll is U); the loop is unrolled over all of them.
// Round 1 measured a full unroll of 24 segments as instruction-cache bound (1.5 "no instruction" stalls per issue);
// with the pair arithmetic the 24-segment wall block is about 900 instructions and 4.4 % faster (DESIGN.md §3).
// TAB (U > 1 only): denominators from the per-track table `tv` (k_rollout_tab) instead of being recomputed.
// CULL (TAB and NS > 0 only): the hit part of a pair runs only where the candidate table tv->cull keeps it (cull_keep).
template <int U, bool TAB = false, int NS = 0, bool CULL = false>
CE_HD bool cast_walls(const EnvState &s, const TrackParams &P, const Tables &T, float dist[kNumRays],
                      unsigned long long *stats, const WarpSeg *ws = nullptr, const TabView *tv = nullptr) {
    const float R0 = kNoHitR;
    float Rp[6], Rm[6], gq[6], gu;
    if (U == kWarpPerEnv) {
#if defined(__CUDA_ARCH__)
        cast_walls_warp(s, T, *ws, Rp, Rm, gq, gu);
#else
        (void)ws; gu = 0.0f;
#pragma unroll
        for (int l = 0; l < 6; ++l) { Rp[l] = R0; Rm[l] = -R0; gq[l] = 0.0f; }
#endif
    } else if (U > 1) {
        WallAcc2 w;
        const float4 *tb[3] = {nullptr, nullptr, nullptr};
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            const int kl = wrap72(s.k + 6 * l);
            const F2 d = T.trig32s[kl];
            w.S[l] = p2(d.y, d.x);
            w.QA[l] = p2(0.0f, 0.0f);
            if (TAB) tb[l] = tv->base + kl * tv->row_f4;
            else w.T64[l] = T.trig64[kl];
        }
        line_origin2(w, s.px, s.py);
#pragma unroll
        for (int l = 0; l < 6; ++l) { w.Rp[l] = R0; w.Rm[l] = -R0; w.gq[l] = 1.0e30f; }
        w.gu = 1.0e30f;
        static_assert(!CULL || (TAB && NS > 0), "the culled pair path is the table kernel's full unroll");
        const unsigned keep = CULL ? cull_keep(tv->cull, s.px, s.py, s.k) : ~0u;
        auto segments = [&](int j0) {                       // segments j0 .. j0 + U - 1
            if (P.segf[j0].chain_start) wall_chain_start2(w, P.segf[j0]);
#pragma unroll
            for (int u = 0; u < U; u += 2)
                wall_pair<TAB>(w, P.segf[j0 + u], P.segd[j0 + u], P.segf[j0 + u + 1], P.segd[j0 + u + 1], s.px, s.py,
                               tb, (j0 + u) >> 1, !CULL || ((keep >> ((j0 + u) >> 1)) & 1u));
        };
        if (NS > 0) {
            // every segment index is a constant: the records are constant-bank operands, no indexed loads, no loop
#pragma unroll
            for (int j0 = 0; j0 < NS; j0 += U) segments(j0);
        } else {
#pragma unroll 1
            for (int j0 = 0; j0 < P.n_seg; j0 += U) segments(j0);
        }
#pragma unroll
        for (int l = 0; l < 6; ++l) { Rp[l] = w.Rp[l]; Rm[l] = w.Rm[l]; gq[l] = w.gq[l]; }
        gu = w.gu;
    } else {
        WallAcc w;
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            const int kl = wrap72(s.k + 6 * l);
            const F2 d = T.trig32s[kl];
            const D2 dd = T.trig64[kl];
            w.c[l] = d.x; w.sn[l] = d.y; w.cd[l] = dd.x; w.sd[l] = dd.y;
        }
        line_origin(w, s.px, s.py);
#pragma unroll
        for (int l = 0; l < 6; ++l) { w.Rp[l] = R0; w.Rm[l] = -R0; w.gq[l] = 1.0e30f; w.qa[l] = 0.0f; }
        w.gu = 1.0e30f;
        if (U == 0) {                                        // big track: geometry from shared memory
#pragma unroll 1
            for (int j = 0; j < P.n_seg; ++j) {
                const SegF f = T.segf[j];
                const SegD g = T.segd[j];
                if (f.chain_start) wall_chain_start(w, f);
                wall_segment<1>(w, f, g, s.px, s.py);
            }
        } else {
#pragma unroll 1
            for (int j = 0; j < P.n_seg; ++j) {
                if (P.segf[j].chain_start) wall_chain_start(w, P.segf[j]);
                wall_segment<1>(w, P.segf[j], P.segd[j], s.px, s.py);
            }
        }
#pragma unroll
        for (int l = 0; l < 6; ++l) { Rp[l] = w.Rp[l]; Rm[l] = w.Rm[l]; gq[l] = w.gq[l]; }
        gu = w.gu;
    }

    // ---- decisions ---------------------------------------------------------------------------
    // Common case (no guard tripped anywhere): branch-free.  One combined flag sends the warp to the
    // careful per-line evaluation below (about 4e-4 of env-steps on the shipped tracks).
    const float r_tiny = frcp(P.tiny_d);
    const float r_coll = 0.1f;                    // d < 10  <=>  1/d > 0.1
    const float r_band = fmul(r_coll, P.coll_band);
    const float g_all = fmin3(fmin3(gq[0], gq[1], gq[2]), fmin3(gq[3], gq[4], gq[5]), 1.0e30f);
    const float r_all = fmaxf(fmax3(fmax3(Rp[0], Rp[1], Rp[2]), fmax3(Rp[3], Rp[4], Rp[5]), 0.0f),
                              -fmin3(fmin3(Rm[0], Rm[1], Rm[2]), fmin3(Rm[3], Rm[4], Rm[5]), 0.0f));
    const float card_hi = fmax3(fmax3(Rp[0], Rp[3], -Rm[0]), -Rm[3], 0.0f);
    const float band_lo = fmin3(fmin3(fabsf(fsub(Rp[0], r_coll)), fabsf(fsub(Rp[3], r_coll)), fabsf(fadd(Rm[0], r_coll))),
                                fabsf(fadd(Rm[3], r_coll)), 1.0e30f);
    bool destroyed = card_hi > r_coll;
#pragma unroll
    for (int l = 0; l < 6; ++l) {
        dist[l] = fminf(frcp(Rp[l]), 1000.0f);          // "if d < best" from best = 1000.0 (lib/car_env.py:198-207)
        dist[l + 6] = fminf(-frcp(Rm[l]), 1000.0f);
    }
    const bool careful = (gu < P.tiny_un) || (g_all < P.eps_qs) || (r_all > r_tiny) || (band_lo < r_band);
    if (careful) {
        const bool redo_all = gu < P.tiny_un;     // car (numerically) on a wall line: sign of u unknown
        destroyed = false;
#pragma unroll
        for (int l = 0; l < 6; ++l) {
            const bool cardinal = (l == 0 || l == 3);
            bool redo = redo_all || (gq[l] < P.eps_qs);
            if (redo) stat_add(stats, kStatLine);
            if (!redo && (Rp[l] > r_tiny || Rm[l] < -r_tiny)) { redo = true; stat_add(stats, kStatTiny); }
            if (!redo && cardinal &&
                (fabsf(fsub(Rp[l], r_coll)) < r_band || fabsf(fadd(Rm[l], r_coll)) < r_band)) {
                redo = true; stat_add(stats, kStatBand);
            }
            if (!redo) {
                if (cardinal) destroyed = destroyed || (Rp[l] > r_coll) || (Rm[l] < -r_coll);
            } else {
                const D2 d0 = T.trig64[wrap72(s.k + 6 * l)], d1 = T.trig64[wrap72(s.k + 6 * l + 36)];
                const double e0 = exact_ray_distance(s.px, s.py, d0.x, d0.y, T.walls64, P.n_seg);
                const double e1 = exact_ray_distance(s.px, s.py, d1.x, d1.y, T.walls64, P.n_seg);
                dist[l] = (float)e0; dist[l + 6] = (float)e1;
                if (cardinal) destroyed = destroyed || (e0 < 10.0) || (e1 < 10.0);
            }
        }
    }
    return destroyed;
}

// ---- observation of a live pose (lib/car_env.py:569-597): normalised position, velocity, heading, rays ------
CE_HD void pose_observation(const EnvState &s, float vx10, float vy10, const float dist[kNumRays], const Tables &T,
                            float obs[kObsDim]) {
    const F2 d = T.trig32[s.k];
    obs[0] = (float)dmul(s.px, 1.0 / 1280.0);
    obs[1] = (float)dmul(s.py, 1.0 / 720.0);
    obs[2] = vx10;
    obs[3] = vy10;
    obs[4] = d.x; obs[5] = d.y;
#pragma unroll
    for (int i = 0; i < kNumRays; ++i) obs[6 + i] = fmul(dist[i], 1.0e-3f);
}

// ---- one CarEnv.step with same-step autoreset --------------------------------------------------
// `final_obs` (optional, 18 floats): receives the observation of the state the step ended in BEFORE the autoreset —
// gymnasium's info["final_observation"]; it equals o.obs wherever the episode did not end.
// `trunc_obs` (optional, 18 floats): receives that observation only in a step that truncates the episode — written
// inside the autoreset branch, so the fused rollouts carry one pointer instead of 18 more live floats.
template <int U, bool TAB = false, int NS = 0, bool CULL = false>
CE_HD void env_step(EnvState &s, int action, double reward_scale, const TrackParams &P, const Tables &T,
                    StepResult &o, unsigned long long *stats, const WarpSeg *ws = nullptr, const TabView *tv = nullptr,
                    float *final_obs = nullptr, float *trunc_obs = nullptr) {
    int thrust, turn;
    decode_action(action, thrust, turn);
    double reward = thrust > 0 ? 0.01 : 0.0;
    const int k_pre = s.k;

    // gate bookkeeping: uses the pose BEFORE this step's turn and move (rays are only refreshed in update)
    o.gate_hit = 0; o.lap = 0;
    if (gate_touched(s, P, T, stats)) {
        reward = dadd(reward, 1.0);
        s.passed += 1;
        o.gate_hit = 1;
        if (s.next_gate == P.n_gates - 1) { reward = dadd(reward, 10.0); s.next_gate = 0; o.lap = 1; }
        else s.next_gate += 1;
    }
    s.k = wrap72(s.k + turn);
    integrate(s, thrust, k_pre, T);

    float dist[kNumRays];
    bool destroyed = cast_walls<U, TAB, NS, CULL>(s, P, T, dist, stats, ws, tv);
    destroyed = destroyed || (P.start_destroyed != 0);
    s.t += 1;
    o.terminated = 0; o.truncated = 0;
    if (destroyed) { o.terminated = 1; reward = dsub(reward, 3.0); }
    else if (s.t >= kTimeLimit) o.truncated = 1;
    o.reward64 = dmul(reward, reward_scale);
    o.reward = (float)o.reward64;
    o.gates_passed = s.passed; o.time_passed = s.t; o.next_gate = s.next_gate;

    // Same-step autoreset.  The live observation is formed for every lane; the reset (state overwrite + the
    // constant reset observation, ~40 select instructions) sits behind a warp vote: an episode ends in about 0.4 %
    // of env-steps, i.e. seven of eight warp-steps skip it with one uniform branch.
    pose_observation(s, (float)dmul(s.vx, 0.1), (float)dmul(s.vy, 0.1), dist, T, o.obs);
    if (final_obs) {
#pragma unroll
        for (int i = 0; i < kObsDim; ++i) final_obs[i] = o.obs[i];
    }
    const bool done = (o.terminated | o.truncated) != 0;
#if defined(__CUDA_ARCH__)
    if (__any_sync(__activemask(), done))
#endif
    {
        if (done) {
            if (trunc_obs && o.truncated) {
#pragma unroll
                for (int i = 0; i < kObsDim; ++i) trunc_obs[i] = o.obs[i];
            }
            s.px = P.start_x; s.py = P.start_y; s.vx = 0.0; s.vy = 0.0;
            s.k = 0; s.t = 0; s.next_gate = 0; s.passed = 0;
#pragma unroll
            for (int i = 0; i < kObsDim; ++i) o.obs[i] = P.reset_obs[i];
        }
    }
}

// Work list of one warp ("slot") of k_rollout_tab_sliced (carenv_kernels.cu).  n_jobs jobs of n_steps steps each are
// laid end to end and cut into n_slots equal intervals of `quota` warp-steps (McNaughton's wrap-around rule); slot s
// owns [s * quota, (s + 1) * quota).  A job cut by a boundary is split IN TIME between the two slots: the slot that
// owns the END of the job's stretch in the linear order runs the job's FIRST steps at the start of its list (item
// `first_job`, steps [0, head_len)), the slot that owns the beginning of the stretch runs the job's LAST steps at the
// end of its list (job last_full + 1, steps [n_steps - tail_len, n_steps)) — so the first part, started at time 0, has
// finished when the second starts at time quota - tail_len >= n_steps - tail_len = head_len (needs n_jobs >= n_slots).
// In between: whole jobs first_job + (head_len > 0) .. last_full.
struct SliceItems { int first_job, head_len, last_full, tail_len; };
CE_HD SliceItems slice_items(int n_jobs, int n_steps, int slot, int n_slots) {
    const long long total = (long long)n_jobs * n_steps;
    const long long quota = (total + n_slots - 1) / n_slots;
    long long lo = (long long)slot * quota;
    if (lo > total) lo = total;
    long long hi = lo + quota;
    if (hi > total) hi = total;
    SliceItems r;
    r.first_job = (int)(lo / n_steps);
    const int off = (int)(lo - (long long)r.first_job * n_steps);
    r.head_len = off > 0 ? n_steps - off : 0;
    r.last_full = (int)(hi / n_steps) - 1;                   // last job that ends at or before hi
    r.tail_len = (int)(hi - (long long)(r.last_full + 1) * n_steps);
    if (lo >= hi) { r.head_len = 0; r.tail_len = 0; r.last_full = r.first_job - 1; }
    return r;
}

// Observation of the start pose (what CarEnv.reset returns, lib/car_env.py:682-688), evaluated
// with the literal float64 formulas; also tells whether the start pose already collides.
CE_HD bool reset_observation(const TrackParams &P, const Tables &T, float obs[kObsDim]) {
    obs[0] = (float)(P.start_x / 1280.0); obs[1] = (float)(P.start_y / 720.0);
    obs[2] = 0.0f; obs[3] = 0.0f;
    obs[4] = (float)T.trig64[0].x; obs[5] = (float)T.trig64[0].y;
    bool destroyed = false;
    for (int i = 0; i < kNumRays; ++i) {
        const D2 d = T.trig64[wrap72(6 * i)];
        const double e = exact_ray_distance(P.start_x, P.start_y, d.x, d.y, T.walls64, P.n_seg);
        obs[6 + i] = (float)(e / 1000.0);
        if (i % 3 == 0 && e < 10.0) destroyed = true;
    }
    return destroyed;
}

}  // namespace carenv
