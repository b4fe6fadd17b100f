// hrp_env.cu -- the fused highway-v0 step / observe / reset kernels (sm_100a).
//
// One warp owns one env for the whole policy step: the 15 simulation frames of
// HighwayEnv._simulate (reference call site training/routine.py:134; algorithm: highway-env
// 1.10.1, SURVEY.md Appendix A) run out of shared memory, then reward/termination, the
// optional in-place respawn, the Kinematics observation and the RoPE/Dist/Rank embedding
// (experiments/rope_embed.py:64-74, dist_embed.py:76-96, rank_embed.py:45-51) are produced by
// the same warp before the state goes back to HBM once.
//
// Lane l of the warp owns vehicles l and l+32 (V <= 64) in registers.  What other vehicles
// need to see of a vehicle lives in a per-warp shared-memory block.  Instead of the
// reference's O(V) scan per neighbour query, vehicles are kept ranked by x (fp64 keys,
// repaired by odd-even transposition each frame) and every lane band has a 64-bit occupancy
// mask in rank order, so "vehicle in front / behind on lane L" is two bit operations.
//
// Numerics.  The kernels are templates over the working type R.  R = float is the product: x and the IDM
// lane-change timer are fp64 (ordering and the 1.0 < timer test are decided exactly as the fp64 reference
// decides them), everything else is fp32 with approximate division / rsqrt / exp2 / log2.  R = double is the
// VALIDATION instantiation (hrp_env_create_ex, HRP_ENV_REAL64): the same code with fp64 state and IEEE fp64
// arithmetic, slow, used by the parity tests to check the kernel's logic -- rank-ordered neighbour search, band
// masks, list-order commits, collision bookkeeping -- bit-exactly against the fp64 oracle on every step, with no
// rounding in the way (tests/test_env_gpu.py).
#include <math.h>

#include "hrp_internal.cuh"

namespace {

constexpr double kPiD = 3.14159265358979323846;

// arithmetic of the working type
template <typename R> struct Ops;
template <> struct Ops<float> {
    static __device__ __forceinline__ float div(float a, float b) { return __fdividef(a, b); }
    static __device__ __forceinline__ float rsqrt(float a) { return rsqrtf(a); }
    static __device__ __forceinline__ float asin(float a) { return asinf(a); }
    static __device__ __forceinline__ float tan(float a) { return tanf(a); }
    // r^d for r >= 0 (<= 2 ulp in r; the result goes through exp2 / log2 anyway)
    static __device__ __forceinline__ float powpos(float r, float d) { return r > 0.f ? exp2f(d * __log2f(r)) : 0.f; }
    // sin and cos of a heading: traffic headings are a few tenths of a radian, where the Taylor polynomials
    // (|error| < 3e-10 for |x| <= 0.5) are exact to fp32 rounding; anything larger takes the library path
    static __device__ __forceinline__ void sincos(float x, float *s, float *c)
    {
        if (fabsf(x) <= 0.5f) {
            float x2 = x * x;
            float ps = fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, 2.7557319e-6f, -1.9841270e-4f), 8.3333333e-3f), -1.6666667e-1f), 1.f);
            float pc = fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, 2.4801587e-5f, -1.3888889e-3f), 4.1666667e-2f), -0.5f), 1.f);
            *s = x * ps;
            *c = pc;
        } else {
            // rare (a spinning crashed vehicle); one lane pulls its whole warp through this branch, so it is the SFU pair
            // on the argument reduced to [-pi, pi] (|error| < 1e-6, inside the heading tolerance of the parity tests),
            // not the library's full-range slow path
            const float r = x - 6.283185307179586f * rintf(x * 0.15915494309189535f);
            __sincosf(r, s, c);
        }
    }
    // ContinuousAction.get_action: float32 lmap of the clipped np.float32 action (exact float32 operation order)
    static __device__ __forceinline__ float lmap_action(float a, float lo, float span)
    {
        return __fadd_rn(lo, __fdiv_rn(__fmul_rn(__fsub_rn(a, -1.0f), span), 2.0f));
    }
};
template <> struct Ops<double> {
    static __device__ __forceinline__ double div(double a, double b) { return a / b; }
    static __device__ __forceinline__ double rsqrt(double a) { return 1.0 / sqrt(a); }
    static __device__ __forceinline__ double asin(double a) { return ::asin(a); }
    static __device__ __forceinline__ double tan(double a) { return ::tan(a); }
    static __device__ __forceinline__ double powpos(double r, double d) { return pow(r, d); }
    static __device__ __forceinline__ void sincos(double x, double *s, double *c) { ::sincos(x, s, c); }
    static __device__ __forceinline__ double lmap_action(double a, double lo, double span)
    {
        // the env's float32 arithmetic, then widened (the oracle does the same)
        return (double)Ops<float>::lmap_action((float)a, (float)lo, (float)span);
    }
};

template <typename R> struct __align__(16) Rec { R xr, v, ch, sh; };  // what a neighbour query reads of a vehicle: one vector load

template <typename R>
struct __align__(16) WarpS {
    double x[HRP_VS];    // absolute longitudinal position
    double key[HRP_VS];  // scratch: observation sort keys
    Rec<R> rec[HRP_VS];  // x - xref (working copy in R), speed, cos / sin of the heading
    R y[HRP_VS], h[HRP_VS], ts[HRP_VS], delta[HRP_VS];
    R impx[HRP_VS], impy[HRP_VS];
    int impkey[HRP_VS];
    float rowd[HRP_VS];  // scratch: per-row normalised distance of the embedding
    ull band[HRP_MAX_LANES];
    unsigned char lane[HRP_VS], tl_old[HRP_VS], tl_new[HRP_VS], order[HRP_VS], rank[HRP_VS];
    unsigned char crash[HRP_VS], queue[HRP_VS], res[2 * HRP_VS], perm[HRP_VS];
    uint32_t skey[HRP_VS];
    int rowveh[HRP_MAX_OBS_ROWS];
    float obs[HRP_MAX_OBS_ROWS * HRP_MAX_FEATURES];
};

template <typename R>
struct Veh {  // what the owning lane keeps in registers
    double x, timer;
    R y, h, v, ts, delta, impx, impy, ch, sh;
    R acc, tb;  // persistent action: acceleration and tan(beta)
    int lane, tlane;
    bool crashed, has_impact;
};

template <typename R> __device__ __forceinline__ R nzf(R x) { return fabs(x) > R(1e-2) ? x : (x >= R(0) ? R(1e-2) : R(-1e-2)); }
template <typename R> __device__ __forceinline__ R clipf(R x, R lo, R hi) { return fmin(fmax(x, lo), hi); }
template <typename R> __device__ __forceinline__ R wrap_to_pi(R x)
{
    const R pi = R(kPiD);
    if (x >= -pi && x < pi) return x;
    return x - R(2) * pi * floor((x + pi) / (R(2) * pi));
}
// first set bit above / last set bit below rank p of a 64-slot occupancy mask.  The mask is shifted so that the
// vehicle's own bit lands on bit 0 (front) / bit 63 (rear) with one funnel shift on the two 32-bit halves -- the
// 64-bit shift / ffs / clz sequences the compiler emits for the one-line versions cost three times as many instructions.
__device__ __forceinline__ int slot_front(ull mask, int p)
{
    const uint32_t lo = (uint32_t)mask, hi = (uint32_t)(mask >> 32);
    const bool big = p >= 32;
    const uint32_t a = big ? hi : lo, b = big ? 0u : hi;       // (b:a) = mask >> (p & 32)
    const uint32_t l2 = __funnelshift_r(a, b, p) & ~1u;         // the shift is taken mod 32; bit 0 = the vehicle itself
    const uint32_t h2 = b >> (p & 31);
    const int r = l2 ? __ffs((int)l2) - 1 : 31 + __ffs((int)h2);
    return (l2 | h2) ? p + r : -1;
}
__device__ __forceinline__ int slot_rear(ull mask, int p)
{
    const uint32_t lo = (uint32_t)mask, hi = (uint32_t)(mask >> 32);
    const int s = 63 - p;                                       // shift left so that bit p lands on bit 63
    const bool big = s >= 32;
    const uint32_t a = big ? lo : hi, b = big ? 0u : lo;       // (a:b) = mask << (s & 32)
    const uint32_t h2 = __funnelshift_l(b, a, s) & 0x7FFFFFFFu;
    const uint32_t l2 = b << (s & 31);
    const int r = h2 ? 63 - __clz((int)h2) : 31 - __clz((int)l2);
    return (l2 | h2) ? r - s : -1;
}
template <typename R> __device__ __forceinline__ int closest_lane(R y, int lanes)
{
    // argmin_i |y - 4 i| with the first minimum winning a tie (RoadNetwork.get_closest_lane_index):
    // ceil(y / 4 - 1/2), clamped.  y / 4 and the subtraction of 0.5 are exact in binary floating point
    // wherever the result can change the answer.
    int i = (int)ceil(y * R(0.25) - R(0.5));
    return max(0, min(lanes - 1, i));
}

// IDMVehicle.desired_gap (SURVEY A.6): e follows f
template <typename R> __device__ __forceinline__ R desired_gap_rec(const Rec<R> &e, const Rec<R> &f)
{
    R dvx = e.v * e.ch - f.v * f.ch;
    R dvy = e.v * e.sh - f.v * f.sh;
    R dv = dvx * e.ch + dvy * e.sh;
    return R(10) + e.v * R(1.5) + e.v * dv * R(0.12909944487358055);  // 1 / (2 sqrt(3*5))
}
// COMFORT_ACC_MAX * (1 - (max(v,0)/|not_zero(v0)|)^delta); v0 already clipped to [0, 30]
template <typename R> __device__ __forceinline__ R idm_free(R v, R v0, R delta)
{
    R r = Ops<R>::div(fmax(v, R(0)), fabs(nzf(v0)));
    return R(3) * (R(1) - Ops<R>::powpos(r, delta));
}
// COMFORT_ACC_MAX * (desired_gap / not_zero(d))^2, e follows f
template <typename R> __device__ __forceinline__ R idm_interaction_rec(const Rec<R> &e, const Rec<R> &f)
{
    R g = Ops<R>::div(desired_gap_rec(e, f), nzf(f.xr - e.xr));
    return R(3) * g * g;
}

// IDMVehicle.mobil for vehicle i and the candidate on `side` (0: lane-1, 1: lane+1).
// Returns candidate lane + 1, or 0.  The free-road term of self_pred_a - self_a cancels.
template <typename R> __device__ int mobil_item(const WarpS<R> &S, const EnvDev &P, int i, int side)
{
    int li = S.lane[i];
    int c = side == 0 ? li - 1 : li + 1;
    if (c < 0 || c >= P.lanes) return 0;
    double xi = S.x[i];
    if (!(fabs(S.y[i] - R(4) * c) <= R(8) && xi >= 0.0 && xi < 10005.0)) return 0;
    const Rec<R> me = S.rec[i];
    if (fabs(me.v) < R(1)) return 0;
    int p = S.rank[i];
    ull mc = S.band[c];
    int sf = slot_front(mc, p), sr = slot_rear(mc, p);
    if (sr >= 0) {
        int nf = S.order[sr];
        bool ctrl = nf > 0 || P.ego_mode == 1;
        R v0 = ctrl ? clipf(S.ts[nf], R(0), R(30)) : R(0);
        const Rec<R> fo = S.rec[nf];
        R a = idm_free(fo.v, v0, S.delta[i]) - idm_interaction_rec(fo, me);
        if (a < R(-2)) return 0;
    }
    R pred = sf >= 0 ? idm_interaction_rec(me, S.rec[S.order[sf]]) : R(0);
    int so = slot_front(S.band[li], p);
    R cur = so >= 0 ? idm_interaction_rec(me, S.rec[S.order[so]]) : R(0);
    R jerk = cur - pred;
    return jerk >= R(0.2) ? c + 1 : 0;
}

// RoadObject.handle_collisions for list-ordered pair (i < j): spherical pre-check, then the
// separating-axis test of utils.are_polygons_intersecting.  The reference walks the 8 edge
// normals (n0, n1, -n0, -n1 of a, then of b); n and -n give the same separation flags, and the
// same |distance| unless one projected interval contains the other, so each of the 4 distinct
// normals is evaluated once and both distance variants feed the minimum in the reference order.
// Returns bit0 = intersecting, bit1 = will_intersect (+ translation).
template <typename R> __device__ int collide_pair(const WarpS<R> &S, int i, int j, R dt, R &tx, R &ty)
{
    const Rec<R> a = S.rec[i], b = S.rec[j];
    const R cay = S.y[i], cby = S.y[j];
    R dx = b.xr - a.xr, dy = cby - cay;
    R lim = R(5.385164807134504) + a.v * dt;  // sqrt(5^2 + 2^2) + v dt
    if (lim < R(0) || dx * dx + dy * dy > lim * lim) return 0;
    R uax = a.ch, uay = a.sh, ubx = b.ch, uby = b.sh;
    R cax = a.xr, cbx = b.xr;
    R rdx = (a.v * uax - b.v * ubx) * dt, rdy = (a.v * uay - b.v * uby) * dt;
    {
        // cheap exit for the common near miss (vehicles side by side on adjacent lanes): if a's lateral
        // axis separates the rectangles now AND after the displacement, both flags end up false whatever
        // the other axes say, which is the reference's "no contact" result
        R nx = -uay, ny = uax;
        R pa = cax * nx + cay * ny, pb = cbx * nx + cby * ny;
        R rb = R(2.5) * fabs(ubx * nx + uby * ny) + fabs(-uby * nx + ubx * ny);
        R gap = fabs(pa - pb) - (R(1) + rb);
        if (gap > R(0) && gap - fabs(nx * rdx + ny * rdy) > R(0)) return 0;
    }
    bool inter = true, will = true;
    R mind = R(INFINITY), ax = R(0), ay = R(0);
    R dneg[2], nnx[2], nny[2], ddn[2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        // reference edge order: -u_a, +w_a, (+u_a, -w_a), -u_b, +w_b, (+u_b, -w_b)
        R nx, ny;
        if (k == 0) { nx = -uax; ny = -uay; }
        else if (k == 1) { nx = -uay; ny = uax; }
        else if (k == 2) { nx = -ubx; ny = -uby; }
        else { nx = -uby; ny = ubx; }
        R pa = cax * nx + cay * ny, pb = cbx * nx + cby * ny;
        R ra = R(2.5) * fabs(uax * nx + uay * ny) + fabs(-uay * nx + uax * ny);
        R rb = R(2.5) * fabs(ubx * nx + uby * ny) + fabs(-uby * nx + ubx * ny);
        R min_a = pa - ra, max_a = pa + ra, min_b = pb - rb, max_b = pb + rb;
        R sd = min_a < min_b ? min_b - max_a : min_a - max_b;
        if (sd > R(0)) inter = false;
        R vp = nx * rdx + ny * rdy;
        if (vp < R(0)) min_a += vp; else max_a += vp;
        R d1 = min_b - max_a, d2 = min_a - max_b;
        R dist = min_a < min_b ? d1 : d2;
        if (dist > R(0)) will = false;
        if (!inter && !will) return 0;
        R dd = (cax - cbx) * nx + (cay - cby) * ny;
        if (fabs(dist) < mind) {
            mind = fabs(dist);
            if (dd > R(0)) { ax = nx; ay = ny; } else { ax = -nx; ay = -ny; }
        }
        dneg[k & 1] = max_a > max_b ? d2 : d1;  // the same edge seen through the opposite normal
        nnx[k & 1] = nx; nny[k & 1] = ny; ddn[k & 1] = dd;
        if (k & 1) {
#pragma unroll
            for (int t = 0; t < 2; ++t)
                if (fabs(dneg[t]) < mind) {
                    mind = fabs(dneg[t]);
                    if (ddn[t] < R(0)) { ax = -nnx[t]; ay = -nny[t]; } else { ax = nnx[t]; ay = nny[t]; }
                }
        }
    }
    tx = mind * ax; ty = mind * ay;
    return (inter ? 1 : 0) | (will ? 2 : 0);
}

// ---------------------------------------------------------------------------------------
// rank bookkeeping
template <typename R> __device__ void rank_full(WarpS<R> &S, int V, int lane)
{
    // rank = number of vehicles ordered before (x, list index); O(V) per vehicle, once per launch
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        if (k < V) {
            double xk = S.x[k];
            int r = 0;
            for (int j = 0; j < V; ++j) {
                double xj = S.x[j];
                r += (xj < xk || (xj == xk && j < k)) ? 1 : 0;
            }
            S.rank[k] = (unsigned char)r;
            S.order[r] = (unsigned char)k;
        }
    }
    __syncwarp();
}
template <typename R> __device__ void rank_repair(WarpS<R> &S, int V, int lane)
{
    // pre-check on the ego-relative working copies: xr = (R)(x - xref) is recomputed from the fp64 x every frame, and
    // the subtraction of a common xref and the rounding to R are both monotone, so an inversion (true gap <= 0) shows
    // up as a working-copy gap <= 0 at any distance from the ego: "every gap >= 4e-3" proves the order without fp64
    // loads
    {
        bool sus = false;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            int s = lane + 32 * q;
            if (s + 1 < V) sus |= S.rec[S.order[s + 1]].xr - S.rec[S.order[s]].xr < R(4e-3);
        }
        if (!__any_sync(HRP_FULL, sus)) return;   // ranks are unchanged, nothing to rewrite
    }
    for (;;) {
        bool inv = false;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            int s = lane + 32 * q;
            if (s + 1 < V) {
                // odd-even transposition keeps (x, list index) order: equal x never swaps back and forth
                int a = S.order[s], b = S.order[s + 1];
                double xa = S.x[a], xb = S.x[b];
                inv |= xa > xb || (xa == xb && a > b);
            }
        }
        if (!__any_sync(HRP_FULL, inv)) break;
#pragma unroll
        for (int par = 0; par < 2; ++par) {
            int s = 2 * lane + par;
            if (s + 1 < V) {
                int a = S.order[s], b = S.order[s + 1];
                double xa = S.x[a], xb = S.x[b];
                if (xa > xb || (xa == xb && a > b)) { S.order[s] = (unsigned char)b; S.order[s + 1] = (unsigned char)a; }
            }
            __syncwarp();
        }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int s = lane + 32 * q;
        if (s < V) S.rank[S.order[s]] = (unsigned char)s;
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------
// state movement HBM <-> registers/shared
template <typename R> __device__ __forceinline__ void publish(WarpS<R> &S, const Veh<R> &u, int k, double xref)
{
    S.x[k] = u.x;
    Rec<R> r;
    r.xr = (R)(u.x - xref); r.v = u.v; r.ch = u.ch; r.sh = u.sh;
    S.rec[k] = r;
    S.y[k] = u.y; S.h[k] = u.h;
    S.ts[k] = u.ts; S.delta[k] = u.delta;
    S.lane[k] = (unsigned char)u.lane; S.tl_old[k] = S.tl_new[k] = (unsigned char)u.tlane;
    S.impkey[k] = -1; S.crash[k] = 0;
}
template <typename R>
__device__ void load_env(const EnvDev &P, WarpS<R> &S, Veh<R> (&u)[2], int e, int lane, double &xref)
{
    size_t base = (size_t)e * HRP_VS;
    xref = P.x[base];  // ego x at the start of the step
    const R *py = (const R *)P.y, *ph = (const R *)P.heading, *pv = (const R *)P.speed, *pts = (const R *)P.tspeed,
            *pde = (const R *)P.delta, *pix = (const R *)P.impx, *piy = (const R *)P.impy;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        if (k < P.V) {
            Veh<R> &w = u[q];
            w.x = P.x[base + k]; w.timer = P.timer[base + k];
            w.y = py[base + k]; w.h = ph[base + k]; w.v = pv[base + k];
            w.ts = pts[base + k]; w.delta = pde[base + k];
            w.impx = pix[base + k]; w.impy = piy[base + k];
            uint32_t f = P.flags[base + k];
            w.lane = f & 0xff; w.tlane = (f >> 8) & 0xff;
            w.crashed = (f >> 16) & 1; w.has_impact = (f >> 17) & 1;
            Ops<R>::sincos(w.h, &w.sh, &w.ch);
            w.acc = R(0); w.tb = R(0);
            publish(S, w, k, xref);
        } else {
            u[q] = Veh<R>{};  // empty slot: the frame code runs on it with selects, its results are never stored
            u[q].ch = R(1);
        }
    }
    __syncwarp();
}
template <typename R> __device__ void store_env(const EnvDev &P, const Veh<R> (&u)[2], int e, int lane)
{
    size_t base = (size_t)e * HRP_VS;
    R *py = (R *)P.y, *ph = (R *)P.heading, *pv = (R *)P.speed, *pts = (R *)P.tspeed, *pde = (R *)P.delta,
      *pix = (R *)P.impx, *piy = (R *)P.impy;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        if (k < P.V) {
            const Veh<R> &w = u[q];
            P.x[base + k] = w.x; P.timer[base + k] = w.timer;
            py[base + k] = w.y; ph[base + k] = w.h; pv[base + k] = w.v;
            pts[base + k] = w.ts; pde[base + k] = w.delta;
            pix[base + k] = w.impx; piy[base + k] = w.impy;
            P.flags[base + k] = (uint32_t)w.lane | ((uint32_t)w.tlane << 8) |
                                ((uint32_t)w.crashed << 16) | ((uint32_t)w.has_impact << 17);
        }
    }
}

// ---------------------------------------------------------------------------------------
// HighwayEnv._create_vehicles / Vehicle.create_random (SURVEY A.3) with Philox draws.
__device__ __forceinline__ float u01f(uint32_t r) { return (float)(r >> 8) * (1.0f / 16777216.0f); }
template <typename R> __device__ int speed_to_index(R speed)
{
    R x = (speed - R(20)) / R(10);
    return (int)clipf(rint(x * R(2)), R(0), R(2));
}
template <typename R>
__device__ void spawn_env(const EnvDev &P, WarpS<R> &S, Veh<R> (&u)[2], int e, int lane, uint32_t episode,
                          double &xref)
{
    const ull gid = P.seed_env ? 0ull : P.env_id_base + (ull)e;
    const ull seed = P.seed_env ? P.seed_env[e] : P.seed;
    double val[2] = {0.0, 0.0};
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        Veh<R> &w = u[q];
        if (k < P.V) {
            uint32_t r[4];
            hrp_philox((uint32_t)k, episode, (uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)seed,
                       (uint32_t)(seed >> 32), r);
            int ln = (int)((double)u01f(r[0]) * (double)P.lanes);
            double speed, spacing;
            if (k == 0) {
                if (P.initial_lane >= 0) ln = P.initial_lane;
                speed = 25.0; spacing = P.ego_spacing;
            } else {
                speed = 21.0 + 3.0 * (double)u01f(r[1]);
                spacing = P.inv_density;
            }
            double offset = spacing * (12.0 + speed) * P.gap_factor;
            double inc = offset * (0.9 + (1.1 - 0.9) * (double)u01f(r[2]));
            val[q] = k == 0 ? 3.0 * offset + inc : inc;
            w.y = R(4) * ln; w.h = R(0); w.v = (R)speed; w.ts = (R)speed;
            w.lane = ln; w.tlane = ln;
            w.delta = k > 0 ? (R)(3.5 + (4.5 - 3.5) * (double)u01f(r[3])) : R(4);
            w.impx = w.impy = R(0); w.crashed = false; w.has_impact = false;
            w.ch = R(1); w.sh = R(0); w.acc = R(0); w.tb = R(0);
            if (k == 0 && P.ego_mode == 1) w.ts = R(20) + R(5) * speed_to_index(w.v);
        }
    }
    // x_k = x_{k-1} + inc_k: inclusive scan over list order (fp64)
#pragma unroll
    for (int q = 0; q < 2; ++q) {
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            double t = __shfl_up_sync(HRP_FULL, val[q], d);
            if (lane >= d) val[q] += t;
        }
    }
    double tot0 = __shfl_sync(HRP_FULL, val[0], 31);
    val[1] += tot0;
    xref = __shfl_sync(HRP_FULL, val[0], 0);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        if (k < P.V) {
            Veh<R> &w = u[q];
            w.x = val[q];
            double t = (w.x + (double)w.y) * 3.14159265358979323846;
            w.timer = k > 0 ? t - floor(t) : 0.0;  // python: (x + y) * pi % 1.0, operands >= 0
            publish(S, w, k, xref);
        }
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------
// KinematicObservation.observe (SURVEY A.8) + embedding wrapper, warp-cooperative.
template <typename R> __device__ double feature_value(const WarpS<R> &S, int code, int k)
{
    switch (code) {
    case HRP_F_PRESENCE: return 1.0;
    case HRP_F_X: return S.x[k];
    case HRP_F_Y: return (double)S.y[k];
    case HRP_F_VX: return (double)S.rec[k].v * (double)S.rec[k].ch;
    case HRP_F_VY: return (double)S.rec[k].v * (double)S.rec[k].sh;
    case HRP_F_HEADING: return (double)S.h[k];
    case HRP_F_COS_H: return (double)S.rec[k].ch;
    case HRP_F_SIN_H: return (double)S.rec[k].sh;
    }
    return 0.0;
}
template <typename R> __device__ void write_row(const EnvDev &P, WarpS<R> &S, int row, int k)
{
    S.rowveh[row] = k;
    for (int f = 0; f < P.F; ++f) {
        int code = P.feat[f];
        double val = feature_value(S, code, k);
        if (k != 0 && !P.absolute && code >= HRP_F_X && code <= HRP_F_VY) val -= feature_value(S, code, 0);
        if (P.normalize && P.has_range[f]) {
            val = -1.0 + (val - P.lo[f]) * 2.0 / (P.hi[f] - P.lo[f]);
            if (P.clip) val = fmin(fmax(val, -1.0), 1.0);
        }
        S.obs[row * P.F + f] = (float)val;
    }
}

// the embedding epilogue on an [N, F] table in shared memory -> out[N, Fout] in global memory.  float32 with the
// reference's operation order (numpy float32 arithmetic): explicit round-to-nearest intrinsics, IEEE division and
// square root, and the full-range sinf / cosf / sincosf of the CUDA math library (this file is NOT compiled with
// --use_fast_math: the angles reach 2 pi, outside the range where the SFU approximations hold their error bound).
__device__ void embed_store(int kind, int edim, int use_euclid, int ego_idx, float max_dist,
                            const float *__restrict__ table, const float *tab, float *rowd, int N,
                            int F, int Fout, int lane, float *__restrict__ out,
                            const float *__restrict__ dist_override = nullptr)
{
    if (dist_override) {  // RotaryEmbedWrapper._apply_rope(obs, dist_norm): caller-supplied distances
        for (int r = lane; r < N; r += 32) rowd[r] = dist_override[r];
        __syncwarp();
    } else if (kind == HRP_EMBED_ROPE || kind == HRP_EMBED_DIST) {
        // rel = obs[:, :2] - obs[ego, :2]; dist = clip(norm(rel) / max_dist, 0, 1), all float32
        float ex = tab[ego_idx * F + 0], ey = F > 1 ? tab[ego_idx * F + 1] : 0.f;
        for (int r = lane; r < N; r += 32) {
            float rx = __fsub_rn(tab[r * F + 0], ex);
            float d;
            if (use_euclid) {
                float ry = __fsub_rn(tab[r * F + 1], ey);
                d = __fsqrt_rn(__fadd_rn(__fmul_rn(rx, rx), __fmul_rn(ry, ry)));
            } else {
                d = fabsf(rx);
            }
            d = __fdiv_rn(d, max_dist);
            rowd[r] = fminf(fmaxf(d, 0.f), 1.f);
        }
        __syncwarp();
    }
    const float two_pi = 6.2831853071795862f;  // float32(2*pi), as numpy's weak python scalar
    int total = N * Fout;
    for (int idx = lane; idx < total; idx += 32) {
        int r = idx / Fout, c = idx - r * Fout;
        float o;
        if (kind == HRP_EMBED_ROPE && c < edim) {
            int p = c >> 1;
            float theta = __fmul_rn(__fmul_rn(two_pi, rowd[r]), table[p]);
            float sn, cs;
            sincosf(theta, &sn, &cs);
            float a = tab[r * F + 2 * p], b = tab[r * F + 2 * p + 1];
            o = (c & 1) ? __fadd_rn(__fmul_rn(a, sn), __fmul_rn(b, cs))
                        : __fsub_rn(__fmul_rn(a, cs), __fmul_rn(b, sn));
        } else if (c < F) {
            o = tab[r * F + c];
        } else if (kind == HRP_EMBED_DIST) {
            int j = c - F, half = edim >> 1;
            float fr = table[j < half ? j : j - half];
            float ang = __fmul_rn(__fmul_rn(two_pi, rowd[r]), fr);
            o = j < half ? sinf(ang) : cosf(ang);
        } else {  // HRP_EMBED_RANK: tanh(table) precomputed by the host
            o = table[r * edim + (c - F)];
        }
        out[idx] = o;
    }
}

template <typename R>
__device__ void observe_env(const EnvDev &P, WarpS<R> &S, int e, int lane, float *__restrict__ obs,
                            const int32_t *__restrict__ perm_in, int32_t *__restrict__ row_vehicle,
                            uint32_t draw)
{
    const int V = P.V, N = P.N, F = P.F;
    for (int i = lane; i < N * F; i += 32) S.obs[i] = 0.f;
    for (int i = lane; i < N; i += 32) S.rowveh[i] = -1;
    // Road.close_objects_to: list order, ||p - p_ego|| < 200 and -10 < dx unless see_behind
    double ex = S.x[0];
    R ey = S.y[0];
    bool close[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        close[q] = false;
        if (k >= 1 && k < V) {
            double dx = S.x[k] - ex, dy = (double)S.y[k] - (double)ey;
            close[q] = (dx * dx + dy * dy < 200.0 * 200.0) && (P.see_behind || dx > -10.0);
            S.key[k] = close[q] ? fabs(dx) : INFINITY;
        }
    }
    ull cm = (ull)__ballot_sync(HRP_FULL, close[0]) | ((ull)__ballot_sync(HRP_FULL, close[1]) << 32);
    // row permutation for order == "shuffled": injected, or rank of Philox keys
    if (!P.sorted && N > 1) {
        if (perm_in) {
            for (int i = lane; i < N - 1; i += 32) S.perm[i] = (unsigned char)perm_in[(size_t)e * (N - 1) + i];
        } else {
            const ull gid = P.seed_env ? 0ull : P.env_id_base + (ull)e;
            const ull seed = P.seed_env ? P.seed_env[e] : P.seed;
            for (int blk = lane; blk * 4 < N - 1; blk += 32) {
                uint32_t r[4];
                hrp_philox((uint32_t)blk, draw, (uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)seed,
                           (uint32_t)(seed >> 32) ^ 0xA5A5A5A5u, r);
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if (blk * 4 + t < N - 1) S.skey[blk * 4 + t] = r[t];
            }
            __syncwarp();
            for (int i = lane; i < N - 1; i += 32) {
                uint32_t ki = S.skey[i];
                int r = 0;
                for (int j = 0; j < N - 1; ++j) {
                    uint32_t kj = S.skey[j];
                    r += (kj < ki || (kj == ki && j < i)) ? 1 : 0;
                }
                S.perm[i] = (unsigned char)r;
            }
        }
    }
    __syncwarp();
    if (lane == 0) write_row(P, S, 0, 0);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        if (close[q]) {
            int r;
            if (P.sorted) {  // stable sort by |dx|: count candidates ordered before k
                double kk = S.key[k];
                r = 0;
                ull m = cm;
                while (m) {
                    int j = __ffsll((long long)m) - 1;
                    m &= m - 1;
                    double kj = S.key[j];
                    r += (kj < kk || (kj == kk && j < k)) ? 1 : 0;
                }
            } else {
                r = __popcll(cm & ((1ull << k) - 1ull));
            }
            if (r < N - 1) {
                int row = 1 + (P.sorted ? r : (int)S.perm[r]);
                write_row(P, S, row, k);
            }
        }
    }
    __syncwarp();
    float *out = obs + (size_t)e * N * P.Fout;
    embed_store(P.embed_kind, P.embed_dim, P.use_euclid, P.ego_idx, P.max_dist, P.table, S.obs, S.rowd, N,
                F, P.Fout, lane, out);
    if (row_vehicle)
        for (int i = lane; i < N; i += 32) row_vehicle[(size_t)e * N + i] = S.rowveh[i];
    __syncwarp();
}

// ---------------------------------------------------------------------------------------
// OccupancyGridObservation.observe (absolute=False, as_image=False; DESIGN.md §3.1), warp-cooperative.  fp64 in both
// instantiations, every operation an explicit round-to-nearest intrinsic: a cell index is a floor, and the fp64
// validation kernel must decide it bit for bit as the sequential fp64 restatement (tests/grid_oracle.py) does, with
// no contraction into FMAs.  Compiled into the grid kernels only (the OBS template parameter below).
__device__ __forceinline__ double grid_lmap(double v, double lo, double hi)     // utils.lmap(v, [lo, hi], [-1, 1])
{
    return __dadd_rn(-1.0, __ddiv_rn(__dmul_rn(__dsub_rn(v, lo), 2.0), __dsub_rn(hi, lo)));
}
__device__ __forceinline__ double grid_unlmap(double v, double lo, double hi)   // utils.lmap(v, [-1, 1], [lo, hi])
{
    return __dadd_rn(lo, __ddiv_rn(__dmul_rn(__dadd_rn(v, 1.0), __dsub_rn(hi, lo)), 2.0));
}
// pos_to_index of an ego-relative position: cell id ix * H + iy, or -1 outside [0, W) x [0, H)
__device__ __forceinline__ int grid_cell(const GridDev &G, double px, double py, double c, double s)
{
    if (G.galign) {   // [[c, s], [-s, c]] @ p
        const double rx = __dadd_rn(__dmul_rn(c, px), __dmul_rn(s, py));
        const double ry = __dadd_rn(__dmul_rn(-s, px), __dmul_rn(c, py));
        px = rx; py = ry;
    }
    const double fx = floor(__ddiv_rn(__dsub_rn(px, G.glo[0]), G.gstep[0]));
    const double fy = floor(__ddiv_rn(__dsub_rn(py, G.glo[1]), G.gstep[1]));
    return (fx >= 0.0 && fx < (double)G.gw && fy >= 0.0 && fy < (double)G.gh) ? (int)fx * G.gh + (int)fy : -1;
}
// Vehicle.to_dict(ego)[code]: x, y, vx, vy relative to the ego, the rest absolute
template <typename R> __device__ __forceinline__ double grid_feature(const WarpS<R> &S, int code, int k)
{
    switch (code) {
    case HRP_F_PRESENCE: return 1.0;
    case HRP_F_X: return __dsub_rn(S.x[k], S.x[0]);
    case HRP_F_Y: return __dsub_rn((double)S.y[k], (double)S.y[0]);
    case HRP_F_VX: return __dsub_rn(__dmul_rn((double)S.rec[k].v, (double)S.rec[k].ch), __dmul_rn((double)S.rec[0].v, (double)S.rec[0].ch));
    case HRP_F_VY: return __dsub_rn(__dmul_rn((double)S.rec[k].v, (double)S.rec[k].sh), __dmul_rn((double)S.rec[0].v, (double)S.rec[0].sh));
    case HRP_F_HEADING: return (double)S.h[k];
    case HRP_F_COS_H: return (double)S.rec[k].ch;
    case HRP_F_SIN_H: return (double)S.rec[k].sh;
    }
    return 0.0;
}
template <typename R>
__device__ void observe_grid(const EnvDev &P, const GridDev &G, WarpS<R> &S, int e, int lane, float *__restrict__ obs,
                             int32_t *__restrict__ cell_vehicle)
{
    const int V = P.V, F = P.F, C = G.gw * G.gh;
    for (int i = lane; i < F * C; i += 32) S.obs[i] = 0.f;   // an empty cell is NaN upstream, and nan_to_num makes it 0
    const double ex = S.x[0], ey = (double)S.y[0];
    const double c = (double)S.rec[0].ch, s = (double)S.rec[0].sh;
    // every vehicle, the ego included: its cell into the shuffle-key scratch (the grid draws no permutation)
    int cell[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int k = lane + 32 * q;
        cell[q] = -1;
        if (k < V) {
            double px = __dsub_rn(S.x[k], ex), py = __dsub_rn((double)S.y[k], ey);
            if (G.gx >= 0) px = grid_unlmap(grid_lmap(px, P.lo[G.gx], P.hi[G.gx]), P.lo[G.gx], P.hi[G.gx]);
            if (G.gy >= 0) py = grid_unlmap(grid_lmap(py, P.lo[G.gy], P.hi[G.gy]), P.lo[G.gy], P.hi[G.gy]);
            cell[q] = grid_cell(G, px, py, c, s);
            S.skey[k] = (uint32_t)cell[q];
        }
    }
    __syncwarp();
    // upstream writes the vehicles in reverse list order, so the lowest index owns a shared cell
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int k = lane + 32 * q;
        bool own = cell[q] >= 0;
        for (int j = 0; j < k && own; ++j) own = S.skey[j] != (uint32_t)cell[q];
        if (!own) continue;
        for (int f = 0; f < F; ++f) {
            const int code = P.feat[f];
            if (code == HRP_F_ON_ROAD) continue;
            double v = grid_feature(S, code, k);
            if (P.has_range[f]) v = grid_lmap(v, P.lo[f], P.hi[f]);
            if (P.clip) v = fmin(fmax(v, -1.0), 1.0);
            S.obs[f * C + cell[q]] = (float)v;
        }
    }
    // fill_road_layer_by_lanes: waypoints ex - 100 + i * min(grid_step), i < ceil(200 / step), clipped to the road,
    // at (w, 4 L) on every lane, spread over the warp
    for (int f = 0; f < F; ++f) {
        if (P.feat[f] != HRP_F_ON_ROAD) continue;
        const double step = fmin(G.gstep[0], G.gstep[1]);
        const double start = __dsub_rn(ex, 100.0);
        const int n = (int)ceil(__ddiv_rn(__dsub_rn(__dadd_rn(ex, 100.0), start), step));
        for (int i = lane; i < P.lanes * n; i += 32) {
            const int L = i / n, w = i - L * n;
            const double wx = fmin(fmax(__dadd_rn(start, __dmul_rn((double)w, step)), 0.0), 10000.0);
            const int cc = grid_cell(G, __dsub_rn(wx, ex), __dsub_rn(4.0 * L, ey), c, s);
            if (cc >= 0) S.obs[f * C + cc] = 1.f;
        }
    }
    __syncwarp();
    float *out = obs + (size_t)e * F * C;
    for (int i = lane; i < F * C; i += 32) out[i] = S.obs[i];
    if (cell_vehicle)
        for (int i = lane; i < C; i += 32) {
            int who = -1;
            for (int j = 0; j < V && who < 0; ++j) who = S.skey[j] == (uint32_t)i ? j : -1;
            cell_vehicle[(size_t)e * C + i] = who;
        }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------
// One simulation frame: Road.act() then Road.step(dt) (SURVEY A.11).  EGO_ONLY: highway-fast-v0's collision rule
// (hrp_cfg.ego_collisions_only; DESIGN.md Appendix C): only the pairs (0, k) are tested.
template <typename R, bool EGO_ONLY = false>
__device__ void simulate_frame(const EnvDev &P, WarpS<R> &S, Veh<R> (&u)[2], int lane, double xref)
{
    const int V = P.V;
    const R dt = (R)P.dt64;
    const R window = (R)P.coll_window;
    const bool ego_ctrl = P.ego_mode == 1;
    const R kPi = R(kPiD);

    // ---- band occupancy masks in rank order: |y - 4L| <= 3 (on_lane with margin 1)
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int s = lane + 32 * q;
        R yy = R(0);
        bool inx = false;
        if (s < V) {
            int veh = S.order[s];
            yy = S.y[veh];
            double xx = S.x[veh];
            inx = xx >= -5.0 && xx < 10005.0;
        }
        for (int L = 0; L < P.lanes; ++L) {
            unsigned b = __ballot_sync(HRP_FULL, inx && fabs(yy - R(4) * L) <= R(3));
            if (lane == 0) reinterpret_cast<unsigned *>(&S.band[L])[q] = b;
        }
    }
    __syncwarp();

    // ---- IDMVehicle.change_lane_policy, part 1: MOBIL decisions of vehicles whose timer fired
    bool fire[2], mid[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        Veh<R> &w = u[q];
        bool idm = k > 0 && k < V && !w.crashed;
        mid[q] = idm && w.lane != w.tlane;
        fire[q] = idm && w.lane == w.tlane && 1.0 < w.timer;
        if (fire[q]) w.timer = 0.0;
    }
    unsigned fm0 = __ballot_sync(HRP_FULL, fire[0]), fm1 = __ballot_sync(HRP_FULL, fire[1]);
    if (fm0 | fm1) {
        unsigned lt = (1u << lane) - 1u;
        int pos[2] = {__popc(fm0 & lt), __popc(fm0) + __popc(fm1 & lt)};
#pragma unroll
        for (int q = 0; q < 2; ++q)
            if (fire[q]) S.queue[pos[q]] = (unsigned char)(lane + 32 * q);
        __syncwarp();
        int nitems = 2 * (__popc(fm0) + __popc(fm1));
        for (int t = lane; t < nitems; t += 32)
            S.res[t] = (unsigned char)mobil_item(S, P, S.queue[t >> 1], t & 1);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 2; ++q)
            if (fire[q]) {
                int r0 = S.res[2 * pos[q]], r1 = S.res[2 * pos[q] + 1];
                if (r0) u[q].tlane = r0 - 1;
                if (r1) u[q].tlane = r1 - 1;  // a later candidate overwrites an earlier one
                S.tl_new[lane + 32 * q] = (unsigned char)u[q].tlane;
            }
        __syncwarp();
    }

    // ---- part 2: vehicles already changing lane abort if someone ahead targets the same lane.
    // List order matters: vehicle k sees this frame's decisions of j < k, last frame's of j > k.
    ull mm = (ull)__ballot_sync(HRP_FULL, mid[0]) | ((ull)__ballot_sync(HRP_FULL, mid[1]) << 32);
    while (mm) {
        int k = __ffsll((long long)mm) - 1;
        mm &= mm - 1;
        int T = S.tl_new[k];
        const Rec<R> rk = S.rec[k];
        bool hit = false;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            int j = lane + 32 * q;
            if (j < V && j != k && (j > 0 || ego_ctrl) && S.lane[j] != T) {
                int tj = j < k ? S.tl_new[j] : S.tl_old[j];
                if (tj == T) {
                    const Rec<R> rj = S.rec[j];
                    // the reference decides "ahead" on the fp64 positions: x_j - x_k > 0
                    R d = rj.xr - rk.xr;
                    if (S.x[j] - S.x[k] > 0.0 && d < desired_gap_rec(rk, rj)) hit = true;
                }
            }
        }
        if (__any_sync(HRP_FULL, hit)) {
            if (lane == (k & 31)) {
                if (k >> 5) u[1].tlane = u[1].lane; else u[0].tlane = u[0].lane;
                S.tl_new[k] = S.lane[k];
            }
        }
        __syncwarp();
    }

    // ---- controls: steering_control + IDM acceleration (or the ego's own action).  Straight-line code with
    // selects: every lane runs the same instructions whether its slot holds a vehicle, a crashed one or none.
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int k = lane + 32 * q;
        Veh<R> &w = u[q];
        const bool valid = k < V;
        const bool act = valid && !w.crashed && (k > 0 || ego_ctrl);  // ContinuousAction ego keeps its action dict
        // ControlledVehicle.steering_control(target_lane) -> tan(beta) without leaving the tangent
        const R lat = w.y - R(4) * w.tlane;
        const R lsc = -(R(1) / R(0.6)) * lat;
        const R rv = Ops<R>::div(R(1), nzf(w.v));
        // clip(asin(clip(c, -1, 1)), -pi/4, pi/4) == asin(clip(c, -sin(pi/4), sin(pi/4))): asin is monotone
        const R hc = Ops<R>::asin(clipf(lsc * rv, R(-0.70710678118654752), R(0.70710678118654752)));
        const R href = clipf(hc, -kPi / R(4), kPi / R(4));
        const R hrc = R(5) * wrap_to_pi(href - w.h);
        const R ss = clipf(R(2.5) * rv * hrc, R(-1), R(1));  // sin(slip)
        const R tslip = ss * Ops<R>::rsqrt(fmax(R(1) - ss * ss, R(0)));  // tan(slip); +-inf at |ss| == 1
        // tan(beta) = clip(2 tan slip, +-tan(pi/3)) / 2
        const R tb_new = clipf(tslip, R(-0.86602540378443865), R(0.86602540378443865));
        // IDMVehicle.acceleration against the front vehicle of the own lane and of the target lane
        const int p = valid ? (int)S.rank[k] : 0;
        const R a0 = idm_free(w.v, clipf(w.ts, R(0), R(30)), w.delta);
        Rec<R> me;
        me.xr = (R)(w.x - xref); me.v = w.v; me.ch = w.ch; me.sh = w.sh;
        const int sf = slot_front(S.band[w.lane], p);
        const R i1 = idm_interaction_rec(me, S.rec[S.order[max(sf, 0)]]);
        R acc = a0 - (sf >= 0 ? i1 : R(0));
        // the front vehicle of the target lane matters only between lanes: the whole warp skips it otherwise
        if (__any_sync(HRP_FULL, valid && w.lane != w.tlane)) {
            const int st = slot_front(S.band[w.tlane], p);
            const R i2 = idm_interaction_rec(me, S.rec[S.order[max(st, 0)]]);
            const R acc_t = a0 - (st >= 0 ? i2 : R(0));
            acc = w.lane != w.tlane ? fmin(acc, acc_t) : acc;
        }
        const R acc_idm = clipf(acc, R(-6), R(6));
        const R acc_mdp = (R(1) / R(0.6)) * (w.ts - w.v);  // MDPVehicle: speed_control
        w.tb = act ? tb_new : w.tb;
        w.acc = act ? (k > 0 ? acc_idm : acc_mdp) : w.acc;
    }
    __syncwarp();  // every read of the frame-start state is done

    // ---- Vehicle.step(dt): clip_actions, kinematic bicycle, pending impact, lane re-assignment
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int k = lane + 32 * q;
        Veh<R> &w = u[q];
        w.timer += k > 0 ? P.dt64 : 0.0;
        w.tb = w.crashed ? R(0) : w.tb;
        w.acc = w.crashed ? R(-1) * w.v : w.acc;
        w.acc = w.v > R(40) ? fmin(w.acc, R(40) - w.v) : (w.v < R(-40) ? fmax(w.acc, R(-40) - w.v) : w.acc);
        const R cb = Ops<R>::rsqrt(R(1) + w.tb * w.tb), sb = w.tb * cb;
        const R c = w.ch * cb - w.sh * sb, s = w.sh * cb + w.ch * sb;
        w.x += (double)(w.v * c * dt);
        w.y += w.v * s * dt;
        w.x += w.has_impact ? (double)w.impx : 0.0;   // pending impact of the previous frame's collision
        w.y += w.has_impact ? w.impy : R(0);
        w.crashed = w.crashed || w.has_impact;
        w.has_impact = false;
        w.impx = w.impy = R(0);
        w.h += w.v * sb * R(0.4) * dt;   // / (LENGTH / 2); the product form saves the IEEE division
        w.v += w.acc * dt;
        w.lane = closest_lane(w.y, P.lanes);
        Ops<R>::sincos(w.h, &w.sh, &w.ch);
        if (k < V) {
            S.x[k] = w.x;
            Rec<R> r;
            r.xr = (R)(w.x - xref); r.v = w.v; r.ch = w.ch; r.sh = w.sh;
            S.rec[k] = r;
            S.y[k] = w.y;
            S.lane[k] = (unsigned char)w.lane;
            S.tl_old[k] = S.tl_new[k] = (unsigned char)w.tlane;
        }
    }
    __syncwarp();
    rank_repair(S, V, lane);

    if constexpr (EGO_ONLY) {
        // ---- collisions of highway-fast-v0: lane l tests pairs (0, l) and (0, l + 32) in one pass.  The ego's
        // partners can sit any number of ranks away (two uncontrolled vehicles between them are not tested against
        // each other), so this is a window on |x_k - x_0|, not the rank-neighbour sweep below.
        const R x0 = S.rec[0].xr;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int k = lane + 32 * q;
            int ev = 0;
            R tx = R(0), ty = R(0);
            if (k >= 1 && k < V && fabs(S.rec[k].xr - x0) <= window) ev = collide_pair(S, 0, k, dt, tx, ty);
            unsigned evm = __ballot_sync(HRP_FULL, ev != 0);
            while (evm) {  // rare: serialise in k order, so that the ego keeps the impact of its last pair
                int src = __ffs(evm) - 1;
                evm &= evm - 1;
                int bv = __shfl_sync(HRP_FULL, ev, src);
                R btx = __shfl_sync(HRP_FULL, tx, src), bty = __shfl_sync(HRP_FULL, ty, src);
                if (lane == 0) {
                    const int bk = src + 32 * q;
                    if (bv & 2) {
                        S.impkey[0] = 64 + bk; S.impx[0] = R(0.5) * btx; S.impy[0] = R(0.5) * bty;
                        S.impkey[bk] = 0; S.impx[bk] = R(-0.5) * btx; S.impy[bk] = R(-0.5) * bty;
                    }
                    if (bv & 1) { S.crash[0] = 1; S.crash[bk] = 1; }
                }
            }
        }
    } else {
        // ---- collisions: pairs within the pre-check radius are neighbours in rank order
        int a[2];
        R xa[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            a[q] = lane + 32 * q < V ? (int)S.order[lane + 32 * q] : -1;
            xa[q] = S.rec[max(a[q], 0)].xr;
        }
        for (int off = 1; off < V; ++off) {
            int b[2];
            bool cand[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                int s2 = lane + 32 * q + off;
                cand[q] = a[q] >= 0 && s2 < V;
                b[q] = 0;
                if (cand[q]) {
                    b[q] = S.order[s2];
                    cand[q] = S.rec[b[q]].xr - xa[q] <= window;  // >= sqrt(29) + max speed * dt
                }
            }
            if (!__any_sync(HRP_FULL, cand[0] || cand[1])) break;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                int ev = 0, ei = 0, ej = 0;
                R tx = R(0), ty = R(0);
                if (cand[q]) {
                    ei = min(a[q], b[q]); ej = max(a[q], b[q]);
                    ev = collide_pair(S, ei, ej, dt, tx, ty);
                }
                unsigned evm = __ballot_sync(HRP_FULL, ev != 0);
                while (evm) {  // rare: serialise so that the last pair in (i, j) order wins the impact
                    int src = __ffs(evm) - 1;
                    evm &= evm - 1;
                    int bv = __shfl_sync(HRP_FULL, ev, src);
                    int bi = __shfl_sync(HRP_FULL, ei, src), bj = __shfl_sync(HRP_FULL, ej, src);
                    R btx = __shfl_sync(HRP_FULL, tx, src), bty = __shfl_sync(HRP_FULL, ty, src);
                    if (lane == 0) {
                        if (bv & 2) {
                            int ki = 64 + bj, kj = bi;  // pairs (i, *) come after every pair (*, i)
                            if (ki > S.impkey[bi]) { S.impkey[bi] = ki; S.impx[bi] = R(0.5) * btx; S.impy[bi] = R(0.5) * bty; }
                            if (kj > S.impkey[bj]) { S.impkey[bj] = kj; S.impx[bj] = R(-0.5) * btx; S.impy[bj] = R(-0.5) * bty; }
                        }
                        if (bv & 1) { S.crash[bi] = 1; S.crash[bj] = 1; }
                    }
                }
            }
        }
    }
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        int k = lane + 32 * q;
        if (k >= V) continue;
        Veh<R> &w = u[q];
        if (S.crash[k]) { w.crashed = true; S.crash[k] = 0; }
        if (S.impkey[k] >= 0) {
            w.has_impact = true; w.impx = S.impx[k]; w.impy = S.impy[k];
            S.impkey[k] = -1;
        }
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------
// FINAL: the instantiation with the final-observation output (hrp_env_step_final).  A compile-time switch, so that the
// default kernels carry none of its code: the step kernel is sensitive to instruction-cache pressure (DESIGN.md §3.1).
// OBS: the observation epilogue, HRP_OBS_KINEMATICS or HRP_OBS_OCCUPANCY_GRID -- compile-time for the same reason, and
// with one call site of observe_env / observe_grid per instantiation.
// EGO_ONLY: highway-fast-v0's ego-only collision pass (simulate_frame) -- compile-time for the same reason.
template <typename R, int WARPS, bool FINAL = false, int OBS = HRP_OBS_KINEMATICS, bool EGO_ONLY = false>
__device__ __forceinline__ void step_body(const EnvDev &P, const float *__restrict__ actions, float *__restrict__ obs,
                                          float *__restrict__ reward, uint8_t *__restrict__ term,
                                          uint8_t *__restrict__ trunc, const int32_t *__restrict__ perm,
                                          int32_t *__restrict__ row_vehicle, float *__restrict__ final_obs = nullptr,
                                          const GridDev &G = GridDev{})
{
    __shared__ WarpS<R> smem[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * WARPS + warp;
    // Launched with programmatic stream serialisation.  The successor in the stream (the policy's first GEMM, or the
    // next step) may be scheduled as CTAs of this grid retire; it waits for this grid to complete before it reads
    // anything.  This kernel reads the simulator state, which its predecessor may have written (a step after a step,
    // a step after a reset), so it waits for the predecessor before the first load: only the index arithmetic above
    // overlaps the predecessor's tail.
    hrp_pdl_release();
    hrp_pdl_wait();
    if (e >= P.E) return;
    if (P.step_mask && !P.step_mask[e]) return;   // multiplexed experiments: this env is not taking a step now
    WarpS<R> &S = smem[warp];
    Veh<R> u[2];
    double xref;
    load_env(P, S, u, e, lane, xref);
    rank_full(S, P.V, lane);

    // ActionType.act on the first frame (SURVEY A.2)
    float a0 = actions[2 * e], a1 = actions[2 * e + 1];
    if (lane == 0) {
        if (P.ego_mode == 0) {
            // ContinuousAction.get_action: float32 lmap of the clipped np.float32 action
            a0 = fminf(fmaxf(a0, -1.f), 1.f); a1 = fminf(fmaxf(a1, -1.f), 1.f);
            u[0].acc = Ops<R>::lmap_action((R)a0, R(-5), R(10));
            R steer = Ops<R>::lmap_action((R)a1, (R)(-0.78539816339744831f), (R)1.5707963267948966f);
            u[0].tb = R(0.5) * Ops<R>::tan(steer);
        } else {
            // MDPVehicle.act(action) / ControlledVehicle.act(action)
            int act = (int)a0;
            Veh<R> &w = u[0];
            if (act == 3 || act == 4) {
                int idx = speed_to_index(w.v) + (act == 3 ? 1 : -1);
                idx = max(0, min(2, idx));
                w.ts = R(20) + R(5) * idx;
                S.ts[0] = w.ts;
            } else if (act == 0 || act == 2) {
                int t = max(0, min(P.lanes - 1, w.tlane + (act == 2 ? 1 : -1)));
                if (fabs(w.y - R(4) * t) <= R(8) && w.x >= 0.0 && w.x < 10005.0) w.tlane = t;
                S.tl_old[0] = S.tl_new[0] = (unsigned char)w.tlane;
            }
        }
    }
    __syncwarp();

    for (int frame = 0; frame < P.frames; ++frame) {
        simulate_frame<R, EGO_ONLY>(P, S, u, lane, xref);
        if (P.trace) {   // validation aid: the intra-step trajectory, for the frame-by-frame parity check
            double *t = P.trace + (((size_t)e * P.frames + frame) * HRP_VS) * HRP_TRACE_FIELDS;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int k = lane + 32 * q;
                if (k < P.V) {
                    const Veh<R> &w = u[q];
                    double *r = t + (size_t)k * HRP_TRACE_FIELDS;
                    r[0] = w.x; r[1] = (double)w.y; r[2] = (double)w.v; r[3] = (double)w.h;
                    r[4] = (double)w.impx; r[5] = (double)w.impy;
                    r[6] = (double)((uint32_t)w.lane | ((uint32_t)w.tlane << 8) | ((uint32_t)w.crashed << 16) |
                                    ((uint32_t)w.has_impact << 17));
                }
            }
        }
    }

    // HighwayEnv._reward / _is_terminated / _is_truncated (SURVEY A.9)
    int done = 0;
    double tnow = 0.0;
    if (lane == 0) {
        const Veh<R> &w = u[0];
        int rl = P.ego_mode == 1 ? w.tlane : w.lane;
        R fs = w.v * w.ch;
        R scaled = (fs - (R)P.rs_lo) / ((R)P.rs_hi - (R)P.rs_lo);
        bool on_road = fabs(w.y - R(4) * w.lane) <= R(2) && w.x >= -5.0 && w.x < 10005.0;
        R r = (R)P.collision_reward * (w.crashed ? R(1) : R(0)) +
              (R)P.right_lane_reward * ((R)rl / (R)max(P.lanes - 1, 1)) +
              (R)P.high_speed_reward * clipf(scaled, R(0), R(1));
        if (P.normalize_reward)
            r = (r - (R)P.collision_reward) / (((R)P.high_speed_reward + (R)P.right_lane_reward) - (R)P.collision_reward);
        r *= on_road ? R(1) : R(0);
        tnow = P.time[e] + P.dtime;
        bool te = w.crashed || (P.offroad_terminal && !on_road);
        bool tr = tnow >= P.duration;
        reward[e] = (float)r; term[e] = te; trunc[e] = tr;
        done = (te || tr) ? 1 : 0;
    }
    done = __shfl_sync(HRP_FULL, done, 0);
    uint32_t draw = P.obs_draw[e];
    if constexpr (FINAL) {
        // Pass 0, finished envs only: the observation of the terminal state into final_obs, before a respawn overwrites
        // it -- the same publish of the headings and the same shuffle draw as the observation of pass 1, so it is bit
        // for bit what an autoreset = 0 handle returns (in shuffled mode both observations of the step use one row
        // permutation; row_vehicle describes `obs` only).  Pass 1 is the default path below.  A loop rather than a
        // second call: with one call site each, observe_env and spawn_env are compiled as in the default kernel, so
        // both observations round exactly as the default kernel's does.
#pragma unroll 1
        for (int pass = done ? 0 : 1; pass < 2; ++pass) {
            if (pass == 1 && done && P.autoreset) {
                uint32_t ep = P.episode[e] + 1;
                spawn_env(P, S, u, e, lane, ep, xref);
                if (lane == 0) { P.episode[e] = ep; tnow = 0.0; }
            } else {
#pragma unroll
                for (int q = 0; q < 2; ++q)
                    if (lane + 32 * q < P.V) S.h[lane + 32 * q] = u[q].h;
                __syncwarp();
            }
            if (pass == 1 && lane == 0) { P.time[e] = tnow; P.obs_draw[e] = draw + 1; }
            if constexpr (OBS == HRP_OBS_OCCUPANCY_GRID)
                observe_grid(P, G, S, e, lane, pass ? obs : final_obs, pass ? row_vehicle : nullptr);
            else
                observe_env(P, S, e, lane, pass ? obs : final_obs, perm, pass ? row_vehicle : nullptr, draw);
        }
    } else {
        if (done && P.autoreset) {
            uint32_t ep = P.episode[e] + 1;
            spawn_env(P, S, u, e, lane, ep, xref);
            if (lane == 0) { P.episode[e] = ep; tnow = 0.0; }
        } else {
#pragma unroll
            for (int q = 0; q < 2; ++q)
                if (lane + 32 * q < P.V) S.h[lane + 32 * q] = u[q].h;
            __syncwarp();
        }
        if (lane == 0) { P.time[e] = tnow; P.obs_draw[e] = draw + 1; }
        if constexpr (OBS == HRP_OBS_OCCUPANCY_GRID)
            observe_grid(P, G, S, e, lane, obs, row_vehicle);
        else
            observe_env(P, S, e, lane, obs, perm, row_vehicle, draw);
    }
    store_env(P, u, e, lane);
}

// The kernels and launchers below are built twice.  This file on its own is the default translation unit: every
// highway-v0 kernel.  hrp_env_fast.cu includes it with HRP_ENV_FAST_TU defined and gets the highway-fast-v0 step
// kernels instead.  A separate translation unit because the compiler's inlining choices for the shared device
// functions depend on how many kernels call them: kept apart, the default kernels compile exactly as they would without
// the fast ones.
#ifndef HRP_ENV_FAST_TU
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA, HRP_STEP_CTAS_PER_SM)
hrp_step_kernel(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                const int32_t *__restrict__ perm, int32_t *__restrict__ row_vehicle)
{
    step_body<float, HRP_WARPS_PER_CTA>(P, actions, obs, reward, term, trunc, perm, row_vehicle);
}
// validation instantiation: fp64 state and arithmetic (two envs per CTA: the per-warp block is twice as large)
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA_F64)
hrp_step_kernel_f64(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                    float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                    const int32_t *__restrict__ perm, int32_t *__restrict__ row_vehicle)
{
    step_body<double, HRP_WARPS_PER_CTA_F64>(P, actions, obs, reward, term, trunc, perm, row_vehicle);
}
// the same two with the final-observation output: final_obs[E, N, F_out] of the envs whose episode ended on this step
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA, HRP_STEP_CTAS_PER_SM)
hrp_step_kernel_final(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                      float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                      const int32_t *__restrict__ perm, int32_t *__restrict__ row_vehicle, float *__restrict__ final_obs)
{
    step_body<float, HRP_WARPS_PER_CTA, true>(P, actions, obs, reward, term, trunc, perm, row_vehicle, final_obs);
}
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA_F64)
hrp_step_kernel_f64_final(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                          float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                          const int32_t *__restrict__ perm, int32_t *__restrict__ row_vehicle,
                          float *__restrict__ final_obs)
{
    step_body<double, HRP_WARPS_PER_CTA_F64, true>(P, actions, obs, reward, term, trunc, perm, row_vehicle, final_obs);
}
// the OccupancyGrid instantiations of the four: obs[E, F, W, H], row_vehicle[E, W * H] (the vehicle of each cell)
template <bool FINAL>
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA, HRP_STEP_CTAS_PER_SM)
hrp_step_kernel_grid(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                     float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                     int32_t *__restrict__ row_vehicle, float *__restrict__ final_obs, const GridDev G)
{
    step_body<float, HRP_WARPS_PER_CTA, FINAL, HRP_OBS_OCCUPANCY_GRID>(P, actions, obs, reward, term, trunc, nullptr,
                                                                        row_vehicle, final_obs, G);
}
template <bool FINAL>
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA_F64)
hrp_step_kernel_f64_grid(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                         float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                         int32_t *__restrict__ row_vehicle, float *__restrict__ final_obs, const GridDev G)
{
    step_body<double, HRP_WARPS_PER_CTA_F64, FINAL, HRP_OBS_OCCUPANCY_GRID>(P, actions, obs, reward, term, trunc,
                                                                             nullptr, row_vehicle, final_obs, G);
}

template <typename R, int WARPS>
__global__ void __launch_bounds__(32 * WARPS)
hrp_observe_kernel(const EnvDev P, float *__restrict__ obs, const int32_t *__restrict__ perm,
                   int32_t *__restrict__ row_vehicle)
{
    __shared__ WarpS<R> smem[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * WARPS + warp;
    if (e >= P.E) return;
    WarpS<R> &S = smem[warp];
    Veh<R> u[2];
    double xref;
    load_env(P, S, u, e, lane, xref);
    uint32_t draw = P.obs_draw[e];
    observe_env(P, S, e, lane, obs, perm, row_vehicle, draw);
    if (lane == 0) P.obs_draw[e] = draw + 1;
}

template <typename R, int WARPS>
__global__ void __launch_bounds__(32 * WARPS)
hrp_reset_kernel(const EnvDev P, const uint8_t *__restrict__ mask, float *__restrict__ obs)
{
    __shared__ WarpS<R> smem[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * WARPS + warp;
    if (e >= P.E) return;
    if (mask && !mask[e]) return;
    WarpS<R> &S = smem[warp];
    Veh<R> u[2];
    double xref;
    spawn_env(P, S, u, e, lane, 0u, xref);
    uint32_t draw = P.obs_draw[e];
    if (lane == 0) { P.episode[e] = 0; P.time[e] = 0.0; P.obs_draw[e] = draw + 1; }
    if (obs) observe_env(P, S, e, lane, obs, nullptr, nullptr, draw);
    store_env(P, u, e, lane);
}

// the two above with the OccupancyGrid observation (the shuffle counter advances as for Kinematics)
template <typename R, int WARPS>
__global__ void __launch_bounds__(32 * WARPS)
hrp_observe_kernel_grid(const EnvDev P, const GridDev G, float *__restrict__ obs, int32_t *__restrict__ cell_vehicle)
{
    __shared__ WarpS<R> smem[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * WARPS + warp;
    if (e >= P.E) return;
    WarpS<R> &S = smem[warp];
    Veh<R> u[2];
    double xref;
    load_env(P, S, u, e, lane, xref);
    observe_grid(P, G, S, e, lane, obs, cell_vehicle);
    if (lane == 0) P.obs_draw[e] += 1;
}

template <typename R, int WARPS>
__global__ void __launch_bounds__(32 * WARPS)
hrp_reset_kernel_grid(const EnvDev P, const GridDev G, const uint8_t *__restrict__ mask, float *__restrict__ obs)
{
    __shared__ WarpS<R> smem[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * WARPS + warp;
    if (e >= P.E) return;
    if (mask && !mask[e]) return;
    WarpS<R> &S = smem[warp];
    Veh<R> u[2];
    double xref;
    spawn_env(P, S, u, e, lane, 0u, xref);
    if (lane == 0) { P.episode[e] = 0; P.time[e] = 0.0; P.obs_draw[e] += 1; }
    if (obs) observe_grid(P, G, S, e, lane, obs, nullptr);
    store_env(P, u, e, lane);
}

// standalone wrapper.observation() over caller-provided [B, N, F] observations
__global__ void __launch_bounds__(128)
hrp_embed_kernel(int kind, int edim, int use_euclid, int ego_idx, float max_dist,
                 const float *__restrict__ table, const float *__restrict__ obs, float *__restrict__ out,
                 long long batch, int N, int F, int Fout, const float *__restrict__ dist_override)
{
    // the [N, F] table is read straight from global memory (L1-resident, a few KB per warp),
    // so F is not limited by the simulator's HRP_MAX_FEATURES here
    __shared__ float rowd[4][HRP_MAX_OBS_ROWS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    long long b = (long long)blockIdx.x * 4 + warp;
    if (b >= batch) return;
    const float *src = obs + (size_t)b * N * F;
    embed_store(kind, edim, use_euclid, ego_idx, max_dist, table, src, rowd[warp], N, F, Fout, lane,
                out + (size_t)b * N * Fout, dist_override ? dist_override + (size_t)b * N : nullptr);
}

#else
// highway-fast-v0 (hrp_cfg.ego_collisions_only = 1): the eight step kernels of the default translation unit with the
// ego-only collision pass, fp32 / fp64 x with and without final_obs x Kinematics / OccupancyGrid.  One parameter list for all of them (perm is
// NULL for a grid, G unused by Kinematics), so that the launcher picks one from a table.
template <bool FINAL, int OBS>
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA, HRP_STEP_CTAS_PER_SM)
hrp_step_kernel_ego(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                    float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                    const int32_t *__restrict__ perm, int32_t *__restrict__ row_vehicle, float *__restrict__ final_obs,
                    const GridDev G)
{
    step_body<float, HRP_WARPS_PER_CTA, FINAL, OBS, true>(P, actions, obs, reward, term, trunc, perm, row_vehicle,
                                                          final_obs, G);
}
template <bool FINAL, int OBS>
__global__ void __launch_bounds__(32 * HRP_WARPS_PER_CTA_F64)
hrp_step_kernel_f64_ego(const EnvDev P, const float *__restrict__ actions, float *__restrict__ obs,
                        float *__restrict__ reward, uint8_t *__restrict__ term, uint8_t *__restrict__ trunc,
                        const int32_t *__restrict__ perm, int32_t *__restrict__ row_vehicle,
                        float *__restrict__ final_obs, const GridDev G)
{
    step_body<double, HRP_WARPS_PER_CTA_F64, FINAL, OBS, true>(P, actions, obs, reward, term, trunc, perm, row_vehicle,
                                                               final_obs, G);
}
#endif
}  // namespace

#ifndef HRP_ENV_FAST_TU
int hrp_launch_step(const EnvDev &P, const GridDev &G, bool ego_only, const float *actions, float *obs, float *reward,
                    uint8_t *term, uint8_t *trunc, const int32_t *perm, int32_t *row_vehicle, cudaStream_t s,
                    float *final_obs)
{
    if (ego_only)
        return hrp_launch_step_ego(P, G, actions, obs, reward, term, trunc, perm, row_vehicle, s, final_obs);
    if (G.obs_type == HRP_OBS_OCCUPANCY_GRID) {
        const int warps = P.real64 ? HRP_WARPS_PER_CTA_F64 : HRP_WARPS_PER_CTA;
        const dim3 grid((P.E + warps - 1) / warps), block(32 * warps);
        if (P.real64)
            HRP_CUDA_OK(hrp_launch_pdl(final_obs ? hrp_step_kernel_f64_grid<true> : hrp_step_kernel_f64_grid<false>, grid,
                                       block, 0, s, P, actions, obs, reward, term, trunc, row_vehicle, final_obs, G));
        else
            HRP_CUDA_OK(hrp_launch_pdl(final_obs ? hrp_step_kernel_grid<true> : hrp_step_kernel_grid<false>, grid, block,
                                       0, s, P, actions, obs, reward, term, trunc, row_vehicle, final_obs, G));
        return 0;
    }
    if (P.real64) {
        int grid = (P.E + HRP_WARPS_PER_CTA_F64 - 1) / HRP_WARPS_PER_CTA_F64;
        if (final_obs) {
            HRP_CUDA_OK(hrp_launch_pdl(hrp_step_kernel_f64_final, dim3(grid), dim3(32 * HRP_WARPS_PER_CTA_F64), 0, s, P,
                                       actions, obs, reward, term, trunc, perm, row_vehicle, final_obs));
            return 0;
        }
        HRP_CUDA_OK(hrp_launch_pdl(hrp_step_kernel_f64, dim3(grid), dim3(32 * HRP_WARPS_PER_CTA_F64), 0, s, P, actions, obs,
                                   reward, term, trunc, perm, row_vehicle));
        return 0;
    }
    int grid = (P.E + HRP_WARPS_PER_CTA - 1) / HRP_WARPS_PER_CTA;
    if (final_obs) {
        HRP_CUDA_OK(hrp_launch_pdl(hrp_step_kernel_final, dim3(grid), dim3(32 * HRP_WARPS_PER_CTA), 0, s, P, actions, obs,
                                   reward, term, trunc, perm, row_vehicle, final_obs));
        return 0;
    }
    HRP_CUDA_OK(hrp_launch_pdl(hrp_step_kernel, dim3(grid), dim3(32 * HRP_WARPS_PER_CTA), 0, s, P, actions, obs, reward, term,
                               trunc, perm, row_vehicle));
    return 0;
}
int hrp_launch_observe(const EnvDev &P, const GridDev &G, float *obs, const int32_t *perm, int32_t *row_vehicle,
                       cudaStream_t s)
{
    if (G.obs_type == HRP_OBS_OCCUPANCY_GRID) {
        const int warps = P.real64 ? HRP_WARPS_PER_CTA_F64 : HRP_WARPS_PER_CTA;
        const int grid = (P.E + warps - 1) / warps;
        if (P.real64)
            hrp_observe_kernel_grid<double, HRP_WARPS_PER_CTA_F64><<<grid, 32 * warps, 0, s>>>(P, G, obs, row_vehicle);
        else
            hrp_observe_kernel_grid<float, HRP_WARPS_PER_CTA><<<grid, 32 * warps, 0, s>>>(P, G, obs, row_vehicle);
    } else if (P.real64) {
        int grid = (P.E + HRP_WARPS_PER_CTA_F64 - 1) / HRP_WARPS_PER_CTA_F64;
        hrp_observe_kernel<double, HRP_WARPS_PER_CTA_F64><<<grid, 32 * HRP_WARPS_PER_CTA_F64, 0, s>>>(P, obs, perm, row_vehicle);
    } else {
        int grid = (P.E + HRP_WARPS_PER_CTA - 1) / HRP_WARPS_PER_CTA;
        hrp_observe_kernel<float, HRP_WARPS_PER_CTA><<<grid, 32 * HRP_WARPS_PER_CTA, 0, s>>>(P, obs, perm, row_vehicle);
    }
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}
int hrp_launch_reset(const EnvDev &P, const GridDev &G, const uint8_t *mask, float *obs, cudaStream_t s)
{
    if (G.obs_type == HRP_OBS_OCCUPANCY_GRID) {
        const int warps = P.real64 ? HRP_WARPS_PER_CTA_F64 : HRP_WARPS_PER_CTA;
        const int grid = (P.E + warps - 1) / warps;
        if (P.real64)
            hrp_reset_kernel_grid<double, HRP_WARPS_PER_CTA_F64><<<grid, 32 * warps, 0, s>>>(P, G, mask, obs);
        else
            hrp_reset_kernel_grid<float, HRP_WARPS_PER_CTA><<<grid, 32 * warps, 0, s>>>(P, G, mask, obs);
    } else if (P.real64) {
        int grid = (P.E + HRP_WARPS_PER_CTA_F64 - 1) / HRP_WARPS_PER_CTA_F64;
        hrp_reset_kernel<double, HRP_WARPS_PER_CTA_F64><<<grid, 32 * HRP_WARPS_PER_CTA_F64, 0, s>>>(P, mask, obs);
    } else {
        int grid = (P.E + HRP_WARPS_PER_CTA - 1) / HRP_WARPS_PER_CTA;
        hrp_reset_kernel<float, HRP_WARPS_PER_CTA><<<grid, 32 * HRP_WARPS_PER_CTA, 0, s>>>(P, mask, obs);
    }
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}
int hrp_launch_embed(int kind, int embed_dim, int use_euclid, int ego_idx, float max_dist,
                     const float *table, const float *obs, float *out, long long batch, int rows,
                     int cols, const float *dist_override, cudaStream_t s)
{
    int fout = kind == HRP_EMBED_DIST || kind == HRP_EMBED_RANK ? cols + embed_dim : cols;
    unsigned grid = (unsigned)((batch + 3) / 4);
    hrp_embed_kernel<<<grid, 128, 0, s>>>(kind, embed_dim, use_euclid, ego_idx, max_dist, table, obs, out,
                                          batch, rows, cols, fout, dist_override);
    HRP_CUDA_OK(cudaGetLastError());
    return 0;
}
#else
int hrp_launch_step_ego(const EnvDev &P, const GridDev &G, const float *actions, float *obs, float *reward,
                        uint8_t *term, uint8_t *trunc, const int32_t *perm, int32_t *row_vehicle, cudaStream_t s,
                        float *final_obs)
{
    typedef void (*StepKernel)(const EnvDev, const float *, float *, float *, uint8_t *, uint8_t *, const int32_t *,
                               int32_t *, float *, const GridDev);
    static const StepKernel kernels[2][2][2] = {   // [real64][final_obs][grid]
        {{hrp_step_kernel_ego<false, HRP_OBS_KINEMATICS>, hrp_step_kernel_ego<false, HRP_OBS_OCCUPANCY_GRID>},
         {hrp_step_kernel_ego<true, HRP_OBS_KINEMATICS>, hrp_step_kernel_ego<true, HRP_OBS_OCCUPANCY_GRID>}},
        {{hrp_step_kernel_f64_ego<false, HRP_OBS_KINEMATICS>, hrp_step_kernel_f64_ego<false, HRP_OBS_OCCUPANCY_GRID>},
         {hrp_step_kernel_f64_ego<true, HRP_OBS_KINEMATICS>, hrp_step_kernel_f64_ego<true, HRP_OBS_OCCUPANCY_GRID>}}};
    const bool grid = G.obs_type == HRP_OBS_OCCUPANCY_GRID;
    const int warps = P.real64 ? HRP_WARPS_PER_CTA_F64 : HRP_WARPS_PER_CTA;
    HRP_CUDA_OK(hrp_launch_pdl(kernels[P.real64 ? 1 : 0][final_obs ? 1 : 0][grid ? 1 : 0],
                               dim3((P.E + warps - 1) / warps), dim3(32 * warps), 0, s, P, actions, obs, reward,
                               term, trunc, grid ? nullptr : perm, row_vehicle, final_obs, G));
    return 0;
}
#endif
