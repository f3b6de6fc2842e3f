// Per-chain device logic of the grid-based Poisson-thinning loop.
//
// One *team* of TEAM consecutive lanes (TEAM = 1: thread per chain, small d; TEAM = 32: warp per chain)
// owns one chain.  Coordinate i is owned by team lane i % TEAM; x and v live in shared memory as
// per-thread-owned strided arrays (bank-conflict free, no cross-thread hazards), all cross-lane traffic is
// shuffle reductions/scans, and every scalar of the thinning state machine is team-uniform in registers.
//
// Reference behaviour replaced (file:line relative to the reference root):
//   build_bound      state.upper_bound_func: AbstractPDMP.jl:121-136 -> UpperBound.jl:18-36 / 92-137 / 203-247
//   fd derivative    UpperBound.jl:50-76
//   next_event       UpperBound.jl:264-273
//   thinning         SamplingLoopInplace.jl:27-39, 65-217
//   jumps            ZigZagSamplers.jl:101-107, BouncyParticleSamplers.jl:50-74,
//                    ForwardEventChainMonteCarlo.jl:60-113,132-218, BoomerangSamplers.jl:49-67
//   record           Composites.jl:239-260
// Quirks of the reference are kept on purpose (SURVEY.md 8a "gotchas"); each is marked QUIRK below.
#pragma once
#include "common.cuh"
#include "philox.cuh"
#include "potentials.cuh"

namespace pdmpflux {

// Dynamic shared memory of the skeleton kernels.  x, v (and the ZigZag line model A, B) are addressed through
// this symbol with per-thread element offsets so the compiler emits LDS/STS (pointers stored in the Chain object
// degrade to generic loads).
// Layout of one state vector (x, v, ...):
//   TEAM == 1: element (coordinate j, thread) at j * kBlockThreads + thread            (bank-conflict free)
//   TEAM  > 1: chain-contiguous, coordinate i of local chain c at c * dpad + i, i.e. owned coordinate j of team
//              lane tl at c * dpad + tl + j * TEAM.  A chain's x (v) is then one contiguous run of d doubles, which
//              is exactly a skeleton row: it is shipped to HBM by a single TMA bulk copy.
extern __shared__ __align__(128) double g_smem[];
#define XS(j) g_smem[off_x + (j) * kStr]
#define VS(j) g_smem[off_v + (j) * kStr]
#define AS(j) g_smem[off_a + (j) * kStr]
#define BS(j) g_smem[off_b + (j) * kStr]
#define M1S(j) g_smem[off_m1 + (j) * kStr]
#define M2S(j) g_smem[off_m2 + (j) * kStr]
// Sticky Zig-Zag: 1.0 / 0.0 activity flag per coordinate; VU = the velocity the flow, the rates and the bounds see
// (`_active_velocity`, SamplingLoopInplace.jl:13-25: frozen coordinates move with velocity zero)
#define ACS(j) g_smem[off_ac + (j) * kStr]
#define VU(j) (kSticky ? VS(j) * ACS(j) : VS(j))
#define BOX(k) g_smem[off_box + (k) * kBStr]
#define CUM(k) g_smem[off_cum + (k) * kBStr]

// PATH selects how the bound and the rates are evaluated:
//   kPathGeneric   every grid node / Brent iterate makes a pass over the coordinates (any potential, any option)
//   kPathFastBrent affine line model + Brent (grid_size = 0)
//   kPathFastGrid  affine line model + grid bound with analytic derivatives
// The fast paths need Pot::kAffine (constant, decoupled Hessian beyond the first kSpecial coordinates): along
// x + t v every such coordinate rate is A_i + t B_i exactly, so
//   * ZigZag:   rate(t) = sum_i max(0, A_i + t B_i) (+ special coordinates), and on a grid cell the reference's
//               tangent construction max(val_l, val_r, inter, 0) collapses to max(val_l, val_r, 0) because the
//               tangents of an affine function are the function itself (inter lies between val_l and val_r);
//   * BPS/FECMC: <grad U(x_t), v> = a + t b with a = sum A_i, b = sum B_i: one reduction per bound instead of one
//               per grid node;
//   * Boomerang (kSpecial == 0): <P x_t, v_t> = sin cos (pvv - pxx) + (cos^2 - sin^2) pxv.
// Results differ from the generic path (and the oracle) only by floating-point reassociation (~1e-16 relative).
// Thread-per-chain Zig-Zag x Brent ("compressed line model"): capacity of the per-chain register list of coordinates
// whose rate changes sign inside the bound's bracket (see Chain::classify_line)
constexpr int kCrossMax = 12;

// NW (Zig-Zag + kPathFastBrent only) is the line model of common.cuh.  kLineRegs: compile-time capacity of the
// owned-coordinate loops; the line model (A_j, B_j) of the owned coordinates then lives in registers (slots >= n_own
// hold A = B = 0) and the ~40 rate evaluations of a Brent bound touch neither shared memory nor any loop counter.
template <int TEAM, int SAMPLER, int POT, int PATH, int NW = kLineShared>
struct Chain {
    using P = Pot<POT>;
    static constexpr bool kFast = (PATH != kPathGeneric);
    static_assert(NW == kLineShared || NW == kLineTransposed || NW == kLineRegs, "NW is one of the kLine* models");
    static constexpr bool kRegLine = (NW == kLineRegs);
    static constexpr int NWW = kRegLine ? kLineRegs : 1;
    static_assert(NW == kLineShared || (SAMPLER == PDMPFLUX_ZIGZAG && PATH == kPathFastBrent), "NW is a Zig-Zag x Brent option");
    // kLineTransposed: "transposed" team Brent -- every lane of the team keeps the chain's compressed line model and
    // evaluates ONE abscissa of a speculative batch of TEAM Brent iterations (see build_bound_brent)
    static constexpr bool kTeamSpec = (NW == kLineTransposed);
    static_assert(!kTeamSpec || TEAM == 8, "transposed Brent: teams of 8 lanes");
    static constexpr int NS = P::kSpecial;
    static constexpr int K = P::K;
    static constexpr int KK = K > 0 ? K : 1;
    static constexpr bool kRot = (SAMPLER == PDMPFLUX_BOOMERANG);
    static constexpr bool kSticky = (SAMPLER == PDMPFLUX_STICKY_ZIGZAG);
    static constexpr bool kSpeedUp = (SAMPLER == PDMPFLUX_SPEEDUP_ZIGZAG);
    static constexpr bool kZZ = (SAMPLER == PDMPFLUX_ZIGZAG) || kSticky || kSpeedUp;   // StickyZigZagSamplers.jl:69-101: same closures
    static_assert(!kSticky || PATH == kPathGeneric, "Sticky Zig-Zag runs on the generic path");
    static_assert(!kSpeedUp || PATH == kPathGeneric, "Speed-Up Zig-Zag runs on the generic path");
    static constexpr int kBT = block_threads_rt(TEAM, SAMPLER, PATH);   // threads per block
    static constexpr int kStr = (TEAM == 1) ? kBT : TEAM;  // stride between a thread's owned elements
    static constexpr int kBStr = (TEAM == 1) ? kBT : 1;    // stride between a chain's box / cum entries

    const KernelParams& p;
    int off_ac;                      // Sticky Zig-Zag: is_active flags of the owned coordinates (1.0 / 0.0)
    double tt;                       // Sticky Zig-Zag: time to thaw (StickySamplingLoop.jl:43)
    int off_m1, off_m2;              // fused-moment accumulators (owned columns, only when p.accumulate_moments)
    int off_x, off_v, off_a, off_b;  // element offsets into g_smem of this thread's owned columns of x, v, A, B
    double* sc0; // scratch owned vectors (FECMC)
    double* sc1;
    double* sc2;
    int tl, d, nown;
    int nfull;               // owned slots j < nfull belong to a coordinate on every lane; slot nfull only where tl < d - TEAM * nfull
    unsigned mask;
    int64_t chain;

    double Lx[KK], Lv[KK];  // functionals of the current (x, v)
    // fast-path line model of the current (x, v)
    // (ZigZag + Brent keeps the per-owned-coordinate A_j, B_j in shared memory: AS(j), BS(j))
    // Speed-Up Zig-Zag (SpeedUpZigZagSamplers.jl:71-83): scalars of the current (x, v) that determine the closed-form flow
    // y = x - v1 x1 v:  <y,y>, <y,v>, <v,v>, <x,x>, v1 x1, and a, c/d, Y0 + sqrt(Y0^2 + a), sqrt(d) v1 of the reference
    double su_yy, su_yv, su_vv, su_xx, su_vx1, su_v1, su_a, su_cd, su_root, su_rate;
    static constexpr bool kCompressed = (TEAM == 1 || kTeamSpec) && (SAMPLER == PDMPFLUX_ZIGZAG) && (PATH == kPathFastBrent);
    double cl_al, cl_be;      // compressed line model: sum of A_i, B_i over the coordinates that are active on the whole bracket
    int cl_n;                 // ... number of sign-changing coordinates kept in ca / cb (unused slots hold 0); > kCrossMax: not compressed
    double ca[kCompressed ? kCrossMax : 1], cb[kCompressed ? kCrossMax : 1];   // registers: only indexed by unrolled loops
    double ra[NWW], rb[NWW];  // kRegLine: A_j, B_j of the owned coordinates (registers: only indexed by unrolled loops)
    double la, lb;          // BPS/FECMC: a = sum A_i, b = sum B_i over the affine coordinates
    double pxx, pxv, pvv;   // Boomerang: <Px,x>, <Px,v>, <Pv,v>

    // PDMPState scalars (Composites.jl:59-83), team-uniform
    double t, horizon, tp, ts, exp_rv, lambda_bar, ar;
    int eb, rej, hh;
    double eva[5];
    bool accept;
    int status;
    int64_t n_builds, n_rates;

    // BoundBox (Composites.jl:15-20), team-uniform, thread-local storage.  Grid nodes are recomputed on
    // demand from (gc, grem, gh): node k = fma(k, gc, k * grem / (G-1)), last node = gh.
    // box_max / cum_sum live in shared memory, one copy per chain (every lane of a team writes the same values;
    // thread-local arrays would be replicated TEAM times in local memory and spill to DRAM behind the row traffic)
    int off_box, off_cum;
    double step, gc, grem, gh;
    int nb;

    // output staging (see record())
    int off_f;               // TEAM == 1: 2 x 3 carry slots (x, v) in shared memory, slot s at off_f + s * kBT
    int fcnt, fskip;         // row stream: elements carried over / leading phantom slots of the first 32-byte group
    int scnt, sskip;         // scalar columns t / horizon / ar: staged events / leading phantom slots
    double st_t[3], st_h[3], st_a[3];
    bool bulk_pending;

    // draws
    DrawKey key;
    uint32_t sE, sU, sN;
    int64_t pE, pU, pN;
    const double *tE, *tU, *tN;
    bool exhausted;

    __device__ Chain(const KernelParams& p_) : p(p_) {}

    // ------------------------------------------------------------------------------------------------
    // draws: tape (parity mode) or Philox
    // ------------------------------------------------------------------------------------------------
    __device__ double rand_exp() {
        if (p.draw_mode) return draw_exp(key, sE++);
        if (pE >= p.nE) { exhausted = true; return 1.0; }
        return __ldg(tE + pE++);
    }
    __device__ double rand_uniform() {
        if (p.draw_mode) return draw_uniform(key, sU++);
        if (pU >= p.nU) { exhausted = true; return 0.5; }
        return __ldg(tU + pU++);
    }
    // normal number `off` of a block of `count` consecutive normals (call normals_reserve first)
    __device__ double rand_normal_at(int64_t off) {
        if (p.draw_mode) return draw_normal(key, sN + (uint32_t)off);
        return exhausted ? 1.0 : __ldg(tN + pN + off);
    }
    // Normals number 2*i and 2*i+1 of the current block (FECMC orthogonal switch: g1[i], g2[i]) -- one Box-Muller.
    __device__ __forceinline__ void rand_normal_two_at(int64_t i, double& z1, double& z2) {
        if (p.draw_mode && !(sN & 1u)) draw_normal_pair(key, (sN >> 1) + (uint32_t)i, z1, z2);
        else { z1 = rand_normal_at(2 * i); z2 = rand_normal_at(2 * i + 1); }
    }
    // Normals for the owned coordinates j0 and j0+1 (slot = coordinate index) of a block of d normals.  In Philox
    // mode neighbouring lanes (tl, tl^1) own the two halves of the same Box-Muller pair at every j, so the even lane
    // evaluates the pair of row j0, the odd lane the pair of row j0+1, and they swap halves with one shuffle:
    // one Box-Muller per lane per two coordinates instead of two.
    __device__ __forceinline__ void rand_normal_rows(int j0, double& z0, double& z1) {
        if constexpr (TEAM >= 2) {
            if (p.draw_mode && !(sN & 1u)) {
                const int odd = tl & 1;
                const int ie = (tl & ~1) + TEAM * (j0 + odd);  // even coordinate of the pair this lane evaluates
                double ne, no;
                draw_normal_pair(key, (sN >> 1) + (uint32_t)(ie >> 1), ne, no);
                const double recv = __shfl_xor_sync(mask, odd ? ne : no, 1);
                z0 = odd ? recv : ne;
                z1 = odd ? no : recv;
                return;
            }
        }
        if constexpr (TEAM == 1) {
            if (p.draw_mode && !((sN + (uint32_t)j0) & 1u)) {  // rows j0, j0+1 are the two halves of one pair
                draw_normal_pair(key, (sN + (uint32_t)j0) >> 1, z0, z1);
                return;
            }
        }
        // tape mode: lanes that do not own the coordinate must not read it (it may lie beyond the chain's tape)
        z0 = owns(j0) ? rand_normal_at(coord(j0)) : 0.0;
        z1 = owns(j0 + 1) ? rand_normal_at(coord(j0 + 1)) : 0.0;
    }
    // v_j <- N(0,1) for every owned coordinate (BPS / Boomerang refresh); returns the lane's partial sum of squares
    __device__ double refresh_velocity_normals() {
        normals_reserve(d);
        double nn = 0.0;
        int j = 0;
        for (; j + 1 < nown; j += 2) {  // every lane takes part in the shuffle, ownership only gates the store
            double z0, z1;
            rand_normal_rows(j, z0, z1);
            if (owns(j)) { VS(j) = z0; nn += z0 * z0; }
            if (owns(j + 1)) { VS(j + 1) = z1; nn += z1 * z1; }
        }
        if (j < nown && owns(j)) {
            const double z = rand_normal_at(coord(j));
            VS(j) = z; nn += z * z;
        }
        normals_advance(d);
        return nn;
    }

    __device__ void normals_reserve(int64_t count) {
        if (!p.draw_mode && pN + count > p.nN) exhausted = true;
    }
    __device__ void normals_advance(int64_t count) {
        if (p.draw_mode) sN += (uint32_t)count;
        else if (!exhausted) pN += count;
    }

    // ------------------------------------------------------------------------------------------------
    // helpers
    // ------------------------------------------------------------------------------------------------
    __device__ __forceinline__ bool owns(int j) const {
        if constexpr (TEAM == 1) return true;  // nown == d
        else return tl + TEAM * j < d;
    }
    __device__ __forceinline__ int coord(int j) const { return tl + TEAM * j; }
    // coordinate i of this lane's chain, owned or not (TEAM > 1: the chain-contiguous run starts tl elements earlier)
    __device__ __forceinline__ double x_all(int i) const { return TEAM == 1 ? XS(i) : g_smem[off_x - tl + i]; }
    __device__ __forceinline__ double v_all(int i) const { return TEAM == 1 ? VS(i) : g_smem[off_v - tl + i]; }
    // f(j) for every owned slot: an unpredicated main loop over the slots every lane owns, then the ragged last slot
    // (U = unroll factor of the main loop: 4 for light bodies, 1 for bodies that draw normals)
    template <int U = 4, class F>
    __device__ __forceinline__ void for_owned(F&& f) const {
#pragma unroll U
        for (int j = 0; j < nfull; ++j) f(j);
        if (tl < d - TEAM * nfull) f(nfull);
    }

    // functionals of the current x and v (one fused multi-value reduction)
    __device__ void compute_functionals() {
        if constexpr (K > 0) {
            double acc[2 * KK];
#pragma unroll
            for (int k = 0; k < 2 * KK; ++k) acc[k] = 0.0;
            for_owned([&](int j) {
                P::accum(p.pot, coord(j), XS(j), acc);
                P::accum(p.pot, coord(j), VU(j), acc + KK);
            });
            team_sum_n<TEAM, 2 * KK>(acc, mask);
#pragma unroll
            for (int k = 0; k < KK; ++k) { Lx[k] = acc[k]; Lv[k] = acc[KK + k]; }
        }
        if constexpr (kSpeedUp) {  // SpeedUpZigZagSamplers.jl:72-76
            const double x1 = team_bcast<TEAM>(XS(0), 0, mask), v1 = team_bcast<TEAM>(VS(0), 0, mask);  // coordinate 0: lane 0, slot 0
            const double vx1 = v1 * x1;
            double r4[4] = {0.0, 0.0, 0.0, 0.0};
            for_owned([&](int j) {
                const double xj = XS(j), vj = VS(j);
                const double yj = xj - vx1 * vj;          // y = x - v[1] * x[1] * v
                r4[0] += yj * yj; r4[1] += yj * vj; r4[2] += vj * vj; r4[3] += xj * xj;
            });
            team_sum_n<TEAM, 4>(r4, mask);
            su_yy = r4[0]; su_yv = r4[1]; su_vv = r4[2]; su_xx = r4[3];
            su_vx1 = vx1; su_v1 = v1;
            const double dd = (double)d;
            const double c = v1 * su_yv;                              // c = v[1] * (y . v)
            su_a = (1 + su_yy) / dd - (c * c) / (dd * dd);            // a = (1 + y . y) / dim - c^2 / dim^2
            su_cd = c / dd;
            const double Y0 = x1 + su_cd;                             // Y_0 = x[1] + c / dim
            su_root = Y0 + sqrt(Y0 * Y0 + su_a);
            su_rate = sqrt(dd) * v1;
        }
    }

    struct Flow {  // x_t = a x + b v ; v_t = c x + e v
        double a, b, c, e;
        // Speed-Up Zig-Zag: x_t = (x - c v) + b v with c = v1 x1, b = v1 X_1(t); speed sqrt(1 + |x_t|^2) at x_t,
        // d/dt of b (so that dx_t/dt = ds v) and d/dt of the speed
        double sp, ds, dsp;
    };
    __device__ __forceinline__ Flow flow_coef(double tt) const {
        Flow f;
        if constexpr (kSpeedUp) {  // SpeedUpZigZagSamplers.jl:71-79
            const double bt = su_root * exp(su_rate * tt);            // b_t = (Y_0 + sqrt(Y_0^2 + a)) exp(sqrt(dim) v[1] t)
            const double X1 = (bt * bt - su_a) / (2 * bt) - su_cd;    // X_1 = (b_t^2 - a) / (2 b_t) - c / dim
            f.a = 1.0; f.e = 1.0;
            f.c = su_vx1;
            f.b = su_v1 * X1;
            f.sp = sqrt(1.0 + (su_yy + 2.0 * f.b * su_yv + X1 * X1 * su_vv));
            f.ds = su_v1 * su_rate * (bt * bt + su_a) / (2 * bt);     // v1 dX_1/dt
            f.dsp = f.ds * (su_yv + f.b * su_vv) / f.sp;              // <x_t, dx_t/dt> / speed
        } else if constexpr (kRot) {  // BoomerangSamplers.jl:31
            double s, c;
            sincos(tt, &s, &c);
            f.a = c; f.b = s; f.c = -s; f.e = c;
        } else {               // ZigZagSamplers.jl:80 (same for BPS, FECMC)
            f.a = 1.0; f.b = tt; f.c = 0.0; f.e = 1.0;
        }
        return f;
    }
    __device__ __forceinline__ void flow_point(const Flow& f, double xi, double vi, double& xt, double& vt) const {
        if constexpr (kSpeedUp) { xt = (xi - f.c * vi) + f.b * vi; vt = vi; }   // y + v[1] * X_1 * v
        else if constexpr (kRot) { xt = xi * f.a + vi * f.b; vt = xi * f.c + vi * f.e; }
        else { xt = xi + vi * f.b; vt = vi; }
    }
    // effective gradient of the Speed-Up Zig-Zag at a point with speed sp: speed grad U - grad speed (:81-83)
    __device__ __forceinline__ double grad_eff(double g, double xt, double sp) const {
        if constexpr (kSpeedUp) return sp * g - xt / sp;
        else return g;
    }
    __device__ __forceinline__ void flow_functionals(const Flow& f, double* Lxt, double* Lvt) const {
#pragma unroll
        for (int k = 0; k < KK; ++k) {
            if constexpr (kSpeedUp) { Lxt[k] = (Lx[k] - f.c * Lv[k]) + f.b * Lv[k]; Lvt[k] = Lv[k]; }
            else if constexpr (kRot) { Lxt[k] = Lx[k] * f.a + Lv[k] * f.b; Lvt[k] = Lx[k] * f.c + Lv[k] * f.e; }
            else { Lxt[k] = Lx[k] + Lv[k] * f.b; Lvt[k] = Lv[k]; }
        }
    }

    // closed-form int_0^tt x_i(s) ds and int_0^tt x_i(s)^2 ds along the flow from the current (x, v); tt may be
    // negative (time-horizon variant stepping back to T), which subtracts the overshoot
    __device__ void accumulate_segment(double tt, const Flow& f) {
        for_owned([&](int j) {
            const double x = XS(j), v = VU(j);
            if constexpr (kRot) {  // x cos s + v sin s  (f.a = cos tt, f.b = sin tt)
                const double s2t = 2.0 * f.b * f.a;
                M1S(j) += x * f.b + v * (1.0 - f.a);
                M2S(j) += x * x * (0.5 * tt + 0.25 * s2t) + v * v * (0.5 * tt - 0.25 * s2t) + x * v * f.b * f.b;
            } else {
                M1S(j) += tt * (x + 0.5 * v * tt);
                M2S(j) += tt * (x * x + tt * (x * v + v * v * tt * (1.0 / 3.0)));
            }
        });
    }

    __device__ void flow_inplace(double tt) {
        wait_row_stores();  // x / v are about to change: the TMA engine must have read the previous row
        const Flow f = flow_coef(tt);
        if (p.accumulate_moments) accumulate_segment(tt, f);
        for_owned([&](int j) {
            double xt, vt;
            flow_point(f, XS(j), VU(j), xt, vt);
            XS(j) = xt;
            if constexpr (kRot) VS(j) = vt;
        });
    }

    __device__ __forceinline__ double extra_rate() const {
        return SAMPLER == PDMPFLUX_FECMC ? 0.0 : p.refresh_rate;
    }

    // ================================================================================================
    // fast-path line model (PATH != kPathGeneric; linear flow unless Boomerang)
    // ================================================================================================
    // signed coordinate rates of the special (non-affine) leading coordinates at time tt: y_k = g_k(x_t) v_k,
    // dy_k = (H(x_t) v)_k v_k; these only depend on the functionals, so every lane evaluates them.
    __device__ __forceinline__ void special_rates(double tt, double* y, double* dy) const {
        if constexpr (NS > 0) {
            double Lxt[KK];
#pragma unroll
            for (int k = 0; k < KK; ++k) Lxt[k] = Lx[k] + Lv[k] * tt;
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                double g, hv;
                P::eval(p.pot, k, Lxt[k], Lv[k], Lxt, Lv, g, hv);
                y[k] = g * Lv[k];
                dy[k] = hv * Lv[k];
            }
        }
    }

    // Build the line model of the current (x, v); called once per (x, v) change, after compute_functionals().
    __device__ void prepare_line() {
        if constexpr (!kFast) return;
        else if constexpr (kRot) {
            double r3[3] = {0.0, 0.0, 0.0};
            for_owned([&](int j) {
                const double xi = XS(j), vi = VS(j);
                double g, hv;
                P::eval(p.pot, coord(j), xi, vi, Lx, Lv, g, hv);
                r3[0] += g * xi; r3[1] += g * vi; r3[2] += hv * vi;
            });
            team_sum_n<TEAM, 3>(r3, mask);
            pxx = r3[0]; pxv = r3[1]; pvv = r3[2];
        } else if constexpr (kZZ) {
            if constexpr (kRegLine) {
#pragma unroll
                for (int j = 0; j < kLineRegs; ++j) {
                    double A = 0.0, B = 0.0;  // A = B = 0 contributes max(0, 0) = 0 for unowned / special / padding slots
                    if (j < nown && owns(j) && coord(j) >= NS) {
                        const double vi = VS(j);
                        double g, hv;
                        P::eval(p.pot, coord(j), XS(j), vi, Lx, Lv, g, hv);
                        A = g * vi; B = hv * vi;
                    }
                    ra[j] = A; rb[j] = B;
                }
            } else if constexpr (kCompressed) {
                // nothing to store: classify_line() compresses the model per bracket
            } else if constexpr (PATH == kPathFastBrent) {
                for (int j = 0; j < nown; ++j) {
                    double A = 0.0, B = 0.0;  // A = B = 0 contributes max(0, 0) = 0 for unowned / special slots
                    if (owns(j) && coord(j) >= NS) {
                        const double vi = VS(j);
                        double g, hv;
                        P::eval(p.pot, coord(j), XS(j), vi, Lx, Lv, g, hv);
                        A = g * vi; B = hv * vi;
                    }
                    AS(j) = A; BS(j) = B;
                }
            }
        } else {  // BPS / FECMC
            double r2[2] = {0.0, 0.0};
            if constexpr (P::kSplit) {
                // coordinate-local parts only; the functional parts are added from (Lx, Lv) after the reduction --
                // the same sums the pass that writes a new velocity accumulates (accept_bps_fused), bit for bit
                for_owned([&](int j) {
                    const double vi = VS(j);
                    double gl, hl;
                    P::eval_local(p.pot, coord(j), XS(j), vi, gl, hl);
                    r2[0] += gl * vi; r2[1] += hl * vi;
                });
                team_sum_n<TEAM, 2>(r2, mask);
                double ca_, cb_;
                P::line_corr(p.pot, Lx, Lv, ca_, cb_);
                la = r2[0] + ca_; lb = r2[1] + cb_;
            } else {
                for_owned([&](int j) {
                    if (NS == 0 || coord(j) >= NS) {
                        const double vi = VS(j);
                        double g, hv;
                        P::eval(p.pot, coord(j), XS(j), vi, Lx, Lv, g, hv);
                        r2[0] += g * vi; r2[1] += hv * vi;
                    }
                });
                team_sum_n<TEAM, 2>(r2, mask);
                la = r2[0]; lb = r2[1];
            }
        }
    }

    // signed scalar rate <grad U(x_t), v_t> and its d/dt from the line model (BPS / FECMC / Boomerang)
    __device__ __forceinline__ void line_scalar(double tt, double& y, double& dy) const {
        if constexpr (kRot) {
            double s, c;
            sincos(tt, &s, &c);
            const double c2 = c * c - s * s, sc = s * c;
            y = sc * (pvv - pxx) + c2 * pxv;
            dy = c2 * (pvv - pxx) - 4.0 * sc * pxv;  // v_t' H v_t - <grad U(x_t), x_t>
        } else {
            y = la + tt * lb;
            dy = lb;
            if constexpr (NS > 0) {
                double ys[NS], dys[NS];
                special_rates(tt, ys, dys);
#pragma unroll
                for (int k = 0; k < NS; ++k) { y += ys[k]; dy += dys[k]; }
            }
        }
    }

    // rotation flow: signed rate and d/dt from sin / cos of the flow time
    __device__ __forceinline__ void line_scalar_sc(double s, double c, double& y, double& dy) const {
        const double c2 = c * c - s * s, sc = s * c;
        y = sc * (pvv - pxx) + c2 * pxv;
        dy = c2 * (pvv - pxx) - 4.0 * sc * pxv;  // v_t' H v_t - <grad U(x_t), x_t>
    }

    // Compressed line model: does any active lane hold a sign-changing coordinate in slots k0 .. k0+3?  Slots past
    // cl_n hold A = B = 0 and add max(0, 0 + t 0) = +0.0 to accumulators that are already >= +0.0, so a group that
    // no lane uses is skipped without changing a bit (C2 keeps about 6 of the 12 slots).  The vote keeps the branch
    // warp-uniform; a lane whose own slots are empty still runs a group some other lane needs, which adds +0.0.
    // Teams only: the thread-per-chain kernel is issue bound and measured 5 % slower at 65536 chains with the votes.
    __device__ __forceinline__ bool crossing_group_used(int k0) const {
        if constexpr (!kTeamSpec) return true;
        else return __any_sync(__activemask(), k0 < cl_n);
    }

    // `sampler.rate` (always the unsigned rate): ZigZagSamplers.jl:83-86, BouncyParticleSamplers.jl:39-42,
    // ForwardEventChainMonteCarlo.jl:20-23, BoomerangSamplers.jl:38-41.  Uses Lx/Lv of the current (x, v).
    __device__ double rate_unsigned(double tt) {
        if constexpr (kFast && !kZZ) {
            double y, dy;
            line_scalar(tt, y, dy);
            return (y > 0.0 ? y : 0.0) + extra_rate();
        } else if constexpr (kRegLine) {
            // max(0, y) = (y + |y|) / 2 exactly in binary floating point; four accumulators, everything in registers
            double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int j = 0; j < kLineRegs; ++j) {
                const double y = fma(tt, rb[j], ra[j]);
                acc[j & 3] += y + fabs(y);
            }
            double sp_ = 0.0;  // special coordinates: independent of the reduction, evaluated while the shuffles fly
            if constexpr (NS > 0) {
                double ys[NS], dys[NS];
                special_rates(tt, ys, dys);
#pragma unroll
                for (int k = 0; k < NS; ++k) sp_ += ys[k] + fabs(ys[k]);
                sp_ *= 0.5;
            }
            const double s = team_sum<TEAM>((acc[0] + acc[1]) + (acc[2] + acc[3]), mask);
            return fma(0.5, s, sp_);
        } else if constexpr (kCompressed) {
            // sum_i max(0, A_i + t B_i) over the affine coordinates = (al + t be) over the always-active ones
            //                                                       + the few coordinates that change sign in the bracket
            double s = 0.0;
            if (cl_n <= kCrossMax) {
                double c[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
                for (int k = 0; k < kCrossMax; ++k) {   // empty slots are A = B = 0: max(0, 0) = 0
                    if ((k & 3) == 0 && !crossing_group_used(k)) break;
                    const double y = fma(tt, cb[k], ca[k]);
                    c[k & 3] += y + fabs(y);
                }
                s = fma(0.5, (c[0] + c[1]) + (c[2] + c[3]), fma(tt, cl_be, cl_al));
            } else {  // more sign changes than the list holds (rare): every coordinate from (x, v)
                double c0 = 0.0;
                for (int i = NS; i < d; ++i) {
                    const double vi = v_all(i);
                    double g, hv;
                    P::eval(p.pot, i, x_all(i), vi, Lx, Lv, g, hv);
                    const double y = fma(tt, hv * vi, g * vi);
                    c0 += y + fabs(y);
                }
                s = 0.5 * c0;
            }
            if constexpr (NS > 0) {
                double ys[NS], dys[NS];
                special_rates(tt, ys, dys);
                double sp_ = 0.0;
#pragma unroll
                for (int k = 0; k < NS; ++k) sp_ += ys[k] + fabs(ys[k]);
                s = fma(0.5, sp_, s);
            }
            return s;
        } else if constexpr (kZZ && PATH == kPathFastBrent) {
            // max(0, y) = (y + |y|) / 2 exactly in binary floating point: one DADD (|.| is an operand modifier)
            // instead of a compare and two selects; the halving is applied once to the sum.
            double s0 = 0.0, s1 = 0.0;  // two accumulators: shorter dependency chain
            int j = 0;
            for (; j + 1 < nown; j += 2) {
                const double y0 = fma(tt, BS(j), AS(j));
                const double y1 = fma(tt, BS(j + 1), AS(j + 1));
                s0 += y0 + fabs(y0);
                s1 += y1 + fabs(y1);
            }
            if (j < nown) {
                const double y0 = fma(tt, BS(j), AS(j));
                s0 += y0 + fabs(y0);
            }
            s0 = 0.5 * (s0 + s1);
            s1 = 0.0;
            double s = team_sum<TEAM>(s0 + s1, mask);
            if constexpr (NS > 0) {
                double ys[NS], dys[NS];
                special_rates(tt, ys, dys);
#pragma unroll
                for (int k = 0; k < NS; ++k) s += (ys[k] > 0.0 ? ys[k] : 0.0);
            }
            return s;
        } else {
            const Flow f = flow_coef(tt);
            double Lxt[KK], Lvt[KK];
            flow_functionals(f, Lxt, Lvt);
            double s = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    double xt, vt;
                    flow_point(f, XS(j), VU(j), xt, vt);
                    const double y = grad_eff(P::grad(p.pot, coord(j), xt, Lxt), xt, f.sp) * vt;
                    if constexpr (kZZ) s += (y > 0.0 ? y : 0.0);
                    else s += y;
                }
            s = team_sum<TEAM>(s, mask);
            if constexpr (kZZ) return s;
            else return (s > 0.0 ? s : 0.0) + extra_rate();
        }
    }

    // rate_unsigned at B times at once (the speculative Brent batches): the same operations in the same order per time
    // as rate_unsigned(), so the values are bit-identical; the B evaluations are independent instruction streams and
    // their team reductions travel together.
    template <int B>
    __device__ __forceinline__ void rate_unsigned_n(const double (&tt)[B], double (&out)[B]) {
        if constexpr (kRegLine) {
            double acc[B][4];
#pragma unroll
            for (int b = 0; b < B; ++b) acc[b][0] = acc[b][1] = acc[b][2] = acc[b][3] = 0.0;
#pragma unroll
            for (int j = 0; j < kLineRegs; ++j)
#pragma unroll
                for (int b = 0; b < B; ++b) {
                    const double y = fma(tt[b], rb[j], ra[j]);
                    acc[b][j & 3] += y + fabs(y);
                }
            double sp_[B], s[B];
#pragma unroll
            for (int b = 0; b < B; ++b) {
                sp_[b] = 0.0;
                if constexpr (NS > 0) {
                    double ys[NS], dys[NS];
                    special_rates(tt[b], ys, dys);
#pragma unroll
                    for (int k = 0; k < NS; ++k) sp_[b] += ys[k] + fabs(ys[k]);
                    sp_[b] *= 0.5;
                }
                s[b] = (acc[b][0] + acc[b][1]) + (acc[b][2] + acc[b][3]);
            }
            team_sum_n<TEAM, B>(s, mask);
#pragma unroll
            for (int b = 0; b < B; ++b) out[b] = fma(0.5, s[b], sp_[b]);
        } else if constexpr (kCompressed) {
            if (cl_n <= kCrossMax) {
                double c[B][4];
#pragma unroll
                for (int b = 0; b < B; ++b) c[b][0] = c[b][1] = c[b][2] = c[b][3] = 0.0;
#pragma unroll
                for (int k = 0; k < kCrossMax; ++k) {
                    if ((k & 3) == 0 && !crossing_group_used(k)) break;
#pragma unroll
                    for (int b = 0; b < B; ++b) {
                        const double y = fma(tt[b], cb[k], ca[k]);
                        c[b][k & 3] += y + fabs(y);
                    }
                }
#pragma unroll
                for (int b = 0; b < B; ++b) {
                    double s = fma(0.5, (c[b][0] + c[b][1]) + (c[b][2] + c[b][3]), fma(tt[b], cl_be, cl_al));
                    if constexpr (NS > 0) {
                        double ys[NS], dys[NS];
                        special_rates(tt[b], ys, dys);
                        double sp_ = 0.0;
#pragma unroll
                        for (int k = 0; k < NS; ++k) sp_ += ys[k] + fabs(ys[k]);
                        s = fma(0.5, sp_, s);
                    }
                    out[b] = s;
                }
            } else {
#pragma unroll
                for (int b = 0; b < B; ++b) out[b] = rate_unsigned(tt[b]);
            }
        } else {
#pragma unroll
            for (int b = 0; b < B; ++b) out[b] = rate_unsigned(tt[b]);
        }
    }

    // range(0, stop=h, length=G) (UpperBound.jl:94,204): Julia's TwicePrecision range gives ~correctly rounded
    // k*h/(G-1) with the last node == h.  Here: c = h/(G-1) rounded, rem = h - c (G-1) exactly (fma), and
    // node k = fma(k, c, k rem/(G-1)) -- one division per bound, at most 1 ulp from the exact quotient.
    __device__ void make_grid(double h, int G) {
        const double m = (double)(G - 1);
        gc = h / m;
        grem = fma(-gc, m, h) * p.inv_gm1;
        gh = h;
        nb = G;
        step = grid_t(1);  // t[2] - t[1] with t[1] = 0
    }
    __device__ __forceinline__ double grid_t(int k) const {
        if (k >= nb - 1) return gh;
        const double kk = (double)k;
        return fma(kk, gc, kk * grem);
    }

    __device__ static __forceinline__ double clamp_pos(double pos, double stp) {
        if (pos != pos) pos = 0.0;              // replace(NaN => 0.0)
        return fmin(fmax(pos, 0.0), stp);       // clamp.(pos, 0, step)
    }
    // one cell of upper_bound_grid_vect for one coordinate (UpperBound.jl:229-241)
    // QUIRK: the tangent intersection is computed as an ABSOLUTE time, clamped to [0, step] and then used as an
    // OFFSET from the left node.
    __device__ __forceinline__ double vect_cell(double vl, double gl, double vr, double gr, double tl_, double tr_) const {
        double pos = (vl - vr + gr * tr_ - gl * tl_) / (gr - gl);
        pos = clamp_pos(pos, step);
        const double inter = vl + gl * pos;
        return fmax(fmax(fmax(vl, vr), inter), 0.0);
    }
    // one cell of upper_bound_grid (UpperBound.jl:123-131)
    __device__ __forceinline__ double scalar_cell(double vl, double gl, double vr, double gr) const {
        double pos = (vl - vr + gr * step) / (gr - gl);
        pos = clamp_pos(pos, step);
        const double inter = vl + gl * pos;
        // QUIRK: BPS/Boomerang signed bound counts the refresh rate twice (inside the rate and via :131)
        return fmax(fmax(fmax(vl, vr), inter), 0.0) + p.bound_refresh;
    }

    // ---- vectorised (ZigZag) bound: value and d/dt of (signed_)rate_vect for one owned coordinate ----
    __device__ __forceinline__ double vect_value(int i, double xi, double vi, double tt) const {
        double Lxt[KK];
        if constexpr (kSpeedUp) {
            const Flow f = flow_coef(tt);
            double Lvt[KK], xt, vt;
            flow_functionals(f, Lxt, Lvt);
            flow_point(f, xi, vi, xt, vt);
            const double y = grad_eff(P::grad(p.pot, i, xt, Lxt), xt, f.sp) * vi;
            return p.signed_bound ? y : (y > 0.0 ? y : 0.0);
        } else {
#pragma unroll
            for (int k = 0; k < KK; ++k) Lxt[k] = Lx[k] + Lv[k] * tt;
            const double y = P::grad(p.pot, i, xi + vi * tt, Lxt) * vi;
            return p.signed_bound ? y : (y > 0.0 ? y : 0.0);
        }
    }
    // Speed-Up Zig-Zag: value and d/dt of the signed coordinate rate grad U_eff,i(x_t) v_i at the flow point f
    // (what ForwardDiff computes through the closed-form flow): dx_t/dt = ds v, d speed/dt = dsp
    __device__ __forceinline__ void speedup_rate_and_slope(int i, double xi, double vi, const Flow& f, double& y, double& dy) const {
        double Lxt[KK], Lvt[KK], Ld[KK], xt, vt;
        flow_functionals(f, Lxt, Lvt);
        flow_point(f, xi, vi, xt, vt);
#pragma unroll
        for (int k = 0; k < KK; ++k) Ld[k] = f.ds * Lv[k];
        const double di = f.ds * vi;
        double g, hd;
        P::eval(p.pot, i, xt, di, Lxt, Ld, g, hd);
        y = (f.sp * g - xt / f.sp) * vi;
        dy = (f.dsp * g + f.sp * hd - di / f.sp + xt * f.dsp / (f.sp * f.sp)) * vi;
    }
    __device__ __forceinline__ void vect_node(int i, double xi, double vi, double tt, double h, double& val,
                                              double& dval) const {
        if (p.deriv_mode == PDMPFLUX_DERIV_JVP) {
            double y, dy;
            if constexpr (kSpeedUp) speedup_rate_and_slope(i, xi, vi, flow_coef(tt), y, dy);
            else {
                double Lxt[KK];
#pragma unroll
                for (int k = 0; k < KK; ++k) Lxt[k] = Lx[k] + Lv[k] * tt;
                double g, hv;
                P::eval(p.pot, i, xi + vi * tt, vi, Lxt, Lv, g, hv);
                y = g * vi; dy = hv * vi;
            }
            if (p.signed_bound) { val = y; dval = dy; }
            else { val = (y > 0.0 ? y : 0.0); dval = (0.0 > y) ? 0.0 : dy; }
        } else {  // finite_difference_derivative, UpperBound.jl:50-76 with start = 0
            val = vect_value(i, xi, vi, tt);
            const double hh_ = kSqrtEps * fmax(1.0, fabs(tt));
            const double xm = fmax(0.0, tt - hh_), xp = fmin(h, tt + hh_);
            if (xp == xm) dval = val - val;
            else {
                const double fp = (xp == tt) ? val : vect_value(i, xi, vi, xp);
                const double fm = (xm == tt) ? val : vect_value(i, xi, vi, xm);
                dval = (fp - fm) / (xp - xm);
            }
        }
    }

    // upper_bound_grid_vect, UpperBound.jl:203-247 -- affine line model (fast path)
    // Cells are processed in register chunks of kCellsV (= 9: the default grid_size = 10 is exactly one chunk).
    static constexpr int kCellsV = 9;
    template <bool FULL>
    __device__ __forceinline__ void vect_affine_chunk(int nc, const double (&tm_)[kCellsV], const double (&th_)[kCellsV],
                                                      double (&bacc)[kCellsV]) {
#pragma unroll 2
        for (int j = 0; j < nown; ++j)
            if (owns(j)) {
                const int i = coord(j);
                if (i < NS) continue;  // special coordinates are added once, after the reduction
                // affine coordinate: max(val_l, val_r, inter, 0) == max(val_l, val_r, 0); holds for the unsigned
                // variant max(0, .) as well (DESIGN.md "affine cells").  With the cell midpoint tm and half width
                // th: max(val_l, val_r) = A + B tm + |B| th, and max(m, 0) = (m + |m|) / 2 -- four FP64 instructions
                // per (coordinate, cell), no compares or selects.
                const double vi = VS(j);
                double g, hv;
                P::eval(p.pot, i, XS(j), vi, Lx, Lv, g, hv);
                const double A = g * vi, B = hv * vi, aB = fabs(B);
#pragma unroll
                for (int u = 0; u < kCellsV; ++u)
                    if (FULL || u < nc) {
                        const double m = fma(aB, th_[u], fma(B, tm_[u], A));
                        bacc[u] += m + fabs(m);
                    }
            }
    }

    __device__ void build_bound_vect_affine(double h) {
        const int G = p.G;
        make_grid(h, G);
        for (int k0 = 0; k0 < G - 1; k0 += kCellsV) {
            const int nc = min(kCellsV, G - 1 - k0);
            double bacc[kCellsV], tm_[kCellsV], th_[kCellsV];
            double tl_ = grid_t(k0);
#pragma unroll
            for (int u = 0; u < kCellsV; ++u) {
                const double tr_ = grid_t(min(k0 + u + 1, G - 1));
                tm_[u] = 0.5 * (tl_ + tr_); th_[u] = 0.5 * (tr_ - tl_);
                bacc[u] = 0.0;
                tl_ = tr_;
            }
            if (nc == kCellsV) vect_affine_chunk<true>(nc, tm_, th_, bacc);
            else vect_affine_chunk<false>(nc, tm_, th_, bacc);
#pragma unroll
            for (int u = 0; u < kCellsV; ++u) bacc[u] *= 0.5;
            team_sum_n<TEAM, kCellsV>(bacc, mask);
            if constexpr (NS > 0) {  // special coordinates: the reference's cell formula, evaluated by every lane
                double yl[NS], dl[NS];
                special_rates(grid_t(k0), yl, dl);
                for (int u = 0; u < nc; ++u) {
                    double yr[NS], dr[NS];
                    special_rates(grid_t(k0 + u + 1), yr, dr);
                    double add = 0.0;
#pragma unroll
                    for (int k = 0; k < NS; ++k) {
                        double vl = yl[k], gl = dl[k], vr = yr[k], gr = dr[k];
                        if (!p.signed_bound) {
                            gl = (0.0 > vl) ? 0.0 : gl; vl = (vl > 0.0 ? vl : 0.0);
                            gr = (0.0 > vr) ? 0.0 : gr; vr = (vr > 0.0 ? vr : 0.0);
                        }
                        add += vect_cell(vl, gl, vr, gr, grid_t(k0 + u), grid_t(k0 + u + 1));
                        yl[k] = yr[k]; dl[k] = dr[k];
                    }
                    BOX(k0 + u) = add;  // stash; merged below
                }
            }
#pragma unroll
            for (int u = 0; u < kCellsV; ++u)
                if (u < nc) {
                    if constexpr (NS > 0) BOX(k0 + u) += bacc[u];
                    else BOX(k0 + u) = bacc[u];
                }
        }
        double cs = 0.0;
        CUM(0) = 0.0;
        for (int k = 0; k < G - 1; ++k) { cs += BOX(k); CUM(k + 1) = cs * step; }
    }

    // upper_bound_grid_vect, UpperBound.jl:203-247 -- generic path
    __device__ void build_bound_vect(double h) {
        if constexpr (kFast) { build_bound_vect_affine(h); return; }
        const int G = p.G;
        make_grid(h, G);
        for (int k0 = 0; k0 < G - 1; k0 += kChunk) {
            const int nc = min(kChunk, G - 1 - k0);
            double bacc[kChunk], tn[kChunk + 1];
#pragma unroll
            for (int u = 0; u < kChunk; ++u) bacc[u] = 0.0;
#pragma unroll
            for (int u = 0; u <= kChunk; ++u) tn[u] = grid_t(min(k0 + u, G - 1));
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const int i = coord(j);
                    const double xi = XS(j), vi = VU(j);
                    double vl, gl;
                    vect_node(i, xi, vi, tn[0], h, vl, gl);
#pragma unroll
                    for (int u = 0; u < kChunk; ++u)
                        if (u < nc) {
                            double vr, gr;
                            vect_node(i, xi, vi, tn[u + 1], h, vr, gr);
                            bacc[u] += vect_cell(vl, gl, vr, gr, tn[u], tn[u + 1]);
                            vl = vr; gl = gr;
                        }
                }
            team_sum_n<TEAM, kChunk>(bacc, mask);
#pragma unroll
            for (int u = 0; u < kChunk; ++u)
                if (u < nc) BOX(k0 + u) = bacc[u];
        }
        // sum_i cumsum_k(BOX(i,k)) * step  ==  cumsum_k(sum_i BOX(i,k)) * step   (UpperBound.jl:243-246)
        double cs = 0.0;
        CUM(0) = 0.0;
        for (int k = 0; k < G - 1; ++k) { cs += BOX(k); CUM(k + 1) = cs * step; }
    }

    // ---- scalar bound function: `signed_rate` / `rate` (AbstractPDMP.jl:104-112) at n <= kChunk times ----
    // outv[u] = value, outd[u] = analytic d/dt (when want_d)
    __device__ void scalar_nodes(const double* tt, int n, bool want_d, double* outv, double* outd) {
        double av[kChunk], ad[kChunk];
        Flow fl[kChunk];
#pragma unroll
        for (int u = 0; u < kChunk; ++u) {
            av[u] = 0.0; ad[u] = 0.0;
            fl[u] = flow_coef(u < n ? tt[u] : 0.0);
        }
        for (int j = 0; j < nown; ++j)
            if (owns(j)) {
                const int i = coord(j);
                const double xi = XS(j), vi = VU(j);
#pragma unroll
                for (int u = 0; u < kChunk; ++u)
                    if (u < n) {
                        double Lxt[KK], Lvt[KK];
                        flow_functionals(fl[u], Lxt, Lvt);
                        double xt, vt;
                        flow_point(fl[u], xi, vi, xt, vt);
                        if (want_d) {
                            double g, hv, y, dy;
                            if constexpr (kSpeedUp) speedup_rate_and_slope(i, xi, vi, fl[u], y, dy);
                            else {
                            P::eval(p.pot, i, xt, vt, Lxt, Lvt, g, hv);  // dx_t/dt = v_t for both flows
                            y = g * vt;
                            dy = hv * vt;
                            }
                            if constexpr (kRot) dy -= g * xt;              // dv_t/dt = -x_t
                            if constexpr (kZZ) {                           // scalar ZigZag: sum(max.(0, g.*v))
                                av[u] += (y > 0.0 ? y : 0.0);
                                ad[u] += (0.0 > y) ? 0.0 : dy;
                            } else { av[u] += y; ad[u] += dy; }
                        } else {
                            const double y = grad_eff(P::grad(p.pot, i, xt, Lxt), xt, fl[u].sp) * vt;
                            if constexpr (kZZ) av[u] += (y > 0.0 ? y : 0.0);
                            else av[u] += y;
                        }
                    }
            }
        team_sum_n<TEAM, kChunk>(av, mask);
        if (want_d) team_sum_n<TEAM, kChunk>(ad, mask);
#pragma unroll
        for (int u = 0; u < kChunk; ++u)
            if (u < n) {
                if constexpr (kZZ) { outv[u] = av[u]; if (want_d) outd[u] = ad[u]; }
                else finish_scalar(av[u], ad[u], outv[u], outd[u]);
            }
    }
    // signed / unsigned post-processing of <grad U, v> (AbstractPDMP.jl:104-112)
    __device__ __forceinline__ void finish_scalar(double y, double dy, double& val, double& dval) const {
        if (p.signed_bound) { val = y + extra_rate(); dval = dy; }
        else { val = (y > 0.0 ? y : 0.0) + extra_rate(); dval = (0.0 > y) ? 0.0 : dy; }
    }

    // upper_bound_grid, UpperBound.jl:92-137
    __device__ void build_bound_scalar(double h) {
        const int G = p.G;
        make_grid(h, G);
        if constexpr (kFast && !kZZ) {  // O(1) nodes from the line model
            // value and d/dt of the bound function at node time tt: analytic, or the reference's
            // finite_difference_derivative (UpperBound.jl:50-76) applied to the closed-form value
            // (rotation flow: s0 = sin tt, c0 = cos tt are supplied by the caller -- the nodes are equally spaced, so they
            // follow from sin / cos of the grid step by the angle-addition recurrence: ONE sincos per bound instead of one
            // per node.  The recurrence error (~k ulp) is common to a node's value and to its finite-difference stencil,
            // which is built from the same (s0, c0), so it is not amplified by 1 / h.)
            auto node = [&](double tt, double s0, double c0, double& val, double& dval) {
                double y, dy;
                if constexpr (kRot) line_scalar_sc(s0, c0, y, dy);
                else line_scalar(tt, y, dy);
                finish_scalar(y, dy, val, dval);
                if (p.deriv_mode != PDMPFLUX_DERIV_JVP) {
                    const double hh_ = kSqrtEps * fmax(1.0, fabs(tt));
                    const double xm = fmax(0.0, tt - hh_), xp = fmin(h, tt + hh_);
                    // value at a stencil point tn = tt + dh.  Rotation flow: sin / cos(tn) by the angle-addition
                    // formulas with sin(dh) = dh, cos(dh) = 1 - dh^2/2 (exact to double precision for |dh| ~ 1e-8) --
                    // one sincos per grid node instead of three; the quotient keeps its O(sqrt(eps)) noise level.
                    auto at = [&](double tn) -> double {
                        double yy, dd, vv_, du;
                        if constexpr (kRot) {
                            const double dh = tn - tt, ch_ = 1.0 - 0.5 * dh * dh;
                            line_scalar_sc(s0 * ch_ + c0 * dh, c0 * ch_ - s0 * dh, yy, dd);
                        } else line_scalar(tn, yy, dd);
                        finish_scalar(yy, dd, vv_, du);
                        return vv_;
                    };
                    if (xp == xm) dval = val - val;
                    else dval = ((xp != tt ? at(xp) : val) - (xm != tt ? at(xm) : val)) / (xp - xm);
                }
            };
            double vl, gl, cs = 0.0;
            CUM(0) = 0.0;
            if constexpr (!kRot && NS == 0) {
                if (p.deriv_mode == PDMPFLUX_DERIV_JVP) {
                    // <grad U(x + t v), v> = a + t b is affine: both tangents of a cell are the function itself, so the
                    // reference's max(val_l, val_r, inter, 0) is max(val_l, val_r, 0) (same for the unsigned variant) --
                    // no division, no clamping.
                    double d0;
                    finish_scalar(la, lb, vl, d0);
                    for (int k = 0; k < G - 1; ++k) {
                        double vr;
                        finish_scalar(fma(grid_t(k + 1), lb, la), lb, vr, d0);
                        const double m = fmax(vl, vr);
                        const double b = 0.5 * (m + fabs(m)) + p.bound_refresh;
                        BOX(k) = b;
                        cs += b;
                        CUM(k + 1) = cs * step;
                        vl = vr;
                    }
                    return;
                }
            }
            double s1 = 0.0, c1 = 1.0, sk = 0.0, ck = 1.0;
            if constexpr (kRot) sincos(step, &s1, &c1);
            node(0.0, sk, ck, vl, gl);
            for (int k = 0; k < G - 1; ++k) {
                double vr, gr;
                if constexpr (kRot) {
                    const double sn = sk * c1 + ck * s1;
                    ck = ck * c1 - sk * s1;
                    sk = sn;
                }
                node(grid_t(k + 1), sk, ck, vr, gr);
                const double b = scalar_cell(vl, gl, vr, gr);
                BOX(k) = b;
                cs += b;
                CUM(k + 1) = cs * step;
                vl = vr; gl = gr;
            }
            return;
        }
        double vals[kMaxGrid], grads[kMaxGrid];
        const bool jvp = (p.deriv_mode == PDMPFLUX_DERIV_JVP);
        for (int k0 = 0; k0 < G; k0 += kChunk) {
            const int n = min(kChunk, G - k0);
            double tt[kChunk], ov[kChunk], od[kChunk];
#pragma unroll
            for (int u = 0; u < kChunk; ++u) tt[u] = grid_t(min(k0 + u, G - 1));
            scalar_nodes(tt, n, jvp, ov, od);
#pragma unroll
            for (int u = 0; u < kChunk; ++u)
                if (u < n) { vals[k0 + u] = ov[u]; grads[k0 + u] = jvp ? od[u] : 0.0; }
        }
        if (!jvp) {  // finite_difference_derivative, UpperBound.jl:50-76 (start = 0, horizon = h)
            for (int k0 = 0; k0 < G; k0 += kChunk) {
                const int n = min(kChunk, G - k0);
                double tp_[kChunk], tm_[kChunk], fp[kChunk], fm[kChunk], dummy[kChunk];
#pragma unroll
                for (int u = 0; u < kChunk; ++u) {
                    const double tt = grid_t(min(k0 + u, G - 1));
                    const double hh_ = kSqrtEps * fmax(1.0, fabs(tt));
                    tm_[u] = fmax(0.0, tt - hh_);
                    tp_[u] = fmin(h, tt + hh_);
                }
                scalar_nodes(tp_, n, false, fp, dummy);
                scalar_nodes(tm_, n, false, fm, dummy);
#pragma unroll
                for (int u = 0; u < kChunk; ++u)
                    if (u < n) {
                        const double tt = grid_t(k0 + u), fx = vals[k0 + u];
                        if (tp_[u] == tm_[u]) grads[k0 + u] = fx - fx;
                        else {
                            const double a = (tp_[u] == tt) ? fx : fp[u];
                            const double b = (tm_[u] == tt) ? fx : fm[u];
                            grads[k0 + u] = (a - b) / (tp_[u] - tm_[u]);
                        }
                    }
            }
        }
        double cs = 0.0;
        CUM(0) = 0.0;
        for (int k = 0; k < G - 1; ++k) {
            const double b = scalar_cell(vals[k], grads[k], vals[k + 1], grads[k + 1]);
            BOX(k) = b;
            cs += b;
            CUM(k + 1) = cs * step;
        }
    }

    // upper_bound_constant, UpperBound.jl:18-36: Optim.jl Brent on t -> -rate(t) over [0, h]
    //
    // The recurrence is Optim's (restated in SURVEY.md Appendix B); it is written here so that
    //   * every rounding is the reference's: Julia does not contract a*b+c, so the few places where nvcc would fuse
    //     (tol, the parabola numerator, the first abscissa) use __dmul_rn / __dadd_rn, which are never contracted --
    //     with bit-identical rate values the iterates are bit-identical to a CPU evaluation of the same recurrence;
    //   * the bookkeeping at the end of an iteration (bracket, best three points) is a fixed set of selects and the
    //     compound conditions are evaluated without short-circuit branches: lanes of a warp belong to different chains,
    //     so both sides of those tiny branches would be executed anyway, plus the divergence bookkeeping
    //     (BSSY / BSYNC / re-convergence) in the hottest loop of the Brent configurations;
    //   * the parabolic step itself (an IEEE division: 124 cycles of latency on B200, measured) stays behind a real
    //     branch: for the piecewise-linear Zig-Zag rates the maximum sits at an end of [0, h], the parabola through
    //     three collinear points is degenerate and Brent takes golden-section steps only (BASELINE config C2: not one
    //     parabolic step in 2.4e4 iterations), so the warps skip the division altogether.
    // Thread-per-chain Zig-Zag x Brent.  On the bracket [0, h] of one bound every affine coordinate rate A_i + t B_i
    // either stays positive (its max(0, .) is the line itself: summed once into al + t be), stays non-positive
    // (contributes nothing) or changes sign (kept individually).  The ~40 rate evaluations of the Brent recurrence and
    // the thinning evaluations that follow (all at times inside the bracket) then cost one fused multiply-add plus a
    // handful of max(0, .) terms instead of a pass over the d coordinates -- and, with a chain per thread, no
    // cross-lane reduction at all.  Same values as the per-coordinate sum up to reassociation.
    __device__ void classify_line(double h) {
        if constexpr (kTeamSpec) { classify_line_team(h); return; }
        double al = 0.0, be = 0.0;
        int n = 0;
        // The sign-changing coordinates are remembered as 6-bit indices packed into two words (d <= 64 on this path;
        // newest in the low bits, the oldest fall off the end) and their (A, B) are re-evaluated into the register list
        // afterwards with static slot indices.  Pushing (A, B) themselves through the 12-slot register list by
        // shift-insert was 48 register moves per sign change, executed by the whole warp for the two lanes that needed
        // them: 19 % of this kernel's instructions at 2.2 active lanes.
        unsigned long long idx_lo = 0ull;   // entries 0 .. 9
        unsigned idx_hi = 0u;               // entries 10, 11
#pragma unroll 2
        for (int j = NS; j < nown; ++j) {
            const double vi = VS(j);
            double g, hv;
            P::eval(p.pot, j, XS(j), vi, Lx, Lv, g, hv);
            const double A = g * vi, B = hv * vi;
            const double yh = fma(h, B, A);
            const bool p0 = A > 0.0, ph = yh > 0.0;
            if (p0 && ph) { al += A; be += B; }
            else if (p0 || ph) {
                idx_hi = (idx_hi << 6) | (unsigned)(idx_lo >> 54);
                idx_lo = (idx_lo << 6) | (unsigned long long)j;
                ++n;    // more than kCrossMax: the oldest entries fall off the end and rate_unsigned() takes the full pass
            }
        }
#pragma unroll
        for (int k = 0; k < kCrossMax; ++k) {
            const int j = (int)((k < 10 ? (idx_lo >> (6 * (k < 10 ? k : 0))) : (unsigned long long)(idx_hi >> (6 * (k < 10 ? 0 : k - 10)))) & 63ull);
            double A = 0.0, B = 0.0;
            if (k < n) {
                const double vi = VS(j);
                double g, hv;
                P::eval(p.pot, j, XS(j), vi, Lx, Lv, g, hv);
                A = g * vi; B = hv * vi;
            }
            ca[k] = A; cb[k] = B;
        }
        cl_al = al; cl_be = be; cl_n = n;
    }

    // The same classification with the coordinates spread over the lanes of a team: always-active sums by one team
    // reduction, the sign-changing coordinates appended to a per-chain list in shared memory (the slots of the A / B
    // vectors; positions from a ballot) and then read back by every lane into its registers -- afterwards each lane
    // evaluates the chain's rate on its own.
    __device__ void classify_line_team(double h) {
        double ab[2] = {0.0, 0.0};
        // the lane's own coordinates: sums of the always-active ones; the sign-changing ones (seldom more than three
        // of a lane's <= 8) wait in registers for their list positions
        double qa0 = 0.0, qa1 = 0.0, qa2 = 0.0, qb0 = 0.0, qb1 = 0.0, qb2 = 0.0;
        int mine = 0;
        for (int j = 0; j < nown; ++j) {
            if (owns(j) && coord(j) >= NS) {
                const double vi = VS(j);
                double g, hv;
                P::eval(p.pot, coord(j), XS(j), vi, Lx, Lv, g, hv);
                const double A = g * vi, B = hv * vi;
                const bool p0 = A > 0.0, ph = fma(h, B, A) > 0.0;
                if (p0 && ph) { ab[0] += A; ab[1] += B; }
                else if (p0 != ph) {
                    qa2 = qa1; qa1 = qa0; qa0 = A;
                    qb2 = qb1; qb1 = qb0; qb0 = B;
                    ++mine;
                }
            }
        }
        // list positions: exclusive scan of the counts over the lanes (shuffles; see team_ballot about ballots)
        int incl = mine;
#pragma unroll
        for (int o = 1; o < TEAM; o <<= 1) {
            const int up = __shfl_up_sync(mask, incl, o, TEAM);
            if (tl >= o) incl += up;
        }
        const int n = __shfl_sync(mask, incl, TEAM - 1, TEAM);
        const int ia = off_a - tl, ib = off_b - tl;   // the chain's list: slots 0 .. kCrossMax-1 of its A / B vectors
        int pos = incl - mine;
        if (mine <= 3) {
            if (mine > 0 && pos < kCrossMax) { g_smem[ia + pos] = qa0; g_smem[ib + pos] = qb0; }
            if (mine > 1 && pos + 1 < kCrossMax) { g_smem[ia + pos + 1] = qa1; g_smem[ib + pos + 1] = qb1; }
            if (mine > 2 && pos + 2 < kCrossMax) { g_smem[ia + pos + 2] = qa2; g_smem[ib + pos + 2] = qb2; }
        } else {  // more than the registers hold: a second pass over the same coordinates (same operations)
            for (int j = 0; j < nown; ++j) {
                if (owns(j) && coord(j) >= NS) {
                    const double vi = VS(j);
                    double g, hv;
                    P::eval(p.pot, coord(j), XS(j), vi, Lx, Lv, g, hv);
                    const double A = g * vi, B = hv * vi;
                    const bool p0 = A > 0.0, ph = fma(h, B, A) > 0.0;
                    if (p0 != ph) {
                        if (pos < kCrossMax) { g_smem[ia + pos] = A; g_smem[ib + pos] = B; }
                        ++pos;
                    }
                }
            }
        }
        team_sum_n<TEAM, 2>(ab, mask);
        __syncwarp(mask);
        // every lane reads the whole list (unconditional loads: api.cu leaves kCrossMax doubles of slack behind the
        // vectors; slots >= n hold stale values and are replaced by A = B = 0)
#pragma unroll
        for (int k = 0; k < kCrossMax; ++k) {
            const double a_ = g_smem[ia + k], b_ = g_smem[ib + k];
            ca[k] = k < n ? a_ : 0.0;
            cb[k] = k < n ? b_ : 0.0;
        }
        __syncwarp(mask);
        cl_al = ab[0]; cl_be = ab[1]; cl_n = n;
    }

    // Speculative batches.  A golden-section step that finds a new best point (the only kind of step the monotone
    // Zig-Zag rates ever produce on the way to an end of the bracket) moves (lo, hi, x) by a rule that does not involve
    // the function values at all.  So the next kSpecB abscissae are predicted from the bracket alone, the rate is
    // evaluated at all of them at once (independent instruction streams, one set of team reductions), and the
    // iterations are then checked side by side against the values: parabola rejected and f(u) < f(x) at every step.
    // If all hold, the state after kSpecB iterations is exactly what the one-at-a-time recurrence produces -- the same
    // operations on the same operands -- at about a quarter of its dependent latency, which is what bounds the 4096-chain
    // configuration (1.7 warps per scheduler).  If any check fails the same iterations are replayed one at a time
    // (brent_step), reusing the batch's values for as long as the abscissae still agree.
    struct Brent { double lo, hi, x, w, v, fx, fw, fv, stp, old; };
    static constexpr double kGolden = 0.3819660112501051;  // (3 - sqrt(5)) / 2
    static constexpr int kSuper = 5;   // transposed team Brent: iterations per lane per pass
    static constexpr int kSpecB = kRegLine ? 4 : 0;   // measured gain only where the team reduction is the latency (+4..13 %); thread-per-chain kernels are issue bound

    // tolerance, midpoint and golden-section abscissa of the iteration that starts from the bracket (lo, hi) and best x
    __device__ static __forceinline__ double brent_golden(double lo, double hi, double x, double& tol, double& mid,
                                                          double& og, double& gstp) {
        tol = __dadd_rn(__dmul_rn(kSqrtEps, fabs(x)), kEps);
        mid = (hi + lo) * 0.5;                                   // (hi + lo) / 2
        og = (x < mid) ? hi - x : lo - x;
        gstp = kGolden * og;
        return x + ((fabs(gstp) >= tol) ? gstp : ((gstp > 0.0) ? tol : -tol));
    }
    // parabola through (x, fx), (w, fw), (v, fv): does the recurrence take it?  Only considered when |old_step| > tol.
    __device__ static __forceinline__ bool brent_parabola(const Brent& s, double tol, double& pp, double& q) {
        const double xw = s.x - s.w, xv = s.x - s.v;
        const double r = xw * (s.fx - s.fv);
        q = xv * (s.fx - s.fw);
        pp = __dadd_rn(__dmul_rn(xv, q), -__dmul_rn(xw, r));
        q = q - r;
        q = q + q;                                               // 2 (q - r)
        pp = (q > 0.0) ? -pp : pp;
        q = fabs(q);                                             // `if q > 0: p = -p else: q = -q`
        const double hx = s.hi - s.x, xl = s.x - s.lo;
        return (int)(fabs(s.old) > tol) & (int)(fabs(pp) < fabs(q * s.old * 0.5)) & (int)(pp < q * hx) & (int)(pp < q * xl);
    }
    // one iteration; true when the stopping rule fires (state untouched).  With HINT, f(hu) = hf is already known.
    template <bool HINT>
    __device__ __forceinline__ bool brent_step(Brent& s, double hu, double hf) {
        double tol, mid, og, gstp;
        double u = brent_golden(s.lo, s.hi, s.x, tol, mid, og, gstp);
        const double tol2 = tol + tol;
        if (fabs(s.x - mid) <= fma(s.hi - s.lo, -0.5, tol2)) return true;  // 2 tol - (hi - lo) / 2: the halving is exact
        double pp, q;
        const bool use_para = brent_parabola(s, tol, pp, q);
        double new_old = og, new_stp = gstp;
        if (use_para) {                                          // parabolic step (an IEEE division: 124 cycles)
            double sp = pp / q;
            const double xt = s.x + sp;
            const bool near_end = (int)((xt - s.lo) < tol2) | (int)((s.hi - xt) < tol2);
            sp = near_end ? ((s.x < mid) ? tol : -tol) : sp;
            new_old = s.stp; new_stp = sp;
            u = s.x + ((fabs(sp) >= tol) ? sp : ((sp > 0.0) ? tol : -tol));
        }
        s.old = new_old; s.stp = new_stp;
        double fu;
        if (HINT && u == hu) fu = hf;
        else fu = -rate_unsigned(u);
        // bookkeeping.  A new best point shifts (x, w, v) <- (u, x, w); the other outcomes are a fixed set of selects
        // on the values before the update.
        const bool left = u < s.x;
        if (fu < s.fx) {
            s.hi = left ? s.x : s.hi;
            s.lo = left ? s.lo : s.x;
            s.v = s.w; s.fv = s.fw; s.w = s.x; s.fw = s.fx; s.x = u; s.fx = fu;
        } else {
            const bool c1 = (int)(fu <= s.fw) | (int)(s.w == s.x);
            const bool c2 = (int)(fu <= s.fv) | (int)(s.v == s.x) | (int)(s.v == s.w);
            s.lo = left ? u : s.lo;
            s.hi = left ? s.hi : u;
            const bool v_u = !c1 & c2;
            s.v = c1 ? s.w : (v_u ? u : s.v);
            s.fv = c1 ? s.fw : (v_u ? fu : s.fv);
            s.w = c1 ? u : s.w;
            s.fw = c1 ? fu : s.fw;
        }
        return false;
    }

    __device__ void build_bound_brent(double h) {
        if constexpr (kCompressed) classify_line(h);
        Brent s;
        s.lo = 0.0; s.hi = h;
        s.x = __dadd_rn(s.lo, __dmul_rn(kGolden, __dadd_rn(s.hi, -s.lo)));
        s.fx = -rate_unsigned(s.x);
        s.stp = 0.0; s.old = 0.0; s.w = s.x; s.v = s.x; s.fw = s.fx; s.fv = s.fx;
        if constexpr (kTeamSpec) {
            // Transposed passes: lane tl of the team takes iterations tl, tl + TEAM, tl + 2 TEAM, ... of the next
            // kSuper * TEAM iterations -- on BASELINE config C2 a whole bound (36 iterations) is one pass.  While golden
            // steps keep finding a new best point the search walks towards one end E of the bracket: that end stays,
            // the other end becomes the previous best point and x <- x + golden (E - x), whatever the function values
            // are.  Every lane runs this three-operation recurrence through all iterations of the pass, noting the
            // points of its own ones; then it does ITS iterations in full, side by side -- tolerance, stopping rule,
            // golden abscissa, the rate there (the compressed line model is complete in every lane: no reduction), the
            // parabola test with the function values of the three iterations before (fetched from the neighbouring
            // lanes) -- and checks that each is of the assumed kind.  The team's votes decide: the first iteration
            // whose stopping rule fires ends the search, provided every iteration before it is vouched for by its lane.
            // Otherwise TEAM iterations are replayed one at a time and the next pass starts from there.  The operations
            // and operands of every iteration are the one-at-a-time recurrence's, so the result is bit-identical.
            constexpr int S = kSuper;
            auto rot = [&](double v, int j) { return __shfl_sync(mask, v, (tl - j) & (TEAM - 1), TEAM); };
            bool done = false;
            for (int it = 0; it < 1000 && !done;) {
                const bool right = s.x < (s.hi + s.lo) * 0.5;
                const double E = right ? s.hi : s.lo;
                double X[S], W[S], V[S];
                {
                    double mx = s.x, mw = s.w, mv = s.v;
#pragma unroll
                    for (int k = 0; k < TEAM - 1; ++k) {
                        if (k < tl) {
                            const double u = __dadd_rn(mx, __dmul_rn(kGolden, E - mx));
                            mv = mw; mw = mx; mx = u;
                        }
                    }
                    __syncwarp(mask);
                    X[0] = mx; W[0] = mw; V[0] = mv;
#pragma unroll
                    for (int b = 1; b < S; ++b) {
#pragma unroll
                        for (int k = 0; k < TEAM; ++k) {
                            const double u = __dadd_rn(mx, __dmul_rn(kGolden, E - mx));
                            mv = mw; mw = mx; mx = u;
                        }
                        X[b] = mx; W[b] = mw; V[b] = mv;
                    }
                }
                double F[S], TOL[S], U[S];
                unsigned long long stopmask = 0ull, goodmask = 0ull;
                bool asok[S];
#pragma unroll
                for (int b = 0; b < S; ++b) {
                    const bool first = (b == 0) && (tl == 0);
                    const double moving = first ? (right ? s.lo : s.hi) : W[b];
                    const double lo_ = right ? moving : s.lo, hi_ = right ? s.hi : moving;
                    double mid, og, gstp;
                    U[b] = brent_golden(lo_, hi_, X[b], TOL[b], mid, og, gstp);
                    const bool stop = fabs(X[b] - mid) <= fma(hi_ - lo_, -0.5, TOL[b] + TOL[b]);
                    asok[b] = ((X[b] < mid) == right) & (fabs(gstp) >= TOL[b]);
                    stopmask |= (unsigned long long)(stop ? 1u : 0u) << (TEAM * b + tl);   // my bits; merged below
                }
                rate_unsigned_n<S>(U, F);   // the S rates side by side (bit-identical to S calls of rate_unsigned)
#pragma unroll
                for (int b = 0; b < S; ++b) F[b] = -F[b];
                const double ulast = U[S - 1];
                {
                    double r1p = 0.0, r2p = 0.0, r3p = 0.0;   // the rotations of the previous block of TEAM iterations
#pragma unroll
                    for (int b = 0; b < S; ++b) {
                        const double r1 = rot(F[b], 1), r2 = rot(F[b], 2), r3 = rot(F[b], 3);
                        Brent m;
                        if (b == 0) {
                            m.fx = tl >= 1 ? r1 : s.fx;
                            m.fw = tl >= 2 ? r2 : (tl == 1 ? s.fx : s.fw);
                            m.fv = tl >= 3 ? r3 : (tl == 2 ? s.fx : (tl == 1 ? s.fw : s.fv));
                        } else {
                            m.fx = tl >= 1 ? r1 : r1p;
                            m.fw = tl >= 2 ? r2 : r2p;
                            m.fv = tl >= 3 ? r3 : r3p;
                        }
                        r1p = r1; r2p = r2; r3p = r3;
                        const bool first = (b == 0) && (tl == 0);
                        const double moving = first ? (right ? s.lo : s.hi) : W[b];
                        m.lo = right ? moving : s.lo;
                        m.hi = right ? s.hi : moving;
                        m.x = X[b]; m.w = W[b]; m.v = V[b]; m.stp = 0.0;
                        m.old = first ? s.old : E - W[b];
                        double pp, qq;
                        const bool para = brent_parabola(m, TOL[b], pp, qq);
                        const bool good = !para & (F[b] < m.fx) & asok[b];
                        goodmask |= (unsigned long long)(good ? 1u : 0u) << (TEAM * b + tl);
                    }
                }
                stopmask = team_or64<TEAM>(stopmask, mask);
                goodmask = team_or64<TEAM>(goodmask, mask);
                constexpr int N = S * TEAM;
                const int nterm = stopmask ? __ffsll((long long)stopmask) - 1 : N;   // first iteration that stops
                const int nbad = __ffsll((long long)~goodmask) - 1;                   // first iteration not as assumed (>= N: none)
                const int nc = min(nterm, min(nbad, N));                              // iterations 0 .. nc-1 stand
                // value a lane noted for iteration `step` (team-uniform argument)
                auto at = [&](const double (&arr)[S], int step) {
                    const int bb = step / TEAM;
                    double sel = arr[0];
#pragma unroll
                    for (int b = 1; b < S; ++b) sel = (bb == b) ? arr[b] : sel;
                    return team_bcast<TEAM>(sel, step & (TEAM - 1), mask);
                };
                it += nc;
                if (nterm <= nbad && nterm < N) {   // the stopping rule fired: only the best value is needed
                    if (nterm >= 1) s.fx = at(F, nterm - 1);
                    done = true;
                } else {
                    if (nc >= 1) {                  // the state at the start of iteration nc
                        const double xn = (nc < N) ? at(X, min(nc, N - 1)) : team_bcast<TEAM>(ulast, TEAM - 1, mask);
                        const double wn = at(X, nc - 1);
                        const double vn = nc >= 2 ? at(X, nc - 2) : s.w;
                        const double f1 = at(F, nc - 1);
                        const double f2 = nc >= 2 ? at(F, nc - 2) : s.fx;
                        const double f3 = nc >= 3 ? at(F, nc - 3) : (nc == 2 ? s.fx : s.fw);
                        s.x = xn; s.w = wn; s.v = vn; s.fx = f1; s.fw = f2; s.fv = f3;
                        s.lo = right ? wn : s.lo;
                        s.hi = right ? s.hi : wn;
                        s.old = E - wn;
                        s.stp = kGolden * s.old;
                    }
                    if (nc < N) {                   // an iteration of another kind: one at a time for a while
#pragma unroll 1
                        for (int k = 0; k < TEAM && !done; ++k) {
                            done = brent_step<false>(s, 0.0, 0.0);
                            ++it;
                        }
                    }
                }
            }
        } else if constexpr (kSpecB > 0) {
            bool done = false;
            for (int it = 0; it < 1000 && !done;) {
                double U[kSpecB], F[kSpecB];
                {
                    double pl = s.lo, ph = s.hi, px = s.x;
#pragma unroll
                    for (int k = 0; k < kSpecB; ++k) {
                        double tol, mid, og, gstp;
                        const double u = brent_golden(pl, ph, px, tol, mid, og, gstp);
                        U[k] = u;
                        const bool left = u < px;
                        ph = left ? px : ph;
                        pl = left ? pl : px;
                        px = u;
                    }
                }
                rate_unsigned_n<kSpecB>(U, F);
#pragma unroll
                for (int k = 0; k < kSpecB; ++k) F[k] = -F[k];
                Brent q = s;
                bool ok = true, term = false;
                double fterm = s.fx;
                int nsteps = 0;
#pragma unroll
                for (int k = 0; k < kSpecB; ++k) {
                    double tol, mid, og, gstp, pp, qq;
                    const double u = brent_golden(q.lo, q.hi, q.x, tol, mid, og, gstp);  // == U[k]
                    const bool stop = fabs(q.x - mid) <= fma(q.hi - q.lo, -0.5, tol + tol);
                    fterm = (!term && stop) ? q.fx : fterm;
                    term |= stop;
                    const bool para = brent_parabola(q, tol, pp, qq);
                    ok &= term | (!para & (F[k] < q.fx));
                    nsteps += term ? 0 : 1;
                    const bool left = u < q.x;
                    q.hi = left ? q.x : q.hi;
                    q.lo = left ? q.lo : q.x;
                    q.v = q.w; q.fv = q.fw; q.w = q.x; q.fw = q.fx; q.x = u; q.fx = F[k];
                    q.old = og; q.stp = gstp;
                }
                if (ok) {
                    it += nsteps;
                    if (term) { s.fx = fterm; done = true; }
                    else s = q;
                } else {
#pragma unroll 1
                    for (int k = 0; k < kSpecB && !done; ++k) {
                        done = brent_step<true>(s, U[k], F[k]);
                        ++it;
                    }
                }
            }
        } else {
            for (int it = 0; it < 1000; ++it)
                if (brent_step<false>(s, 0.0, 0.0)) break;
        }
        const double fx = s.fx;
        BOX(0) = -fx + 0.0;  // init_state passes no refresh here (AbstractPDMP.jl:122-125)
        CUM(0) = 0.0; CUM(1) = BOX(0) * (h - 0.0);
        step = h - 0.0;
        nb = 2; gh = h; gc = h; grem = 0.0;
    }

    __device__ void build_bound(double h) {
        ++n_builds;
        if constexpr (PATH == kPathFastBrent) build_bound_brent(h);
        else if constexpr (PATH == kPathFastGrid) {
            if constexpr (kZZ) build_bound_vect(h); else build_bound_scalar(h);
        } else {
            if (p.G == 0) build_bound_brent(h);
            else if (kZZ && p.vectorized) build_bound_vect(h);
            else build_bound_scalar(h);
        }
    }

    // next_event, UpperBound.jl:264-273
    __device__ void next_event(double e, double& tp_out, double& lb_out) const {
        // searchsortedfirst(cum_sum, e): cum_sum is non-decreasing (box_max >= 0), so the first index with
        // cum_sum[idx] >= e is the number of entries below e -- counted without a data-dependent loop exit, which
        // would make the lanes of a warp (different chains) leave one by one.
        int idx = 0;
        for (int k = 0; k < nb; ++k) idx += (CUM(k) < e) ? 1 : 0;
        if (idx >= nb) { tp_out = CUDART_INF; lb_out = BOX(nb - 2); return; }
        if (idx == 0) { tp_out = CUDART_NAN; lb_out = BOX(0); return; }  // e <= 0 cannot happen (randexp > 0)
        tp_out = grid_t(idx - 1) + (e - CUM(idx - 1)) / (CUM(idx) - CUM(idx - 1)) * step;
        lb_out = BOX(idx - 1);
    }

    // ------------------------------------------------------------------------------------------------
    // velocity jumps (x already moved; functionals of x are recomputed here)
    // ------------------------------------------------------------------------------------------------
    __device__ void jump_zigzag() {  // ZigZagSamplers.jl:101-107 + Distributions.jl categorical CDF scan
        // lambda_i = max(0, g_i v_i), p = lambda / S, m = first index with cumsum(p)_m > u (else the last index).
        // cumsum(p)_m > u  <=>  cumsum(lambda)_m > u S, so the d divisions are not needed; isprobvec(p) (all p >= 0,
        // sum p ~ 1, else the reference's Categorical constructor throws) holds iff S is finite and positive.
        double S = 0.0;
        const double sp0 = kSpeedUp ? sqrt(1.0 + su_xx) : 1.0;  // speed(x) at the current point (compute_functionals ran on it)
        for (int j = 0; j < nown; ++j)
            if (owns(j)) {
                const double y = grad_eff(P::grad(p.pot, coord(j), XS(j), Lx), XS(j), sp0) * VS(j);
                S += (y > 0.0 ? y : 0.0);
            }
        S = team_sum<TEAM>(S, mask);
        if (!(S > 0.0) || !(S < CUDART_INF)) { status = PDMPFLUX_CHAIN_NOT_PROBVEC; return; }
        const double uS = rand_uniform() * S;
        double carry = 0.0;
        int m = d - 1;
        for (int j = 0; j < nown; ++j) {
            double lj = 0.0;
            if (owns(j)) {
                const double y = grad_eff(P::grad(p.pot, coord(j), XS(j), Lx), XS(j), sp0) * VS(j);
                lj = (y > 0.0 ? y : 0.0);
            }
            const double incl = team_scan_incl<TEAM>(lj, mask, tl) + carry;
            const bool hit = owns(j) && (incl > uS);
            int first = -1;
            if constexpr (TEAM == 1) first = hit ? 0 : -1;
            else {
                const unsigned b = team_ballot<TEAM>(hit, tl, mask);
                first = b ? (__ffs(b) - 1) : -1;
            }
            if (first >= 0) { m = first + TEAM * j; break; }
            carry = team_bcast<TEAM>(incl, TEAM - 1, mask);
        }
        if (m % TEAM == tl) { const int j = m / TEAM; VS(j) = -VS(j); }
    }

    __device__ void jump_bps() {  // BouncyParticleSamplers.jl:50-74
        double r2[2] = {0.0, 0.0};
        for_owned([&](int j) {
            const double g = P::grad(p.pot, coord(j), XS(j), Lx);
            r2[0] += g * VS(j);
            r2[1] += g * g;
        });
        team_sum_n<TEAM, 2>(r2, mask);
        const double gv = r2[0], gg = r2[1];
        const double bounce = (gv > 0.0 ? gv : 0.0);
        const double prob = bounce / (bounce + p.refresh_rate);
        const double u = rand_uniform();
        if (u < prob) {
            if (gg == 0) return;
            const double scale = 2 * gv / gg;
            for_owned([&](int j) {
                const double g = P::grad(p.pot, coord(j), XS(j), Lx);
                VS(j) = VS(j) - scale * g;
            });
        } else {
            double nn = refresh_velocity_normals();
            if (!p.gaussian_velocity) {
                nn = 1.0 / sqrt(team_sum<TEAM>(nn, mask));
                for_owned([&](int j) { VS(j) = VS(j) * nn; });
            }
        }
    }

    // if_accept! for BPS on the affine fast path (SamplingLoopInplace.jl:170-186 + BouncyParticleSamplers.jl:50-74).
    // The literal sequence is six passes over the coordinates per event: flow, functionals of the moved point, gradient
    // and its two inner products, the new velocity, and -- for the next bound -- functionals and the line model again.
    // Here the functionals ride along: those of the moved x with the flow pass, those of the reflected v with the pass
    // that writes it (same summation order as compute_functionals, so the values are bit-identical and everything after
    // an event stays a pure function of the recorded (x, v): resuming from a history column reproduces the run bit for
    // bit).  For `kSplit` potentials the line model (a, b) of the new state is accumulated in that last pass too -- the
    // very sums prepare_line() would form from the stored (x, v') -- so a reflection is three passes and the next bound
    // starts right away (`line_ready`).  Returns true when (Lx, Lv) are the functionals of the new state.
    // `T`: total flow time (deferred horizon moves included).
    __device__ bool accept_bps_fused(double T, bool& line_ready) {
        line_ready = false;
        wait_row_stores();  // x / v are about to change: the TMA engine must have read the previous row
        if (p.accumulate_moments) accumulate_segment(T, flow_coef(T));
        double ax[KK];
#pragma unroll
        for (int k = 0; k < KK; ++k) ax[k] = 0.0;
        for_owned([&](int j) {
            const double xn = XS(j) + VS(j) * T;
            XS(j) = xn;
            if constexpr (K > 0) P::accum(p.pot, coord(j), xn, ax);
        });
        if constexpr (K > 0) {
            team_sum_n<TEAM, KK>(ax, mask);
#pragma unroll
            for (int k = 0; k < KK; ++k) Lx[k] = ax[k];
        }
        double r2[2] = {0.0, 0.0};
        for_owned([&](int j) {
            const double g = P::grad(p.pot, coord(j), XS(j), Lx);
            r2[0] += g * VS(j);
            r2[1] += g * g;
        });
        team_sum_n<TEAM, 2>(r2, mask);
        const double gv = r2[0], gg = r2[1];
        const double bounce = (gv > 0.0 ? gv : 0.0);
        const double prob = bounce / (bounce + p.refresh_rate);
        const double u = rand_uniform();
        if (u < prob) {
            if (gg == 0) return true;   // v unchanged: Lv still valid
            const double scale = 2 * gv / gg;
            if constexpr (P::kSplit) {   // functionals AND line model of the new velocity in the pass that writes it
                double av[KK + 2];
#pragma unroll
                for (int k = 0; k < KK + 2; ++k) av[k] = 0.0;
                for_owned([&](int j) {
                    const double xj = XS(j);
                    const double g = P::grad(p.pot, coord(j), xj, Lx);
                    const double vn = VS(j) - scale * g;
                    VS(j) = vn;
                    double gl, hl;
                    P::eval_local(p.pot, coord(j), xj, vn, gl, hl);
                    av[0] += gl * vn; av[1] += hl * vn;
                    if constexpr (K > 0) P::accum(p.pot, coord(j), vn, av + 2);
                });
                team_sum_n<TEAM, KK + 2>(av, mask);
#pragma unroll
                for (int k = 0; k < KK; ++k) Lv[k] = K > 0 ? av[2 + k] : Lv[k];
                double ca_, cb_;
                P::line_corr(p.pot, Lx, Lv, ca_, cb_);
                la = av[0] + ca_; lb = av[1] + cb_;
                line_ready = true;
                return true;
            }
            double av[KK];
#pragma unroll
            for (int k = 0; k < KK; ++k) av[k] = 0.0;
            for_owned([&](int j) {
                const double g = P::grad(p.pot, coord(j), XS(j), Lx);
                const double vn = VS(j) - scale * g;
                VS(j) = vn;
                if constexpr (K > 0) P::accum(p.pot, coord(j), vn, av);
            });
            if constexpr (K > 0) {
                team_sum_n<TEAM, KK>(av, mask);
#pragma unroll
                for (int k = 0; k < KK; ++k) Lv[k] = av[k];
            }
            return true;
        }
        double nn = refresh_velocity_normals();
        if (!p.gaussian_velocity) {
            nn = 1.0 / sqrt(team_sum<TEAM>(nn, mask));
            for_owned([&](int j) { VS(j) = VS(j) * nn; });
        }
        return false;
    }

    __device__ void jump_boomerang() {  // BoomerangSamplers.jl:49-67
        // QUIRK: the jump uses grad U(x) - x although the rates use grad U (BoomerangSamplers.jl:38-46 vs :51-52)
        double r2[2] = {0.0, 0.0};
        for_owned([&](int j) {
            const double g = P::grad(p.pot, coord(j), XS(j), Lx) - XS(j);
            r2[0] += g * VS(j);
            r2[1] += g * g;
        });
        team_sum_n<TEAM, 2>(r2, mask);
        const double gv = r2[0];
        const double bounce = (gv > 0.0 ? gv : 0.0);
        const double prob = bounce / (bounce + p.refresh_rate);
        const double u = rand_uniform();
        if (u < prob) {
            const double ing = 1.0 / sqrt(r2[1]);
            // <v, e> = <v, g> / |g| (r2[0] is already reduced)
            const double ve = r2[0] * ing;
            for_owned([&](int j) {
                const double e = (P::grad(p.pot, coord(j), XS(j), Lx) - XS(j)) * ing;
                VS(j) = VS(j) - 2 * ve * e;
            });
        } else {  // QUIRK: refresh draws from the global RNG in the reference (:65); on a tape it is the N stream
            refresh_velocity_normals();
        }
    }

    // ForwardEventChainMonteCarlo.jl:132-218 (+ :60-88, :105-113), fused.
    //
    // The reference builds the new velocity through a chain of d-vectors (n, v_o, g1, g2, e1, e2, v_rot, proposal: seven
    // passes over three scratch vectors).  Every one of them lies in span{v, n, z1, z2} (z1, z2 the two rows of the
    // randn(2, d) draw), so the result is  v' = c_v v + c_1 z1 + c_2 z2 + c_n n  with coefficients that depend only on
    // eight inner products.  Here: one pass for |g|^2, <v, g>, |v|^2; one pass that draws z1, z2 and accumulates the
    // eight products; scalar Gram-Schmidt algebra; one pass that writes v'.  z1, z2 are the only vectors kept between
    // passes (two scratch vectors, written once and read once).  Differences from the literal sequence are
    // reassociation only (~1e-15 relative; parity is held at 1e-10).  The degenerate case |v_o| ~ 0 (a redraw of v_o,
    // probability ~0) takes the literal multi-pass path below.
    __device__ void jump_fecmc() {
        const double sf = p.speed_factor;
        const double u = rand_uniform();
        double rho = -sqrt(1 - pow(u, 2.0 / (d - 1)));
        if (sf != 1.0) rho = sf * rho;
        double r3[3] = {0.0, 0.0, 0.0};
        for_owned([&](int j) {
            const double g = P::grad(p.pot, coord(j), XS(j), Lx), vj = VS(j);
            r3[0] += g * g; r3[1] += vj * g; r3[2] += vj * vj;
        });
        team_sum_n<TEAM, 3>(r3, mask);
        const double ng = sqrt(r3[0]);
        const double inv_ng = ng == 0 ? 0.0 : 1.0 / ng;   // n = g / |g| (zero vector if the norm is 0)
        const double vn = r3[1] * inv_ng;                  // <v, n>
        const double nn = ng == 0 ? 0.0 : 1.0;             // <n, n>
        double nvo = r3[2] - vn * vn * nn;                 // |v - <v,n> n|^2
        if (!(nvo > 1e-3 * r3[2])) {                       // cancellation (or the degenerate redraw): literal path
            jump_fecmc_literal(rho);
            return;
        }
        const double u2 = rand_uniform();
        const double rad = (sf != 1.0) ? sqrt(sf * sf - rho * rho) : sqrt(1 - rho * rho);
        if (u2 >= p.mix_p) {  // keep the direction of v_o: v' = v_o / |v_o| sqrt(1 - rho^2) + rho n
            const double sc_ = rad / sqrt(nvo);
            const double cn = (rho - sc_ * vn) * inv_ng;
            for_owned([&](int j) { VS(j) = fma(sc_, VS(j), cn * P::grad(p.pot, coord(j), XS(j), Lx)); });
            return;
        }
        double* __restrict__ z1s = sc0;
        double* __restrict__ z2s = sc1;
        if (p.switch_) {  // _orthogonal_switch; randn(key, 2, dim) is column-major: g1[i] = N[2i], g2[i] = N[2i+1]
            normals_reserve(2 * (int64_t)d);
            double a[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
            for_owned<1>([&](int j) {
                double z1, z2;
                rand_normal_two_at(coord(j), z1, z2);
                z1s[j * kStr] = z1; z2s[j * kStr] = z2;
                const double n = P::grad(p.pot, coord(j), XS(j), Lx) * inv_ng;
                const double vo = fma(-vn, n, VS(j));
                a[0] += z1 * n; a[1] += z2 * n; a[2] += z1 * z1; a[3] += z2 * z2; a[4] += z1 * z2;
                a[5] += vo * z1; a[6] += vo * z2; a[7] += vo * vo;
            });
            normals_advance(2 * (int64_t)d);
            team_sum_n<TEAM, 8>(a, mask);
            nvo = a[7];
            // Gram-Schmidt on (g1, g2) = (z1 - a0 n, z2 - a1 n):  e1 = g1 / N1,  e2 = (g2 - b e1) / N2
            const double N1 = sqrt(a[2] - a[0] * a[0] * nn);
            const double b = (a[4] - a[0] * a[1] * nn) / N1;
            const double N2 = sqrt(a[3] - a[1] * a[1] * nn - b * b);
            const double c1 = a[5] / N1;               // <v_o, e1>   (<v_o, n> = 0)
            const double c2 = (a[6] - b * c1) / N2;    // <v_o, e2>
            double p1 = c2, p2 = c1;                   // swap of the (e1, e2) components
            if (p.ran_p) {
                const double th = rand_uniform() * 2 * 3.14159265358979323846;
                double st, ct;
                sincos(th, &st, &ct);
                p1 = ct * c1 + st * c2; p2 = st * c1 - ct * c2;
            }
            // proposal = v_o + q1 e1 + q2 e2
            const double q1 = p1 - c1, q2 = p2 - c2;
            const double vop = nvo + q1 * c1 + q2 * c2;                              // <v_o, proposal>
            const double pp2 = nvo + 2.0 * (q1 * c1 + q2 * c2) + q1 * q1 + q2 * q2;  // |proposal|^2
            double sgn = 1.0;
            if (p.positive) sgn = (vop > 0) ? 1.0 : ((vop < 0) ? -1.0 : vop);        // sign(0) = 0, sign(NaN) = NaN
            const double sc_ = sgn * rad / sqrt(pp2 * (sgn * sgn));                  // sign(0) = 0 -> NaN as in the reference
            const double gam = q2 / N2, bet = (q1 - gam * b) / N1;
            const double cz1 = sc_ * bet, cz2 = sc_ * gam;
            const double cn = (rho - sc_ * (bet * a[0] + gam * a[1]) - sc_ * vn) * inv_ng;
            for_owned([&](int j) {
                const double g = P::grad(p.pot, coord(j), XS(j), Lx);
                VS(j) = fma(sc_, VS(j), fma(cz1, z1s[j * kStr], fma(cz2, z2s[j * kStr], cn * g)));
            });
        } else {  // _full_refresh: w = z / |z|, proposal = w - <w, n> n, v' = proposal rad / |proposal| + rho n
            normals_reserve(d);
            double a[2] = {0.0, 0.0};
            for_owned<1>([&](int j) {
                const double z = rand_normal_at(coord(j));
                z1s[j * kStr] = z;
                a[0] += z * (P::grad(p.pot, coord(j), XS(j), Lx) * inv_ng);
                a[1] += z * z;
            });
            normals_advance(d);
            team_sum_n<TEAM, 2>(a, mask);
            const double k = rad / sqrt(a[1] - a[0] * a[0] * nn);
            const double cn = (rho - k * a[0]) * inv_ng;
            for_owned([&](int j) { VS(j) = fma(k, z1s[j * kStr], cn * P::grad(p.pot, coord(j), XS(j), Lx)); });
        }
    }

    // the reference's sequence of vector operations, pass by pass (used for the degenerate / ill-conditioned case)
    __device__ void jump_fecmc_literal(double rho) {
        const double sf = p.speed_factor;
        double* __restrict__ vo = sc0;
        // n = grad U(x) / |grad U(x)| (zero vector if the norm is 0)
        double r2[2] = {0.0, 0.0};
        for (int j = 0; j < nown; ++j)
            if (owns(j)) {
                const double g = P::grad(p.pot, coord(j), XS(j), Lx);
                r2[0] += g * g;
            }
        const double ng = sqrt(team_sum<TEAM>(r2[0], mask));
        // n_i = g_i / |g|: multiplied by the reciprocal (1 ulp from the reference's division, 25x cheaper)
        const double inv_ng = ng == 0 ? 0.0 : 1.0 / ng;
        auto nvec = [&](int j) -> double { return P::grad(p.pot, coord(j), XS(j), Lx) * inv_ng; };
        double vn = 0.0;
        for (int j = 0; j < nown; ++j)
            if (owns(j)) vn += VS(j) * nvec(j);
        vn = team_sum<TEAM>(vn, mask);
        double nvo = 0.0;
        for (int j = 0; j < nown; ++j)
            if (owns(j)) {
                const double o = VS(j) - vn * nvec(j);
                vo[j * kStr] = o;
                nvo += o * o;
            }
        nvo = team_sum<TEAM>(nvo, mask);
        if (sqrt(nvo) < 1e-10) {  // degenerate orthogonal part: redraw
            normals_reserve(d);
            double a = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double z = rand_normal_at(coord(j));
                    vo[j * kStr] = z;
                    a += z * nvec(j);
                }
            normals_advance(d);
            a = team_sum<TEAM>(a, mask);
            nvo = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double o = vo[j * kStr] - a * nvec(j);
                    vo[j * kStr] = o;
                    nvo += o * o;
                }
            nvo = team_sum<TEAM>(nvo, mask);
        }
        const double u2 = rand_uniform();
        const double rad = (sf != 1.0) ? sqrt(sf * sf - rho * rho) : sqrt(1 - rho * rho);
        if (u2 >= p.mix_p) {
            const double sc_ = rad / sqrt(nvo);
            for (int j = 0; j < nown; ++j)
                if (owns(j)) VS(j) = vo[j * kStr] * sc_ + rho * nvec(j);
            return;
        }
        double* __restrict__ prop = sc1;
        if (p.switch_) {  // _orthogonal_switch; randn(key, 2, dim) is column-major: g1[i] = N[2i], g2[i] = N[2i+1]
            double* e1 = sc1;
            double* __restrict__ e2 = sc2;
            normals_reserve(2 * (int64_t)d);
            double a[2] = {0.0, 0.0};
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    double z1, z2;
                    rand_normal_two_at(coord(j), z1, z2);
                    e1[j * kStr] = z1; e2[j * kStr] = z2;
                    const double n = nvec(j);
                    a[0] += z1 * n; a[1] += z2 * n;
                }
            normals_advance(2 * (int64_t)d);
            team_sum_n<TEAM, 2>(a, mask);
            double n1 = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double n = nvec(j);
                    const double g1 = e1[j * kStr] - a[0] * n;
                    e1[j * kStr] = g1;
                    e2[j * kStr] = e2[j * kStr] - a[1] * n;
                    n1 += g1 * g1;
                }
            n1 = 1.0 / sqrt(team_sum<TEAM>(n1, mask));
            double b = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double q = e1[j * kStr] * n1;
                    e1[j * kStr] = q;
                    b += e2[j * kStr] * q;
                }
            b = team_sum<TEAM>(b, mask);
            double n2 = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double q = e2[j * kStr] - b * e1[j * kStr];
                    e2[j * kStr] = q;
                    n2 += q * q;
                }
            n2 = 1.0 / sqrt(team_sum<TEAM>(n2, mask));
            double c[2] = {0.0, 0.0};
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double q = e2[j * kStr] * n2;
                    e2[j * kStr] = q;
                    c[0] += vo[j * kStr] * e1[j * kStr];
                    c[1] += vo[j * kStr] * q;
                }
            team_sum_n<TEAM, 2>(c, mask);
            double ct = 0.0, st = 0.0;
            if (p.ran_p) {
                const double th = rand_uniform() * 2 * 3.14159265358979323846;
                sincos(th, &st, &ct);
            }
            double r3[2] = {0.0, 0.0};  // <vo, prop>, <prop, prop>
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double q1 = e1[j * kStr], q2 = e2[j * kStr], o = vo[j * kStr];
                    const double vr = o - c[0] * q1 - c[1] * q2;
                    double pr;
                    if (p.ran_p) pr = vr + (ct * q1 + st * q2) * c[0] + (st * q1 - ct * q2) * c[1];
                    else pr = vr + q2 * c[0] + q1 * c[1];
                    prop[j * kStr] = pr;  // prop aliases e1: e1[j] is dead from here on
                    r3[0] += o * pr;
                    r3[1] += pr * pr;
                }
            team_sum_n<TEAM, 2>(r3, mask);
            double sgn = 1.0;
            if (p.positive) sgn = (r3[0] > 0) ? 1.0 : ((r3[0] < 0) ? -1.0 : r3[0]);  // sign(0)=0, sign(NaN)=NaN
            const double sc_ = sgn * rad / sqrt(r3[1] * (sgn * sgn));  // sign(0) = 0 -> 0/0 = NaN as in the reference
            for (int j = 0; j < nown; ++j)
                if (owns(j)) VS(j) = prop[j * kStr] * sc_ + rho * nvec(j);
        } else {  // _full_refresh
            normals_reserve(d);
            double nw = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double z = rand_normal_at(coord(j));
                    prop[j * kStr] = z;
                    nw += z * z;
                }
            normals_advance(d);
            nw = 1.0 / sqrt(team_sum<TEAM>(nw, mask));
            double a = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double q = prop[j * kStr] * nw;
                    prop[j * kStr] = q;
                    a += q * nvec(j);
                }
            a = team_sum<TEAM>(a, mask);
            double np_ = 0.0;
            for (int j = 0; j < nown; ++j)
                if (owns(j)) {
                    const double q = prop[j * kStr] - a * nvec(j);
                    prop[j * kStr] = q;
                    np_ += q * q;
                }
            np_ = rad / sqrt(team_sum<TEAM>(np_, mask));
            for (int j = 0; j < nown; ++j)
                if (owns(j)) VS(j) = prop[j * kStr] * np_ + rho * nvec(j);
        }
    }

    // if_accept! for ZigZag with a linear flow, fused into one pass over the coordinates:
    //   x <- x + tp v (flow), lambda_i = max(0, g_i(x) v_i) at the new x, categorical draw, flip.
    // `S` = sum lambda_i is exactly the rate just evaluated at tp for the accept test (same point, same formula), and
    // the functionals of the new x follow from linearity (L(x + tp v) = L(x) + tp L(v)), so the reference's separate
    // passes (flow, grad, sum, cdf scan: ZigZagSamplers.jl:80, :101-107) collapse into this loop.  S > 0 is implied
    // by the acceptance (u < S / lambda_bar), hence Categorical's isprobvec check cannot fail here.
    __device__ void accept_zigzag(double tt, double S) {
        wait_row_stores();
        if (p.accumulate_moments) accumulate_segment(tt, flow_coef(tt));
        double Lxn[KK];
#pragma unroll
        for (int k = 0; k < KK; ++k) Lxn[k] = Lx[k] + Lv[k] * tt;
        const double uS = rand_uniform() * S;
        if constexpr (TEAM == 1) {
            double cum = 0.0;
            int m = d - 1;
            bool found = false;
            for (int j = 0; j < nown; ++j) {
                const double vi = VS(j);
                const double xn = XS(j) + vi * tt;
                XS(j) = xn;
                const double y = P::grad(p.pot, j, xn, Lxn) * vi;
                cum += (y > 0.0 ? y : 0.0);
                if (!found && cum > uS) { m = j; found = true; }
            }
            VS(m) = -VS(m);
        } else {
            // The categorical scan runs over the coordinates in order.  With the strided ownership of the other passes
            // that is one team-wide scan per owned row (n_own serial scans); here the team instead splits the chain's
            // contiguous shared-memory row into TEAM blocks of n_own consecutive coordinates: a serial pass inside the
            // lane, ONE scan over the lanes' block totals, and a short search inside the block that holds the index.
            __syncwarp(mask);  // x / v written under the strided ownership are visible to the whole team
            const int cbx = off_x - tl, cbv = off_v - tl;  // element offset of the chain's coordinate 0
            const int i0 = tl * nown, i1 = min(d, i0 + nown);
            double tot = 0.0;
            for (int i = i0; i < i1; ++i) {
                const double vi = g_smem[cbv + i];
                const double xn = g_smem[cbx + i] + vi * tt;
                g_smem[cbx + i] = xn;
                const double y = P::grad(p.pot, i, xn, Lxn) * vi;
                tot += (y > 0.0 ? y : 0.0);
            }
            const double incl = team_scan_incl<TEAM>(tot, mask, tl);
            double excl = __shfl_up_sync(mask, incl, 1, TEAM);
            if (tl == 0) excl = 0.0;
            const unsigned b = team_ballot<TEAM>((i0 < i1) && (incl > uS), tl, mask);
            const int first = b ? (__ffs(b) - 1) : -1;
            if (first < 0) {  // rounding left the total below u S: the reference's scan ends on the last index
                if (tl == (d - 1) / nown) g_smem[cbv + d - 1] = -g_smem[cbv + d - 1];
            } else if (tl == first) {
                double cum = excl;
                int m = i1 - 1;
                for (int i = i0; i < i1; ++i) {
                    const double y = P::grad(p.pot, i, g_smem[cbx + i], Lxn) * g_smem[cbv + i];
                    cum += (y > 0.0 ? y : 0.0);
                    if (cum > uS) { m = i; break; }
                }
                g_smem[cbv + m] = -g_smem[cbv + m];
            }
            __syncwarp(mask);
        }
    }

    __device__ void velocity_jump() {
        // functionals of the moved x (v's are refreshed by the next compute_functionals before a bound build)
        compute_functionals();
        if constexpr (kZZ) jump_zigzag();   // Sticky: the jump sees the FULL velocity, frozen coordinates included
                                            // (QUIRK: if_accept! passes state.v, SamplingLoopInplace.jl:178)
        else if constexpr (SAMPLER == PDMPFLUX_BPS) jump_bps();
        else if constexpr (SAMPLER == PDMPFLUX_FECMC) jump_fecmc();
        else jump_boomerang();
    }

    // ------------------------------------------------------------------------------------------------
    // thinning state machine: SamplingLoopInplace.jl, flattened
    // ------------------------------------------------------------------------------------------------
    // The reference nests three loops (events -> `while !accept` one_step_of_thinning! -> `while tp < horizon`
    // ac_step!).  Lanes of a warp that own different chains need different trip counts (extra bound builds after
    // horizon hits, extra proposals after rejections), and nested loops would make every chain wait for the
    // slowest one at every loop exit.  Here the nest is flattened into one loop whose body is
    //   [bound build + first proposal, if this chain needs one]  then  [one accept/reject step, if it has a proposal]
    // so a chain that finished its event immediately starts the next one.  The sequence of operations per chain
    // (and hence the draw order) is exactly the reference's.
    __device__ void begin_event(int64_t ev) {  // get_event_state!, :28-31
        eb = 0; rej = 0; hh = 0;
#pragma unroll
        for (int k = 0; k < 5; ++k) eva[k] = 0.0;
        key.event = (uint32_t)(p.event0 + ev + 1);
        sE = sU = sN = 0;
    }

    __device__ int64_t run_events(int64_t c, bool valid) {  // returns the number of events recorded
        int64_t ev = 0;
        int steps = 0;
        bool need_build = true, half = false;
        // BPS / ForwardECMC on the affine fast path: a horizon move changes neither v nor the line's slope, so the line
        // model (and the functionals) of the moved point follow in O(1) -- a <- a + h b -- and the move itself is
        // deferred: x stays at the last event until the next event (or the end of the launch) flows it by the summed
        // time.  0.7 horizon moves per event on BASELINE config C3, each formerly a flow pass, a functionals pass and a
        // line-model pass over the coordinates.  Same path, one rounding instead of one per move (~1e-16 relative).
        constexpr bool kDefer = kFast && !kRot && !kZZ;
        double pend = 0.0;        // flow time not yet applied to x
        bool line_valid = false;  // (la, lb, Lx) already describe the point x + pend v
        bool funcs_valid = false; // (Lx, Lv) are the functionals of the current (x, v) (computed along with the jump)
        auto horizon_move = [&](double h) {
            if constexpr (kDefer) {
                pend += h;
                la = fma(h, lb, la);
#pragma unroll
                for (int k = 0; k < KK; ++k) Lx[k] = fma(h, Lv[k], Lx[k]);
                line_valid = true;
            } else flow_inplace(h);
        };
        accept = false;
        begin_event(0);
        // time-horizon variant: `while state.t < T` (src/sample.jl:360)
        if (p.use_t_stop && status == 0 && !(t < p.t_stop)) status = PDMPFLUX_CHAIN_DONE;
        bool live = valid && status == 0 && p.n_events > 0;
        // Every lane of the warp stays in this loop until the whole warp is done; the warp-wide vote at the loop
        // head is the reconvergence point of each iteration, and both blocks of the body are plain ifs, so the
        // lanes that build a bound do it together and the lanes that have a proposal test it together.
        while (__any_sync(0xffffffffu, live)) {
            if (live && need_build) {
                if (++steps > p.max_steps) { status = PDMPFLUX_CHAIN_STEP_LIMIT; live = false; }
                else {
                    double h = horizon;
                    if (!half) {  // one_step_of_thinning!, :65-85
                        if (!(kDefer && line_valid)) {
                            if (!(kDefer && funcs_valid)) compute_functionals();
                            prepare_line();
                        }
                        funcs_valid = false;
                    } else h = horizon / 2;  // erroneous_acceptance_rate!, :131-151 (same x, v: line model still valid)
                    build_bound(h);
                    const double e = rand_exp();
                    next_event(e, tp, lambda_bar);
                    exp_rv = e;
                    if (exhausted) { status = PDMPFLUX_CHAIN_TAPE_EXHAUSTED; live = false; }
                    else if (half) {
                        // QUIRK: a non-adaptive chain keeps the full horizon although the live bound covers half of it
                        horizon = p.adaptive ? h : horizon;
                        eb += 1;
                        {   // error_value_ar[errored_bound % 5 + 1] = ar, without dynamic indexing (keeps the state in registers)
                            const int slot = eb % 5;
#pragma unroll
                            for (int k = 0; k < 5; ++k)
                                if (k == slot) eva[k] = ar;
                        }
                        half = false;
                        need_build = false;  // back in moves_until_horizon!; a proposal beyond the horizon restarts below
                    } else if (tp > horizon) {  // move_to_horizon!, :87-101 (need_build stays set)
                        horizon_move(horizon);
                        ts += horizon;
                        hh += 1;
                        horizon = p.adaptive ? horizon * 1.01 : horizon;
                    } else need_build = false;
                }
            }
            if (live && !need_build) {
                // moves_until_horizon!, :103-111: `while tp < horizon && !accept` -- otherwise a fresh outer step
                if (!(tp < horizon)) need_build = true;
                else {
                    // ac_step!, :113-129
                    ++n_rates;
                    const double lt = rate_unsigned(tp);
                    ar = lt / lambda_bar;
                    if (ar > 1.0) { need_build = true; half = true; }
                    else if (rand_uniform() < ar) {  // ac_step_with_proxy!, :153-168 -> if_accept!, :170-186
                        if (p.use_t_stop && t + tp + ts > p.t_stop) {
                            // The event falls beyond T: the skeleton ends with the point at exactly t = T reached by
                            // the deterministic flow, with zeroed event statistics (src/sample.jl:385-420).  The
                            // state is at time t + ts here, so the remaining flow time may be negative when horizon
                            // moves already carried it past T (the flows are groups: same point as flowing the
                            // pre-event state by T - t).
                            flow_inplace(p.t_stop - (t + ts) + pend);
                            pend = 0.0; line_valid = false;
                            t = p.t_stop;
                            ar = 0.0; eb = 0; rej = 0; hh = 0;
#pragma unroll
                            for (int k = 0; k < 5; ++k) eva[k] = 0.0;
                            record(c, p.col0 + ev);
                            ++ev;
                            status = PDMPFLUX_CHAIN_DONE;
                            live = false;
                        } else {
                        if constexpr (kZZ && !kSticky && !kSpeedUp) accept_zigzag(tp, lt);
                        else if constexpr (kDefer && SAMPLER == PDMPFLUX_BPS) {
                            funcs_valid = accept_bps_fused(tp + pend, line_valid);
                            pend = 0.0;
                        } else {
                            flow_inplace(tp + pend);
                            pend = 0.0; line_valid = false;
                            velocity_jump();
                        }
                        t = t + tp + ts;
                        ts = 0.0;
                        tp = 0.0;
                        if (exhausted) { status = PDMPFLUX_CHAIN_TAPE_EXHAUSTED; live = false; }
                        else if (status != 0) live = false;
                        else {
                            record(c, p.col0 + ev);
                            ++ev;
                            steps = 0;
                            begin_event(ev);
                            need_build = true;
                            live = ev < p.n_events;
                            if (p.use_t_stop && !(t < p.t_stop)) { status = PDMPFLUX_CHAIN_DONE; live = false; }
                        }
                        }
                    } else {  // if_reject!, :188-203
                        const double e3 = exp_rv + rand_exp();
                        next_event(e3, tp, lambda_bar);
                        horizon = p.adaptive ? horizon / 1.04 : horizon;  // QUIRK: shrink before the horizon check
                        exp_rv = e3;
                        rej += 1;
                        if (exhausted) { status = PDMPFLUX_CHAIN_TAPE_EXHAUSTED; live = false; }
                        else if (tp > horizon) {  // move_to_horizon2!, :205-217 (no horizon growth here)
                            horizon_move(horizon);
                            ts += horizon;
                            hh += 1;
                            need_build = true;
                        }
                    }
                }
            }
        }
        if constexpr (kDefer) {
            if (pend != 0.0) flow_inplace(pend);  // a chain stopped inside an event: its stored state is the moved point
        }
        return ev;
    }

    // ------------------------------------------------------------------------------------------------
    // Sticky Zig-Zag: get_event_state!(state, ::StickyPDMP) (SamplingLoopInplace.jl:49-63) and its loop body
    // (StickySamplingLoop.jl:30-164), with the masked variants of the shared steps (SamplingLoopInplace.jl:87-217).
    // Every accepted flip, every sticking and every thawing is a skeleton point.  Written with the reference's own
    // nesting (this is the row after the hot path: parity first).  Quirks kept: the velocity jump after an accepted
    // event sees the full velocity, frozen coordinates included; thawing adds tt but not the time already spent in
    // horizon moves (ts) to the clock (:160-161); axis crossings are only looked for at the start of an outer step
    // (:52-60) and the time to the axis is -x_j v_j (|v_j| = 1 is assumed, :81-83).
    // ------------------------------------------------------------------------------------------------
    __device__ double frozen_rate() {  // sum of kappa_i over the frozen coordinates (StickySamplingLoop.jl:37-42, :143-148)
        double r = 0.0;
        for_owned([&](int j) { if (ACS(j) == 0.0) r += __ldg(p.kappa + coord(j)); });
        return team_sum<TEAM>(r, mask);
    }

    __device__ void sticky_move_to_axes_and_stick() {  // StickySamplingLoop.jl:73-107
        double best = CUDART_INF;
        int bi = 0x7fffffff;
        for_owned([&](int j) {
            if (ACS(j) != 0.0) {
                const double dj = XS(j) * VS(j);
                if (dj < 0 && -dj < best) { best = -dj; bi = coord(j); }   // per lane in increasing coordinate order
            }
        });
        if constexpr (TEAM > 1) {  // lexicographic minimum of (time, coordinate): the reference keeps the first minimum
#pragma unroll
            for (int o = TEAM / 2; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(mask, best, o);
                const int oi = __shfl_xor_sync(mask, bi, o);
                if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
            }
        }
        if (!(best < CUDART_INF)) { status = PDMPFLUX_CHAIN_STEP_LIMIT; return; }  // "erronous t_togo": cannot happen
        flow_inplace(best);
        if (bi % TEAM == tl) ACS(bi / TEAM) = 0.0;   // freeze the coordinate
        t += best + ts;
        ts = 0.0;
    }

    __device__ void sticky_thaw_one_coordinate() {  // StickySamplingLoop.jl:138-164
        flow_inplace(tt);
        const double total = frozen_rate();
        const double u = rand_uniform() * total;
        // first frozen coordinate (in coordinate order) whose cumulative kappa reaches u
        double carry = 0.0;
        int m = -1;
        for (int j = 0; j < nown && m < 0; ++j) {
            const double kj = (owns(j) && ACS(j) == 0.0) ? __ldg(p.kappa + coord(j)) : 0.0;
            const double incl = team_scan_incl<TEAM>(kj, mask, tl) + carry;
            const bool hit = owns(j) && ACS(j) == 0.0 && (incl >= u);
            if constexpr (TEAM == 1) { if (hit) m = j; }
            else {
                const unsigned b = team_ballot<TEAM>(hit, tl, mask);
                if (b) m = (__ffs(b) - 1) + TEAM * j;
            }
            carry = team_bcast<TEAM>(incl, TEAM - 1, mask);
        }
        if (m >= 0 && m % TEAM == tl) ACS(m / TEAM) = 1.0;   // thaw it
        // QUIRK: the clock advances by tt only; the horizon moves made since the last event (ts) are dropped
        t += tt;
        ts = 0.0;
    }

    __device__ int64_t run_events_sticky(int64_t c, bool valid) {
        int64_t ev = 0;
        bool live = valid && status == 0 && p.n_events > 0;
        while (live) {
            begin_event(ev);
            accept = false;
            bool stick = false;
            int steps = 0;
            while (!accept && !stick && live) {   // get_event_state!
                if (++steps > p.max_steps) { status = PDMPFLUX_CHAIN_STEP_LIMIT; live = false; break; }
                // one_step_of_thinning_or_sticking_or_thawing, StickySamplingLoop.jl:30-67
                compute_functionals();
                build_bound(horizon);
                const double e = rand_exp();
                next_event(e, tp, lambda_bar);
                exp_rv = e;
                const double rt = frozen_rate();
                tt = (rt == 0) ? CUDART_INF : rand_exp() / rt;
                if (exhausted) { status = PDMPFLUX_CHAIN_TAPE_EXHAUSTED; live = false; break; }
                const double event_time = fmin(fmin(tp, horizon), tt);
                bool crossed = false;
                for_owned([&](int j) {
                    const double xj = XS(j);
                    crossed = crossed || (xj * (xj + VU(j) * event_time) < 0);
                });
                if constexpr (TEAM > 1) crossed = team_ballot<TEAM>(crossed, tl, mask) != 0u;
                if (crossed) {
                    sticky_move_to_axes_and_stick();
                    stick = true;
                } else if (fmin(tp, tt) > horizon) {  // move_to_horizon!, SamplingLoopInplace.jl:87-101
                    flow_inplace(horizon);
                    ts += horizon;
                    hh += 1;
                    horizon = p.adaptive ? horizon * 1.01 : horizon;
                } else {  // moves_until_horizon_or_axes, StickySamplingLoop.jl:121-132
                    while (fmin(tp, tt) < horizon && !accept && !stick && live) {
                        if (tp < tt) {  // ac_step!, SamplingLoopInplace.jl:113-129
                            ++n_rates;
                            const double lt = rate_unsigned(tp);
                            ar = lt / lambda_bar;
                            if (ar > 1.0) {  // erroneous_acceptance_rate!, :131-151
                                const double h2 = horizon / 2;
                                build_bound(h2);
                                const double e2 = rand_exp();
                                next_event(e2, tp, lambda_bar);
                                exp_rv = e2;
                                horizon = p.adaptive ? h2 : horizon;
                                eb += 1;
                                const int slot = eb % 5;
#pragma unroll
                                for (int k = 0; k < 5; ++k)
                                    if (k == slot) eva[k] = ar;
                            } else if (rand_uniform() < ar) {  // if_accept!, :170-186
                                flow_inplace(tp);
                                velocity_jump();
                                t = t + tp + ts;
                                ts = 0.0;
                                tp = 0.0;
                                accept = true;
                            } else {  // if_reject!, :188-203
                                const double e3 = exp_rv + rand_exp();
                                next_event(e3, tp, lambda_bar);
                                horizon = p.adaptive ? horizon / 1.04 : horizon;
                                exp_rv = e3;
                                rej += 1;
                                if (fmin(tp, tt) > horizon) {  // move_to_horizon2!, :205-217
                                    flow_inplace(horizon);
                                    ts += horizon;
                                    hh += 1;
                                }
                            }
                        } else {
                            sticky_thaw_one_coordinate();
                            stick = true;
                        }
                        if (exhausted) { status = PDMPFLUX_CHAIN_TAPE_EXHAUSTED; live = false; }
                        else if (status != 0) live = false;
                        if (++steps > p.max_steps) { status = PDMPFLUX_CHAIN_STEP_LIMIT; live = false; }
                    }
                }
                if (status != 0) live = false;
            }
            if (!live) break;
            record(c, p.col0 + ev);
            ++ev;
            live = ev < p.n_events;
        }
        return ev;
    }

    // ------------------------------------------------------------------------------------------------
    // record!, Composites.jl:239-260 (chain-major slabs) -- HBM write path
    // ------------------------------------------------------------------------------------------------
    // Every byte of a PDMPHistory row is written exactly once and in full 32-byte sectors wherever alignment
    // allows (a partially written sector costs a DRAM read-modify-write):
    //   X, V rows   TEAM > 1: one TMA bulk copy per row straight from the chain-contiguous shared-memory state
    //               TEAM == 1: each lane streams its chain's rows as aligned groups of 4 doubles (256-bit stores);
    //                          up to 3 doubles are carried to the next event in shared memory
    //   t, horizon, ar   staged in registers for 4 events, one 256-bit store per column
    //   error_value_ar, errored_bound, rejected, hitting_horizon   almost always zero: the host zero-fills the
    //               columns (DMA fill at full bandwidth) and only non-zero entries are written here
    __device__ __forceinline__ void wait_row_stores() {
        if constexpr (TEAM > 1) {
            if (bulk_pending) {
                if (tl == 0) bulk_wait_read();
                __syncwarp(mask);
                bulk_pending = false;
            }
        }
    }

    __device__ void init_output(int64_t c) {
        bulk_pending = false;
        const int64_t o0 = c * p.ld_cols + p.col0;
        const int64_t r0 = c * p.ld_rows + p.col0_rows;
        scnt = sskip = (int)(o0 & 3);
        fcnt = fskip = (int)((r0 * d) & 3);
    }

    // TEAM == 1: the ng complete 32-byte groups of the stream (carry[0..R) ++ row) of one thread's chain.  R is a
    // template argument so that which element comes from the carry and which from the row is decided at compile time:
    // a group is four shared-memory loads with immediate offsets and one 256-bit store (the run-time variant spent a
    // compare, an address select and a load per element: 6.5 % of config C1's instructions).
    template <int R>
    __device__ __forceinline__ void row_groups_tm1(double* G, int64_t gfirst, int ng, int off_src, int off_carry) {
        if (ng <= 0) return;
        double* dst = G + gfirst;
        {
            double vq[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) vq[k] = k < R ? g_smem[off_carry + k * kBT] : g_smem[off_src + (k - R) * kBT];
            if (fskip > 0) {  // first group of this launch starts mid-sector: scalar stores for the real part
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (k >= fskip) dst[k] = vq[k];
            } else st256(dst, vq[0], vq[1], vq[2], vq[3]);
        }
        int o = off_src + (4 - R) * kBT;
#pragma unroll 2
        for (int q = 1; q < ng; ++q) {
            dst += 4;
            st256(dst, g_smem[o], g_smem[o + kBT], g_smem[o + 2 * kBT], g_smem[o + 3 * kBT]);
            o += 4 * kBT;
        }
    }
    __device__ __forceinline__ void row_stream_tm1(double* G, int64_t gfirst, int ng, int r, int off_src, int off_carry) {
        switch (r) {
        case 0: row_groups_tm1<0>(G, gfirst, ng, off_src, off_carry); break;
        case 1: row_groups_tm1<1>(G, gfirst, ng, off_src, off_carry); break;
        case 2: row_groups_tm1<2>(G, gfirst, ng, off_src, off_carry); break;
        default: row_groups_tm1<3>(G, gfirst, ng, off_src, off_carry); break;
        }
    }

    __device__ void record(int64_t c, int64_t col) {
        const int64_t o = c * p.ld_cols + col;                                // scalar columns
        const int64_t orow = c * p.ld_rows + (col - p.col0) + p.col0_rows;    // X / V rows
        // ---- X, V rows ----
        if constexpr (TEAM > 1) {
            if (p.bulk_rows) {
                fence_async_smem();   // make this lane's generic-proxy writes of x / v visible to the TMA engine
                __syncwarp(mask);
                if (tl == 0) {
                    if (p.X) bulk_store(p.X + orow * d, &g_smem[off_x], (uint32_t)d * 8u);
                    if (p.V) bulk_store(p.V + orow * d, &g_smem[off_v], (uint32_t)d * 8u);
                    bulk_commit();
                }
                bulk_pending = true;
            } else {
                if (p.X)
                    for (int j = 0; j < nown; ++j)
                        if (owns(j)) p.X[orow * d + coord(j)] = XS(j);
                if (p.V)
                    for (int j = 0; j < nown; ++j)
                        if (owns(j)) p.V[orow * d + coord(j)] = VS(j);
            }
        } else {
            if (p.vec32) {
                const int r = fcnt;                  // carried (or phantom) elements in front of this row
                const int total = r + d;
                const int ng = total >> 2;
                const int64_t gfirst = orow * d - r;    // 4-aligned element index of the combined stream's start
                if (p.X) row_stream_tm1(p.X, gfirst, ng, r, off_x, off_f);
                if (p.V) row_stream_tm1(p.V, gfirst, ng, r, off_v, off_f + 3 * kBT);
                const int rem = total - 4 * ng;
                if (ng > 0) {
                    for (int k = 0; k < rem; ++k) {  // tail of the row becomes the next carry
                        const int pos = 4 * ng + k;
                        g_smem[off_f + k * kBT] = g_smem[off_x + (pos - r) * kBT];
                        g_smem[off_f + (3 + k) * kBT] = g_smem[off_v + (pos - r) * kBT];
                    }
                    fskip = 0;
                } else {  // d < 4 and the group is still open: append
                    for (int k = r; k < total; ++k) {
                        g_smem[off_f + k * kBT] = g_smem[off_x + (k - r) * kBT];
                        g_smem[off_f + (3 + k) * kBT] = g_smem[off_v + (k - r) * kBT];
                    }
                }
                fcnt = rem;
            } else {
                if (p.X)
                    for (int j = 0; j < nown; ++j) p.X[orow * d + j] = XS(j);
                if (p.V)
                    for (int j = 0; j < nown; ++j) p.V[orow * d + j] = VS(j);
            }
        }
        if constexpr (kSticky) {  // is_active[:, k] (Composites.jl:254-258), one byte per coordinate
            if (p.ACT) for_owned([&](int j) { p.ACT[orow * d + coord(j)] = ACS(j) != 0.0 ? 1 : 0; });
        }
        if (tl != 0) return;
        // ---- t, horizon, ar: 4 events per 256-bit store ----
        if (p.vec32) {
            if (scnt < 3) {
                if (scnt == 0) { st_t[0] = t; st_h[0] = horizon; st_a[0] = ar; }
                else if (scnt == 1) { st_t[1] = t; st_h[1] = horizon; st_a[1] = ar; }
                else { st_t[2] = t; st_h[2] = horizon; st_a[2] = ar; }
                ++scnt;
            } else {
                if (sskip == 0) {
                    if (p.T) st256(p.T + o - 3, st_t[0], st_t[1], st_t[2], t);
                    if (p.H) st256(p.H + o - 3, st_h[0], st_h[1], st_h[2], horizon);
                    if (p.AR) st256(p.AR + o - 3, st_a[0], st_a[1], st_a[2], ar);
                } else {
                    flush_scalars(o);  // slots [sskip, 3) are real, the current event follows
                    if (p.T) p.T[o] = t;
                    if (p.H) p.H[o] = horizon;
                    if (p.AR) p.AR[o] = ar;
                }
                scnt = 0; sskip = 0;
            }
        } else {
            if (p.T) p.T[o] = t;
            if (p.H) p.H[o] = horizon;
            if (p.AR) p.AR[o] = ar;
        }
        // ---- sparse diagnostic columns ----
        if (!p.sparse_cols || eb != 0) {
            if (p.EB) p.EB[o] = eb;
            if (p.EVA) {
#pragma unroll
                for (int k = 0; k < 5; ++k) p.EVA[o * 5 + k] = eva[k];
            }
        }
        if ((!p.sparse_cols || rej != 0) && p.REJ) p.REJ[o] = rej;
        if ((!p.sparse_cols || hh != 0) && p.HH) p.HH[o] = hh;
    }

    // staged scalar slots [sskip, scnt) belong to elements o_next - scnt + k
    __device__ void flush_scalars(int64_t o_next) {
#pragma unroll
        for (int k = 0; k < 3; ++k)
            if (k >= sskip && k < scnt) {
                const int64_t o = o_next - scnt + k;
                if (p.T) p.T[o] = st_t[k];
                if (p.H) p.H[o] = st_h[k];
                if (p.AR) p.AR[o] = st_a[k];
            }
    }

    // end of launch: write what is still staged (scalar stores) and drain the TMA engine
    __device__ void finish_output(int64_t c, int64_t n_recorded) {
        const int64_t o_next = c * p.ld_cols + p.col0 + n_recorded;
        const int64_t r_next = c * p.ld_rows + p.col0_rows + n_recorded;
        if constexpr (TEAM == 1) {
            if (p.vec32) {
                for (int k = fskip; k < fcnt; ++k) {
                    const int64_t g = r_next * d - fcnt + k;
                    if (p.X) p.X[g] = g_smem[off_f + k * kBT];
                    if (p.V) p.V[g] = g_smem[off_f + (3 + k) * kBT];
                }
            }
        } else {
            if (bulk_pending && tl == 0) bulk_wait_all();
        }
        if (tl == 0 && p.vec32) flush_scalars(o_next);
    }
};

// One launch advances every chain by p.n_events accepted events (or just records the current state when
// n_events == 0 and col0 names the column).  Grid = ceil(n_chains / (kBT / TEAM)).
constexpr int kMinBlocksGrid = 4;   // grid-bound kernels of teams of 1 / 8: blocks per SM (3 measured -10 .. -13 %)
template <int TEAM, int SAMPLER, int POT, int PATH, int NW = kLineShared>
__global__ void __launch_bounds__(block_threads_rt(TEAM, SAMPLER, PATH), PATH == kPathGeneric ? 1 : (PATH == kPathFastBrent ? (TEAM == 1 && SAMPLER == PDMPFLUX_ZIGZAG ? 4 : 2) : (TEAM == 32 ? 3 : kMinBlocksGrid))) skeleton_kernel(const __grid_constant__ KernelParams p) {
    constexpr int kBT = block_threads_rt(TEAM, SAMPLER, PATH);
    constexpr int CPB = kBT / TEAM;  // chains per block
    const int c_local = threadIdx.x / TEAM;
    // A block normally owns one group of CPB chains (grid = number of groups).  With p.n_groups > gridDim.x the grid is
    // persistent (one block per resident slot) and walks over the groups: the per-block scratch vectors in global
    // memory are then indexed by the resident block, stay in the L2 and are rewritten in place instead of being
    // flushed to DRAM behind the history rows (ForwardECMC at large d).
    // (only the warp-per-chain and the ForwardECMC kernels are ever launched that way; for the others the loop is compiled away)
    constexpr bool kPersistent = (TEAM == 32) || (SAMPLER == PDMPFLUX_FECMC);
    int64_t grp = blockIdx.x;
    do {
    const int64_t c_raw = grp * CPB + c_local;
    const bool valid = c_raw < p.n_chains;  // out-of-range lanes stay (warp-wide votes) but never touch memory
    const int64_t c = valid ? c_raw : 0;

    Chain<TEAM, SAMPLER, POT, PATH, NW> ch(p);
    ch.tl = threadIdx.x % TEAM;
    ch.mask = team_mask<TEAM>();
    ch.d = p.d;
    ch.nown = p.n_own;
    ch.nfull = p.d / TEAM;
    ch.chain = c;
    // shared-memory state vectors: [x | v | (A | B) | (scratch x3) | (row carry)]
    const int vec = p.vec_elems;
    const int toff = (TEAM == 1) ? (int)threadIdx.x : c_local * p.dpad + ch.tl;  // this thread's offset in a vector
    ch.off_x = toff;
    ch.off_v = vec + toff;
    constexpr int kVectors = state_vectors(SAMPLER, PATH, TEAM, NW);
    int used = kVectors;
    ch.off_a = ch.off_b = 0;
    if constexpr (kVectors == 4) {
        ch.off_a = 2 * vec + toff;
        ch.off_b = 3 * vec + toff;
    }
    {
        double* base = p.scratch_in_smem ? g_smem + (size_t)used * vec + toff
                                         : (p.scratch ? p.scratch + (size_t)blockIdx.x * 3 * vec + toff : nullptr);
        ch.sc0 = base;
        ch.sc1 = base + vec;
        ch.sc2 = base + 2 * (size_t)vec;
        if (p.scratch_in_smem && SAMPLER == PDMPFLUX_FECMC) used += 3;
    }
    ch.off_ac = 0;
    ch.tt = CUDART_INF;
    if constexpr (SAMPLER == PDMPFLUX_STICKY_ZIGZAG) {
        ch.off_ac = used * vec + toff;
        used += 1;
        ch.for_owned([&](int j) { g_smem[ch.off_ac + j * ch.kStr] = p.sact[c * p.d + ch.coord(j)] ? 1.0 : 0.0; });
    }
    ch.off_m1 = ch.off_m2 = 0;
    if (p.accumulate_moments) {
        ch.off_m1 = used * vec + toff;
        ch.off_m2 = (used + 1) * vec + toff;
        used += 2;
        for (int j = 0; j < ch.nown; ++j)
            if (ch.owns(j)) {
                g_smem[ch.off_m1 + j * ch.kStr] = p.M1[c * p.d + ch.coord(j)];
                g_smem[ch.off_m2 + j * ch.kStr] = p.M2[c * p.d + ch.coord(j)];
            }
    }
    ch.off_f = used * vec + (int)threadIdx.x;  // TEAM == 1 only: 6 carry slots per thread
    {
        const int gb = p.G > 2 ? p.G : 2;      // entries per array (Brent uses 1 + 2)
        const int base = used * vec + (TEAM == 1 ? 6 * kBT : 0);
        if constexpr (TEAM == 1) {
            ch.off_box = base + (int)threadIdx.x;
            ch.off_cum = base + gb * kBT + (int)threadIdx.x;
        } else {
            ch.off_box = base + c_local * 2 * gb;
            ch.off_cum = ch.off_box + gb;
        }
    }
    // load PDMPState
    ch.for_owned([&](int j) {
        g_smem[ch.off_x + j * ch.kStr] = p.sx[c * p.d + ch.coord(j)];
        g_smem[ch.off_v + j * ch.kStr] = p.sv[c * p.d + ch.coord(j)];
    });
    ch.t = p.st[c];
    ch.horizon = p.shorizon[c];
    ch.ar = p.sar[c];
    ch.tp = 0.0; ch.ts = 0.0; ch.exp_rv = 0.0; ch.lambda_bar = 0.0;
    ch.eb = 0; ch.rej = 0; ch.hh = 0;
#pragma unroll
    for (int k = 0; k < 5; ++k) ch.eva[k] = 0.0;
    ch.accept = false;
    ch.status = p.status[c];
    ch.n_builds = p.counters[2 * c];
    ch.n_rates = p.counters[2 * c + 1];
    ch.exhausted = false;
    const uint64_t gchain = (uint64_t)(p.chain_offset + c);
    ch.key.k0 = (uint32_t)p.seed; ch.key.k1 = (uint32_t)(p.seed >> 32);
    ch.key.chain_lo = (uint32_t)gchain; ch.key.chain_hi8 = (uint32_t)(gchain >> 32) << 8;
    ch.tE = p.tE + c * p.nE; ch.tU = p.tU + c * p.nU; ch.tN = p.tN + c * p.nN;
    ch.pE = p.tape_pos[3 * c]; ch.pU = p.tape_pos[3 * c + 1]; ch.pN = p.tape_pos[3 * c + 2];
    ch.init_output(c);
    if constexpr (TEAM > 1) __syncwarp(ch.mask);

    if (p.n_events == 0) {
        if (valid) {
            ch.record(c, p.col0);
            ch.finish_output(c, 1);
            if (ch.tl == 0) p.ncols[c] += 1;
        }
        continue;
    }
    int64_t n_rec;
    if constexpr (SAMPLER == PDMPFLUX_STICKY_ZIGZAG) n_rec = ch.run_events_sticky(c, valid);
    else n_rec = ch.run_events(c, valid);
    if (!valid) continue;   // (only whole teams are invalid, and only in the last group)
    if constexpr (SAMPLER == PDMPFLUX_STICKY_ZIGZAG)
        ch.for_owned([&](int j) { p.sact[c * p.d + ch.coord(j)] = g_smem[ch.off_ac + j * ch.kStr] != 0.0 ? 1 : 0; });
    ch.finish_output(c, n_rec);
    // store PDMPState
    for (int j = 0; j < ch.nown; ++j)
        if (ch.owns(j)) {
            p.sx[c * p.d + ch.coord(j)] = g_smem[ch.off_x + j * ch.kStr];
            p.sv[c * p.d + ch.coord(j)] = g_smem[ch.off_v + j * ch.kStr];
        }
    if (p.accumulate_moments)
        for (int j = 0; j < ch.nown; ++j)
            if (ch.owns(j)) {
                p.M1[c * p.d + ch.coord(j)] = g_smem[ch.off_m1 + j * ch.kStr];
                p.M2[c * p.d + ch.coord(j)] = g_smem[ch.off_m2 + j * ch.kStr];
            }
    if (ch.tl == 0) {
        p.st[c] = ch.t;
        p.shorizon[c] = ch.horizon;
        p.sar[c] = ch.ar;
        p.status[c] = ch.status;
        p.counters[2 * c] = ch.n_builds;
        p.counters[2 * c + 1] = ch.n_rates;
        p.tape_pos[3 * c] = ch.pE; p.tape_pos[3 * c + 1] = ch.pU; p.tape_pos[3 * c + 2] = ch.pN;
        p.ncols[c] += n_rec;
    }
    } while (kPersistent && (grp += gridDim.x) < p.n_groups);
}

}  // namespace pdmpflux
