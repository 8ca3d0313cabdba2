// vag_grid.cuh -- K0: per-parameter-set adaptive (phi, theta, t) grid.
//
// Restates auto_grid and its callees (src/core/grid-refinement.h:40-706,
// src/core/grid-refinement.cpp:140-197, Coord::detect_symmetry src/core/mesh.h:120-185) for the
// typed jets / isotropic media, i.e. symmetry >= phi_symmetric and no spreading.
//
// Execution model: ONE WARP builds one model's grid.  The algorithm is written as uniform code
// (every lane executes it redundantly -- the same latency as one lane -- so scalar state stays in
// registers and needs no broadcast) interleaved with `par.for_each(n, f)` regions whose index
// space is strided over the 32 lanes and whose results go to a per-model scratch slab:
//   * the 512-point jet-profile scans, the 101-point pdf pre-scans, the 200 CDF sample abscissae
//   * the six stage evaluations of every dopri5 attempt of the CDF quadrature (a pure quadrature:
//     the pdf does not depend on the state, so the stages are independent) and its dense output
//   * the inverse-CDF look-ups, the per-theta symmetry probes, t_dec and the time-bound scan.
// Order-dependent reductions (running peaks, sums whose rounding matters, first-hit searches) stay
// in uniform code over the precomputed values, so results equal the sequential restatement's.
// On the host (oracle/hostemu) `Par` is a plain loop.
#pragma once

#include "vag_dopri5.cuh"
#include "vag_model.cuh"

namespace vag {

enum Symmetry : int { SYM_STRUCTURED = 0, SYM_PHI_SYMMETRIC = 1, SYM_PIECEWISE = 2, SYM_ISOTROPIC = 3 };

// Per-model grid header (device resident).
struct GridHeader {
    int n_theta, n_phi, n_phi_eff, n_t;
    int n_reps, symmetry, phi_mirrored, status;
    int t_num_tot, t_num_base, has_early, is_rvs;
    double t_end, min_t_start, min_t_early;
    int spreading, structured;
    // rows3d: structured model with axisymmetric = False -- one ODE row per (phi_i, theta_j) on its own time lattice
    // (build_time_grid, grid-refinement.h:612-619); row index r = i * n_theta + j, n_reps = n_phi * n_theta
    int rows3d, pad_;
    double t_obs_min;  // first observation time (code units): the per-row lattice bounds of a rows3d model derive from it
    double theta_s;  // jet_spreading_edge (spreading models)
    int quad_attempts_theta, quad_attempts_phi;  // dopri5 attempts of the two CDF quadratures (work counters)
};

// Slab of per-model arrays (capacities fixed per batch by the host).
struct GridSlab {
    double* theta;   // [cap_theta]
    double* phi;     // [cap_phi]
    int* reps;       // [cap_theta]
    double* t_dec;   // [cap_theta]  t_dec of each representative row
    double* work;    // scratch: grid_work_doubles(cap_theta, cap_phi)
    int cap_theta, cap_phi;
};

// sequential executor (host emulation, single-thread fallback inside tests)
struct SeqPar {
    template <class F>
    VAG_HD void for_each(int n, F f) const {
        for (int i = 0; i < n; ++i) f(i);
    }
    // smallest j in [begin, end) with pred(j), or end
    template <class P>
    VAG_HD int first_true(int begin, int end, P pred) const {
        for (int j = begin; j < end; ++j)
            if (pred(j)) return j;
        return end;
    }
    // while (active) active = round();  -- see GroupPar::lockstep
    template <class R>
    VAG_HD void lockstep(bool active, R round) const {
        while (active) active = round();
    }
};
#if defined(__CUDACC__)
// one warp: index space strided over the lanes, warp barrier (with memory ordering) afterwards
struct WarpPar {
    int lane;
    template <class F>
    __device__ __forceinline__ void for_each(int n, F f) const {
        __syncwarp();
        for (int i = lane; i < n; i += 32) f(i);
        __syncwarp();
    }
    // first-hit search of an order-independent predicate: 32 candidates per ballot, in index order
    template <class P>
    __device__ __forceinline__ int first_true(int begin, int end, P pred) const {
        for (int j0 = begin; j0 < end; j0 += 32) {
            const int j = j0 + lane;
            const unsigned hits = __ballot_sync(0xffffffffu, j < end && pred(j));
            if (hits) return j0 + __ffs(hits) - 1;
        }
        return end;
    }
    template <class R>
    __device__ __forceinline__ void lockstep(bool active, R round) const {
        while (active) active = round();
    }
};
// G lanes of a warp (G = 2 ... 32): the same contract for a sub-warp group, so that 32 / G models share one warp.
// The grid builder is mostly uniform (scalar) code that every cooperating lane executes redundantly;
// with narrower groups the same instruction stream serves 32 / G models at once, while the strided
// regions keep all lanes busy.  Groups synchronise with their own lane mask (they diverge freely).
template <int G>
struct GroupPar {
    int lane;       // 0 .. G-1 within the group
    unsigned mask;  // lanes of this group within the warp
    int shift;      // first lane of the group
    template <class F>
    __device__ __forceinline__ void for_each(int n, F f) const {
        __syncwarp(mask);
        for (int i = lane; i < n; i += G) f(i);
        __syncwarp(mask);
    }
    template <class P>
    __device__ __forceinline__ int first_true(int begin, int end, P pred) const {
        for (int j0 = begin; j0 < end; j0 += G) {
            const int j = j0 + lane;
            const unsigned hits = (__ballot_sync(mask, j < end && pred(j)) & mask) >> shift;
            if (hits) return j0 + __ffs(hits) - 1;
        }
        return end;
    }
    // `while (active) active = round();` for a loop whose trip count differs between models.  The groups that enter
    // together run their rounds together until the last of them is done (a finished group idles): a group that needs
    // another round does not leave the others to run theirs alone later, so the warp issues each round's stage
    // evaluations and uniform code once for all of its groups instead of once per group.
    template <class R>
    __device__ __forceinline__ void lockstep(bool active, R round) const {
        const unsigned peers = __activemask();
        while (__any_sync(peers, active))
            if (active) active = round();
    }
};
#endif

constexpr int GRID_NSCAN = 513;  // longest scan (find_theta_range visits at most 513 nodes)

VAG_HD size_t grid_work_doubles(int cap_theta, int cap_phi) {
    // base_theta[cap_theta] + 5 per-theta arrays + 2 scan arrays + CDF samples + stage values
    return (size_t)6 * cap_theta + 2 * (GRID_NSCAN + 7) + 2 * dflt::theta_samples + cap_phi + 32;
}

// ---------------------------------------------------------------------------------------------------
// BIT-EXACT SECTION.  Everything from here to estimate_t_dec determines, or is determined by, the step
// positions of the reference's adaptive CDF quadratures (theta grid, then the phi grid whose pdf sums over
// the theta nodes).  Those quadratures are chaotic in the last bit (vag_libm.cuh header), so this section
// reproduces the REFERENCE BUILD's arithmetic operation by operation: the instruction sequence g++ emits for
// src/core/grid-refinement.h under the reference's flags (CMakeLists.txt:10-16: -O3 -ffp-contract=fast
// -freciprocal-math on an FMA target), read off oracle/_ref/libvagref.so.  What that means concretely:
//   * a product feeding a sum is ONE fma exactly where gcc fused it (first product of an a*b + c*d pair), and
//     two roundings everywhere else -- written with gl::mul / gl::add / gl::fma, which no compiler re-contracts;
//   * a division by a compile-time constant is a multiplication by its rounded reciprocal (x / 100 -> x * 0.01,
//     the dense-output constants of Boost's dopri5), divisions by variables are true divisions;
//   * libm calls go through gl:: (the host libm's own algorithms and tables).
// oracle/hostemu runs the same source on the host; tests/test_grid_exact.py demands bit-equal theta / phi nodes
// against the unmodified reference there, and the -m gpu tier demands bit-equal nodes between device and host.
// ---------------------------------------------------------------------------------------------------
VAG_HD double structure_weight(double Gamma) {  // grid-refinement.h:11-13
    const double w0 = gl::mul(gl::sub(Gamma, 1.0), Gamma);
    const double s = (0.0 > w0) ? 0.0 : gl::sqrt(w0);
    return gl::mul(Gamma, s);
}
// physics::relativistic::gamma_to_beta (src/core/physics.h:36-40) as compiled
VAG_HD double gamma_to_beta_x(double Gamma) {
    return gl::div(gl::sqrt(gl::mul(gl::add(Gamma, 1.0), gl::sub(Gamma, 1.0))), Gamma);
}

// xt::linspace(a, b, n)[i] (external/xtensor/generators/xbuilder.hpp:199-222,460-468):
// fma(i, step, a) with the last element forced to b.
VAG_HD double linspace_at(double a, double b, int n, int i) {
    const double step = gl::div(gl::sub(b, a), fmax(1.0, (double)(n - 1)));
    if (n > 1 && i == n - 1) return b;
    return gl::fma((double)i, step, a);
}

// ---- find_jet_jumps: grid-refinement.h:40-86 -------------------------------------------------
template <class Par>
VAG_HD int find_jet_jumps(const Par& par, const ModelCfg& m, double gamma_cut, double* jumps, int cap, double* G) {
    constexpr int n_scan = 512;
    constexpr double eps = dflt::binary_search_eps;
    constexpr double theta_lo = dflt::theta_min;
    constexpr double theta_hi = con::pi / 2;
    constexpr double dtheta = (theta_hi - theta_lo) / (n_scan - 1);
    if (jet_Gamma0(m, theta_hi) >= gamma_cut) {
        jumps[0] = theta_hi;
        return 1;
    }
    auto node = [&](int j) { return j == 0 ? theta_lo : gl::fma((double)j, dtheta, theta_lo); };
    // A plain top-hat profile (Gamma0 inside theta_c, 1 outside; Gamma0 >= gamma_cut) has exactly one candidate, the
    // first node with !(theta_j < theta_c): it is located directly on the same node expression instead of evaluating
    // and scanning all 512 nodes -- same j, same refinement below.
    const bool tophat = m.jet_type == VAG_JET_TOPHAT && !m.ejecta && m.Gamma0 >= gamma_cut;
    int j_top = n_scan;
    if (tophat) {
        int j = (int)((m.theta_c - theta_lo) / dtheta);
        j = j < 0 ? 0 : (j > n_scan - 1 ? n_scan - 1 : j);
        while (j > 0 && !(node(j - 1) < m.theta_c)) --j;
        while (j < n_scan && node(j) < m.theta_c) ++j;
        j_top = (j >= 1) ? j : n_scan;  // theta_c <= theta_lo: the profile is 1 everywhere, no candidate
    } else {
        par.for_each(n_scan, [&](int j) { G[j] = jet_Gamma0(m, node(j)); });
    }
    // The walk's jump test at node j reads only G[j-1] and G[j]: the candidates are found with an
    // order-preserving parallel search, each hit is then refined exactly as the sequential walk does.
    int n = 0;
    auto is_jump = [&](int j) {
        const double prev_G = G[j - 1], cur_G = G[j];
        if (!(prev_G >= gamma_cut || cur_G >= gamma_cut)) return false;
        const double dG = fabs(cur_G - prev_G);
        const double scale = vmax(prev_G - 1, cur_G - 1);
        return scale > 0 && dG > 0.5 * scale;
    };
    auto next_jump = [&](int from) {
        if (tophat) return (from <= j_top) ? j_top : n_scan;
        return par.first_true(from, n_scan, is_jump);
    };
    for (int j = next_jump(1); j < n_scan; j = next_jump(j + 1)) {
        const double prev_th = (j - 1 == 0) ? theta_lo : gl::fma((double)(j - 1), dtheta, theta_lo);
        const double cur_th = gl::fma((double)j, dtheta, theta_lo);
        const double prev_G = tophat ? m.Gamma0 : G[j - 1], cur_G = tophat ? 1.0 : G[j];
        double lo = prev_th, hi = cur_th;
        while (hi - lo > eps) {
            const double mid = 0.5 * (lo + hi);
            const double G_mid = jet_Gamma0(m, mid);
            if (fabs(G_mid - prev_G) < fabs(G_mid - cur_G)) {
                lo = mid;
            } else {
                hi = mid;
            }
        }
        if (n >= cap) return -1;  // more discontinuities than the compiled capacity: reported, never truncated
        jumps[n++] = prev_G > cur_G ? lo : hi;
    }
    return n;
}

// ---- find_theta_range: grid-refinement.h:88-111 ----------------------------------------------
// The reference walks th -= step / th += step with early exit; the node sequence (a running sum,
// so not j*step) is generated in uniform code, the profile evaluated at all nodes in parallel,
// and the first hit taken in walk order.
// The two node sequences are running sums of compile-time constants -- the same 513 + 513 doubles for every model --
// so they are generated ONCE (ThetaWalk: on the device by k_init_tables at vag_create, on the host at first use) by the
// reference's own loop; a per-model copy cost every model a 1026-long dependent DADD chain and 8 KB of scratch writes.
struct ThetaWalk {
    double down[GRID_NSCAN + 7], up[GRID_NSCAN + 7];
    int n_down, n_up;
};
VAG_HD void build_theta_walk(ThetaWalk& w) {
    constexpr int n_scan = 512;
    const double theta_lo = dflt::theta_min;
    const double theta_hi = con::pi / 2;
    const double step = (theta_hi - theta_lo) / n_scan;
    int n = 0;
    for (double th = theta_hi; th >= theta_lo && n < GRID_NSCAN + 6; th -= step) w.down[n++] = th;
    w.n_down = n;
    n = 0;
    for (double th = theta_lo; th <= theta_hi && n < GRID_NSCAN + 6; th += step) w.up[n++] = th;
    w.n_up = n;
}
#if defined(__CUDACC__)
__device__ ThetaWalk g_theta_walk;
#endif
VAG_HD const ThetaWalk& theta_walk() {
#if defined(__CUDA_ARCH__)
    return g_theta_walk;
#else
    static const ThetaWalk w = [] {
        ThetaWalk t;
        build_theta_walk(t);
        return t;
    }();
    return w;
#endif
}
// The profile is evaluated inside the order-preserving first-hit search (G lanes per round, stop at the first round
// with a hit -- the reference's early exit): an on-axis core ends the upward walk in its first round.
template <class Par>
VAG_HD void find_theta_range(const Par& par, const ModelCfg& m, double gamma_cut, double& theta_min, double& theta_max) {
    const ThetaWalk& tw = theta_walk();
    theta_max = con::pi / 2;
    theta_min = dflt::theta_min;
    {
        const int n = tw.n_down;
        int j;
        if (m.jet_type == VAG_JET_TOPHAT && !m.ejecta && m.Gamma0 >= gamma_cut) {
            // top-hat: the hit test is theta < theta_c on a strictly descending sequence -- bisection finds the same first hit
            int lo = 0, hi = n;  // first q with down[q] < theta_c
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (tw.down[mid] < m.theta_c)
                    hi = mid;
                else
                    lo = mid + 1;
            }
            j = lo;
        } else {
            j = par.first_true(0, n, [&](int q) { return jet_Gamma0(m, tw.down[q]) >= gamma_cut; });
        }
        if (j < n) theta_max = tw.down[j];
    }
    {
        const int n = tw.n_up;
        const int j = par.first_true(0, n, [&](int q) { return jet_Gamma0(m, tw.up[q]) >= gamma_cut; });
        if (j < n) theta_min = tw.up[j];
    }
}

// ---- the scalar quadrature stepper of inverse_CFD_sampling ----------------------------------------
// Boost.odeint's dense_output_runge_kutta<controlled_runge_kutta<runge_kutta_dopri5<double>>> driving
// dx/dt = pdf(t) (the state never enters the right-hand side), as g++ compiled it into inverse_CFD_sampling:
//   stage abscissae   fma(a_i, dt, t) for a = 1/5, 3/10, 4/5, 8/9 and t + dt for the last two
//   new state         x + (dt c1) k1 + (dt c3) k3 + (dt c4) k4 + (dt c5) k5 + (dt c6) k6 as one fma chain, left to right
//   error             ((dt dc3) k3 rounded) then the fma chain dc1 k1, dc4 k4, dc5 k5, dc6 k6, dc7 k7
//   error norm        |e| / fma(eps, fma(|dt|, |k1|, |x|), eps)           (controlled_runge_kutta.hpp:64-90)
//   rejected          dt = max(0.9 pow(err, -1/3), 0.2) dt                (:114-129)
//   accepted          t += dt;  err < 0.5:  dt *= (err > 5^-5) ? 0.9 pow(err, -1/5) : 4.5   (:131-153)
//   dense output      Hairer's continuous extension with the reciprocal-constant weights below (dopri5.hpp:229-275)
// VARIANT: g++ compiled the stepper twice.  Inlined into the theta-grid sampler (VARIANT = 0) the unused stage
// states were eliminated, so dt * a2 has one use and fuses into the first stage abscissa, and the error-norm scale is
// fma(|dt|, |k1|, |x|).  The phi-grid sampler (VARIANT = 1) calls the out-of-line do_step, which keeps the stage states:
// dt * b21 (= dt * a2) is shared with them, hence rounded before it is added to t, and the scale is |x| + (|dt| |k1|
// rounded).  Everything else is identical.
template <int VARIANT>
struct CdfQuad {
    double x, k1, t, dt;           // current state, FSAL derivative, time, next step size
    double xo, ko, to;             // state / derivative / time at the start of the last accepted step
    double k3, k4, k5, k6;         // stages of the last accepted step
    bool deriv_ready;
    static constexpr double a2 = 1.0 / 5, a3 = 3.0 / 10, a4 = 4.0 / 5, a5 = 8.0 / 9;
    static constexpr double c1 = 35.0 / 384, c3 = 500.0 / 1113, c4 = 125.0 / 192, c5 = -2187.0 / 6784, c6 = 11.0 / 84;
    static constexpr double dc1 = c1 - 5179.0 / 57600, dc3 = c3 - 7571.0 / 16695, dc4 = c4 - 393.0 / 640,
                            dc5 = c5 - (-92097.0 / 339200), dc6 = c6 - 187.0 / 2100, dc7 = -1.0 / 40;

    VAG_HD void initialize(double t0, double dt0) {
        x = 0;
        t = to = t0;
        dt = dt0;
        deriv_ready = false;
    }
    // abscissa of stage s = 0..5 (k2 .. k7) of an attempt from (t, dt)
    VAG_HD static double stage_time(double t, double dt, int s) {
        const double a = (s == 0) ? a2 : (s == 1) ? a3 : (s == 2) ? a4 : a5;
        if (VARIANT == 1 && s == 0) return gl::add(gl::mul(a2, dt), t);
        return s < 4 ? gl::fma(a, dt, t) : gl::add(dt, t);
    }
    // one attempt with the six stage values kk[0..5] = pdf(stage_time(t, dt, s)); true = accepted
    VAG_HD bool try_step(const double* kk, double eps) {
        const double K3 = kk[1], K4 = kk[2], K5 = kk[3], K6 = kk[4], K7 = kk[5];
        double xn = gl::fma(gl::mul(dt, c1), k1, x);
        xn = gl::fma(gl::mul(dt, c3), K3, xn);
        xn = gl::fma(gl::mul(dt, c4), K4, xn);
        xn = gl::fma(gl::mul(dt, c5), K5, xn);
        xn = gl::fma(gl::mul(dt, c6), K6, xn);
        double e = gl::mul(gl::mul(dt, dc3), K3);
        e = gl::fma(gl::mul(dt, dc1), k1, e);
        e = gl::fma(gl::mul(dt, dc4), K4, e);
        e = gl::fma(gl::mul(dt, dc5), K5, e);
        e = gl::fma(gl::mul(dt, dc6), K6, e);
        e = gl::fma(gl::mul(dt, dc7), K7, e);
        const double scale = (VARIANT == 1) ? gl::add(fabs(x), gl::mul(fabs(dt), fabs(k1))) : gl::fma(fabs(dt), fabs(k1), fabs(x));
        const double den = gl::fma(eps, scale, eps);
        const double err = fabs(gl::div(fabs(e), den));
        if (err > 1.0) {
            dt = gl::mul(vmax(0.2, gl::mul(gl::pow(err, -1.0 / 3.0), 0.9)), dt);
            return false;
        }
        xo = x;
        ko = k1;
        to = t;
        k3 = K3;
        k4 = K4;
        k5 = K5;
        k6 = K6;
        x = xn;
        k1 = K7;
        t = gl::add(dt, t);
        if (err < 0.5) dt = gl::mul(dt, (err > 0.00032) ? gl::mul(gl::pow(err, -1.0 / 5.0), 0.9) : 4.5);
        return true;
    }
    // dense output at tq inside the last accepted step
    VAG_HD double calc_state(double tq) const {
        constexpr double b1 = c1, b3 = c3, b4 = c4, b5 = c5, b6 = c6;
        const double h = gl::sub(t, to);
        const double th = gl::div(gl::sub(tq, to), h);
        const double X1 = gl::mul(gl::mul(gl::fnma(31403016.0, th, 2558722523.0), 5.0), 1.0 / 11282082432.0);
        const double X3 = gl::mul(gl::mul(gl::fnma(15701508.0, th, 882725551.0), 100.0), 1.0 / 32700410799.0);
        const double X4 = gl::mul(gl::mul(gl::fnma(31403016.0, th, 443332067.0), 25.0), 1.0 / 1880347072.0);
        const double X5 = gl::mul(gl::mul(gl::fnma(3489224.0, th, 23143187.0), 32805.0), 1.0 / 199316789632.0);
        const double X6 = gl::mul(gl::mul(gl::fnma(7076736.0, th, 29972135.0), 55.0), 1.0 / 822651844.0);
        const double X7 = gl::mul(gl::mul(gl::fnma(829305.0, th, 7414447.0), 10.0), 1.0 / 29380423.0);
        const double thm1 = gl::sub(th, 1.0);
        const double thsq = gl::mul(th, th);
        const double A = gl::mul(gl::fnma(2.0, th, 3.0), thsq);
        const double B = gl::mul(thsq, thm1);
        const double C = gl::mul(B, thm1);
        const double D0 = gl::mul(thm1, th);
        double w1 = gl::fms(A, b1, gl::mul(X1, C));
        w1 = gl::fma(D0, thm1, w1);
        const double w3 = gl::fma(A, b3, gl::mul(X3, C));
        const double w4 = gl::fms(A, b4, gl::mul(X4, C));
        const double w5 = gl::fma(A, b5, gl::mul(X5, C));
        const double w6 = gl::fms(A, b6, gl::mul(X6, C));
        const double w7 = gl::fma(C, X7, B);
        double r = gl::fma(gl::mul(w1, h), ko, xo);
        r = gl::fma(gl::mul(w3, h), k3, r);
        r = gl::fma(gl::mul(w4, h), k4, r);
        r = gl::fma(gl::mul(w5, h), k5, r);
        r = gl::fma(gl::mul(w6, h), k6, r);
        r = gl::fma(gl::mul(w7, h), k1, r);
        return r;
    }
};

// ---- inverse_CFD_sampling: grid-refinement.h:137-189 -----------------------------------------
// pdf(x) functor; writes num nodes to x_out.  x_i / cdf_i: n_samp doubles each, kk: 8 doubles.
// Returns the number of quadrature attempts (6 pdf evaluations each): the work counter behind bench.py's K0 roofline entry.
template <int VARIANT, class Par, class Pdf>
VAG_HD int inverse_cdf_sampling(const Par& par, const Pdf& pdf, double lo, double hi, int num, bool log_sample,
                                bool midpoint, double* x_out, double* x_i, double* cdf_i, double* kk) {
    constexpr int n_samp = dflt::theta_samples;
    constexpr double rtol = dflt::ode_rtol;
    {
        const double a = log_sample ? gl::log10(lo) : lo, b = log_sample ? gl::log10(hi) : hi;
        par.for_each(n_samp, [&](int i) {
            const double v = linspace_at(a, b, n_samp, i);
            x_i[i] = log_sample ? gl::pow(10.0, v) : v;
            cdf_i[i] = 0;
        });
    }
    CdfQuad<VARIANT> st;
    st.initialize(lo, gl::mul(gl::sub(hi, lo), 1.0 / 1e3));
    int k = 1, attempts = 0, steps = 0, fails = 0;
    // one attempt per round: while st.t <= hi, up to 500 attempts per step, at most max_ode_steps accepted steps
    par.lockstep(st.t <= hi, [&]() {
        if (!st.deriv_ready) {
            st.k1 = pdf(st.t);
            st.deriv_ready = true;
        }
        const double t0 = st.t, dt = st.dt;
        // the six stage evaluations of an attempt are independent (a pure quadrature): one lane each
        par.for_each(6, [&](int s) { kk[s] = pdf(CdfQuad<VARIANT>::stage_time(t0, dt, s)); });
        ++attempts;
        if (!st.try_step(kk, rtol)) return ++fails < 500;
        fails = 0;
        if (++steps > dflt::max_ode_steps) return false;
        // dense output for every sample abscissa the accepted step passed
        // m = number of sample abscissae the step passed: first q >= k with !(st.t > x_i[q]), searched G at a time
        const double t_now = st.t;
        const int m = par.first_true(k, n_samp, [&](int q) { return !(t_now > x_i[q]); }) - k;
        if (m > 0) {
            const int k0 = k;
            par.for_each(m, [&](int i) { cdf_i[k0 + i] = st.calc_state(x_i[k0 + i]); });
            k += m;
        }
        return st.t <= hi;
    });
    const double c0 = cdf_i[0], c1 = cdf_i[n_samp - 1];
    // first j with target <= cdf_i[j].  A lane visits its queries in ascending q, hence (c1 >= c0) ascending target, and
    // every sample below the previous hit has already failed the test for a smaller target: the scan resumes there
    // instead of restarting at 0 (same result as the reference's scan from 0 for any cdf_i, monotone or not).
    int j_resume = 0;
    double target_prev = -kInf;
    par.for_each(num, [&](int q) {
        // midpoint quantiles: front + (back - front) * (q + 0.5) / num, evaluated lazily by xtensor per element
        const double target = midpoint ? gl::add(c0, gl::div(gl::mul(gl::sub(c1, c0), gl::add((double)q, 0.5)), (double)num))
                                       : linspace_at(c0, c1, num, q);
        int j = (target >= target_prev) ? j_resume : 0;
        for (;;) {  // the sequential scan, four candidates per round: independent loads, tests in scan order
            const int last = n_samp - 1;
            const double c0 = cdf_i[imin(j, last)], c1 = cdf_i[imin(j + 1, last)], c2 = cdf_i[imin(j + 2, last)],
                         c3 = cdf_i[imin(j + 3, last)];
            if (!(j < n_samp) || target <= c0) break;
            if (!(j + 1 < n_samp) || target <= c1) {
                j += 1;
                break;
            }
            if (!(j + 2 < n_samp) || target <= c2) {
                j += 2;
                break;
            }
            if (!(j + 3 < n_samp) || target <= c3) {
                j += 3;
                break;
            }
            j += 4;
        }
        j_resume = j;
        target_prev = target;
        double xo = 0;
        if (j < n_samp) {
            if (j == 0) {
                xo = x_i[0];
            } else {
                const double denom = gl::sub(cdf_i[j], cdf_i[j - 1]);
                if (denom > 0) {
                    const double slope = gl::div(gl::sub(x_i[j], x_i[j - 1]), denom);
                    xo = gl::fma(slope, gl::sub(target, cdf_i[j - 1]), x_i[j - 1]);
                } else {
                    xo = x_i[j - 1];
                }
            }
        }
        x_out[q] = xo;
    });
    return attempts;
}

// ---- adaptive_theta_grid: grid-refinement.h:199-291 ------------------------------------------
struct ThetaPdf {
    const ModelCfg& m;
    double theta_v, cw_Gpsq, vw_Gvsq, Gamma_peak_sq, Gamma_v_sq, doppler_alpha, floor_weight;
    VAG_HD double operator()(double theta) const {
        const double Gamma = jet_Gamma0<true>(m, theta);
        const double dtheta = gl::sub(theta, theta_v);
        const double beta = gamma_to_beta_x(Gamma);
        const double c = gl::cos(dtheta);
        const double doppler = gl::div(gl::sub(1.0, beta), gl::fnma(c, beta, 1.0));
        const double structure = structure_weight(Gamma);
        const double a1 = gl::fma(doppler, doppler_alpha, 1.0);
        const double core = gl::div(gl::mul(cw_Gpsq, theta), gl::fma(gl::mul(Gamma_peak_sq, theta), theta, 1.0));
        const double view = gl::div(gl::mul(vw_Gvsq, fabs(dtheta)), gl::fma(gl::mul(dtheta, Gamma_v_sq), dtheta, 1.0));
        return gl::add(gl::fma(a1, structure, gl::add(view, core)), floor_weight);
    }
};

// scratch: A[>=101], B[>=101], samples x_i/cdf_i [2*theta_samples], kk[8]
template <class Par>
VAG_HD int adaptive_theta_grid(const Par& par, const ModelCfg& m, double theta_min, double theta_max, int base_pts,
                               double theta_v, double theta_resol, double* out, int cap, double* A, double* B,
                               double* samp, double* kk, int* attempts = nullptr) {
    constexpr double core_beam_coeff = 55.0, view_beam_coeff = 25.0, doppler_alpha0 = 12.0, floor_fraction = 0.25;
    constexpr int scan_pts = 100;
    const double theta_extent = gl::sub(theta_max, theta_min);
    double peak_weight = 0, Gamma_peak = 1.0, struct_sum = 0, Gamma_v = 1.0;
    int last_bright = 0;
    par.for_each(scan_pts + 1, [&](int i) {
        const double theta = gl::fma(gl::mul((double)i, theta_extent), 0.01, theta_min);
        const double Gamma = jet_Gamma0(m, theta);
        const double dth = gl::sub(theta, theta_v);
        A[i] = Gamma;
        B[i] = gl::div(Gamma, gl::sqrt(gl::fma(gl::mul(gl::mul(Gamma, Gamma), dth), dth, 1.0)));
    });
    for (int i = 0; i <= scan_pts; ++i) {
        const double Gamma = A[i];
        const double w = structure_weight(Gamma);
        struct_sum = gl::add(struct_sum, w);
        if (w > peak_weight) {
            peak_weight = w;
            Gamma_peak = Gamma;
            last_bright = i;
        } else if (w > gl::mul(peak_weight, 0.01)) {
            last_bright = i;
        }
        Gamma_v = vmax(Gamma_v, B[i]);
    }
    const double floor_weight = gl::mul(floor_fraction, peak_weight);
    const double CDF_est = gl::mul(theta_extent, gl::fma(struct_sum, 0.01, floor_weight));
    const double theta_bright = gl::fma(gl::mul((double)last_bright, theta_extent), 0.01, theta_min);

    Gamma_peak = vmax(Gamma_peak, Gamma_v);
    const double sw_v = structure_weight(Gamma_v);
    const double doppler_alpha = gl::mul(gl::sqrt((1.0 > sw_v) ? peak_weight : gl::div(peak_weight, sw_v)), doppler_alpha0);

    const double Gamma_peak_sq = gl::mul(Gamma_peak, Gamma_peak);
    const double Gamma_v_sq = gl::mul(Gamma_v, Gamma_v);
    // compute_beam_pts(log_decades, coeff, offset) = size_t(max(0, log_decades - offset) * resol * coeff)
    auto decades = [&](double arg, double offset) {  // max(0, log10(max(1, arg)) - offset)
        if (!(arg > 1.0)) return 0.0;
        const double d = gl::sub(gl::log10(arg), offset);
        return (d > 0.0) ? d : 0.0;
    };
    const double core_real =
        gl::mul(gl::mul(decades(gl::mul(gl::sub(theta_bright, theta_min), Gamma_peak), 1.0), theta_resol), core_beam_coeff);
    const long long core_beam_pts = (long long)core_real;
    const double theta_v_left = gl::sub(theta_v, theta_min);
    const double theta_v_right = gl::sub(theta_max, theta_v);
    double view_real = 0;
    long long view_beam_pts = 0;
    if (gl::mul(theta_v, Gamma_peak) > 3.0) {
        view_real = gl::mul(gl::mul(decades(gl::mul(vmax(theta_v_left, theta_v_right), Gamma_v), 0.0), theta_resol), view_beam_coeff);
        view_beam_pts = (long long)view_real;
    }
    const long long total_pts = base_pts + core_beam_pts + view_beam_pts;
    if (total_pts > cap) return -(int)total_pts;

    auto calibrate = [&](long long n_pts, double beam_cdf) -> double {
        return (n_pts > 0 && beam_cdf > 0) ? gl::div(gl::mul(gl::div((double)n_pts, (double)base_pts), CDF_est), beam_cdf) : 0.0;
    };
    const double core_cdf = gl::mul(
        gl::log(gl::div(gl::fma(gl::mul(theta_max, Gamma_peak_sq), theta_max, 1.0), gl::fma(gl::mul(theta_min, Gamma_peak_sq), theta_min, 1.0))),
        0.5);
    const double core_weight = calibrate(core_beam_pts, core_cdf);
    const double view_cdf = gl::mul(gl::add(gl::log(gl::fma(gl::mul(Gamma_v_sq, theta_v_right), theta_v_right, 1.0)),
                                            gl::log(gl::fma(gl::mul(theta_v_left, Gamma_v_sq), theta_v_left, 1.0))),
                                    0.5);
    const double view_weight = calibrate(view_beam_pts, view_cdf);

    const ThetaPdf pdf{m,          theta_v,      gl::mul(Gamma_peak_sq, core_weight), gl::mul(Gamma_v_sq, view_weight), Gamma_peak_sq,
                       Gamma_v_sq, doppler_alpha, floor_weight};
    // an Ejecta's profile is a std::function call the optimiser cannot see through: the stage states stay alive (VARIANT 1)
    int na;
    if (m.ejecta)
        na = inverse_cdf_sampling<1>(par, pdf, theta_min, theta_max, (int)total_pts, /*log=*/true, /*midpoint=*/false, out, samp,
                                     samp + dflt::theta_samples, kk);
    else
        na = inverse_cdf_sampling<0>(par, pdf, theta_min, theta_max, (int)total_pts, /*log=*/true, /*midpoint=*/false, out, samp,
                                     samp + dflt::theta_samples, kk);
    if (attempts) *attempts = na;
    return (int)total_pts;
}

// ---- jump_refinement_grid (grid-refinement.cpp:140-164) + merge_grids (grid-refinement.h:362-393)
VAG_HD int jump_refinement_grid(const double* jumps, int n_jumps, double theta_min, double theta_max,
                                double avg_spacing, double* pts) {
    int n = 0;
    const double tight = avg_spacing * 0.125;
    for (int idx = 0; idx < n_jumps; ++idx) {
        const double jt = jumps[idx];
        if (jt >= con::pi / 2 - 0.01) continue;
        if (jt - tight >= theta_min) pts[n++] = jt - tight;
        if (jt + tight <= theta_max) pts[n++] = jt + tight;
        if (jt >= theta_min && jt <= theta_max) pts[n++] = jt;
    }
    // sort + unique (tiny n: insertion sort)
    for (int i = 1; i < n; ++i) {
        const double v = pts[i];
        int j = i - 1;
        while (j >= 0 && pts[j] > v) {
            pts[j + 1] = pts[j];
            --j;
        }
        pts[j + 1] = v;
    }
    int u = 0;
    for (int i = 0; i < n; ++i)
        if (u == 0 || pts[u - 1] != pts[i]) pts[u++] = pts[i];
    return u;
}

VAG_HD int merge_grids(const double* a, int na, const double* b, int nb, double* out, int cap) {
    int n = 0, i = 0, j = 0;
    double last = 0;
    auto add_unique = [&](double v) {
        if (n == 0 || last != v) {
            if (n < cap) out[n] = v;
            last = v;
            ++n;
        }
    };
    while (i < na && j < nb) {
        if (a[i] <= b[j]) {
            add_unique(a[i++]);
            if (a[i - 1] == b[j]) j++;
        } else {
            add_unique(b[j++]);
        }
    }
    while (i < na) add_unique(a[i++]);
    while (j < nb) add_unique(b[j++]);
    return n;
}

// ---- adaptive_phi_grid: grid-refinement.h:295-360 --------------------------------------------
// Per-theta invariants (beta, structure weight, cos/sin theta, dcos) are hoisted out of the
// pdf: every typed jet is phi-independent, so the hoisted values are the ones the reference
// recomputes inside phi_weight on every call.
struct PhiPdf {
    const double *beta, *sw, *dcos, *ct_ctv, *st_stv;  // beta, structure weight, dcos, cos(theta), sin_tv sin(theta)
    int n_theta;
    double cos_tv, floor_weight;
    VAG_HD double weight(double phi) const {
        const double cos_phi = gl::cos(phi);
        double w = 0;
        for (int it = 0; it < n_theta; ++it) {
            // cos_alpha = fma(cos_tv, cos(theta), (sin_tv sin(theta)) cos_phi);  a = (1 - beta) / fnma(cos_alpha, beta, 1)
            const double cos_alpha = gl::fma(cos_tv, ct_ctv[it], gl::mul(st_stv[it], cos_phi));
            const double a = gl::div(gl::sub(1.0, beta[it]), gl::fnma(cos_alpha, beta[it], 1.0));
            w = gl::fma(gl::mul(sw[it], a), dcos[it], w);
        }
        return w;
    }
    VAG_HD double operator()(double phi) const { return gl::add(weight(phi), floor_weight); }
};

// scratch: per-theta arrays pt[5*n_theta], A[>=101], samples [2*theta_samples], kk[8]
template <class Par>
VAG_HD int adaptive_phi_grid(const Par& par, const ModelCfg& m, int phi_num, double theta_v, const double* theta,
                             int n_theta, bool is_axisymmetric, double phi_max, double self_boost_cap, double* out,
                             int cap, double* pt, double* A, double* samp, double* kk, int* attempts = nullptr) {
    if (theta_v == 0 && is_axisymmetric) {
        if (phi_num > cap) return -phi_num;
        par.for_each(phi_num, [&](int i) { out[i] = linspace_at(0., 2 * con::pi, phi_num, i); });
        return phi_num;
    }
    const bool half_range = phi_max < 2 * con::pi;
    double* beta = pt;
    double* sw = beta + n_theta;
    double* ct = sw + n_theta;      // cos(theta)
    double* st = ct + n_theta;      // sin_tv * sin(theta)
    double* dcos_arr = st + n_theta;
    const double cos_tv = gl::cos(theta_v), sin_tv = gl::sin(theta_v);
    par.for_each(n_theta, [&](int it) {
        const double left = (it == 0) ? 0.0 : 0.5 * (theta[it - 1] + theta[it]);
        const double right = (it == n_theta - 1) ? theta[it] : 0.5 * (theta[it] + theta[it + 1]);
        dcos_arr[it] = fabs(gl::sub(gl::cos(left), gl::cos(right)));
        const double Gamma = jet_Gamma0(m, theta[it]);
        beta[it] = gamma_to_beta_x(Gamma);
        sw[it] = structure_weight(Gamma);
        ct[it] = gl::cos(theta[it]);
        st[it] = gl::mul(sin_tv, gl::sin(theta[it]));
    });
    PhiPdf pdf{beta, sw, dcos_arr, ct, st, n_theta, cos_tv, 0.0};

    constexpr int scan_pts = 100;
    par.for_each(scan_pts + 1, [&](int s) { A[s] = pdf.weight(gl::mul(gl::mul(phi_max, (double)s), 0.01)); });
    double peak_weight = 0, sum_weight = 0;
    for (int s = 0; s <= scan_pts; ++s) {
        peak_weight = vmax(peak_weight, A[s]);
        sum_weight = gl::add(sum_weight, A[s]);
    }
    const double floor_weight = gl::mul(0.05, peak_weight);
    if (self_boost_cap > 0 && peak_weight > 0) {
        const double mean_pdf = gl::fma(sum_weight, 1.0 / (scan_pts + 1), floor_weight);
        const double concentration = gl::div(gl::add(peak_weight, floor_weight), mean_pdf);
        const double boost = vclamp(gl::mul(concentration, 0.2), 1.0, self_boost_cap);
        phi_num = (int)(long long)gl::mul((double)phi_num, boost);
    }
    if (phi_num > cap) return -phi_num;
    pdf.floor_weight = floor_weight;
    const int na = inverse_cdf_sampling<1>(par, pdf, 0, phi_max, phi_num, /*log=*/false, /*midpoint=*/half_range, out, samp,
                                           samp + dflt::theta_samples, kk);
    if (attempts) *attempts = na;
    return phi_num;
}

// ---- estimate_t_dec: grid-refinement.h:401-453 -----------------------------------------------
VAG_HD double estimate_t_dec(const ModelCfg& m, double theta) {
    const double gamma = jet_Gamma0(m, theta);
    const double beta = gamma_to_beta(gamma);
    double m_jet = jet_eps_k(m, theta) / (gamma * con::c2);
    m_jet /= (1.0 + m.sigma0);  // HasSigma branch (grid-refinement.h:407-409); exact no-op for sigma0 = 0
    const double target = m_jet / gamma;
    constexpr double r_min = 1e-3;
    const double r_max = r_min * pow(10.0, 40.0);
    if (target <= 0) return r_min * (1 - beta) / (beta * con::c);

    if (m.medium_type == VAG_MEDIUM_ISM) {
        const double rho = m.rho_ism;
        if (rho > 0) {
            const double r3_dec = r_min * r_min * r_min + 3 * target / rho;
            const double r_dec = cbrt(vmax(r3_dec, 0.0));
            return vmin(r_dec, r_max) * (1 - beta) / (beta * con::c);
        }
        return r_max * (1 - beta) / (beta * con::c);
    }
    constexpr int N = 256;
    const double u_min = log(1e-3);
    const double u_max = u_min + 40 * log(10.0);
    const double du = (u_max - u_min) / N;
    double mass = 0;
    double r_prev = exp(u_min);
    double f_prev = medium_rho(m, r_prev) * r_prev * r_prev;
    for (int i = 1; i <= N; ++i) {
        const double r_i = exp(u_min + i * du);
        const double f_i = medium_rho(m, r_i) * r_i * r_i;
        const double dr = r_i - r_prev;
        mass += 0.5 * (f_prev + f_i) * dr;
        if (mass >= target) {
            const double r_dec = r_prev + (target - (mass - 0.5 * (f_prev + f_i) * dr)) / f_i;
            return r_dec * (1 - beta) / (beta * con::c);
        }
        f_prev = f_i;
        r_prev = r_i;
    }
    return exp(u_max) * (1 - beta) / (beta * con::c);
}

// ---- time lattice: grid-refinement.h:516-581, grid-refinement.cpp:166-197 ---------------------
VAG_HD double logspace_at(double la, double lb, int n, int i) { return pow(10.0, linspace_at(la, lb, n, i)); }

// The lattice builders fill grid[idx] for idx = tid, tid + nthr, ... (tid = 0, nthr = 1: the whole row): every node is
// an independent expression of the segment bounds, so a warp builds a row's lattice in parallel (k_lattice).
// logspace_with_band_refinement(ts, t_end, b_lo, b_hi, n, factor) -> grid[n]
VAG_HD void logspace_with_band_refinement(double ts, double t_end, double b_lo, double b_hi, int n, double factor,
                                          double* grid, int tid = 0, int nthr = 1) {
    b_lo = vmax(b_lo, ts);
    b_hi = vmin(b_hi, t_end);
    if (!(b_hi > b_lo) || n < 8) {
        const double la = log10(ts), lb = log10(t_end);
        for (int i = tid; i < n; i += nthr) grid[i] = logspace_at(la, lb, n, i);
        return;
    }
    const double l0 = log10(ts), l1 = log10(b_lo), l2 = log10(b_hi), l3 = log10(t_end);
    const double w1 = l1 - l0, w2 = factor * (l2 - l1), w3 = l3 - l2;
    const long long segs = n - 1;
    long long n1 = (long long)round((double)segs * w1 / (w1 + w2 + w3));
    long long n3 = (long long)round((double)segs * w3 / (w1 + w2 + w3));
    n1 = n1 < segs - 2 ? n1 : segs - 2;
    n3 = n3 < segs - 1 - n1 - 1 ? n3 : segs - 1 - n1 - 1;
    const long long n2 = segs - n1 - n3;
    for (long long idx = tid; idx < n1 + n2 + n3 + 1; idx += nthr) {
        double v;
        if (idx < n1) {
            v = pow(10.0, l0 + (l1 - l0) * (double)idx / (double)n1);
        } else if (idx < n1 + n2) {
            v = pow(10.0, l1 + (l2 - l1) * (double)(idx - n1) / (double)n2);
        } else {
            const long long k = idx - n1 - n2;
            v = pow(10.0, (n3 > 0) ? l2 + (l3 - l2) * (double)k / (double)n3 : l3);
        }
        grid[idx] = v;
    }
}

// logspace_with_cross_refinement(t_start, t_end, t_refine, t_num, base_t_num) -> grid[t_num]
VAG_HD void logspace_with_cross_refinement(double t_start, double t_end, double t_refine, int t_num, int base_t_num,
                                           double* grid, int tid = 0, int nthr = 1) {
    t_refine = vclamp(t_refine, t_start, t_end);
    if (t_refine <= t_start || t_refine >= t_end) {
        const double la = log10(t_start), lb = log10(t_end);
        for (int i = tid; i < t_num; i += nthr) grid[i] = logspace_at(la, lb, t_num, i);
        return;
    }
    const double log_total = log10(t_end / t_start);
    const double log_after = log10(t_end / t_refine);
    long long n_post = (long long)((double)base_t_num * log_after / log_total);
    if (n_post < 2) n_post = 2;
    if (n_post >= t_num) n_post = t_num / 2;
    const long long n_pre = t_num + 1 - n_post;
    const double la0 = log10(t_start), lb0 = log10(t_refine), lb1 = log10(t_end);
    // nodes [0, n_pre): first segment; then k = 1 .. n_post - 1 of the second while the array has room; the rest stay 0
    for (long long idx = tid; idx < t_num; idx += nthr) {
        double v = 0;
        if (idx < n_pre) {
            v = logspace_at(la0, lb0, (int)n_pre, (int)idx);
        } else {
            const long long k = idx - n_pre + 1;
            if (k < n_post) v = logspace_at(lb0, lb1, (int)n_post, (int)k);
        }
        grid[idx] = v;
    }
}

// Lattice of one representative row: make_time_grid + store_time_grid (grid-refinement.h:571-591).
// Symmetric models share the global start / early point; a `structured` (spreading) model gives every
// row its own (build_time_grid, grid-refinement.h:612-619): row_start = max(t_raw, cut),
// row_early = 0.99 min(t_raw, cut), left by build_grid in the model's scratch slab.
VAG_HD void build_row_lattice(const GridHeader& h, double t_dec, double T0, double row_start, double row_early,
                              double* t_row, int tid = 0, int nthr = 1) {
    double* grid = t_row + (h.has_early ? 1 : 0);
    const double ts = h.structured ? row_start : h.min_t_start;
    if (h.is_rvs) {
        const double t_cross_limit = vmax(t_dec, T0);
        logspace_with_cross_refinement(ts, h.t_end, 10 * t_cross_limit, h.t_num_tot, h.t_num_base, grid, tid, nthr);
    } else {
        logspace_with_band_refinement(ts, h.t_end, t_dec / 3, 3 * t_dec, h.t_num_tot, 3.0, grid, tid, nthr);
    }
    if (h.has_early && tid == 0) t_row[0] = h.structured ? row_early : h.min_t_early;
}

// scan_time_bounds (grid-refinement.h:471-514): raw lattice start of cell (phi_i, theta_j)
VAG_HD double raw_row_start(const ModelCfg& m, double t_obs_min, double th, double G, double cos_tv, double sin_tv,
                            double phi) {
    const double b = gamma_to_beta(G);
    const double cos_a = cos(th) * cos_tv + sin(th) * sin_tv * cos(phi);
    return 0.99 * t_obs_min * (1 - b) / (1 - cos_a * b) / (1 + m.z);
}
// lattice guard of theta row j (same source): min(0.01 t_dec, 1e-2 s[, 0.01 T0 with a reverse shock])
VAG_HD double row_start_cut(const ModelCfg& m, bool is_rvs, double t_dec) {
    double cut = vmin(0.01 * t_dec, 1e-2 * unit::sec);
    if (is_rvs) cut = vmin(cut, 0.01 * m.T0);
    return cut;
}

// ---- auto_grid: grid-refinement.h:638-706 (axisymmetric, typed jets) --------------------------
template <class Par>
VAG_HD void build_grid(const Par& par, const ModelCfg& m, double t_obs_min, double t_obs_max, GridHeader& h,
                       const GridSlab& s) {
    h.status = 0;
    h.is_rvs = m.has_rvs ? 1 : 0;
    const double theta_view = m.theta_v;
    const double theta_cut = con::pi / 2;
    auto fail_capacity = [&]() {
        h.status |= VAG_ST_CAPACITY;
        h.n_theta = h.n_phi = h.n_phi_eff = h.n_t = h.n_reps = 0;
    };

    // scratch carve-up (grid_work_doubles)
    double* base_theta = s.work;                       // [cap_theta]
    double* pt = base_theta + s.cap_theta;             // [5*cap_theta] per-theta arrays
    double* A = pt + 5 * (size_t)s.cap_theta;          // [GRID_NSCAN+7]
    double* B = A + (GRID_NSCAN + 7);                  // [GRID_NSCAN+7]
    double* samp = B + (GRID_NSCAN + 7);               // [2*theta_samples]
    double* kk = samp + 2 * dflt::theta_samples;       // [8]

    // A steep smooth profile trips the jump test too (adjacent scan nodes differing by more than half):
    // a Gaussian core of theta_c ~ 0.014 rad yields 14 "jumps", the most any typed profile produces.
    constexpr int JUMP_CAP = 48;
    double jumps[JUMP_CAP];
    const int n_jumps = find_jet_jumps(par, m, con::Gamma_cut, jumps, JUMP_CAP, A);
    if (n_jumps < 0) return fail_capacity();
    double inner_edge, outer_edge;
    find_theta_range(par, m, con::Gamma_cut, inner_edge, outer_edge);
    for (int i = 0; i < n_jumps; ++i) outer_edge = vmax(outer_edge, jumps[i]);
    const double theta_min = vmax(dflt::theta_min, inner_edge);
    const double theta_max = vmin(outer_edge, theta_cut);

    const int theta_num =
        dflt::min_theta_points + (int)(long long)((theta_max - theta_min) * 180 / con::pi * m.theta_resol);

    h.quad_attempts_theta = h.quad_attempts_phi = 0;
    const int n_base = adaptive_theta_grid(par, m, theta_min, theta_max, theta_num, theta_view, m.theta_resol,
                                           base_theta, s.cap_theta, A, B, samp, kk, &h.quad_attempts_theta);
    if (n_base < 0) return fail_capacity();
    const double avg_spacing = (theta_max - theta_min) / n_base;
    double feat[3 * JUMP_CAP];
    const int n_feat = jump_refinement_grid(jumps, n_jumps, theta_min, theta_max, avg_spacing, feat);
    const int n_theta = merge_grids(base_theta, n_base, feat, n_feat, s.theta, s.cap_theta);
    if (n_theta > s.cap_theta) return fail_capacity();
    h.n_theta = n_theta;

    // phi grid (grid-refinement.h:664-693)
    const bool axis = m.axisymmetric != 0;
    const long long phi_base_ll = (long long)(360 * m.phi_resol);
    const int phi_base = (int)(phi_base_ll > 1 ? phi_base_ll : 1);
    const bool mirror_phi = axis && theta_view != 0 && phi_base > 4;
    int n_phi;
    if (mirror_phi) {
        const int n_half = (phi_base + 1) / 2;
        n_phi = adaptive_phi_grid(par, m, n_half, theta_view, s.theta, n_theta, axis, con::pi, 5.0, s.phi, s.cap_phi, pt,
                                  A, samp, kk, &h.quad_attempts_phi);
        h.phi_mirrored = 1;
    } else {
        const double doppler_sharpness = jet_Gamma0(m, theta_view) * sin(theta_view);
        const double phi_boost = sqrt(vmax(doppler_sharpness / (2 * con::pi), 1.0));
        long long phi_num = (long long)(phi_base * phi_boost);
        if (phi_num < 1) phi_num = 1;
        if (phi_num > (long long)phi_base * 5) phi_num = (long long)phi_base * 5;
        if (phi_num <= 2) {
            n_phi = (int)phi_num;
            if (n_phi <= s.cap_phi)
                for (int i = 0; i < n_phi; ++i) s.phi[i] = linspace_at(0., 2 * con::pi, n_phi, i);
            else
                n_phi = -n_phi;
        } else {
            n_phi = adaptive_phi_grid(par, m, (int)phi_num, theta_view, s.theta, n_theta, axis, 2 * con::pi, 0.0, s.phi,
                                      s.cap_phi, pt, A, samp, kk, &h.quad_attempts_phi);
        }
        if (n_phi >= 2) {
            const double shift = 0.5 * (s.phi[1] - s.phi[0]);
            const int np = n_phi;
            par.for_each(1, [&](int) {
                for (int i = 0; i < np; ++i) s.phi[i] += shift;
            });
        }
        h.phi_mirrored = 0;
    }
    if (n_phi < 0) return fail_capacity();
    h.n_phi = n_phi;
    // Observer::build_time_grid (src/core/observer.cpp:211-222): axisymmetric shock tables have
    // phi extent 1 (jet_3d = 0), so an on-axis observer needs a single phi sample; with
    // axisymmetric=False the tables carry every phi (jet_3d = 1) and all of them are observed.
    h.n_phi_eff = (theta_view == 0 && axis) ? 1 : n_phi;

    // jet_spreading_edge (grid-refinement.h:113-135): angle of the steepest decline of Gamma0 between the
    // first and last theta node.  The walk's nodes are a running sum; the profile is evaluated at all of
    // them (and their clamped neighbours) in parallel, the minimum is taken in walk order.
    h.spreading = m.spreading;
    h.structured = m.structured;
    h.theta_s = 0;
    if (m.spreading) {
        const double th_min = s.theta[0], th_max = s.theta[n_theta - 1];
        const double step = (th_max - th_min) / 256;
        int nn = 0;
        for (double th = th_min; th <= th_max && nn < GRID_NSCAN + 6; th += step) A[nn++] = th;
        {
            const int cnt = nn;
            par.for_each(cnt, [&](int q) {
                const double th = A[q];
                const double lo = vmax(th - step, th_min), hi = vmin(th + step, th_max);
                B[q] = (jet_Gamma0(m, hi) - jet_Gamma0(m, lo)) / (hi - lo);
            });
        }
        double theta_s = th_min, dp_min = 0;
        for (int q = 0; q < nn; ++q)
            if (B[q] < dp_min) {
                dp_min = B[q];
                theta_s = A[q];
            }
        if (dp_min == 0) theta_s = th_max;
        h.theta_s = theta_s;
    }

    // detect_symmetry (mesh.h:120-185): a spreading jet is `structured` (every theta row is solved)
    // per-theta probes in parallel: pt[0..n) = eps_k, pt[n..2n) = Gamma0, then an ordered scan.
    double* e_arr = pt;
    double* g_arr = pt + n_theta;
    double* ts_arr = pt + 2 * (size_t)n_theta;
    const double t_end = 1.01 * t_obs_max / (1 + m.z);
    const double cos_tv = cos(theta_view), sin_tv = sin(theta_view);
    // scan_time_bounds walks phi_size = (axisymmetric ? 1 : N_phi) azimuths (grid-refinement.h:597,484-511);
    // every bound it keeps is monotone in the raw start time, so the per-theta minimum over phi suffices
    const int n_phi_scan = axis ? 1 : n_phi;
    par.for_each(n_theta, [&](int j) {
        const double th = s.theta[j];
        const double G = jet_Gamma0(m, th);
        e_arr[j] = jet_eps_k(m, th);
        g_arr[j] = G;
        // scan_time_bounds (grid-refinement.h:471-514): raw start time of cell (i, j)
        double ts_min = kInf;
        for (int i = 0; i < n_phi_scan; ++i) ts_min = vmin(ts_min, raw_row_start(m, t_obs_min, th, G, cos_tv, sin_tv, s.phi[i]));
        ts_arr[j] = ts_min;
    });
    int n_reps = 0;
    s.reps[n_reps++] = 0;
    for (int j = 1; j < n_theta; ++j)
        if (m.structured || e_arr[j - 1] != e_arr[j] || g_arr[j - 1] != g_arr[j]) s.reps[n_reps++] = j;
    h.n_reps = n_reps;
    h.symmetry = m.structured ? SYM_STRUCTURED
                             : (n_reps == 1) ? SYM_ISOTROPIC : (n_reps < n_theta ? SYM_PIECEWISE : SYM_PHI_SYMMETRIC);

    // build_time_grid (grid-refinement.h:593-636) with phi_size = 1.  t_dec only depends on
    // (eps_k, Gamma0), so it is evaluated once per representative group.
    {
        const int nr = n_reps;
        par.for_each(nr, [&](int r) { s.t_dec[r] = estimate_t_dec(m, s.theta[s.reps[r]]); });
    }
    double min_raw = t_end, min_guarded = t_end, min_cut = t_end, max_ref = 0;
    {
        int r = -1;
        double td = 0;
        for (int j = 0; j < n_theta; ++j) {
            if (r + 1 < n_reps && s.reps[r + 1] == j) td = s.t_dec[++r];
            const double ts = ts_arr[j];
            const double cut = row_start_cut(m, h.is_rvs != 0, td);
            if (h.is_rvs) max_ref = vmax(max_ref, 10.0 * vmax(td, m.T0));
            min_raw = vmin(min_raw, ts);
            min_guarded = vmin(min_guarded, vmax(ts, cut));
            min_cut = vmin(min_cut, cut);
            if (m.structured) {  // per-row lattice bounds (TimeScanResult::t_start / early_t); e_arr is dead by now
                base_theta[j] = vmax(ts, cut);
                pt[j] = 0.99 * vmin(ts, cut);
            }
        }
    }
    h.min_t_early = min_raw;
    h.min_t_start = min_guarded;
    h.has_early = (min_raw < min_cut) ? 1 : 0;
    h.t_end = t_end;
    // compute_time_grid_size (grid-refinement.h:516-528)
    const long long t_num_base = (long long)(vmax(log10(t_end / min_guarded), 1.0) * m.t_resol);
    long long extra = 0;
    if (h.is_rvs && max_ref > min_guarded) {
        const double log_pre_span = log10(vmin(max_ref, t_end) / min_guarded);
        extra = (long long)((2.0 - 1.0) * log_pre_span * m.t_resol);
    }
    h.t_num_base = (int)t_num_base;
    h.t_num_tot = (int)(t_num_base + extra);
    h.n_t = h.t_num_tot + h.has_early;
    // structured + axisymmetric = False: every (phi, theta) cell is its own ODE row (k1_lattice_body derives the
    // row's lattice bounds from t_obs_min; the minima above already run over every phi)
    h.t_obs_min = t_obs_min;
    h.rows3d = (m.structured && !axis) ? 1 : 0;
    h.pad_ = 0;
    if (h.rows3d) h.n_reps = n_phi * n_theta;
}

}  // namespace vag
