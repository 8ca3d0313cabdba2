// vag_observer.cuh -- K3: equal-arrival-time-surface flux integration for one model.
//
// Restates Observer::observe for non-spreading axisymmetric jets (calc_eat_non_spreading +
// finalize_log_grids, src/core/observer.cpp:143-205,439-454; compute_dphi :17-37) fused with
// Observer::specific_flux (src/core/observer.h:355-445, grid form) and specific_flux_series
// (:447-538, series form).  The reference materialises lg2_t / lg2_doppler / lg2_geom_factor for
// every (phi,theta,t) cell and a broadcast photon object per cell; here the EAT geometry is
// recomputed on the fly per row from the UNIQUE shock rows, staged in shared memory together with
// the per-node log2-luminosities, and never written to HBM.
//
// The work of one CTA is expressed as barrier-separated phases, each an HD function of the
// thread index, so the same code runs as a CUDA block (vag_b200.cu) and as a sequential
// host emulation in the CPU test-suite (oracle/hostemu).
#pragma once

#include "vag_grid.cuh"
#include "vag_ic.cuh"
#include "vag_radiation.cuh"

namespace vag {

constexpr int EATS_NU_TILE = 8;     // frequencies handled per pass in grid mode
constexpr int EATS_ROW_CHUNK = 8;   // max (phi,theta) rows staged per pass

// Everything the EATS stage needs about one model (device pointers into the batch workspace).
struct EatsModel {
    const GridHeader* h;
    const double* theta;     // [n_theta]
    const double* phi;       // [n_phi]
    const int* rep_of;       // [n_theta] -> index of the representative row of theta_j
    const double* t_rows;    // [n_reps][n_t] engine-frame lattice
    const double* r;         // [n_reps][n_t]
    const double* Gamma;     // [n_reps][n_t]
    const double* geo_u;     // [n_reps][n_t] sqrt((Gamma-1)(Gamma+1))
    const double* geo_lg2r2; // [n_reps][n_t] 2 log2(r)
    const double* coef;      // [PH_NCOEF][n_reps][n_t]  photon coefficients (SoA)
    long coef_stride;        // distance between coefficient planes (= total cells of the batch)
    double smooth_thick, log2_x_far;
    double one_plus_z, lumi_dist, theta_v;
    // emission model of this pass: 0 synchrotron, 1 synchrotron with the IC correction of a shock
    // with ssc=True, 2 SSC (per-cell tables)
    int mode;
    const IcCell* ic;         // [n_reps][n_t]
    const IcTable* ictab_h;   // [n_reps][n_t]
    const double* ictab;      // [n_reps][n_t][IC_CAP_OUT]
    int* breach;              // model status word: gets VAG_ST_IC_BAND when an SSC query leaves the clamped band
    const double* sp_lut;     // log2_softplus table (vag_math.cuh), in shared memory on the device
    // spreading jets (calc_t_obs / calc_solid_angle, observer.cpp:51-141): theta varies along k, so the line
    // of sight cosine and the solid angle are per-node quantities built from these per-cell tables
    int spreading;
    const double* geo_cth;    // [n_reps][n_t] cos(theta(k))
    const double* geo_sth;    // [n_reps][n_t] sin(theta(k))
    const double* geo_dcos;   // [n_reps][n_t] cos(theta_hi(k)) - cos(theta_lo(k))
};

// compute_dphi: src/core/observer.cpp:17-37
VAG_HD double compute_dphi(const GridHeader& h, const double* phi, int i) {
    const int n = h.n_phi_eff;
    if (n == 1) return 2 * con::pi;
    const int last = n - 1;
    if (h.phi_mirrored) {
        const double left = (i > 0) ? 0.5 * (phi[i - 1] + phi[i]) : 0.0;
        const double right = (i < last) ? 0.5 * (phi[i] + phi[i + 1]) : con::pi;
        return 2 * (right - left);
    }
    return 0.5 * (phi[imin(i + 1, last)] - phi[i > 0 ? i - 1 : 0]);
}

// Row constants of calc_eat_non_spreading (observer.cpp:167-192): t_coeff and log2(dOmega)
// Spreading models reuse the record as (cos(phi) sin(theta_obs), cos(theta_obs), dphi, rep).
struct RowGeom {
    double cos_v, t_coeff, lg2_dOmega;
    int rep;  // representative row index
};

VAG_HD RowGeom row_geometry(const EatsModel& M, int i, int j) {
    const GridHeader& h = *M.h;
    const double cos_obs = cos(M.theta_v), sin_obs = sin(M.theta_v);
    const double cos_phi = cos(M.phi[i] - 0.0);  // coord.phi_view is never set by auto_grid: 0
    const double th = M.theta[j];
    const double ct = cos(th), st = sin(th);
    RowGeom g;
    if (M.spreading) {
        g.cos_v = cos_phi * sin_obs;
        g.t_coeff = cos_obs;
        g.lg2_dOmega = compute_dphi(h, M.phi, i);
        g.rep = h.rows3d ? i * h.n_theta + j : M.rep_of[j];
        return g;
    }
    g.cos_v = st * cos_phi * sin_obs + ct * cos_obs;
    g.t_coeff = (1 - g.cos_v) / con::c * M.one_plus_z;
    const int last = h.n_theta - 1;
    const double cos_th_lo = (j == 0) ? ct : cos(0.5 * (M.theta[j - 1] + th));
    const double cos_th_hi = (j == last) ? ct : cos(0.5 * (th + M.theta[j + 1]));
    const double dOmega = fabs((cos_th_hi - cos_th_lo) * compute_dphi(h, M.phi, i));
    g.lg2_dOmega = rlog2(dOmega);
    g.rep = h.rows3d ? i * h.n_theta + j : M.rep_of[j];
    return g;
}

// line-of-sight cosine of node o of a spreading row (observer.cpp:82)
VAG_HD double spread_cos_v(const EatsModel& M, const RowGeom& g, long o) {
    return M.geo_sth[o] * g.cos_v + M.geo_cth[o] * g.t_coeff;
}

// Linear observer time of node k of a row (observer.cpp:201; spreading: :87)
VAG_HD double node_time(const EatsModel& M, const RowGeom& g, int n_t, int k) {
    const long o = (long)g.rep * n_t + k;
    if (M.spreading) return (M.t_rows[o] + (1 - spread_cos_v(M, g, o)) * M.r[o] / con::c) * M.one_plus_z;
    return M.t_rows[o] * M.one_plus_z + g.t_coeff * M.r[o];
}

// log2 grids of one node: finalize_log_grids (observer.cpp:439-454) on the pre-logged geometry path, or on
// the linear dOmega r^2 of a spreading jet (observer.cpp:131-139)
// dop_lin = Gamma - u cos(v) = 2^-lg2_dop, the linear quantity the log was taken of
VAG_HD void node_logs(const EatsModel& M, const RowGeom& g, int n_t, int k, double& lg2_t, double& lg2_dop,
                      double& lg2_geom, double& dop_lin) {
    const long o = (long)g.rep * n_t + k;
    if (M.spreading) {
        const double cos_v = spread_cos_v(M, g, o);
        dop_lin = M.Gamma[o] - M.geo_u[o] * cos_v;
        const double time = (M.t_rows[o] + (1 - cos_v) * M.r[o] / con::c) * M.one_plus_z;
        const double dOmega = fabs(M.geo_dcos[o] * g.lg2_dOmega);
        lg2_dop = -rlog2(dop_lin);
        lg2_t = rlog2(time);
        lg2_geom = rlog2(dOmega * M.r[o] * M.r[o]) + 3.0 * lg2_dop;
        return;
    }
    dop_lin = M.Gamma[o] - M.geo_u[o] * g.cos_v;
    const double time = M.t_rows[o] * M.one_plus_z + g.t_coeff * M.r[o];
    lg2_dop = -rlog2(dop_lin);
    lg2_t = rlog2(time);
    lg2_geom = (g.lg2_dOmega + M.geo_lg2r2[o]) + 3.0 * lg2_dop;
}

// MODE is a compile-time copy of EatsModel::mode so that the plain synchrotron instantiation of
// k_eats carries no inverse-Compton code (registers, branches)
template <int MODE>
VAG_HD double cell_log2_I_nu(const EatsModel& M, int rep, int n_t, int k, double log2_nu) {
    const long cell = (long)rep * n_t + k;
    if (MODE == 2) {
        bool breach = false;
        const double v = ic_table_log2_I_nu(M.ictab_h[cell], M.ictab + (size_t)cell * IC_CAP_OUT, log2_nu, breach);
        if (breach && M.breach) {
#if defined(__CUDA_ARCH__)
            atomicOr(M.breach, VAG_ST_IC_BAND);
#else
            *M.breach |= VAG_ST_IC_BAND;
#endif
        }
        return v;
    }
    const double* base = M.coef + cell;
    const long stride = M.coef_stride;
    if (MODE == 1)
        return photon_log2_I_nu_ic([&](int c) { return base[c * stride]; }, M.smooth_thick, M.log2_x_far, M.ic[cell],
                                   log2_nu);
    const SynCoefRegs cr = load_syn_coefs([&](int c) { return base[c * stride]; });
    return photon_log2_I_nu_fast(cr, M.sp_lut, M.smooth_thick, M.log2_x_far, log2_nu);
}

// Interval lookup on a row's log2 observer-time lattice.
//   grid form   (iterate_to,      observer.h:309-313,405-433): t_row[k] <= x <  t_row[k+1]
//   series form (iterate_through, observer.h:316-320,494):     t_row[k] <  x <= t_row[k+1], x == t_row[0] -> k = 0
// Returns -1 when the row does not contribute to x.
VAG_HD int find_interval(const double* t_row, int n_t, double x, bool series) {
    if (!(x >= t_row[0])) return -1;
    int lo = 0, hi = n_t;  // count nodes (strictly) below / not above x
    if (series) {
        while (lo < hi) {  // cnt = #nodes < x
            const int mid = (lo + hi) >> 1;
            if (t_row[mid] < x)
                lo = mid + 1;
            else
                hi = mid;
        }
        const int k = lo > 0 ? lo - 1 : 0;
        return (k <= n_t - 2) ? k : -1;
    }
    while (lo < hi) {  // cnt = #nodes <= x
        const int mid = (lo + hi) >> 1;
        if (t_row[mid] <= x)
            lo = mid + 1;
        else
            hi = mid;
    }
    const int k = lo - 1;
    return (k >= 0 && k <= n_t - 2) ? k : -1;
}

// log-log interpolation inside interval k (observer.h:417-433 / :515-520); returns the linear
// contribution exp2(...) or 0 when the slope is not finite.
VAG_HD double interp_contrib2(double lo, double hi, double inv_dt, double dx) {
    const double s = (hi - lo) * inv_dt;
    if (!isfinite(s)) return 0.0;
    return rexp2(lo + dx * s);
}
VAG_HD double interp_contrib(double lo, double hi, double t_lo, double t_hi, double x) {
    return interp_contrib2(lo, hi, vdiv(1.0, t_hi - t_lo), x - t_lo);  // a zero interval gives a non-finite slope: no contribution
}

// ---------------------------------------------------------------------------------------------
// CTA work description.  Shared memory layout (doubles):
//   lg2t   [ROW_CHUNK][n_t]
//   lg2dop [ROW_CHUNK][n_t]          (series mode only)
//   lg2geo [ROW_CHUNK][n_t]          (series mode only)
//   bv     [ROW_CHUNK][n_t][nu_tile] (grid mode only)
// ---------------------------------------------------------------------------------------------
struct EatsShared {
    const RowGeom* rowg;  // row constants of the current chunk (global memory, written by k_rowgeom)
    double* lg2t;
    double* lg2dop;
    double* lg2geo;
    double* bv;
    int nu_tile;  // stride of bv along the node axis (= frequencies staged per pass, <= EATS_NU_TILE)
};

struct EatsRequest {
    int series;            // 0: grid (t x nu), 1: series (t[i], nu[i])
    int n_t_obs, n_nu;     // series: n_nu == n_t_obs (per-point frequencies)
    const double* lg2_t_obs;   // [n_t_obs]  log2(t * unit::sec)
    const double* lg2_nu_obs;  // [n_nu]     log2(nu * unit::Hz)   (without the 1+z shift)
    const double* nu_obs_lin;  // [n_nu]     nu * unit::Hz
    const double* nu23_obs;    // [n_nu]     (nu * unit::Hz)^(2/3) = exp2(2/3 lg2_nu_obs)
    const double* t_obs_lin;   // [n_t_obs]  t * unit::sec
    int i0, ni;                // block of observation points handled by the current pass
    // Banded series (n_bands > 0): the points of a series request share <= EATS_NU_TILE distinct frequencies.  The
    // boundary luminosities are then staged per (node, band) exactly as in grid mode -- lg2_nu_obs / nu_obs_lin /
    // nu23_obs hold the n_bands distinct frequencies -- and a point reads the column band_of[i] of its two
    // bracketing nodes instead of evaluating both spectra itself (same evaluation points as observer.h:494-520).
    int n_bands;
    const int* band_of;        // [n_t_obs] band index of every point
    int acc_stride;            // accumulator columns per frequency: eats_acc_stride(n_t_obs)
};

constexpr int EATS_T_BLOCK = 256;   // observation points accumulated per pass
// accumulator columns actually staged: short requests (100 epochs) do not pay for 256 columns of shared memory
VAG_HD int eats_acc_stride(int n_t_obs) { return n_t_obs >= EATS_T_BLOCK ? EATS_T_BLOCK : ((n_t_obs + 31) & ~31); }

// row_chunk <= EATS_ROW_CHUNK rows are staged per pass (the host lowers it when n_t is large)
VAG_HD size_t eats_shared_doubles(int n_t, bool series, int row_chunk, int nu_tile) {
    size_t n = (size_t)row_chunk * n_t;
    if (series)
        n += 2 * (size_t)row_chunk * n_t;
    else
        n += (size_t)row_chunk * n_t * nu_tile;
    return n;
}

VAG_HD EatsShared eats_carve(double* base, int n_t, bool series, int row_chunk, int nu_tile) {
    EatsShared s;
    s.nu_tile = nu_tile;
    s.rowg = nullptr;
    double* p = base;
    s.lg2t = p;
    p += (size_t)row_chunk * n_t;
    if (series) {
        s.lg2dop = p;
        p += (size_t)row_chunk * n_t;
        s.lg2geo = p;
        s.bv = nullptr;
    } else {
        s.lg2dop = s.lg2geo = nullptr;
        s.bv = p;
    }
    return s;
}

// Rows staged per pass for a lattice of n_t nodes: the count <= row_chunk that wastes the fewest
// thread slots of the last phase-1 round (thread <-> (row, node), nthr threads)
VAG_HD int eats_rows_per_pass(int n_t, int row_chunk, int nthr) {
    int best = row_chunk;
    double best_fill = 0;
    for (int r = row_chunk; r >= 1 && 2 * r > row_chunk; --r) {
        const int items = r * n_t;
        const double fill = (double)items / (double)(((items + nthr - 1) / nthr) * nthr);
        if (fill > best_fill + 1e-9) {
            best_fill = fill;
            best = r;
        }
    }
    return best;
}

// phase 1: node logs (+ boundary luminosities for the frequency tile [l0, l0+nl) in grid mode)
// POINT: per-point series layout (node logs only, the spectra are evaluated per point in phase 2); otherwise the
// (node, frequency) tile of grid mode / banded series.  A compile-time switch: the kernel instantiations of the
// three request kinds then carry only their own code (k_eats runs under a 64-register cap, and every path it does
// not take still costs it registers).
template <int MODE, bool POINT>
VAG_HD void eats_phase1(const EatsModel& M, const EatsRequest& rq, const EatsShared& sh, int nrows, int l0, int nl,
                        int tid, int nthr) {
    const int n_t = M.h->n_t;
    const double lg2_1pz = fast_log2(M.one_plus_z);
    const double w_lo = rq.t_obs_lin[rq.i0], w_hi = rq.t_obs_lin[rq.i0 + rq.ni - 1];
    for (int it = tid; it < nrows * n_t; it += nthr) {
        const int r = it / n_t, k = it - r * n_t;
        const RowGeom g = sh.rowg[r];
        double lt, ld, lg, dop_lin;
        node_logs(M, g, n_t, k, lt, ld, lg, dop_lin);
        sh.lg2t[it] = lt;
        if (POINT) {
            sh.lg2dop[it] = ld;
            sh.lg2geo[it] = lg;
        } else {
            // observed_window (observer.h:324-338) skips nodes no observation interval touches;
            // here a node is evaluated when one of its two adjacent intervals can hold a point.
            const bool need = (k + 1 >= n_t || node_time(M, g, n_t, k + 1) >= w_lo) &&
                              (k == 0 || node_time(M, g, n_t, k - 1) <= w_hi);
            double* bv = sh.bv + (size_t)it * sh.nu_tile;
            if (need) {
                if (MODE == 0) {
                    // the cell's coefficients are read once and serve every frequency of the tile
                    const double* base = M.coef + ((long)g.rep * n_t + k);
                    const long stride = M.coef_stride;
                    const SynCoefRegs cr = load_syn_coefs<true>([&](int c) { return base[c * stride]; });
                    // The two exponentials of a spectrum point factor into a cell part and a frequency part (comoving
                    // nu' = nu_obs (1 + z) dop_lin):  (nu' / nu_m)^(2/3) = x23_cell nu_obs^(2/3),  nu' / nu_M = cut_cell nu_obs.
                    // One exp2 per cell serves the whole tile instead of two per frequency.
                    const double x23_cell = rexp2((-2. / 3) * (ld + cr.log2_nu_m - lg2_1pz));
                    const double cut_cell = con::log2e * cr.inv_nu_M * (M.one_plus_z * dop_lin);
                    for (int l = 0; l < nl; ++l) {
                        const double lg2_nu_src = rq.lg2_nu_obs[l0 + l] + lg2_1pz;
                        bv[l] = photon_log2_I_nu_tile(cr, M.sp_lut, M.smooth_thick, M.log2_x_far, lg2_nu_src - ld,
                                                      x23_cell * rq.nu23_obs[l0 + l], cut_cell * rq.nu_obs_lin[l0 + l]) + lg;
                    }
                } else if (MODE == 1) {
                    // synchrotron of a shock with ssc: the same tile scheme with the IC correction of the thin branch
                    const long cell = (long)g.rep * n_t + k;
                    const double* base = M.coef + cell;
                    const long stride = M.coef_stride;
                    const SynCoefRegs cr = load_syn_coefs<true>([&](int c) { return base[c * stride]; });
                    const double log2_nu_c = base[PH_LOG2_NU_C * stride];
                    const double x23_cell = rexp2((-2. / 3) * (ld + cr.log2_nu_m - lg2_1pz));
                    const double nu_cell = M.one_plus_z * dop_lin;  // comoving nu = nu_cell nu_obs
                    const double cut_cell = con::log2e * cr.inv_nu_M * nu_cell;
                    for (int l = 0; l < nl; ++l) {
                        const double lg2_nu_src = rq.lg2_nu_obs[l0 + l] + lg2_1pz;
                        const double nu_o = rq.nu_obs_lin[l0 + l];
                        bv[l] = photon_log2_I_nu_ic_tile(cr, log2_nu_c, M.sp_lut, M.smooth_thick, M.log2_x_far, M.ic[cell],
                                                         lg2_nu_src - ld, x23_cell * rq.nu23_obs[l0 + l], cut_cell * nu_o,
                                                         nu_cell * nu_o) + lg;
                    }
                } else {
                    for (int l = 0; l < nl; ++l) {
                        const double lg2_nu_src = rq.lg2_nu_obs[l0 + l] + lg2_1pz;
                        bv[l] = cell_log2_I_nu<MODE>(M, g.rep, n_t, k, lg2_nu_src - ld) + lg;
                    }
                }
            }
        }
    }
}

// Phase-2 work assignment of one warp over a block of `ni` observation points.  A warp with a full complement takes
// one point per lane and every staged row.  The warp holding the block's remainder (100 epochs on 128 threads leave it
// 4 points) would run the whole row loop for a handful of lanes; it instead deals the rows to S = 32 / R row slices
// (R = its point count rounded up to a power of two <= 16), every lane sums its slice and the slices are added with a
// fixed shuffle tree -- the row loop of that warp shrinks S-fold.  (Device only: the host emulation keeps one point per
// thread; the two differ by the association of the row sum.)
struct P2Lane {
    int ii;       // point of this lane within the block, or -1
    int slice;    // first row of this lane
    int n_slices; // row stride
    int r_width;  // R: lanes per slice (shuffle tree starts at this offset); 32 = no tree
};
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ P2Lane p2_lane(int w0, int ni, int lane) {
    const int cnt = imin(32, ni - w0);
    P2Lane m;
    if (cnt > 16) {
        m.ii = lane < cnt ? w0 + lane : -1;
        m.slice = 0;
        m.n_slices = 1;
        m.r_width = 32;
    } else {
        int R = 1;
        while (R < cnt) R <<= 1;
        const int q = lane & (R - 1);
        m.ii = q < cnt ? w0 + q : -1;
        m.slice = lane / R;
        m.n_slices = 32 / R;
        m.r_width = R;
    }
    return m;
}
__device__ __forceinline__ double p2_reduce(double v, int r_width) {
    for (int off = r_width; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
#endif

// phase 2 (grid): thread <-> observation time; accumulates the chunk's rows into acc[l][idx]
// acc layout: [nu_tile][rq.acc_stride] (thread-owned columns, no atomics).  NLC = compile-time number of
// frequencies of the tile: their NLC interpolation exponentials are evaluated as one interleaved batch.
// exp2 arguments are clamped to [-1000, 1020]: below, the reference's term is < 1e-301 of anything it is
// added to (it underflows there); above, it would have overflowed.
template <int NLC>
VAG_HD void eats_phase2_grid_n(const EatsModel& M, const EatsRequest& rq, const EatsShared& sh, int nrows, double* acc,
                               int tid, int nthr) {
    const int n_t = M.h->n_t;
#if defined(__CUDA_ARCH__)
    for (int w0 = tid & ~31; w0 < rq.ni; w0 += nthr) {
        const P2Lane pl = p2_lane(w0, rq.ni, tid & 31);
        const int ii = pl.ii, r_first = pl.ii >= 0 ? pl.slice : nrows, r_step = pl.n_slices;  // idle lanes skip the rows
        const double x = rq.lg2_t_obs[rq.i0 + (ii >= 0 ? ii : w0)];
#else
    for (int ii = tid; ii < rq.ni; ii += nthr) {
        const int r_first = 0, r_step = 1;
        const double x = rq.lg2_t_obs[rq.i0 + ii];
#endif
        double sum[NLC];
#pragma unroll
        for (int l = 0; l < NLC; ++l) sum[l] = 0;
        for (int r = r_first; r < nrows; r += r_step) {
            const double* t_row = sh.lg2t + (size_t)r * n_t;
            const int k = find_interval(t_row, n_t, x, false);
            if (k < 0) continue;
            const double* b_lo = sh.bv + ((size_t)r * n_t + k) * sh.nu_tile;
            const double* b_hi = b_lo + sh.nu_tile;
            const double inv_dt = vdiv(1.0, t_row[k + 1] - t_row[k]), dx = x - t_row[k];  // zero interval -> non-finite slope -> skipped
            double arg[NLC], val[NLC];
            bool fin[NLC];
#pragma unroll
            for (int l = 0; l < NLC; ++l) {  // interp_contrib2 (observer.h:417-433)
                const double lo = b_lo[l];
                const double s = (b_hi[l] - lo) * inv_dt;
                fin[l] = isfinite(s);
                const double a = lo + dx * s;
                arg[l] = fin[l] ? vclamp(a, -1000.0, 1020.0) : 0.0;
            }
            dexp2_nc_vec<NLC>(arg, val);
#pragma unroll
            for (int l = 0; l < NLC; ++l) sum[l] += fin[l] ? val[l] : 0.0;
        }
#if defined(__CUDA_ARCH__)
#pragma unroll
        for (int l = 0; l < NLC; ++l) sum[l] = p2_reduce(sum[l], pl.r_width);
        if (ii < 0 || r_first != 0) continue;
#endif
#pragma unroll
        for (int l = 0; l < NLC; ++l) acc[l * rq.acc_stride + ii] += sum[l];
    }
}
VAG_HD void eats_phase2_grid(const EatsModel& M, const EatsRequest& rq, const EatsShared& sh, int nrows, int nl,
                             double* acc, int tid, int nthr) {
    switch (nl) {
        case 1: return eats_phase2_grid_n<1>(M, rq, sh, nrows, acc, tid, nthr);
        case 2: return eats_phase2_grid_n<2>(M, rq, sh, nrows, acc, tid, nthr);
        case 3: return eats_phase2_grid_n<3>(M, rq, sh, nrows, acc, tid, nthr);
        case 4: return eats_phase2_grid_n<4>(M, rq, sh, nrows, acc, tid, nthr);
        case 5: return eats_phase2_grid_n<5>(M, rq, sh, nrows, acc, tid, nthr);
        case 6: return eats_phase2_grid_n<6>(M, rq, sh, nrows, acc, tid, nthr);
        case 7: return eats_phase2_grid_n<7>(M, rq, sh, nrows, acc, tid, nthr);
        default: return eats_phase2_grid_n<8>(M, rq, sh, nrows, acc, tid, nthr);
    }
}

// phase 2 (series): thread <-> data point (t_s, nu_s); acc[EATS_T_BLOCK]
template <int MODE>
VAG_HD void eats_phase2_series(const EatsModel& M, const EatsRequest& rq, const EatsShared& sh, int nrows, double* acc,
                               int tid, int nthr) {
    const int n_t = M.h->n_t;
    const double lg2_1pz = fast_log2(M.one_plus_z);
#if defined(__CUDA_ARCH__)
    for (int w0 = tid & ~31; w0 < rq.ni; w0 += nthr) {
        const P2Lane pl = p2_lane(w0, rq.ni, tid & 31);
        const int ii = pl.ii, r_first = pl.ii >= 0 ? pl.slice : nrows, r_step = pl.n_slices;  // idle lanes skip the rows
        const int s = rq.i0 + (ii >= 0 ? ii : w0);
#else
    for (int ii = tid; ii < rq.ni; ii += nthr) {
        const int r_first = 0, r_step = 1;
        const int s = rq.i0 + ii;
#endif
        const double x = rq.lg2_t_obs[s];
        const double lg2_nu = rq.lg2_nu_obs[s] + lg2_1pz;
        double sum = 0;
        for (int r = r_first; r < nrows; r += r_step) {
            const size_t ro = (size_t)r * n_t;
            const double* t_row = sh.lg2t + ro;
            const int k = find_interval(t_row, n_t, x, true);
            if (k < 0) continue;
            const int rep = sh.rowg[r].rep;
            const double lo = cell_log2_I_nu<MODE>(M, rep, n_t, k, lg2_nu - sh.lg2dop[ro + k]) + sh.lg2geo[ro + k];
            const double hi = cell_log2_I_nu<MODE>(M, rep, n_t, k + 1, lg2_nu - sh.lg2dop[ro + k + 1]) + sh.lg2geo[ro + k + 1];
            sum += interp_contrib(lo, hi, t_row[k], t_row[k + 1], x);
        }
#if defined(__CUDA_ARCH__)
        sum = p2_reduce(sum, pl.r_width);
        if (ii < 0 || r_first != 0) continue;
#endif
        acc[ii] += sum;
    }
}

// phase 2 (banded series): thread <-> data point; the interval is located with the series rule and the two boundary
// luminosities of the point's band come from the staged tile
VAG_HD void eats_phase2_banded(const EatsModel& M, const EatsRequest& rq, const EatsShared& sh, int nrows, double* acc,
                               int tid, int nthr) {
    const int n_t = M.h->n_t;
    for (int ii = tid; ii < rq.ni; ii += nthr) {
        const int s = rq.i0 + ii;
        const double x = rq.lg2_t_obs[s];
        const int b = rq.band_of[s];
        double sum = 0;
        for (int r = 0; r < nrows; ++r) {
            const double* t_row = sh.lg2t + (size_t)r * n_t;
            const int k = find_interval(t_row, n_t, x, true);
            if (k < 0) continue;
            const double* bv = sh.bv + ((size_t)r * n_t + k) * sh.nu_tile + b;
            sum += interp_contrib(bv[0], bv[sh.nu_tile], t_row[k], t_row[k + 1], x);
        }
        acc[ii] += sum;
    }
}

}  // namespace vag
