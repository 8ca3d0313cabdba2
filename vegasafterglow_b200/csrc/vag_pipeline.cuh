// vag_pipeline.cuh -- batch workspace layout in HBM and the body of every kernel of the path.
//
// Pipeline for a batch of parameter sets sharing one observation request
// (the batched form of PyModel::compute_emission, pybind/pymodel.h:922-961):
//   K0  grid        thread / model          -> GridHeader, theta[], phi[], reps[], t_dec[]
//   K0b scan        one CTA                 -> row / cell offsets of the ragged batch, totals
//   K0c rowmap      thread / model          -> row -> (model, rep) map, theta_j -> rep map
//   K1  dynamics    thread / unique row     -> time lattice + shock tables (SoA, [row][k])
//   K2  radiation   CTA / unique row        -> photon coefficients (SoA planes, coalesced in k)
//   K3  EATS        CTA / (model, split, shock) -> flux [comp][nu][t] (vag_observer.cuh)
//   K4  chi2        warp / model            -> chi^2 of the series against data
// Each body is an HD function so the CPU test-suite can execute the identical code sequentially.
#pragma once

#include <climits>

#include "vag_grid.cuh"
#include "vag_ic.cuh"
#include "vag_observer.cuh"
#include "vag_radiation.cuh"
#include "vag_shock.cuh"

namespace vag {

enum { TOT_ROWS = 0, TOT_MAX_NT, TOT_MAX_NTHETA, TOT_MAX_EROWS, TOT_STATUS_OR, TOT_ANY_SSC, TOT_ANY_PAIR, TOT_ANY_FWD_ONLY,
       TOT_ANY_SPREAD, TOT_N };

struct BatchWs {
    int n_models;
    int dbg_max_ode_steps, dbg_max_ode_fails;  // > 0: override the ODE step / consecutive-rejection limits (tests)
    int cap_theta, cap_phi;
    size_t work_per_model;  // doubles
    const vag_params* params;
    ModelCfg* cfg;
    GridHeader* hdr;
    double* theta;   // [n][cap_theta]
    double* phi;     // [n][cap_phi]
    double* t_dec;   // [n][cap_theta]
    double* work;    // [n][work_per_model]
    int* reps;       // [n][cap_theta]
    int* rep_of;     // [n][cap_theta]
    int* row_off;    // [n+1]
    long long* cell_off;  // [n+1]
    int* totals;     // [TOT_N]
    int* status;     // [n]
    // per unique row
    int* row_model;
    int* row_rep;
    int* inj_idx;
    RowDyn* row_dyn;          // ODE kernel -> finishing pass (raw-state bookkeeping, crossing state)
    long long* row_cell_off;  // first global cell of each row
    // per unique cell
    long long n_cells;
    double* t_rows;
    double* fwd[6];  // t_comv, r, Gamma, Gamma_th, B, N_p
    double* rvs[6];
    double* coef_fwd;  // [PH_NCOEF][n_cells]
    double* coef_rvs;
    double* geo_u;     // [n_cells] sqrt((Gamma-1)(Gamma+1)) of the forward table (EATS Doppler factor)
    double* geo_lg2r2; // [n_cells] 2 log2(r)                                   (EATS geometry factor)
    // spreading models only (allocated when the batch has one): Shock::theta and the per-node EATS geometry
    double* sh_theta;  // [n_cells] theta(k) of the row
    double* geo_cth;   // [n_cells] cos theta(k)
    double* geo_sth;   // [n_cells] sin theta(k)
    double* geo_dcos;  // [n_cells] cos(theta_hi) - cos(theta_lo) against the neighbour rows (observer.cpp:112-122)
    // inverse-Compton data: allocated only when some model of the batch has ssc=True
    int any_ssc;
    int max_n_t, max_erows;   // batch maxima (known after K0b)
    IcCell* ic[2];            // [n_cells] per shock
    IcTable* ictab_h[2];      // [n_cells]
    double* ictab[2];         // [n_cells][IC_CAP_OUT]
    double* rowcos;           // [n_models][max_erows]  cos of the angle to the line of sight per (phi,theta) row
    double* dop_min;          // [n_models][max_n_t]    min / max over rows of the linear Doppler denominator
    double* dop_max;
    const KnLut* lut;
    double* ic_scratch;       // [n_ic_warps][IC_SCRATCH_DOUBLES]
    const double* nu_range;   // [2] log2 of min / max observation frequency (code units); ragged request: [n_models][2]
    const double* sp_lut;     // [SPL_DOUBLES] log2_softplus table (vag_math.cuh)
    RowGeom* rowgeom;         // [n_models][max_erows] EATS row constants (k_rowgeom)
};

// ---- K0 ---------------------------------------------------------------------------------------
template <class Par>
VAG_HD void k0_grid_body(const Par& par, const BatchWs& w, int mi, double t_obs_min, double t_obs_max) {
    ModelCfg cfg = make_cfg(w.params[mi]);
    if (w.dbg_max_ode_steps > 0) cfg.max_ode_steps = w.dbg_max_ode_steps;
    if (w.dbg_max_ode_fails > 0) cfg.max_ode_fails = w.dbg_max_ode_fails;
    w.cfg[mi] = cfg;
    GridSlab s;
    s.theta = w.theta + (size_t)mi * w.cap_theta;
    s.phi = w.phi + (size_t)mi * w.cap_phi;
    s.reps = w.reps + (size_t)mi * w.cap_theta;
    s.t_dec = w.t_dec + (size_t)mi * w.cap_theta;
    s.work = w.work + (size_t)mi * w.work_per_model;
    s.cap_theta = w.cap_theta;
    s.cap_phi = w.cap_phi;
    GridHeader h;
    build_grid(par, cfg, t_obs_min * unit::sec, t_obs_max * unit::sec, h, s);
    w.hdr[mi] = h;
    w.status[mi] = h.status;
}

// ---- K0b: exclusive scan over models (single CTA; `tid`-strided two-pass is overkill for the
// few thousand models of a batch, so thread 0 of the CTA walks the headers) -------------------------
VAG_HD void k0b_scan_body(const BatchWs& w) {
    int rows = 0, max_nt = 0, max_nth = 0, max_erows = 0, st = 0;
    long long cells = 0;
    for (int mi = 0; mi < w.n_models; ++mi) {
        const GridHeader& h = w.hdr[mi];
        w.row_off[mi] = rows;
        w.cell_off[mi] = cells;
        rows += h.n_reps;
        cells += (long long)h.n_reps * h.n_t;
        max_nt = imax(max_nt, h.n_t);
        max_nth = imax(max_nth, h.n_theta);
        max_erows = imax(max_erows, h.n_theta * h.n_phi_eff);
        st |= h.status;
    }
    w.row_off[w.n_models] = rows;
    w.cell_off[w.n_models] = cells;
    w.totals[TOT_ROWS] = rows;
    w.totals[TOT_MAX_NT] = max_nt;
    w.totals[TOT_MAX_NTHETA] = max_nth;
    w.totals[TOT_MAX_EROWS] = max_erows;
    w.totals[TOT_STATUS_OR] = st;
    int any = 0;
    for (int mi = 0; mi < w.n_models; ++mi) any |= (w.cfg[mi].fwd.ssc || (w.cfg[mi].has_rvs && w.cfg[mi].rvs.ssc)) ? 1 : 0;
    w.totals[TOT_ANY_SSC] = any;
    int any_pair = 0, any_fwd = 0;
    for (int mi = 0; mi < w.n_models; ++mi) (w.cfg[mi].has_rvs ? any_pair : any_fwd) = 1;
    w.totals[TOT_ANY_PAIR] = any_pair;
    w.totals[TOT_ANY_FWD_ONLY] = any_fwd;
    int any_spread = 0;
    for (int mi = 0; mi < w.n_models; ++mi) any_spread |= w.cfg[mi].spreading;
    w.totals[TOT_ANY_SPREAD] = any_spread;
}

// ---- K0c --------------------------------------------------------------------------------------
VAG_HD void k0c_rowmap_body(const BatchWs& w, int mi) {
    const GridHeader& h = w.hdr[mi];
    const int* reps = w.reps + (size_t)mi * w.cap_theta;
    int* rep_of = w.rep_of + (size_t)mi * w.cap_theta;
    const int ro = w.row_off[mi];
    for (int r = 0; r < h.n_reps; ++r) {
        w.row_model[ro + r] = mi;
        w.row_rep[ro + r] = r;
        w.row_cell_off[ro + r] = w.cell_off[mi] + (long long)r * h.n_t;
        if (h.rows3d) continue;  // row r = i * n_theta + j: no representative list (eats_rep)
        const int j0 = reps[r];
        const int j1 = (r + 1 < h.n_reps) ? reps[r + 1] : h.n_theta;
        for (int j = j0; j < j1; ++j) rep_of[j] = r;
    }
    if (h.rows3d)
        for (int j = 0; j < h.n_theta; ++j) rep_of[j] = j;
}

// theta index of ODE row r, and the ODE row behind EATS row (phi_i, theta_j)
VAG_HD int row_theta_index(const BatchWs& w, int mi, const GridHeader& h, int r) {
    return h.rows3d ? r % h.n_theta : w.reps[(size_t)mi * w.cap_theta + r];
}
VAG_HD int eats_rep(const GridHeader& h, const int* rep_of, int i, int j) {
    return h.rows3d ? i * h.n_theta + j : rep_of[j];
}

VAG_HD ShockRow shock_row(double* const* planes, long long off) {
    ShockRow s;
    s.t_comv = planes[0] + off;
    s.r = planes[1] + off;
    s.Gamma = planes[2] + off;
    s.Gamma_th = planes[3] + off;
    s.B = planes[4] + off;
    s.N_p = planes[5] + off;
    return s;
}

// ---- K1 ---------------------------------------------------------------------------------------
// The shock-table planes double as the raw-state store of the ODE kernel (vag_shock.cuh RawRow):
// component c of the state vector -> forward plane c (c < 6) or reverse plane c - 6.
VAG_HD RawRow raw_row(const BatchWs& w, long long off) {
    RawRow raw;
    for (int c = 0; c < 6; ++c) raw.c[c] = w.fwd[c] + off;
    for (int c = 6; c < 11; ++c) raw.c[c] = w.rvs[c - 6] + off;
    raw.theta = w.sh_theta ? w.sh_theta + off : nullptr;
    return raw;
}

// K1: sequential part of one row -- time lattice + dopri5 integration, raw node states only
constexpr int K1_COL_DOUBLES = Dopri5S<FREqn::N>::kDoublesPerThread;  // stage-vector column of one row
// K1a: engine-time lattice of one unique row, nodes strided over (tid, nthr) (every node is an independent pow(10, .))
VAG_HD void k1_lattice_body(const BatchWs& w, int row, int tid, int nthr) {
    const int mi = w.row_model[row];
    const int r = w.row_rep[row];
    const GridHeader& h = w.hdr[mi];
    const ModelCfg& cfg = w.cfg[mi];
    const long long off = w.cell_off[mi] + (long long)r * h.n_t;
    // per-row lattice bounds of a structured model: work[j] and work[cap_theta + j] (build_grid); a rows3d model
    // derives them for its own (phi_i, theta_j) (scan_time_bounds, grid-refinement.h:485-499)
    const double* work = w.work + (size_t)mi * w.work_per_model;
    double t_dec, row_start = 0.0, row_early = 0.0;
    if (h.rows3d) {
        const int i = r / h.n_theta, j = r - i * h.n_theta;
        const double th = w.theta[(size_t)mi * w.cap_theta + j];
        t_dec = w.t_dec[(size_t)mi * w.cap_theta + j];
        const double ts = raw_row_start(cfg, h.t_obs_min, th, jet_Gamma0(cfg, th), cos(cfg.theta_v), sin(cfg.theta_v),
                                        w.phi[(size_t)mi * w.cap_phi + i]);
        const double cut = row_start_cut(cfg, h.is_rvs != 0, t_dec);
        row_start = vmax(ts, cut);
        row_early = 0.99 * vmin(ts, cut);
    } else {
        t_dec = w.t_dec[(size_t)mi * w.cap_theta + r];
        if (h.structured) {
            row_start = work[r];
            row_early = work[w.cap_theta + r];
        }
    }
    build_row_lattice(h, t_dec, cfg.T0, row_start, row_early, w.t_rows + off, tid, nthr);
    // grid-refinement.h:633-635: every thread re-reads the nodes it wrote itself (and thread 0 the early point)
    bool finite = true;
    for (int k = tid + (h.has_early ? 1 : 0); k < h.n_t; k += nthr) finite = finite && isfinite(w.t_rows[off + k]);
    if (tid == 0 && h.has_early) finite = finite && isfinite(w.t_rows[off]);
    if (!finite) {
#if defined(__CUDA_ARCH__)
        atomicOr(&w.status[mi], VAG_ST_GRID_NONFINITE);
#else
        w.status[mi] |= VAG_ST_GRID_NONFINITE;
#endif
    }
}

template <bool PAIR>
VAG_HD void k1_dynamics_body(const BatchWs& w, int row, double* col, int col_stride) {
    const int mi = w.row_model[row];
    const int r = w.row_rep[row];
    const GridHeader& h = w.hdr[mi];
    const ModelCfg& cfg = w.cfg[mi];
    const long long off = w.cell_off[mi] + (long long)r * h.n_t;
    double* t_row = w.t_rows + off;  // written by k1_lattice_body
    const int jth = row_theta_index(w, mi, h, r);
    const double t_dec = w.t_dec[(size_t)mi * w.cap_theta + (h.rows3d ? jth : r)];
    const double theta = w.theta[(size_t)mi * w.cap_theta + jth];
    int st = 0;  // (a non-finite lattice node was flagged by k1_lattice_body)
    const ShockRow sf = shock_row(w.fwd, off);
    const RawRow raw = raw_row(w, off);
    RowDyn rd;
    if (PAIR) {
        const ShockRow sr = shock_row(w.rvs, off);
        st |= solve_pair_row(cfg, theta, t_dec, t_row, h.n_t, sf, sr, raw, rd, col, col_stride);
    } else {
        (void)col;
        (void)col_stride;
        const double ths = h.theta_s;
        if (cfg.spreading)
            st |= cfg.has_magnetar ? solve_fwd_row<true, true>(cfg, theta, ths, t_dec, t_row, h.n_t, sf, raw, rd)
                                   : solve_fwd_row<false, true>(cfg, theta, ths, t_dec, t_row, h.n_t, sf, raw, rd);
        else
            st |= cfg.has_magnetar ? solve_fwd_row<true, false>(cfg, theta, ths, t_dec, t_row, h.n_t, sf, raw, rd)
                                   : solve_fwd_row<false, false>(cfg, theta, ths, t_dec, t_row, h.n_t, sf, raw, rd);
    }
    w.row_dyn[row] = rd;
    w.inj_idx[row] = rd.injection_idx;
    if (st) {
#if defined(__CUDA_ARCH__)
        atomicOr(&w.status[mi], st);
#else
        w.status[mi] |= st;
#endif
    }
}

// K1b: per-cell completion of the shock tables from the raw node states (save_fwd_shock_state /
// save_rvs_shock_state, forward-shock.tpp:151-173, reverse-shock.tpp:403-426); one thread per (row, k)
struct RowCtx {
    int mi, n_t, has_rvs;
    long long off;
    double theta;
};
VAG_HD RowCtx row_ctx(const BatchWs& w, int row) {
    RowCtx c;
    c.mi = w.row_model[row];
    const int r = w.row_rep[row];
    c.n_t = w.hdr[c.mi].n_t;
    c.has_rvs = w.cfg[c.mi].has_rvs;
    c.off = w.cell_off[c.mi] + (long long)r * c.n_t;
    c.theta = w.theta[(size_t)c.mi * w.cap_theta + row_theta_index(w, c.mi, w.hdr[c.mi], r)];
    return c;
}
VAG_HD void k1b_finish_cell(const BatchWs& w, int row, const RowCtx& c, int k) {
    const ModelCfg& cfg = w.cfg[c.mi];
    const RowDyn& rd = w.row_dyn[row];
    const ShockRow sf = shock_row(w.fwd, c.off);
    const RawRow raw = raw_row(w, c.off);
    if (c.has_rvs)
        finish_pair_cell(cfg, c.theta, rd, sf, shock_row(w.rvs, c.off), raw, k);
    else
        finish_fwd_cell(cfg, rd, sf, raw, k);
}
// K1c: reverse_shock_early_extrap of node k (after every cell of the row is finished and idx_cut,
// the first node with Gamma_th above the thermal cut, is known)
VAG_HD void k1c_extrap_cell(const BatchWs& w, int row, const RowCtx& c, int idx_cut, int k) {
    if (!c.has_rvs || w.row_dyn[row].n_saved < 0) return;
    if (k < idx_cut && extrap_applies(idx_cut, c.n_t, w.row_dyn[row].injection_idx))
        extrap_cell(shock_row(w.rvs, c.off), idx_cut, k);
}
// K1d: node-only pieces of the EATS geometry (observer.cpp:158,200), shared by every (phi,theta) row
// that maps onto this representative row
VAG_HD void k1d_geo_cell(const BatchWs& w, const RowCtx& c, int k) {
    const double g = w.fwd[2][c.off + k];
    w.geo_u[c.off + k] = sqrt((g - 1) * (g + 1));
    w.geo_lg2r2[c.off + k] = 2.0 * rlog2(w.fwd[1][c.off + k]);
}
// K1e (spreading models): per-node trigonometry and solid-angle width of calc_t_obs / calc_solid_angle
// (observer.cpp:51-141).  Row j's boundaries at engine time t(j,k) use the neighbour rows' theta
// interpolated at that time; with every theta row a representative, the neighbours are rows +-1.
VAG_HD double interp_theta_nb(const double* t_nb, const double* th_nb, int n_t, double t_target) {
    int h = 0;  // the reference's monotone k_hint walk, restarted (same result for an ascending lattice)
    int lo = 0, hi = n_t - 1;  // largest h with t_nb[h] < t_target for h >= 1 (0 if none)
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (t_nb[mid] < t_target)
            lo = mid;
        else
            hi = mid - 1;
    }
    h = lo;
    if (h + 1 >= n_t) return th_nb[n_t - 1];
    const double wgt = (t_target - t_nb[h]) / (t_nb[h + 1] - t_nb[h]);
    return th_nb[h] + wgt * (th_nb[h + 1] - th_nb[h]);
}
VAG_HD void k1e_spread_geo_cell(const BatchWs& w, int row, const RowCtx& c, int k) {
    const GridHeader& hh = w.hdr[c.mi];
    const int j = hh.rows3d ? w.row_rep[row] % hh.n_theta : w.row_rep[row];  // neighbours in theta, within the row's phi
    const int last = (hh.rows3d ? hh.n_theta : hh.n_reps) - 1;
    const long long o = c.off + k;
    const double th = w.sh_theta[o];
    w.geo_cth[o] = cos(th);
    w.geo_sth[o] = sin(th);
    const double t_target = w.t_rows[o];
    double th_lo = th, th_hi = th;
    if (j > 0) th_lo = 0.5 * (th + interp_theta_nb(w.t_rows + c.off - c.n_t, w.sh_theta + c.off - c.n_t, c.n_t, t_target));
    if (j < last) th_hi = 0.5 * (th + interp_theta_nb(w.t_rows + c.off + c.n_t, w.sh_theta + c.off + c.n_t, c.n_t, t_target));
    w.geo_dcos[o] = cos(th_hi) - cos(th_lo);
}

// ---- K2 ---------------------------------------------------------------------------------------
// one (row, k) cell of one shock (which = 0 forward, 1 reverse)
VAG_HD void k2_radiation_cell(const BatchWs& w, int row, int k, int which) {
    const int mi = w.row_model[row];
    const GridHeader& h = w.hdr[mi];
    const ModelCfg& cfg = w.cfg[mi];
    const long long off = w.cell_off[mi] + (long long)w.row_rep[row] * h.n_t;
    double* const* pl = which ? w.rvs : w.fwd;
    const RadCfg& rad = which ? cfg.rvs : cfg.fwd;
    auto load = [&](int kk) {
        CellShock c;
        c.t_comv = pl[0][off + kk];
        c.r = pl[1][off + kk];
        c.Gamma_th = pl[3][off + kk];
        c.B = pl[4][off + kk];
        c.N_p = pl[5][off + kk];
        return c;
    };
    const CellShock cs = load(k);
    const int inj = which ? w.inj_idx[row] : h.n_t;
    const bool relic = k >= inj;
    const CellShock ics = relic ? load(inj - 1) : cs;
    double coef[PH_NCOEF];
    radiation_cell(rad, cs, relic, ics, coef);
    double* out = (which ? w.coef_rvs : w.coef_fwd) + off + k;
#pragma unroll
    for (int c = 0; c < PH_NCOEF; ++c) out[(long long)c * w.n_cells] = coef[c];
}

// ---- K2 for shocks with ssc=True: IC cooling along one row (sequential in k) ----------------------
VAG_HD void k2_ic_cool_row(const BatchWs& w, int row, int which) {
    const int mi = w.row_model[row];
    const GridHeader& h = w.hdr[mi];
    const ModelCfg& cfg = w.cfg[mi];
    const long long off = w.cell_off[mi] + (long long)w.row_rep[row] * h.n_t;
    double* const* pl = which ? w.rvs : w.fwd;
    const RadCfg& rad = which ? cfg.rvs : cfg.fwd;
    const int inj = which ? w.inj_idx[row] : h.n_t;
    double* coef = (which ? w.coef_rvs : w.coef_fwd) + off;
    const long long plane = w.n_cells;
    ic_cool_row(rad, h.n_t, inj, pl[0] + off, pl[1] + off, pl[3] + off, pl[4] + off, pl[5] + off, w.ic[which] + off,
                [&](int k, int q, double v) { coef[(long long)q * plane + k] = v; });
}

// ---- per-row line-of-sight cosine and per-k Doppler extrema (SSC output band, pymodel.h:897-909) ---
VAG_HD EatsModel make_eats_model(const BatchWs& w, int mi, int which);
VAG_HD void k_rowcos_body(const BatchWs& w, int mi, int q) {
    const EatsModel M = make_eats_model(w, mi, 0);
    const int n_theta = M.h->n_theta;
    w.rowcos[(size_t)mi * w.max_erows + q] = row_geometry(M, q / n_theta, q % n_theta).cos_v;
}
// row constants of calc_eat_non_spreading for row q of model mi (observer.cpp:167-192)
VAG_HD void k_rowgeom_body(const BatchWs& w, int mi, int q) {
    const EatsModel M = make_eats_model(w, mi, 0);
    const int n_theta = M.h->n_theta;
    w.rowgeom[(size_t)mi * w.max_erows + q] = row_geometry(M, q / n_theta, q % n_theta);
}
VAG_HD void k_dop_extrema_body(const BatchWs& w, int mi, int k) {
    const GridHeader& h = w.hdr[mi];
    const int erows = h.n_theta * h.n_phi_eff;
    const double* Gam = w.fwd[2] + w.cell_off[mi];
    const int* rep_of = w.rep_of + (size_t)mi * w.cap_theta;
    const double* rc = w.rowcos + (size_t)mi * w.max_erows;
    // spreading jets: the line-of-sight cosine is a per-node quantity (observer.cpp:82); rowcos then holds
    // cos(phi) sin(theta_obs) and the node tables supply cos / sin of theta(k)
    const bool spread = w.cfg[mi].spreading && w.sh_theta;
    const double cos_obs = cos(w.cfg[mi].theta_v);
    double lo = kInf, hi = -kInf;
    for (int q = 0; q < erows; ++q) {
        const size_t o = (size_t)eats_rep(h, rep_of, q / h.n_theta, q % h.n_theta) * h.n_t + k;
        const double g = Gam[o];
        const long long cell = w.cell_off[mi] + (long long)o;
        const double cos_v = spread ? w.geo_sth[cell] * rc[q] + w.geo_cth[cell] * cos_obs : rc[q];
        const double d = g - sqrt((g - 1) * (g + 1)) * cos_v;
        lo = vmin(lo, d);
        hi = vmax(hi, d);
    }
    w.dop_min[(size_t)mi * w.max_n_t + k] = lo;
    w.dop_max[(size_t)mi * w.max_n_t + k] = hi;
}

// ---- K2b: SSC spectrum of one cell (one warp) -------------------------------------------------------
template <class Par>
VAG_HD int k2b_ic_spectrum_cell(const Par& par, const BatchWs& w, int row, int k, int which, double* scratch) {
    const int mi = w.row_model[row];
    const GridHeader& h = w.hdr[mi];
    const ModelCfg& cfg = w.cfg[mi];
    const long long cell = w.cell_off[mi] + (long long)w.row_rep[row] * h.n_t + k;
    const RadCfg& rad = which ? cfg.rvs : cfg.fwd;
    const IcCell& c = w.ic[which][cell];
    const double* base = (which ? w.coef_rvs : w.coef_fwd) + cell;
    const long long stride = w.n_cells;
    double smooth_thick, log2_x_far;
    photon_p_consts(rad.p, smooth_thick, log2_x_far);
    auto seed = [&](double log2_nu) {
        return photon_log2_I_nu_ic([&](int q) { return base[(long long)q * stride]; }, smooth_thick, log2_x_far, c, log2_nu);
    };
    // comoving evaluation band of this time index (pybind/pymodel.h:897-909): lg2_doppler = -log2(dop_lin)
    const double lg2_1pz = fast_log2(1 + cfg.z);
    const double lg2_dop_max = -rlog2(w.dop_min[(size_t)mi * w.max_n_t + k]);
    const double lg2_dop_min = -rlog2(w.dop_max[(size_t)mi * w.max_n_t + k]);
    const double nu_eval_min = fast_exp2((w.nu_range[0] + lg2_1pz) - lg2_dop_max);
    const double nu_eval_max = fast_exp2((w.nu_range[1] + lg2_1pz) - lg2_dop_min);
    IcTable hdr;
    const int st = ic_generate(par, c, seed, rad.kn != 0, *w.lut, nu_eval_min, nu_eval_max, scratch, hdr,
                               w.ictab[which] + (size_t)cell * IC_CAP_OUT);
    w.ictab_h[which][cell] = hdr;
    return st;
}

VAG_HD EatsModel make_eats_model(const BatchWs& w, int mi, int which) {
    const GridHeader& h = w.hdr[mi];
    const ModelCfg& cfg = w.cfg[mi];
    const long long off = w.cell_off[mi];
    EatsModel M;
    M.h = &w.hdr[mi];
    M.theta = w.theta + (size_t)mi * w.cap_theta;
    M.phi = w.phi + (size_t)mi * w.cap_phi;
    M.rep_of = w.rep_of + (size_t)mi * w.cap_theta;
    M.t_rows = w.t_rows + off;
    M.r = w.fwd[1] + off;      // the pair solver gives both shocks identical kinematics
    M.Gamma = w.fwd[2] + off;  // (pybind/pymodel.h:943-950): one EAT geometry serves both
    M.geo_u = w.geo_u + off;
    M.geo_lg2r2 = w.geo_lg2r2 + off;
    const int shock = which & 1;  // which: 0 fwd sync, 1 rvs sync, 2 fwd ssc, 3 rvs ssc
    const RadCfg& rad = shock ? cfg.rvs : cfg.fwd;
    M.coef = (shock ? w.coef_rvs : w.coef_fwd) + off;
    M.coef_stride = (long)w.n_cells;
    photon_p_consts(rad.p, M.smooth_thick, M.log2_x_far);
    M.mode = (which >= 2) ? 2 : (rad.ssc ? 1 : 0);
    M.ic = (w.any_ssc && rad.ssc) ? w.ic[shock] + off : nullptr;
    M.ictab_h = (w.any_ssc && rad.ssc) ? w.ictab_h[shock] + off : nullptr;
    M.ictab = (w.any_ssc && rad.ssc) ? w.ictab[shock] + (size_t)off * IC_CAP_OUT : nullptr;
    M.breach = nullptr;
    M.sp_lut = w.sp_lut;
    M.spreading = (cfg.spreading && w.sh_theta) ? 1 : 0;
    M.geo_cth = M.spreading ? w.geo_cth + off : nullptr;
    M.geo_sth = M.spreading ? w.geo_sth + off : nullptr;
    M.geo_dcos = M.spreading ? w.geo_dcos + off : nullptr;
    M.one_plus_z = 1 + cfg.z;
    M.lumi_dist = cfg.lumi_dist;
    M.theta_v = cfg.theta_v;
    (void)h;
    return M;
}

// Final scaling of Observer::specific_flux (observer.h:442) and the unit conversion of
// PyModel::flux_density_grid (pybind/pymodel.cpp:507)
VAG_HD double flux_scale(const EatsModel& M, double F) {
    return F * (M.one_plus_z / (M.lumi_dist * M.lumi_dist)) / unit::flux_den_cgs;
}

// ---- K4: chi^2 of one model (VegasAfterglow/fitting/fitter.py:497-501) ---------------------------
VAG_HD double chi2_term(double lnF_obs, double F_model, double sigma_ln, double wgt) {
    const double d = (lnF_obs - log(vmax(F_model, 1e-300))) / sigma_ln;
    return wgt * d * d;
}

// ---- parameter checks and capacity bounds: one definition for the host and for the device planning (k_plan) ----------
// Why vag_params_validate rejects a parameter set; vag_b200.cu maps each reason to its message.  The order of the checks
// decides which reason a set with several faults gets.
enum ParamsReason {
    PR_OK = 0, PR_JET_TYPE, PR_MEDIUM_TYPE, PR_THETA_C, PR_E_ISO, PR_GAMMA0, PR_DURATION, PR_K_EG, PR_E_ISO_W, PR_GAMMA0_W,
    PR_THETA_W, PR_THETA_W_ORDER, PR_SIGMA0, PR_MAG_L0, PR_MAG_T0, PR_MAG_Q, PR_MAG_WING, PR_N_ISM, PR_A_STAR, PR_N0, PR_K_M,
    PR_LUMI_DIST, PR_Z, PR_THETA_OBS, PR_PHI_OBS,
    PR_FWD_EPS_E, PR_FWD_EPS_B, PR_FWD_XI_E, PR_FWD_P,  // the reverse shock's four follow in the same order
    PR_RVS_EPS_E, PR_RVS_EPS_B, PR_RVS_XI_E, PR_RVS_P, PR_RTOL, PR_NONFINITE_RES
};

VAG_HD bool finite_pos(double x) { return isfinite(x) && x > 0; }
VAG_HD bool in_open_closed(double v, double lo, double hi) { return isfinite(v) && v > lo && v <= hi; }

// PyRadiation (pybind/pymodel.h:303-313); base = PR_FWD_EPS_E or PR_RVS_EPS_E
VAG_HD int radiation_check(const vag_radiation& r, int base) {
    if (!in_open_closed(r.eps_e, 0.0, 1.0)) return base;
    if (!in_open_closed(r.eps_B, 0.0, 1.0)) return base + 1;
    if (!in_open_closed(r.xi_e, 0.0, 1.0)) return base + 2;
    if (!(isfinite(r.p) && r.p > 1.0)) return base + 3;
    return PR_OK;
}

// The checks of the reference constructors (pybind/pymodel.cpp:47-186, pybind/pymodel.h:190-204,303-313,613-649)
VAG_HD int params_check(const vag_params& p) {
    if (p.jet_type < 0 || p.jet_type > 5) return PR_JET_TYPE;
    if (p.medium_type < 0 || p.medium_type > 1) return PR_MEDIUM_TYPE;
    // PyTophatJet / PyGaussianJet / PyPowerLawJet: pybind/pymodel.cpp:47-95
    if (!in_open_closed(p.theta_c, 0.0, con::pi / 2)) return PR_THETA_C;
    const bool has_core = p.jet_type != VAG_JET_POWERLAW_WING;
    const bool has_wing = p.jet_type >= VAG_JET_TWO_COMPONENT;
    if (has_core && !finite_pos(p.E_iso)) return PR_E_ISO;
    if (has_core && !(isfinite(p.Gamma0) && p.Gamma0 > 1.0)) return PR_GAMMA0;
    if (!finite_pos(p.duration)) return PR_DURATION;
    if ((p.jet_type == VAG_JET_POWERLAW || p.jet_type == VAG_JET_STEP_POWERLAW || p.jet_type == VAG_JET_POWERLAW_WING) &&
        (!finite_pos(p.k_e) || !finite_pos(p.k_g)))
        return PR_K_EG;
    // PyTwoComponentJet / PyStepPowerLawJet / PyPowerLawWing: pybind/pymodel.cpp:97-146
    if (has_wing) {
        if (!finite_pos(p.E_iso_w)) return PR_E_ISO_W;
        if (!(isfinite(p.Gamma0_w) && p.Gamma0_w > 1.0)) return PR_GAMMA0_W;
    }
    if (p.jet_type == VAG_JET_TWO_COMPONENT) {
        if (!in_open_closed(p.theta_w, 0.0, con::pi / 2)) return PR_THETA_W;
        if (!(p.theta_w > p.theta_c)) return PR_THETA_W_ORDER;
    }
    if (!(isfinite(p.sigma0) && p.sigma0 >= 0)) return PR_SIGMA0;
    if (p.has_magnetar) {  // PyMagnetar: pybind/pymodel.h:45-49
        if (!finite_pos(p.magnetar_L0)) return PR_MAG_L0;
        if (!finite_pos(p.magnetar_t0)) return PR_MAG_T0;
        if (!finite_pos(p.magnetar_q)) return PR_MAG_Q;
        if (p.jet_type == VAG_JET_POWERLAW_WING) return PR_MAG_WING;
    }
    // PyISM / PyWind: pybind/pymodel.cpp:148-186
    if (p.medium_type == VAG_MEDIUM_ISM) {
        if (!(isfinite(p.n_ism) && p.n_ism >= 0)) return PR_N_ISM;
    } else {
        if (!finite_pos(p.A_star)) return PR_A_STAR;
        if (!(isfinite(p.n_ism) && p.n_ism >= 0)) return PR_N_ISM;
        if (!(p.n0 > 0)) return PR_N0;
        if (!isfinite(p.wind_k_m)) return PR_K_M;
    }
    // PyObserver: pybind/pymodel.h:190-204
    if (!finite_pos(p.lumi_dist)) return PR_LUMI_DIST;
    if (!(isfinite(p.z) && p.z >= 0)) return PR_Z;
    if (!(isfinite(p.theta_obs) && p.theta_obs >= 0 && p.theta_obs <= con::pi)) return PR_THETA_OBS;
    if (!isfinite(p.phi_obs)) return PR_PHI_OBS;
    if (const int r = radiation_check(p.fwd, PR_FWD_EPS_E)) return r;
    if (p.has_rvs)
        if (const int r = radiation_check(p.rvs, PR_RVS_EPS_E)) return r;
    // PyModel ctor: pybind/pymodel.h:642-647 (a non-positive value selects the default)
    if (p.rtol > 0 && !(p.rtol < 1)) return PR_RTOL;
    if (!isfinite(p.rtol) || !isfinite(p.phi_resol) || !isfinite(p.theta_resol) || !isfinite(p.t_resol))
        return PR_NONFINITE_RES;
    return PR_OK;
}

struct Caps {
    int theta, phi;
};

// (int)x as the x86-64 host converts it (cvttsd2si: truncation, INT_MIN for NaN and for values outside int's range) and
// int sums that wrap.  The device's own conversion saturates: spelled out, the bound of a record with, e.g., an unused
// Gamma0_w = inf is the same number on both sides.
VAG_HD int host_int(double x) { return (x > -2147483649.0 && x < 2147483648.0) ? (int)x : INT_MIN; }
VAG_HD int wrap_add(int a, int b) { return (int)((unsigned)a + (unsigned)b); }

// Grid nodes one parameter set can need (upper bounds of auto_grid's node counts,
// src/core/grid-refinement.h:246-262,655,664-677).  log10 is glibc's on the host and its bit-exact restatement on the
// device (vag_libm.cuh): CUDA's log10 can differ by an ulp, which can move the integer bound at a boundary.
VAG_HD Caps caps_of(const vag_params& p) {
    const bool r = p.has_rvs != 0;
    const double th_res = p.theta_resol > 0 ? p.theta_resol : (r ? 0.2 : 0.15);
    const double ph_res = p.phi_resol > 0 ? p.phi_resol : 0.06;
    const double g = vmax(1.0, vmax(p.Gamma0, p.Gamma0_w) * 1.5708);
#if defined(__CUDA_ARCH__)
    const double lg = gl::log10(g);
#else
    const double lg = std::log10(g);
#endif
    int ct = wrap_add(36, host_int(90 * th_res));
    ct = wrap_add(ct, host_int(vmax(0.0, lg - 1) * th_res * 55));
    ct = wrap_add(ct, host_int(lg * th_res * 25));
    ct = wrap_add(ct, 64);
    const int cp = wrap_add((int)((unsigned)imax(host_int(360 * ph_res), 1) * 5u), 8);
    return Caps{ct, cp};
}

// ---- host only: batch planning shared by vag_b200.cu and the host emulation (oracle/hostemu/hostemu.cpp) -----
// capacities of a batch from host-side parameters
inline Caps caps_for(const vag_params* p, size_t n) {
    Caps c{64, 8};
    for (size_t i = 0; i < n; ++i) {
        const Caps b = caps_of(p[i]);
        c.theta = std::max(c.theta, b.theta);
        c.phi = std::max(c.phi, b.phi);
    }
    return c;
}

// Banded series: the boundary luminosities of every (node, band) are staged once per row instead of two spectra per
// (point, row): n_bands * n_t tile evaluations against 2 * n_points per-point ones.  Measured on the config-5 batch
// (5 bands, ~100-node lattices, scripts/series_ab.py): 3.18 ms banded, flat in the number of points, against 1.97 ms
// per 100 points -- the break-even is n_bands * n_t ~ 3 n_points.  n_bands: distinct frequencies of the request (0
// when not banded at all), max_n_t: longest time lattice of the batch, series_mode as vag_set_series_mode.
inline bool series_banded(int n_bands, int max_n_t, size_t n_points, int series_mode) {
    return n_bands >= 1 && n_bands <= EATS_NU_TILE && (series_mode == 2 || (size_t)n_bands * max_n_t <= 3 * n_points);
}

// A ragged request (several data sets, vag_chi2_multi) runs banded when every data set passes series_banded with the
// batch's max_n_t.  With max_bands = the largest count of distinct frequencies of a set and min_q = the smallest
// floor(3 n / n_bands) of a set, that is this test: n_bands * max_n_t <= 3 n  <=>  max_n_t <= floor(3 n / n_bands).
inline bool series_banded_sets(int max_bands, int min_q, int max_n_t, int series_mode) {
    return max_bands >= 1 && max_bands <= EATS_NU_TILE && (series_mode == 2 || max_n_t <= min_q);
}

}  // namespace vag
