// TEST INFRASTRUCTURE ONLY: sequential host execution of the *same* kernel bodies that
// vegasafterglow_b200/csrc/vag_b200.cu launches on the GPU (every body is an HD function of the
// thread index; barriers become loop boundaries).  Lets the CPU-only test tier compare the
// device algorithm against the reference stage by stage.  It is never built into, linked with or
// called by the product library (libvag_b200.so).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../vegasafterglow_b200/csrc/vag_libm.cuh"
#include "../../vegasafterglow_b200/csrc/vag_pipeline.cuh"

using namespace vag;

namespace {

struct HostBatch {
    BatchWs w{};
    std::vector<void*> allocs;
    template <class T>
    T* alloc(size_t n) {
        T* p = static_cast<T*>(std::calloc(std::max<size_t>(n, 1), sizeof(T)));
        allocs.push_back(p);
        return p;
    }
    ~HostBatch() {
        for (void* p : allocs) std::free(p);
    }
};

const double* softplus_table() {
    static std::vector<double> lut;
    if (lut.empty()) {
        lut.resize(SPL_DOUBLES);
        build_softplus_lut(lut.data());
    }
    return lut.data();
}

void run_front(HostBatch& hb, const vag_params* params, size_t n, double t_min, double t_max) {
    BatchWs& w = hb.w;
    w.n_models = (int)n;
    w.sp_lut = softplus_table();
    const Caps caps = caps_for(params, n);  // vag_b200.cu plans its host-buffer batches the same way
    w.cap_theta = caps.theta;
    w.cap_phi = caps.phi;
    w.work_per_model = grid_work_doubles(w.cap_theta, w.cap_phi);
    w.params = params;
    w.cfg = hb.alloc<ModelCfg>(n);
    w.hdr = hb.alloc<GridHeader>(n);
    w.theta = hb.alloc<double>(n * w.cap_theta);
    w.phi = hb.alloc<double>(n * w.cap_phi);
    w.t_dec = hb.alloc<double>(n * w.cap_theta);
    w.work = hb.alloc<double>(n * w.work_per_model);
    w.reps = hb.alloc<int>(n * w.cap_theta);
    w.rep_of = hb.alloc<int>(n * w.cap_theta);
    w.row_off = hb.alloc<int>(n + 1);
    w.cell_off = hb.alloc<long long>(n + 1);
    w.totals = hb.alloc<int>(TOT_N);
    w.status = hb.alloc<int>(n);
    for (size_t i = 0; i < n; ++i) k0_grid_body(SeqPar{}, w, (int)i, t_min, t_max);
    k0b_scan_body(w);
    const int rows = w.totals[TOT_ROWS];
    const long long cells = w.cell_off[n];
    w.n_cells = cells;
    w.row_model = hb.alloc<int>(rows);
    w.row_rep = hb.alloc<int>(rows);
    w.inj_idx = hb.alloc<int>(rows);
    w.row_dyn = hb.alloc<RowDyn>(rows);
    w.row_cell_off = hb.alloc<long long>(rows + 1);
    w.t_rows = hb.alloc<double>(cells);
    for (int a = 0; a < 6; ++a) {
        w.fwd[a] = hb.alloc<double>(cells);
        w.rvs[a] = hb.alloc<double>(cells);
    }
    w.geo_u = hb.alloc<double>(cells);
    w.geo_lg2r2 = hb.alloc<double>(cells);
    w.sh_theta = w.geo_cth = w.geo_sth = w.geo_dcos = nullptr;
    if (w.totals[TOT_ANY_SPREAD]) {
        w.sh_theta = hb.alloc<double>(cells);
        w.geo_cth = hb.alloc<double>(cells);
        w.geo_sth = hb.alloc<double>(cells);
        w.geo_dcos = hb.alloc<double>(cells);
    }
    w.coef_fwd = hb.alloc<double>((size_t)cells * PH_NCOEF);
    w.coef_rvs = hb.alloc<double>((size_t)cells * PH_NCOEF);
    w.max_n_t = std::max(w.totals[TOT_MAX_NT], 1);
    w.max_erows = std::max(w.totals[TOT_MAX_EROWS], 1);
    w.any_ssc = w.totals[TOT_ANY_SSC];
    for (size_t i = 0; i < n; ++i) k0c_rowmap_body(w, (int)i);
    for (int r = 0; r < rows; ++r) k1_lattice_body(w, r, 0, 1);
    for (int r = 0; r < rows; ++r) {
        double col[K1_COL_DOUBLES];
        if (w.cfg[w.row_model[r]].has_rvs)
            k1_dynamics_body<true>(w, r, col, 1);
        else
            k1_dynamics_body<false>(w, r, col, 1);
    }
    for (int r = 0; r < rows; ++r) {
        const RowCtx c = row_ctx(w, r);
        for (int k = 0; k < c.n_t; ++k) k1b_finish_cell(w, r, c, k);
        if (c.has_rvs && w.row_dyn[r].n_saved >= 0) {
            const int idx_cut = extrap_scan(shock_row(w.rvs, c.off), c.n_t, 0, 1);
            for (int k = 0; k < c.n_t; ++k) k1c_extrap_cell(w, r, c, idx_cut, k);
        }
        for (int k = 0; k < c.n_t; ++k) {
            k1d_geo_cell(w, c, k);
            if (w.cfg[c.mi].spreading && w.sh_theta) k1e_spread_geo_cell(w, r, c, k);
        }
    }
    if (w.any_ssc) {
        for (int sft = 0; sft < 2; ++sft) {
            w.ic[sft] = hb.alloc<IcCell>(cells);
            w.ictab_h[sft] = hb.alloc<IcTable>(cells);
            w.ictab[sft] = hb.alloc<double>((size_t)cells * IC_CAP_OUT);
        }
        w.rowcos = hb.alloc<double>(n * w.max_erows);
        w.dop_min = hb.alloc<double>(n * w.max_n_t);
        w.dop_max = hb.alloc<double>(n * w.max_n_t);
        KnLut* lut = hb.alloc<KnLut>(1);
        for (int i = 0; i < KN_LUT_N; ++i) kn_lut_entry(i, lut->ratio[i], lut->lg2_ratio[i]);
        w.lut = lut;
        w.ic_scratch = hb.alloc<double>(IC_SCRATCH_DOUBLES);
    }
    for (int r = 0; r < rows; ++r) {
        const GridHeader& h = w.hdr[w.row_model[r]];
        const ModelCfg& cfg = w.cfg[w.row_model[r]];
        for (int sft = 0; sft < (cfg.has_rvs ? 2 : 1); ++sft) {
            if ((sft ? cfg.rvs : cfg.fwd).ssc) {
                k2_ic_cool_row(w, r, sft);
            } else {
                for (int k = 0; k < h.n_t; ++k) k2_radiation_cell(w, r, k, sft);
            }
        }
    }
}

// SSC tables need the observation band: run after the request is known
void run_ic_tables(HostBatch& hb, const double* nu_range) {
    BatchWs& w = hb.w;
    if (!w.any_ssc) return;
    w.nu_range = nu_range;
    for (int mi = 0; mi < w.n_models; ++mi) {
        const GridHeader& h = w.hdr[mi];
        for (int q = 0; q < h.n_theta * h.n_phi_eff; ++q) k_rowcos_body(w, mi, q);
        for (int k = 0; k < h.n_t; ++k) k_dop_extrema_body(w, mi, k);
    }
    const int rows = w.totals[TOT_ROWS];
    for (int r = 0; r < rows; ++r) {
        const int mi = w.row_model[r];
        const GridHeader& h = w.hdr[mi];
        const ModelCfg& cfg = w.cfg[mi];
        for (int sft = 0; sft < (cfg.has_rvs ? 2 : 1); ++sft) {
            if (!(sft ? cfg.rvs : cfg.fwd).ssc) continue;
            for (int k = 0; k < h.n_t; ++k) w.status[mi] |= k2b_ic_spectrum_cell(SeqPar{}, w, r, k, sft, w.ic_scratch);
        }
    }
}

// sequential emulation of the K3 CTA (vag_b200.cu: k_eats) for one (model, shock)
void eats_emulate(const BatchWs& w, int mi, int which, const EatsRequest& rq0, double* out /*[n_nu][n_t] or [n]*/) {
    const int NTHR = 128;
    EatsModel M = make_eats_model(w, mi, which);
    const GridHeader& h = *M.h;
    const int n_t = h.n_t;
    const int erows = h.n_theta * h.n_phi_eff;
    const bool series = rq0.series != 0;
    const bool banded = rq0.n_bands > 0;
    const int nu_tile = series ? (banded ? rq0.n_bands : 1) : std::min(EATS_NU_TILE, rq0.n_nu);
    std::vector<double> smem(eats_shared_doubles(n_t, series && !banded, EATS_ROW_CHUNK, nu_tile) + 8);
    std::vector<double> acc(EATS_NU_TILE * EATS_T_BLOCK);
    EatsShared sh = eats_carve(smem.data(), n_t, series && !banded, EATS_ROW_CHUNK, nu_tile);
    std::vector<RowGeom> rowg(erows);
    for (int q = 0; q < erows; ++q) rowg[q] = row_geometry(M, q / h.n_theta, q % h.n_theta);
    const int rows_per_pass = eats_rows_per_pass(n_t, EATS_ROW_CHUNK, NTHR);
    EatsRequest rq = rq0;
    const int n_nu_tiles = series ? 1 : (rq.n_nu + nu_tile - 1) / nu_tile;
    for (int tile = 0; tile < n_nu_tiles; ++tile) {
        const int l0 = tile * nu_tile;
        const int nl = series ? (banded ? rq.n_bands : 1) : std::min(nu_tile, rq.n_nu - l0);
        for (int i0 = 0; i0 < rq.n_t_obs; i0 += EATS_T_BLOCK) {
            rq.i0 = i0;
            rq.ni = std::min(EATS_T_BLOCK, rq.n_t_obs - i0);
            std::fill(acc.begin(), acc.end(), 0.0);
            for (int q0 = 0; q0 < erows; q0 += rows_per_pass) {
                const int nrows = std::min(rows_per_pass, erows - q0);
                sh.rowg = rowg.data() + q0;
                for (int tid = 0; tid < NTHR; ++tid) {
                    const bool point = series && !banded;
                    if (M.mode == 0) point ? eats_phase1<0, true>(M, rq, sh, nrows, l0, nl, tid, NTHR) : eats_phase1<0, false>(M, rq, sh, nrows, l0, nl, tid, NTHR);
                    if (M.mode == 1) point ? eats_phase1<1, true>(M, rq, sh, nrows, l0, nl, tid, NTHR) : eats_phase1<1, false>(M, rq, sh, nrows, l0, nl, tid, NTHR);
                    if (M.mode == 2) point ? eats_phase1<2, true>(M, rq, sh, nrows, l0, nl, tid, NTHR) : eats_phase1<2, false>(M, rq, sh, nrows, l0, nl, tid, NTHR);
                }
                for (int tid = 0; tid < NTHR; ++tid) {
                    if (banded) {
                        eats_phase2_banded(M, rq, sh, nrows, acc.data(), tid, NTHR);
                    } else if (!series) {
                        eats_phase2_grid(M, rq, sh, nrows, nl, acc.data(), tid, NTHR);
                    } else {
                        if (M.mode == 0) eats_phase2_series<0>(M, rq, sh, nrows, acc.data(), tid, NTHR);
                        if (M.mode == 1) eats_phase2_series<1>(M, rq, sh, nrows, acc.data(), tid, NTHR);
                        if (M.mode == 2) eats_phase2_series<2>(M, rq, sh, nrows, acc.data(), tid, NTHR);
                    }
                }
            }
            if (series) {
                for (int ii = 0; ii < rq.ni; ++ii) out[i0 + ii] = flux_scale(M, acc[ii]);
            } else {
                for (int l = 0; l < nl; ++l)
                    for (int ii = 0; ii < rq.ni; ++ii)
                        out[(size_t)(l0 + l) * rq.n_t_obs + i0 + ii] = flux_scale(M, acc[l * rq.acc_stride + ii]);
            }
        }
    }
}

int g_series_mode = 0;  // as vag_set_series_mode (include/vag.h)

int run_flux(const vag_params* params, size_t n, const double* t, size_t n_t, const double* nu, size_t n_nu,
             bool series, double* out, int32_t* status) {
    HostBatch hb;
    const double t_min = *std::min_element(t, t + n_t), t_max = *std::max_element(t, t + n_t);
    run_front(hb, params, n, t_min, t_max);
    std::vector<double> lg2t(n_t), tl(n_t), lg2nu(n_nu), nul(n_nu), nu23(n_nu);
    for (size_t i = 0; i < n_t; ++i) {
        tl[i] = t[i] * unit::sec;
        lg2t[i] = std::log2(tl[i]);
    }
    for (size_t i = 0; i < n_nu; ++i) {
        nul[i] = nu[i] * unit::Hz;
        lg2nu[i] = std::log2(nul[i]);
        nu23[i] = std::exp2((2. / 3) * lg2nu[i]);
    }
    EatsRequest rq{};
    rq.series = series ? 1 : 0;
    rq.n_t_obs = (int)n_t;
    rq.n_nu = (int)n_nu;
    rq.lg2_t_obs = lg2t.data();
    rq.lg2_nu_obs = lg2nu.data();
    rq.nu_obs_lin = nul.data();
    rq.nu23_obs = nu23.data();
    rq.t_obs_lin = tl.data();
    rq.acc_stride = eats_acc_stride((int)n_t);
    // banded series (vag_b200.cu run_flux_pass / k_series_bands): distinct frequencies in order of first appearance
    std::vector<int> band_of(n_t, 0);
    std::vector<double> b_lg2, b_lin, b_23;
    if (series && g_series_mode != 1) {
        bool ok = true;
        for (size_t i = 0; i < n_nu && ok; ++i) {
            int q = -1;
            for (size_t b = 0; b < b_lg2.size(); ++b)
                if (b_lg2[b] == lg2nu[i]) q = (int)b;
            if (q < 0) {
                if ((int)b_lg2.size() >= EATS_NU_TILE || !(lg2nu[i] == lg2nu[i])) {
                    ok = false;
                    break;
                }
                q = (int)b_lg2.size();
                b_lg2.push_back(lg2nu[i]);
                b_lin.push_back(nul[i]);
                b_23.push_back(nu23[i]);
            }
            band_of[i] = q;
        }
        if (series_banded(ok ? (int)b_lg2.size() : 0, hb.w.max_n_t, n_t, g_series_mode)) {
            rq.n_bands = (int)b_lg2.size();
            rq.band_of = band_of.data();
            rq.lg2_nu_obs = b_lg2.data();
            rq.nu_obs_lin = b_lin.data();
            rq.nu23_obs = b_23.data();
        }
    }
    const size_t comp = series ? n_t : n_nu * n_t;
    double nu_range[2] = {*std::min_element(lg2nu.begin(), lg2nu.end()), *std::max_element(lg2nu.begin(), lg2nu.end())};
    run_ic_tables(hb, nu_range);
    for (size_t mi = 0; mi < n; ++mi) {
        double* o = out + mi * VAG_NCOMP * comp;
        std::memset(o, 0, sizeof(double) * VAG_NCOMP * comp);
        if (hb.w.hdr[mi].status & VAG_ST_CAPACITY) continue;
        eats_emulate(hb.w, (int)mi, 0, rq, o + VAG_C_FWD_SYNC * comp);
        if (params[mi].has_rvs) eats_emulate(hb.w, (int)mi, 1, rq, o + VAG_C_RVS_SYNC * comp);
        if (params[mi].fwd.ssc) eats_emulate(hb.w, (int)mi, 2, rq, o + VAG_C_FWD_SSC * comp);
        if (params[mi].has_rvs && params[mi].rvs.ssc) eats_emulate(hb.w, (int)mi, 3, rq, o + VAG_C_RVS_SSC * comp);
        for (size_t i = 0; i < comp; ++i)
            o[i] = o[VAG_C_FWD_SYNC * comp + i] + o[VAG_C_FWD_SSC * comp + i] + o[VAG_C_RVS_SYNC * comp + i] +
                   o[VAG_C_RVS_SSC * comp + i];
        if (status) status[mi] = hb.w.status[mi];
    }
    return 0;
}

}  // namespace

extern "C" {
void vagemu_set_series_mode(int mode) { g_series_mode = mode; }

// max |log2_softplus_lut - log2(1 + 2^x)| over n points of [-20, 20] (reference in long double)
double vagemu_softplus_lut_maxerr(int n) {
    const double* lut = softplus_table();
    double worst = 0;
    for (int i = 0; i <= n; ++i) {
        const double x = -20.0 + 40.0 * (double)i / n;
        const long double ref = log2l(1.0L + exp2l((long double)x));
        worst = std::max(worst, (double)fabsl((long double)log2_softplus_lut(lut, x) - ref));
    }
    return worst;
}

int vagemu_flux_density_grid(const vag_params* params, size_t n, const double* t, size_t n_t, const double* nu,
                             size_t n_nu, double* out, int32_t* status) {
    return run_flux(params, n, t, n_t, nu, n_nu, false, out, status);
}

int vagemu_flux_density_series(const vag_params* params, size_t n, const double* t, const double* nu, size_t npts,
                               double* out, int32_t* status) {
    return run_flux(params, n, t, npts, nu, npts, true, out, status);
}

// same contract as vag_details (include/vag.h) + photon coefficient planes
int vagemu_details(const vag_params* p, double t_min, double t_max, vag_grid_info* info, double* theta, double* phi,
                   int32_t* reps, double* t_rows, double* fwd_shock, double* rvs_shock, int32_t* inj_idx,
                   double* coef_fwd, double* coef_rvs) {
    HostBatch hb;
    run_front(hb, p, 1, t_min, t_max);
    const BatchWs& w = hb.w;
    const GridHeader& h = w.hdr[0];
    if (info) {
        info->n_phi = h.n_phi;
        info->n_theta = h.n_theta;
        info->n_t = h.n_t;
        info->n_reps = h.n_reps;
        info->symmetry = h.symmetry;
        info->phi_mirrored = h.phi_mirrored;
        info->n_phi_eff = h.n_phi_eff;
        info->status = w.status[0];
    }
    const size_t cells = (size_t)h.n_reps * h.n_t;
    if (theta) std::memcpy(theta, w.theta, sizeof(double) * h.n_theta);
    if (phi) std::memcpy(phi, w.phi, sizeof(double) * h.n_phi);
    if (reps)
        for (int r = 0; r < h.n_reps; ++r) reps[r] = h.rows3d ? r % h.n_theta : w.reps[r];
    if (t_rows) std::memcpy(t_rows, w.t_rows, sizeof(double) * cells);
    auto dump = [&](double* const* pl, double* o) {
        // order t_comv, r, theta, Gamma, Gamma_th, B, N_p
        const int map[7] = {0, 1, -1, 2, 3, 4, 5};
        for (int a = 0; a < 7; ++a)
            for (int r = 0; r < h.n_reps; ++r)
                for (int k = 0; k < h.n_t; ++k)
                    o[((size_t)a * h.n_reps + r) * h.n_t + k] =
                        map[a] < 0 ? (w.sh_theta ? w.sh_theta[(size_t)r * h.n_t + k] : w.theta[h.rows3d ? r % h.n_theta : w.reps[r]]) : pl[map[a]][(size_t)r * h.n_t + k];
    };
    if (fwd_shock) dump(w.fwd, fwd_shock);
    if (rvs_shock && p->has_rvs) dump(w.rvs, rvs_shock);
    if (inj_idx) std::memcpy(inj_idx, w.inj_idx, sizeof(int) * h.n_reps);
    if (coef_fwd) std::memcpy(coef_fwd, w.coef_fwd, sizeof(double) * cells * PH_NCOEF);
    if (coef_rvs && p->has_rvs) std::memcpy(coef_rvs, w.coef_rvs, sizeof(double) * cells * PH_NCOEF);
    return 0;
}

// gl:: functions of vag_libm.cuh (use_ref = 0) or the live libm they restate (use_ref = 1), elementwise.
// fn: 0 exp, 1 exp2, 2 log, 3 log2, 4 log10, 5 pow(x, y), 6 sin, 7 cos
int vagemu_libm_eval(int fn, const double* x, const double* y, double* out, size_t n, int use_ref) {
    for (size_t i = 0; i < n; ++i) {
        const double a = x[i], b = y ? y[i] : 0.0;
        double r;
        switch (fn) {
            case 0: r = use_ref ? std::exp(a) : gl::exp(a); break;
            case 1: r = use_ref ? std::exp2(a) : gl::exp2(a); break;
            case 2: r = use_ref ? std::log(a) : gl::log(a); break;
            case 3: r = use_ref ? std::log2(a) : gl::log2(a); break;
            case 4: r = use_ref ? std::log10(a) : gl::log10(a); break;
            case 5: r = use_ref ? std::pow(a, b) : gl::pow(a, b); break;
            case 6: r = use_ref ? std::sin(a) : gl::sin(a); break;
            case 7: r = use_ref ? std::cos(a) : gl::cos(a); break;
            default: return -1;
        }
        out[i] = r;
    }
    return 0;
}

}  // extern "C"
