/*
 * vag.h -- C ABI of the B200-native VegasAfterglow model-evaluation path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b): plain pointers and sizes, no
 * torch / pybind / xtensor types.  Every entry point names the reference interface it
 * replaces (paths relative to the reference repository root).
 *
 * Units at this boundary are the reference's *Python-facing* units (pybind/pymodel.cpp:498-514,
 * pybind/pymodel.h:246): seconds, Hz, cm, erg, cm^-3 in; erg cm^-2 s^-1 Hz^-1 out.
 *
 * All compute entry points run on the GPU (sm_100a kernels).  There is no CPU fallback: when no
 * CUDA device is usable they return VAG_ERR_CUDA and vag_last_error() says why.
 */
#ifndef VAG_H_
#define VAG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------- */
/* status codes                                                                                 */
/* ------------------------------------------------------------------------------------------- */
enum {
    VAG_OK = 0,
    VAG_ERR_INVALID = 1, /* argument validation failed: mirrors AFTERGLOW_REQUIRE -> ValueError
                            (pybind/error_handling.h:31-69) */
    VAG_ERR_CUDA = 2,    /* CUDA runtime error / no device                                       */
    VAG_ERR_UNSUPPORTED = 3, /* a switch of the reference that this path does not implement (Python-callable
                                Ejecta / Medium profiles cannot be expressed in vag_params at all)  */
    VAG_ERR_CAPACITY = 4     /* a per-model grid exceeded the compiled capacity                  */
};

/* jet / medium enumerations: the typed variants of JetVariant / MediumVariant
 * (src/environment/jet.h:272, src/environment/medium.h:144). */
enum {
    VAG_JET_TOPHAT = 0,
    VAG_JET_GAUSSIAN = 1,
    VAG_JET_POWERLAW = 2,
    /* closed-form members of the reference's Ejecta family (pybind/pymodel.cpp:97-146,
     * src/environment/jet.h:403-470) as enumerated device profiles */
    VAG_JET_TWO_COMPONENT = 3, /* TwoComponentJet(theta_c, E_iso, Gamma0, theta_w, E_iso_w, Gamma0_w)        */
    VAG_JET_STEP_POWERLAW = 4, /* StepPowerLawJet(theta_c, E_iso, Gamma0, E_iso_w, Gamma0_w, k_e, k_g)       */
    VAG_JET_POWERLAW_WING = 5  /* PowerLawWing(theta_c, E_iso_w, Gamma0_w, k_e, k_g)                         */
};
enum { VAG_MEDIUM_ISM = 0, VAG_MEDIUM_WIND = 1 };

/* per-model status bits written by the kernels (SURVEY.md section 5: the reference prints a
 * warning on stderr and leaves the row at its initial values; we mirror that and set a bit). */
enum {
    VAG_ST_ODE_STEP_CAP = 1,  /* forward-shock.tpp:196-200 / reverse-shock.tpp:555-559           */
    VAG_ST_ODE_STALLED = 2,   /* reverse-shock.tpp:560-566                                       */
    VAG_ST_ODE_FAIL500 = 4,   /* boost max_step_checker.hpp:99-106 (reference throws)            */
    VAG_ST_GRID_NONFINITE = 8, /* grid-refinement.h:633-635                                      */
    VAG_ST_CAPACITY = 16,     /* grid / SSC lattice larger than compiled capacity; model output is NaN */
    VAG_ST_IC_BAND = 32,      /* an SSC query left the clamped output band (inverse-compton.h:622-635:
                                 the reference would rebuild that cell's full-range spectrum)      */
    VAG_ST_INVALID = 64       /* the entry points that plan on the device (vag_chi2_dev, vag_flux_band_dev): the
                                 reference constructors reject this parameter set; flux NaN, chi2 +inf */
};

/* Radiation(eps_e, eps_B, p, xi_e=1, ssc=False, kn=False): pybind/pymodel.h:303-313 */
typedef struct vag_radiation {
    double eps_e, eps_B, p, xi_e;
    int32_t ssc, kn;
} vag_radiation;

/* One parameter set = everything Model.__init__ receives (pybind/pybind.cpp:384-422,
 * pybind/pymodel.h:613-649) for the typed jet/medium variants. */
typedef struct vag_params { /* 320 bytes, mirrored by vegasafterglow_b200/abi.py PARAMS_DTYPE */
    /* jet: TophatJet/GaussianJet/PowerLawJet(theta_c, E_iso, Gamma0[, k_e, k_g], spreading,
     * duration)  pybind/pymodel.cpp:47-95; two-component / step-power-law / power-law-wing :97-146 */
    int32_t jet_type;
    int32_t spreading; /* spreading=True of the jet factories: lateral spreading (forward-shock models) and
                          Symmetry::structured lattices; with axisymmetric = 0 one ODE row per (phi, theta) cell */
    double theta_c, E_iso, Gamma0, k_e, k_g, duration;
    double theta_w, E_iso_w, Gamma0_w; /* wing of the two-component / step-power-law / power-law-wing jets */
    double sigma0;                     /* ejecta magnetisation (constant; the reference expresses it through
                                          Ejecta(sigma0=...)); 0 = unmagnetised */
    /* medium: ISM(n_ism) / Wind(A_star, n_ism=0, n0=inf, k_m=2)  pybind/pymodel.cpp:148-186 */
    int32_t medium_type;
    int32_t pad0_;
    double n_ism, A_star, n0;
    /* Observer(lumi_dist[cm], z, theta_obs, phi_obs=0)  pybind/pymodel.h:190-204 */
    double lumi_dist, z, theta_obs, phi_obs;
    /* radiation */
    vag_radiation fwd;
    vag_radiation rvs;
    int32_t has_rvs;
    int32_t axisymmetric;       /* default 1 */
    int32_t radiative_fireball; /* default 1 */
    int32_t pad1_;
    /* resolutions=(phi, theta, t); a value <= 0 selects the reference default
     * (0.06,0.15,6) forward-only or (0.06,0.2,10) with a reverse shock
     * (src/config/simulation-defaults.h:71-83, pybind/pymodel.h:633-640) */
    double phi_resol, theta_resol, t_resol;
    double rtol; /* <= 0 selects defaults::solver::dynamics_rtol = 1e-6 */
    /* magnetar=Magnetar(L0 [erg/s], t0 [s], q) of the jet factories (pybind/pymodel.h:34-58): energy injection
     * L0 (1 + t/t0)^-q for theta <= theta_c (src/environment/jet.h:518-528).  As in the reference the jet then
     * takes the generic-Ejecta code path (pybind/pymodel.cpp:53-59). */
    int32_t has_magnetar;
    int32_t pad2_;
    double magnetar_L0, magnetar_t0, magnetar_q;
    /* Wind(..., k_m): density slope of the wind, rho = A / (r0^k + r^k) + rho_ism.  2 (or <= 0) selects the typed
     * Wind of the reference; any other value takes its generic-Medium path (pybind/pymodel.cpp:169-185:
     * numeric enclosed mass / thermal energy, CGS profile behind convert_unit_medium). */
    double wind_k_m;
} vag_params;

/* Fill *p with the reference defaults (Tophat/ISM values are NOT set, only the switches). */
void vag_params_default(vag_params* p);

/* Validate one parameter set exactly like the reference constructors do
 * (pybind/pymodel.cpp:47-186, pybind/pymodel.h:190-204,303-313,613-649).
 * Returns VAG_OK or VAG_ERR_INVALID / VAG_ERR_UNSUPPORTED; message via vag_last_error(). */
int vag_params_validate(const vag_params* p);

/* ------------------------------------------------------------------------------------------- */
/* context                                                                                      */
/* ------------------------------------------------------------------------------------------- */
typedef struct vag_context vag_context;

/* Create a context bound to CUDA device `device` (owns a stream and growable workspaces). */
int vag_create(int device, vag_context** out);
void vag_destroy(vag_context* ctx);
const char* vag_last_error(void);
const char* vag_version(void);

/* Output component order of every flux entry point: PyFlux (pybind/pymodel.h:394-400). */
enum { VAG_C_TOTAL = 0, VAG_C_FWD_SYNC = 1, VAG_C_FWD_SSC = 2, VAG_C_RVS_SYNC = 3, VAG_C_RVS_SSC = 4, VAG_NCOMP = 5 };

/* ------------------------------------------------------------------------------------------- */
/* batched model evaluation, HOST buffers (copies inside)                                       */
/* ------------------------------------------------------------------------------------------- */

/* Replaces PyModel::flux_density_grid (pybind/pymodel.cpp:498-514) for n_models parameter sets
 * sharing one (t, nu) request.  t ascending [s], nu [Hz].
 * out[n_models][VAG_NCOMP][n_nu][n_t]  (components a model does not have are 0; total = sum,
 * pybind/pymodel.cpp:350-364).  status[n_models] receives VAG_ST_* bits (may be NULL). */
int vag_flux_density_grid(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, size_t n_t,
                          const double* nu, size_t n_nu, double* out, int32_t* status);

/* Replaces PyModel::flux_density (pybind/pymodel.cpp:373-389): series of (t[i], nu[i]) points,
 * t ascending.  out[n_models][VAG_NCOMP][n]. */
int vag_flux_density_series(vag_context* ctx, const vag_params* params, size_t n_models, const double* t,
                            const double* nu, size_t n, double* out, int32_t* status);

/* Replaces PyModel::flux_density_exposures (pybind/pymodel.cpp:412-496): point i is the average over its exposure
 * expo_time[i] > 0 of num_points samples t[i] + j dt, dt = expo_time[i] / (num_points - 1), j = 0 .. num_points-1 (product
 * and sum rounded separately).  t need not be sorted.  All n * num_points samples are sorted stably by time (ties: point
 * index, then j) and run as ONE shared series request -- exactly vag_flux_density_series on them, with its series modes
 * and output modes -- and a kernel averages on the device: a point's samples added to 0.0 in sorted order, divided by
 * num_points.  Only out[n_models][VAG_NCOMP][n] crosses PCIe.  The result equals that series call followed by that host
 * averaging bit for bit.  status as vag_flux_density_series.  Launches: those of vag_flux_density_series on the samples
 * + 1.  Checks, all before any work is enqueued, in this order and with the messages of the reference's: num_points >= 2,
 * every expo_time[i] finite and > 0, n > 0, t and nu finite and > 0; n * num_points within a 32-bit int. */
int vag_flux_density_exposures(vag_context* ctx, const vag_params* params, size_t n_models, const double* t,
                               const double* nu, const double* expo_time, size_t n, size_t num_points, double* out,
                               int32_t* status);

/* Replaces PyModel::flux (pybind/pymodel.cpp:391-410) = Observer::flux (src/core/observer.h:555-567):
 * flux integrated over [nu_min, nu_max] Hz with Boole weights on num_nu log-spaced frequencies
 * (src/core/quadrature.h:138-191).  out[n_models][VAG_NCOMP][n_t] in erg cm^-2 s^-1. */
int vag_flux_band(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, size_t n_t,
                  double nu_min, double nu_max, size_t num_nu, double* out, int32_t* status);

/* Replaces Fitter._evaluate + _chi2_sum for point data (VegasAfterglow/fitting/fitter.py:497-522):
 * chi2[m] = sum_i w[i] * ((lnF_obs[i] - ln max(F_model[i], 1e-300)) / sigma_ln[i])^2
 * over the series (t[i], nu[i]); non-finite chi2 is returned as +inf (samplers.py:63-70 maps it
 * to logL = -inf).  t ascending. */
int vag_chi2_series(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, const double* nu,
                    const double* lnF_obs, const double* sigma_ln, const double* w, size_t n, double* chi2,
                    int32_t* status);

/* One band-integrated data set of the likelihood (VegasAfterglow/fitting/fitter.py BandObs, :525-531): observed
 * band fluxes [erg cm^-2 s^-1] at ascending epochs t[n], compared with Model.flux(t, nu_min, nu_max, num_nu). */
typedef struct vag_band_obs {
    const double* t;        /* [n] seconds, ascending                                   */
    const double* lnF_obs;  /* [n] ln(observed band flux)                               */
    const double* sigma_ln; /* [n] err / flux                                           */
    const double* w;        /* [n] weights                                              */
    size_t n;
    double nu_min, nu_max;  /* Hz                                                        */
    size_t num_nu;          /* frequency nodes of the Boole quadrature (>= 2)            */
} vag_band_obs;

/* Replaces Fitter._evaluate (fitter.py:503-533) for a batch: chi2[i] = sum over the point data (as vag_chi2_series;
 * n_points may be 0) + sum over every band data set of w ((lnF_obs - ln max(F_band, 1e-300)) / sigma_ln)^2.
 * A non-finite sum, or a model whose ODE hit Boost's 500-rejection limit (VAG_ST_ODE_FAIL500 -- an exception in the
 * reference, logL = -inf in its samplers, samplers.py:63-70), gives chi2 = +inf.  status[i] = OR over all terms. */
int vag_chi2(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, const double* nu,
             const double* lnF_obs, const double* sigma_ln, const double* w, size_t n_points, const vag_band_obs* bands,
             size_t n_bands, double* chi2, int32_t* status);

/* vag_chi2 with host-galaxy extinction fitted per model (Fitter with an extinction law, fitter.py:512-519): the point
 * term compares model m with lnF_obs[i] + A_V[m] * ext_k[i] (product rounded, then sum) instead of lnF_obs[i]; band
 * terms are unchanged.  ext_k[n_points] is in the order of the points (time-sorted) and must be finite; A_V[n_models]
 * is not range-checked (a non-finite A_V gives chi2 = +inf).  ext_k and A_V are both NULL (exactly vag_chi2) or both
 * set, and then n_points > 0.  Same launches as vag_chi2 on the same data. */
int vag_chi2_ext(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, const double* nu,
                 const double* lnF_obs, const double* sigma_ln, const double* w, const double* ext_k, size_t n_points,
                 const double* A_V, const vag_band_obs* bands, size_t n_bands, double* chi2, int32_t* status);

/* ---- several light curves in one batch: every model has its own data set ------------------------------------------
 * The points of all data sets are concatenated into t / nu (and lnF_obs / sigma_ln / w / ext_k) of n_points_total
 * entries; data set d is the slice [sets[d].offset, sets[d].offset + sets[d].n), ascending in time.  Model m is
 * evaluated on data set dataset_of[m] only: its grid window, time lattice and values are those that
 * vag_flux_density_series / vag_chi2_series / vag_chi2_ext give for it on that data set alone (bit for bit when
 * neither call splits the rows of a model over several CTAs -- i.e. from 2368 (model x shock) CTAs on 148 SMs -- and both
 * stage the same number of rows per pass; otherwise to rounding).  An SSC model's tables span its own data set's band.
 * Series modes (vag_set_series_mode) apply to the batch as a whole: it runs banded only when EVERY data set passes the
 * banded test of a single request with the batch's longest time lattice -- mode 0: n_bands(d) <= 8 and
 * n_bands(d) * max_n_t <= 3 n(d) for every d; 1: never; 2: whenever every data set has at most 8 distinct frequencies.
 * Otherwise every model runs per point.
 * Checks, all before any work is enqueued (VAG_ERR_INVALID, the message names the data set or the model): every set
 * non-empty, inside the arrays, ascending, finite and > 0 in t, finite and > 0 in nu; 0 <= dataset_of[m] < n_sets;
 * parameter sets as vag_params_validate.  A data set no model uses is allowed.  Batches over 32768 models run in
 * passes as the other entry points do.  Launches: those of vag_chi2_series / vag_flux_density_series on the same
 * total data, whatever n_sets (one CTA per data set inside the band search kernel).
 * Band-integrated data per data set: vag_flux_band_multi, vag_chi2_multi_bands below; on device buffers, planned on the
 * device: vag_chi2_multi_bands_dev (further below).  A per-model grid (t x nu) request: vag_flux_density_grid_multi.
 * Not provided here: a device-buffer (_dev) variant of the two flux calls.
 * The output mode (vag_set_output_mode) does not apply: every plane of `out` is written. */
typedef struct vag_series_set {
    size_t offset, n; /* slice of the concatenated points */
} vag_series_set;

/* out: model m's [VAG_NCOMP][n of its data set] block starts at element VAG_NCOMP * off[m], off[m] = the sum of the
 * sizes of the data sets of models 0 .. m-1 (out has VAG_NCOMP * off[n_models] elements). */
int vag_flux_density_series_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                                  const vag_series_set* sets, size_t n_sets, const double* t, const double* nu,
                                  size_t n_points_total, double* out, int32_t* status);

/* chi2[m] of vag_chi2_series (ext_k / A_V NULL) or of vag_chi2_ext's point term (both set: ext_k[n_points_total] finite,
 * in point order; A_V[n_models], a non-finite A_V gives +inf) for model m on its data set.  VAG_ST_ODE_FAIL500 gives
 * +inf. */
int vag_chi2_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                   const vag_series_set* sets, size_t n_sets, const double* t, const double* nu, const double* lnF_obs,
                   const double* sigma_ln, const double* w, const double* ext_k, size_t n_points_total, const double* A_V,
                   double* chi2, int32_t* status);

/* ---- band-integrated data in a batch of several light curves ------------------------------------------------------
 * Every (model, band) pair of a call is one evaluation of a single ragged grid request: its own band times x its own
 * frequency nodes (band_grid of vag_flux_band), run through the pipeline once for all evaluations and reduced with each
 * band's weights.  Model m's values are those of vag_flux_band / vag_chi2_ext for that model on that band (data set)
 * alone: bit for bit when neither call splits the rows of a model over several CTAs (from 2368 (evaluation x shock)
 * CTAs on 148 SMs) and both stage the same number of rows per pass; otherwise to rounding.  The pass sizes its
 * shared-memory stage from the longest band and widest node set of the batch: that can lower the rows staged per pass
 * (long lattices), never the frequency tiles -- a model tiles its own num_nu nodes by min(8, widest num_nu) >=
 * min(8, its num_nu), which gives the tiles of its own call (one of num_nu nodes when num_nu <= 8, of 8 and the
 * remainder otherwise), so the same eats_phase2_grid instantiation sums the same terms.  An SSC model's tables span its
 * own band's nodes.  Batches over 32768 evaluations run in passes.  Checks, all before any work is enqueued
 * (VAG_ERR_INVALID, messages name the data set, the band or the model; a failed call leaves the context usable): every
 * band n > 0, t ascending, finite and > 0, nu_min / nu_max / num_nu as vag_flux_band; indices in range; parameter sets
 * as vag_params_validate.  Bands and data sets no model uses are allowed.  The output mode does not apply. */

/* Model.flux of model m on bands[band_of[m]]: only t, n, nu_min, nu_max and num_nu of a band are read (the data
 * pointers may be NULL).  out: model m's [VAG_NCOMP][n of its band] block starts at element VAG_NCOMP * off[m], off[m] =
 * the sum of the sizes of the bands of models 0 .. m-1 (the layout of vag_flux_density_series_multi).  Launches: those
 * of vag_flux_band on one band. */
int vag_flux_band_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* band_of,
                        const vag_band_obs* bands, size_t n_bands, double* out, int32_t* status);

/* One data set of vag_chi2_multi_bands: a slice of the concatenated points (n = 0: no point data) and its band-integrated
 * data bands[band0 .. band0 + n_bands), in this order.  n > 0 or n_bands > 0. */
typedef struct vag_multi_set {
    size_t offset, n;
    size_t band0, n_bands;
} vag_multi_set;

/* chi2[m] and status[m] of vag_chi2_ext (vag_chi2 when ext_k and A_V are NULL) for model m on its data set's points and
 * bands alone: the point term (0 without points), then each band's term in the set's order, added as band + chi2 with
 * the band sum sum_i F(nu_i) w_i in node order; VAG_ST_ODE_FAIL500 of the run a term came from gives +inf.  status = the
 * OR over the terms when the set has bands, the point run's status otherwise.  Point arrays as vag_chi2_multi (NULL
 * only when n_points_total == 0; every set with points passes vag_chi2_multi's checks, and those sets alone decide its
 * series mode); ext_k / A_V as vag_chi2_multi, and A_V[m] is not read for a model whose set has no points.  Band data
 * pointers must be set.  Launches, whatever n_sets and the number of bands: L(points) + L(bands) + 2, where L(points) =
 * those of vag_chi2_multi on the models with points (0 when none has one), L(bands) = those of vag_flux_band_multi on
 * all evaluations (0 when no model has a band), and the 2 are the device gather of the evaluations' parameter records
 * from the models' and the band chi-squared (a warp per model). */
int vag_chi2_multi_bands(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                         const vag_multi_set* sets, size_t n_sets, const double* t, const double* nu, const double* lnF_obs,
                         const double* sigma_ln, const double* w, const double* ext_k, size_t n_points_total,
                         const double* A_V, const vag_band_obs* bands, size_t n_bands_total, double* chi2, int32_t* status);

/* vag_chi2_multi_bands with exposure-averaged points.  expo_time[n_points_total] (point order, each finite and >= 0) and
 * num_expo[n_sets] (>= 2 for every set with a point whose expo_time > 0; not read otherwise).  A point with e = expo_time
 * > 0 of set d is the average of num_expo[d] samples over its exposure, by the rule of vag_flux_density_exposures; a point
 * with e = 0 is one sample at its time (its value is that sample's flux exactly).  The series request of set d is all its
 * samples, sorted stably by time (ties: point index, then j); that window also sets the set's grid.  The chi-squared rule
 * is unchanged: w ((lnF_obs + A_V ext_k - ln max(F_avg, 1e-300)) / sigma_ln)^2, and so are the band terms, the status OR,
 * VAG_ST_ODE_FAIL500 -> +inf, the passes of 32768 models and the series modes (applied to the sets of samples).  With
 * every expo_time = 0 the result equals vag_chi2_multi_bands bit for bit.  The point pass runs the samples without the
 * fused chi-squared, then one launch averages them (a CTA per point model) and one k_chi2 compares the averages with the
 * points' data.  Launches, when the point models fit one pass of 32768: those of vag_chi2_multi_bands on the sets of
 * samples + 1.  Checks, all before any work is enqueued (messages name the data set or the point; a failed call leaves
 * the context usable): those of vag_chi2_multi_bands, then expo_time and num_expo, every sample time finite, and the
 * samples of all sets within a 32-bit int.  Not provided: exposures on band data, a device-buffer (_dev) form. */
int vag_chi2_multi_bands_exposures(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                                   const vag_multi_set* sets, size_t n_sets, const double* t, const double* nu,
                                   const double* lnF_obs, const double* sigma_ln, const double* w, const double* ext_k,
                                   size_t n_points_total, const double* A_V, const double* expo_time,
                                   const int32_t* num_expo, const vag_band_obs* bands, size_t n_bands_total, double* chi2,
                                   int32_t* status);

/* ---- a (t x nu) grid request per model, and posterior-predictive bands across models ------------------------------
 * The times and frequencies of all grid sets are concatenated into t[n_t_total] and nu[n_nu_total]; set d is the times
 * t[t0 .. t0 + n_t), ascending, finite and > 0, crossed with the frequencies nu[nu0 .. nu0 + n_nu) [Hz], finite and > 0.
 * Model m is evaluated on set dataset_of[m] alone, as one evaluation of a single ragged grid request (the run of the band
 * section above, with frequencies in Hz through the same unit conversion as vag_flux_density_grid's).  Its values are
 * those of vag_flux_density_grid for that model on that set alone: bit for bit under the conditions stated for
 * vag_flux_band_multi (no row split in either call -- from 2368 (model x shock) CTAs on 148 SMs -- and the same rows
 * staged per pass; a model tiles its own n_nu as its own call does), otherwise to rounding.  An SSC model's tables span
 * its own set's frequencies.  Batches over 32768 models run in passes.  The output mode does not apply.
 * Checks, all before any work is enqueued (VAG_ERR_INVALID, the message names the set or the model; a failed call
 * leaves the context usable and the outputs untouched): every set n_t > 0 and n_nu > 0, inside the arrays, its times
 * ascending, finite and > 0, its frequencies finite and > 0; 0 <= dataset_of[m] < n_sets; parameter sets as
 * vag_params_validate; n_t_total, n_nu_total, n_sets and n_models within a 32-bit int.  Sets no model uses are allowed.
 * Not provided: device-buffer (_dev) forms of the two calls, bands of components other than total, weighted quantiles. */
typedef struct vag_grid_set {
    size_t t0, n_t;   /* slice of the concatenated times       */
    size_t nu0, n_nu; /* slice of the concatenated frequencies */
} vag_grid_set;

/* PyModel::flux_density_grid (pybind/pymodel.cpp:498-514) of model m on its own set: model m's [VAG_NCOMP][n_nu][n_t]
 * block starts at element VAG_NCOMP * off[m], off[m] = the sum of n_nu * n_t over the sets of models 0 .. m-1 (the
 * layout of vag_flux_density_series_multi); every plane is written.  Launches: those of vag_flux_density_grid on one
 * request, whatever n_sets. */
int vag_flux_density_grid_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                                const vag_grid_set* sets, size_t n_sets, const double* t, size_t n_t_total,
                                const double* nu, size_t n_nu_total, double* out, int32_t* status);

/* Posterior-predictive bands of many fits in one call: the run of vag_flux_density_grid_multi, then for every set d, every
 * q[j] and every (nu, t) column, numpy.quantile(F_total[members of d], q[j], axis=0, method="linear") -- bit for bit (the
 * sign of a zero aside) with numpy's rule on the same flux: h = (n - 1) q, lo = floor(h), hi = min(lo + 1, n - 1),
 * g = h - lo, result a + (b - a) g, or b - (b - a) (1 - g) when g >= 0.5, with a, b the order statistics lo and hi.  The
 * members of d are its models (dataset_of[m] == d) whose status has neither VAG_ST_ODE_FAIL500 (the reference throws)
 * nor VAG_ST_CAPACITY (NaN output); the kernels read that from the run's status on the device.  A column with a NaN among
 * its members gives NaN; a set without members gives NaN and n_used = 0.  The flux never leaves the device: the full
 * ragged output sits in the context's output workspace, 8 * VAG_NCOMP * sum_m n_nu * n_t bytes.
 * out: set d's [n_q][n_nu][n_t] block starts at n_q * the sum of n_nu * n_t over sets 0 .. d-1.  n_used[n_sets]: the
 * members of every set.  status[n_models] may be NULL.  D2H traffic: out, n_used and status only.
 * Checks: those of vag_flux_density_grid_multi, n_q >= 1 and every q[j] finite in [0, 1].
 * Launches: those of vag_flux_density_grid_multi + 2 (the members of every set, a CTA per set; the selection, a CTA per
 * set and 4 consecutive columns, a warp per column, exact MSB radix select over the order-preserving 64-bit image of the
 * fluxes, in shared memory while the set's members fit 160 KB of staged keys, from global memory otherwise). */
int vag_flux_quantiles_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                             const vag_grid_set* sets, size_t n_sets, const double* t, size_t n_t_total, const double* nu,
                             size_t n_nu_total, const double* q, size_t n_q, double* out, int64_t* n_used,
                             int32_t* status);

/* ok[i] = 1 where vag_params_validate accepts params[i], else 0 (no error is raised for rejected sets). */
int vag_params_validate_batch(const vag_params* params, size_t n, int32_t* ok);

/* ------------------------------------------------------------------------------------------- */
/* batched model evaluation, DEVICE buffers (no copies; asynchronous on `stream`)               */
/* ------------------------------------------------------------------------------------------- */
/* Same contracts as above; every pointer is a device pointer on ctx's device; `stream` is a
 * cudaStream_t passed as void* (NULL = the context's own stream).  The calls are stream-ordered;
 * they synchronise the stream once internally (to size the ragged workspace after the grid
 * kernel) and return with the remaining kernels enqueued: call vag_synchronize / sync the stream
 * before reading the outputs.  t must be ascending (not checked on the device path).
 * vag_chi2_dev and vag_flux_band_dev below also plan on the device, which synchronises the stream
 * once more, before the grid kernel. */
int vag_flux_density_grid_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t,
                              size_t n_t, const double* d_nu, size_t n_nu, double* d_out, int32_t* d_status,
                              void* stream);
int vag_flux_density_series_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t,
                                const double* d_nu, size_t n, double* d_out, int32_t* d_status, void* stream);
int vag_chi2_series_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t,
                        const double* d_nu, const double* d_lnF_obs, const double* d_sigma_ln, const double* d_w,
                        size_t n, double* d_chi2, int32_t* d_status, void* stream);
int vag_synchronize(vag_context* ctx);
/* The *_dev entry points cannot see the parameters on the host, so they use the context's grid
 * capacities (theta nodes / phi nodes per model; defaults 384 / 128).  The host-buffer entry
 * points derive tight capacities from the parameters themselves.  A model that needs more nodes
 * than the capacity gets VAG_ST_CAPACITY and NaN output. */
int vag_set_capacity(vag_context* ctx, int cap_theta, int cap_phi);

/* ------------------------------------------------------------------------------------------- */
/* DEVICE buffers, planned on the device: the likelihood of a sampler whose walkers stay in HBM  */
/* ------------------------------------------------------------------------------------------- */
/* Device counterpart of vag_params_validate_batch: d_ok[i] = 1 where vag_params_validate accepts d_params[i], else 0,
 * and caps = {theta, phi} node capacities the accepted records need (the host path's capacities for them).  One kernel;
 * synchronises `stream` to return caps. */
int vag_params_validate_batch_dev(vag_context* ctx, const vag_params* d_params, size_t n, int32_t* d_ok, int caps[2],
                                  void* stream);

/* vag_flux_band and vag_chi2_ext on device buffers, each parameter set checked on the device as vag_params_validate
 * checks it, and the grids sized from the parameters as the host-buffer entry points size them (not by
 * vag_set_capacity).  A rejected set runs as a fixed valid stand-in (an on-axis tophat in ISM) and its results are then
 * overwritten: status VAG_ST_INVALID, flux NaN, chi2 +inf -- the reference raises there, and its samplers map that to
 * logL = -inf (samplers.py:63-70).  The stand-ins are members of the batch: series mode 0 (vag_set_series_mode) sees
 * their lattices too.  Planning is one extra kernel before and one after the call's work, and one D2H of two ints with
 * one more synchronisation of `stream`, before the grid kernel: the capacities size the workspaces on the host.
 * Not checked on the device path: the time order of d_t and of every band's t, and the finiteness of d_ext_k.
 * vag_flux_band_dev: d_out[n_models][VAG_NCOMP][n_t]; the band's frequency nodes and weights are made on the host.
 * vag_chi2_dev: the terms and rules of vag_chi2_ext (ext_k / A_V both NULL or both set, and then n_points > 0; at least
 * one term; status OR over terms only with band terms); `bands` is a host array whose t / lnF_obs / sigma_ln / w are
 * device pointers. */
int vag_flux_band_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t, size_t n_t,
                      double nu_min, double nu_max, size_t num_nu, double* d_out, int32_t* d_status, void* stream);
int vag_chi2_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t, const double* d_nu,
                 const double* d_lnF_obs, const double* d_sigma_ln, const double* d_w, const double* d_ext_k, size_t n_points,
                 const double* d_A_V, const vag_band_obs* bands, size_t n_bands, double* d_chi2, int32_t* d_status,
                 void* stream);

/* vag_chi2_multi_bands on device buffers, planned on the device: several light curves with points and bands in one batch
 * whose records, data and results stay in HBM.  d_params, d_t ... d_ext_k, d_A_V, d_chi2 and d_status (may be NULL) are
 * device pointers; dataset_of, sets and `bands` are host arrays, read only during the call, and the bands' t / lnF_obs /
 * sigma_ln / w are device pointers (vag_chi2_dev's convention).  The output offsets, the point and evaluation lists and
 * the passes of 32768 models are planned on the host, as in vag_chi2_multi_bands.
 * Planning: k_plan checks every record as vag_params_validate does and takes the capacities of the accepted ones; one D2H
 * brings back the two capacities and the ok flags, with one synchronisation of `stream`.  A rejected record is left out
 * of the batch, not run as a stand-in (unlike vag_chi2_dev): the lists hold the accepted models only, and a final k_reject
 * writes chi2 = +inf and status VAG_ST_INVALID for the rejected ones.  For every accepted model, chi2 and status equal
 * those of vag_chi2_multi_bands called on the accepted models alone with host copies of the same arrays, bit for bit, in
 * every series mode: it is the same batch, and the plan's capacities are the host's.  The result does not depend on what
 * the rejected records contain.
 * The accepted models' records, and the point models' A_V, are gathered from d_params / d_A_V on the device (one launch);
 * every band's t / lnF_obs / sigma_ln / w are copied into the concatenated band workspace by one more launch (a CTA per
 * band); the bands' frequency nodes and weights are made on the host.
 * Launches: 2 when no record is accepted (k_plan, k_reject); otherwise L + 2 + (1 when any accepted model has a band),
 * where L = the launches of vag_chi2_multi_bands on the accepted models (L(points) + L(bands) + 2, see there) -- whatever
 * the number of data sets, bands or models.  Synchronisations: those of vag_chi2_multi_bands plus the plan's; the call
 * returns with its work enqueued on `stream`.  n_models == 0: VAG_OK, nothing enqueued.
 * Checks before any work (VAG_ERR_INVALID, messages name the data set, the band or the model; a failed call leaves the
 * context usable): the structural checks of vag_chi2_multi_bands -- set and band ranges, dataset_of in range, n > 0 or
 * n_bands > 0 per set, nu_min / nu_max / num_nu, NULL pointers, the 32-bit limits, ext_k / A_V both set or both NULL and
 * then points.  Not checked on the device path: the time order and finiteness of d_t, d_nu and the band times, and the
 * finiteness of d_ext_k. */
int vag_chi2_multi_bands_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const int32_t* dataset_of,
                             const vag_multi_set* sets, size_t n_sets, const double* d_t, const double* d_nu,
                             const double* d_lnF_obs, const double* d_sigma_ln, const double* d_w, const double* d_ext_k,
                             size_t n_points_total, const double* d_A_V, const vag_band_obs* bands, size_t n_bands_total,
                             double* d_chi2, int32_t* d_status, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* introspection (tests, profiling): stage tables of ONE model, the analogue of                 */
/* PyModel::details (pybind/pymodel.cpp:315-348)                                                */
/* ------------------------------------------------------------------------------------------- */
typedef struct vag_grid_info {
    int32_t n_phi, n_theta, n_t;   /* Coord shape (src/core/mesh.h:55-83)                        */
    int32_t n_reps;                /* coord.theta_reps.size()                                    */
    int32_t symmetry;              /* Symmetry enum value (src/core/mesh.h:49-54)                */
    int32_t phi_mirrored;
    int32_t n_phi_eff;             /* Observer::eff_phi_grid (src/core/observer.cpp:218-222)     */
    int32_t status;
} vag_grid_info;

/* Runs grid + dynamics (+radiation) for one model and the observation window [t_min, t_max] s.
 * Any output pointer may be NULL.  Sizes: theta[n_theta], phi[n_phi], reps[n_reps],
 * t_rows[n_reps][n_t] (engine-frame lattice of each representative row, code units),
 * fwd_shock / rvs_shock [7][n_reps][n_t] in the order t_comv, r, theta, Gamma, Gamma_th, B, N_p
 * (code units, src/dynamics/shock.h:33-39), inj_idx[n_reps] (reverse shock injection_idx).
 * Call once with all NULL to get *info, then allocate. */
int vag_details(vag_context* ctx, const vag_params* p, double t_min, double t_max, vag_grid_info* info,
                double* theta, double* phi, int32_t* reps, double* t_rows, double* fwd_shock, double* rvs_shock,
                int32_t* inj_idx);

/* Photon tables of one model (same front end as vag_details): for each shock [6][n_reps][n_t] in the order
 * log2 nu_m, log2 nu_c, log2 nu_a, log2 nu_M, log2 I_nu_max (code units) and 1/nu_M -- what
 * save_photon_details exports (pybind/pymodel.cpp:263-291).  rvs may be NULL; it is untouched without a
 * reverse shock.  For a shock with ssc=True these are the photons after inverse-Compton cooling. */
int vag_details_photons(vag_context* ctx, const vag_params* p, double t_min, double t_max, double* fwd, double* rvs);

/* Electron and inverse-Compton bookkeeping of the shocks with ssc=True, after KN_cooling / Thomson_cooling
 * (pybind/pymodel.cpp:234-291, 303): for each shock [VAG_IC_DETAIL_PLANES][n_reps][n_t] in the order gamma_m, gamma_c,
 * gamma_a, gamma_M, gamma_m_hat, gamma_c_hat, Y_T.  Planes of a shock without ssc are zero; rvs may be NULL. */
#define VAG_IC_DETAIL_PLANES 7
int vag_details_ic(vag_context* ctx, const vag_params* p, double t_min, double t_max, double* fwd, double* rvs);

/* Output transfer policy of the HOST-buffer flux entry points.
 * VAG_OUT_DENSE (default): every one of the VAG_NCOMP planes of `out` is written (absent components 0).
 * VAG_OUT_PRESENT: planes of components that NO model of the batch has (reverse shock: has_rvs;
 * SSC: fwd.ssc / rvs.ssc) are neither transferred nor written -- the caller's buffer is left
 * untouched there.  This mirrors the reference's FluxDict, whose absent components are empty
 * arrays that are never materialised (pybind/pymodel.h:361-383), and saves 3/5 of the device-to-host
 * traffic of a forward-shock synchrotron batch.  VAG_C_TOTAL and VAG_C_FWD_SYNC are always present. */
enum { VAG_OUT_DENSE = 0, VAG_OUT_PRESENT = 1, VAG_OUT_PRESENT_ALIAS_TOTAL = 2 };
int vag_set_output_mode(vag_context* ctx, int mode);
/* VAG_OUT_PRESENT_ALIAS_TOTAL: as VAG_OUT_PRESENT, and when exactly ONE emission component exists in the whole batch
 * (e.g. forward-shock synchrotron only) the `total` plane -- which is then that component bit for bit -- is not
 * transferred either: vag_last_total_alias() returns the component index (VAG_C_*) whose plane holds the total of the
 * most recent host-buffer call, or -1 when `total` was written.  (The pybind mirror hands the same array out twice.) */
int vag_last_total_alias(vag_context* ctx);

/* Series requests (vag_flux_density_series, vag_chi2*) whose points share at most 8 distinct frequencies -- multi-band
 * light curves -- are evaluated "banded": the boundary luminosities of every lattice node are staged once per band and
 * a point interpolates its band's column, instead of every point evaluating both bracketing spectra itself (the
 * evaluation points are those of Observer::specific_flux_series, src/core/observer.h:494-520; results agree to
 * rounding).  mode 0 (default): chosen per request by cost; 1: never; 2: whenever the request has <= 8 frequencies. */
int vag_set_series_mode(vag_context* ctx, int mode);

/* Lanes that cooperate on one model's grid (K0): 0 (default) chooses by batch size -- the widest group whose launch
 * still fits into one wave on the device; 4, 8, 16 or 32 forces that width for every batch.  The grid
 * is the same bit for bit at every width; forcing one is for tests and A/B timing. */
int vag_set_grid_lanes(vag_context* ctx, int lanes);

/* per-stage device time of the most recent batched call on this context, milliseconds:
 * [0]=grid (K0) [1]=dynamics (K1) [2]=radiation (K2) [3]=EATS flux (K3) [4]=likelihood (K4)
 * Only filled when vag_set_profiling(ctx, 1) was called (adds event records + one sync). */
int vag_set_profiling(vag_context* ctx, int enable);
int vag_last_stage_ms(vag_context* ctx, float ms[8]);
/* Work counters of the most recent profiled pass (the denominators of bench.py's roofline entries): [0] forward-only ODE
 * rows, [1] forward+reverse ODE rows, [2] shock-table cells x shocks, [3] EATS cells (shocks x n_phi_eff x n_theta x n_t),
 * [4] EATS rows, [5] theta-quadrature attempts, [6] phi-quadrature attempts x n_theta, [7] sum of n_theta. */
int vag_last_work(vag_context* ctx, double work[8]);
/* number of kernel launches issued by the most recent batched call */
int vag_last_launch_count(vag_context* ctx);
/* dependent-free DFMA throughput of the device in TFLOP/s (FP64 roofline denominator) */
int vag_measure_fp64_peak(vag_context* ctx, double* tflops);
/* Test hook: lower the shock ODE's accepted-step limit (defaults::solver::max_ode_steps = 100000 -> VAG_ST_ODE_STEP_CAP,
 * forward-shock.tpp:196-200) and / or the consecutive-rejection limit (Boost's 500 -> VAG_ST_ODE_FAIL500) so that the failure
 * semantics can be exercised; 0 restores the reference value. */
int vag_debug_set_ode_limits(vag_context* ctx, int max_steps, int max_fails);
/* Device self-test of the libm-exact functions the grid kernel evaluates (csrc/vag_libm.cuh):
 * out[i] = fn(x[i]) with fn 0 exp, 1 exp2, 2 log, 3 log2, 4 log10, 5 pow(x[i], y[i]), 6 sin, 7 cos; host buffers.
 * The results must equal the host libm's bit for bit (the reference's theta / phi grids depend on it,
 * src/core/grid-refinement.h:137-189); y is NULL except for pow. */
int vag_selftest_libm(vag_context* ctx, int fn, const double* x, const double* y, double* out, size_t n);

#ifdef __cplusplus
}
#endif
#endif /* VAG_H_ */
