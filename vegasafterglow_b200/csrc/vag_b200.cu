// vag_b200.cu -- sm_100a kernels and the C ABI (include/vag.h) of the B200-native
// VegasAfterglow model-evaluation path.  Kernel bodies live in vag_pipeline.cuh / vag_observer.cuh.
//
// Launch geometry (B200: 148 SMs, FP64 path, no tensor cores -- nothing here is a contraction):
//   k_grid<G>        : G = 4 / 8 / 16 / 32 lanes per model (32 / G models share a warp's scalar instruction stream)
//   k_dynamics<PAIR> : one thread per unique ODE row, 8 rows per warp for small batches; forward-only rows on a
//                      register-resident dopri5, pair rows with the stage vectors in shared memory
//   k_radiation      : one 64-thread CTA per unique row: finishes the shock tables from the raw node states,
//                      EATS node geometry, photon coefficients (SoA planes, stores coalesced along k)
//   k_eats<MODE,KIND>: one 128-thread CTA per (model, row-split, shock), 8 CTAs / SM; staged rows, the
//                      log2_softplus table and the accumulators in dynamic shared memory
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/vag.h"
#include "vag_libm.cuh"
#include "vag_pipeline.cuh"
#include "vag_quantile.cuh"
#include "vag_exposure.cuh"

using namespace vag;

static_assert(sizeof(vag_params) == 320, "vag_params layout must match vegasafterglow_b200/abi.py");

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
// A ragged series request (vag_flux_density_series_multi, vag_chi2_multi) gives every model its own data set: a slice
// of the concatenated points, sorted by time within the slice.  Its distinct frequencies (banded runs) sit at
// [set * EATS_NU_TILE] of the band tables.  Model m's output is [VAG_NCOMP][n of its set] at point offset
// out_off[m] - out_off[0] of the pass's output.  A ragged grid request (the band pass of vag_flux_band_multi and
// vag_chi2_multi_bands) gives every model a slice of the concatenated times and one of the concatenated frequency nodes;
// its output is [VAG_NCOMP][n_nu][n] at out_off[m] - out_off[0], out_off counting (time x node) points.  The kernels that
// take `bool RAGGED` run either request: their ragged instantiation rebases the request on the model's data set, so
// every model's arithmetic is that of the shared-request kernel on its own data set.  The table (SetsDev sd) is their
// last parameter: placed earlier, it would move the parameter offsets of the shared instantiations and change their code.
struct SeriesSet {
    int off, n;  // slice of the concatenated points (grid request: of the concatenated times)
    int n_nu;    // series: distinct frequencies of the slice (k_series_bands_sets); grid: frequency nodes of the slice
    int nu_off;  // grid: first node of the slice in the concatenated nodes; the points of an exposure-averaged series
                 // request (k_expo_average): the slice's first point in the sample plan
};
struct SetsDev {
    const int* set_of;         // [models of the pass] data set of each model
    SeriesSet* sets;           // [n_sets]
    const long long* out_off;  // [models of the pass + 1] first output point of each model (prefix sums over the batch)
};
// points of model mi's ragged output block, per component
__device__ __forceinline__ size_t ragged_comp_size(const SetsDev& sd, int mi) {
    return (size_t)(sd.out_off[mi + 1] - sd.out_off[mi]);
}

// K0: G lanes per model (vag_grid.cuh GroupPar), 32 / G models per warp, 4 warps per CTA.  Narrow groups
// share the scalar instruction stream between more models (throughput, large batches); wide groups
// finish one model sooner (latency, small batches).  The observation window is the request's, or (RAGGED) the
// model's data set's.
#ifndef GRID_MIN_BLOCKS
#define GRID_MIN_BLOCKS 4
#endif
template <int G, bool RAGGED>
__global__ void __launch_bounds__(128, GRID_MIN_BLOCKS) k_grid(BatchWs w, const double* __restrict__ t_obs, int n_t_obs,
                                                               SetsDev sd) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int mi = gt / G;
    if (mi >= w.n_models) return;  // whole groups exit together
    const int lane = threadIdx.x & 31;
    const int shift = lane & ~(G - 1);
    const GroupPar<G> par{lane & (G - 1), (G == 32 ? 0xffffffffu : ((1u << (G & 31)) - 1u)) << shift, shift};
    if constexpr (RAGGED) {
        const SeriesSet s = sd.sets[sd.set_of[mi]];
        k0_grid_body(par, w, mi, t_obs[s.off], t_obs[s.off + s.n - 1]);
    } else {
        k0_grid_body(par, w, mi, t_obs[0], t_obs[n_t_obs - 1]);
    }
}

// K0b: exclusive scan of the ragged row / cell counts over the models of the batch + totals.
// One CTA of 1024 threads; thread i owns a contiguous slice of models (k0b_scan_body is the
// sequential statement of the same result).
__global__ void __launch_bounds__(1024) k_scan(BatchWs w) {
    __shared__ int s_rows[1024];
    __shared__ long long s_cells[1024];
    __shared__ int s_max[3][32];
    __shared__ int s_or[32];
    const int tid = threadIdx.x, n = w.n_models;
    const int per = (n + 1023) / 1024;
    const int m0 = min(tid * per, n), m1 = min(m0 + per, n);
    int rows = 0, max_nt = 0, max_nth = 0, max_er = 0, st = 0;
    long long cells = 0;
    for (int mi = m0; mi < m1; ++mi) {
        const GridHeader& h = w.hdr[mi];
        const ModelCfg& cfg = w.cfg[mi];
        if (cfg.fwd.ssc || (cfg.has_rvs && cfg.rvs.ssc)) st |= (1 << 30);  // carries "any ssc" through the OR
        st |= cfg.has_rvs ? (1 << 29) : (1 << 28);                         // "any pair rows" / "any forward-only rows"
        if (cfg.spreading) st |= (1 << 27);                                // "any spreading model"
        rows += h.n_reps;
        cells += (long long)h.n_reps * h.n_t;
        max_nt = max(max_nt, h.n_t);
        max_nth = max(max_nth, h.n_theta);
        max_er = max(max_er, h.n_theta * h.n_phi_eff);
        st |= h.status;
    }
    s_rows[tid] = rows;
    s_cells[tid] = cells;
    __syncthreads();
    // Hillis-Steele inclusive scan over the 1024 slice totals
    for (int off = 1; off < 1024; off <<= 1) {
        int r = 0;
        long long c = 0;
        if (tid >= off) {
            r = s_rows[tid - off];
            c = s_cells[tid - off];
        }
        __syncthreads();
        s_rows[tid] += r;
        s_cells[tid] += c;
        __syncthreads();
    }
    int row0 = s_rows[tid] - rows;
    long long cell0 = s_cells[tid] - cells;
    for (int mi = m0; mi < m1; ++mi) {
        const GridHeader& h = w.hdr[mi];
        w.row_off[mi] = row0;
        w.cell_off[mi] = cell0;
        row0 += h.n_reps;
        cell0 += (long long)h.n_reps * h.n_t;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        max_nt = max(max_nt, __shfl_xor_sync(0xffffffffu, max_nt, o));
        max_nth = max(max_nth, __shfl_xor_sync(0xffffffffu, max_nth, o));
        max_er = max(max_er, __shfl_xor_sync(0xffffffffu, max_er, o));
        st |= __shfl_xor_sync(0xffffffffu, st, o);
    }
    if ((tid & 31) == 0) {
        s_max[0][tid >> 5] = max_nt;
        s_max[1][tid >> 5] = max_nth;
        s_max[2][tid >> 5] = max_er;
        s_or[tid >> 5] = st;
    }
    __syncthreads();
    if (tid == 0) {
        for (int i = 1; i < 32; ++i) {
            max_nt = max(max_nt, s_max[0][i]);
            max_nth = max(max_nth, s_max[1][i]);
            max_er = max(max_er, s_max[2][i]);
            st |= s_or[i];
        }
        w.row_off[n] = s_rows[1023];
        w.cell_off[n] = s_cells[1023];
        w.totals[TOT_ROWS] = s_rows[1023];
        w.totals[TOT_MAX_NT] = max_nt;
        w.totals[TOT_MAX_NTHETA] = max_nth;
        w.totals[TOT_MAX_EROWS] = max_er;
        w.totals[TOT_STATUS_OR] = st & ~(15 << 27);
        w.totals[TOT_ANY_SPREAD] = (st >> 27) & 1;
        w.totals[TOT_ANY_SSC] = (st >> 30) & 1;
        w.totals[TOT_ANY_PAIR] = (st >> 29) & 1;
        w.totals[TOT_ANY_FWD_ONLY] = (st >> 28) & 1;
    }
}

__global__ void k_rowmap(BatchWs w) {
    const int mi = blockIdx.x * blockDim.x + threadIdx.x;
    if (mi >= w.n_models) return;
    k0c_rowmap_body(w, mi);
}

// K1: one thread per unique row, `lanes` rows per 32-thread CTA.  The ODE is a dependent-latency chain
// and rows of one warp diverge (different accept/reject histories, branches of the RHS), so a small
// batch is spread thinly -- few rows per warp, about two warps per scheduler -- and only large batches
// fill whole warps.  The dopri5 stage vectors sit in shared memory, [slot][component][lane]
// (conflict-free: a lane only ever touches its own column).
// PAIR selects the rows a launch integrates (forward+reverse pairs with the shared-memory stepper, or
// forward-only rows with the register-resident one, which needs no shared memory).
// K1a: one warp per unique ODE row builds its time lattice (n_t independent pow(10, .) evaluations)
__global__ void __launch_bounds__(128) k_lattice(BatchWs w, int n_rows) {
    const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (row < n_rows) k1_lattice_body(w, row, threadIdx.x & 31, 32);
}

template <bool PAIR>
__global__ void __launch_bounds__(32) k_dynamics(BatchWs w, int n_rows, int lanes) {
    __shared__ double s_col[PAIR ? K1_COL_DOUBLES * 32 : 1];
    if ((int)threadIdx.x >= lanes) return;
    const int row = blockIdx.x * lanes + threadIdx.x;
    if (row >= n_rows) return;
    if ((w.cfg[w.row_model[row]].has_rvs != 0) != PAIR) return;
    k1_dynamics_body<PAIR>(w, row, s_col + threadIdx.x, 32);
}

// K1b + K2: one CTA per unique row.  Finishes the row's shock tables from the raw node states the ODE
// kernel left (thread <-> node), applies the early-time reverse-shock extrapolation, derives the EATS
// node geometry and then builds the photon coefficients of both shocks (thread <-> node, SoA plane
// stores coalesced along k).
__global__ void __launch_bounds__(64) k_radiation(BatchWs w) {
    __shared__ int s_cut;
    const int row = blockIdx.x;
    const RowCtx c = row_ctx(w, row);
    const int tid = threadIdx.x, nthr = blockDim.x;
    if (tid == 0) s_cut = c.n_t;
    for (int k = tid; k < c.n_t; k += nthr) k1b_finish_cell(w, row, c, k);
    __syncthreads();
    if (c.has_rvs && w.row_dyn[row].n_saved >= 0) {
        const int mine = extrap_scan(shock_row(w.rvs, c.off), c.n_t, tid, nthr);
        if (mine < c.n_t) atomicMin(&s_cut, mine);
        __syncthreads();
        const int idx_cut = s_cut;
        for (int k = tid; k < c.n_t; k += nthr) k1c_extrap_cell(w, row, c, idx_cut, k);
        __syncthreads();
    }
    const ModelCfg& cfg = w.cfg[c.mi];
    for (int k = tid; k < c.n_t; k += nthr) {
        k1d_geo_cell(w, c, k);
        if (cfg.spreading && w.sh_theta) k1e_spread_geo_cell(w, row, c, k);
        if (!cfg.fwd.ssc) k2_radiation_cell(w, row, k, 0);  // ssc shocks: k_ic_cooling
        if (cfg.has_rvs && !cfg.rvs.ssc) k2_radiation_cell(w, row, k, 1);
    }
}

// K2 for shocks with ssc=True: one thread per (row, shock), sequential in k (IC cooling of cell k
// starts from gamma_c of cell k-1)
__global__ void __launch_bounds__(32) k_ic_cooling(BatchWs w, int n_rows) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    const int which = blockIdx.y;
    if (row >= n_rows) return;
    const int mi = w.row_model[row];
    if (which && !w.cfg[mi].has_rvs) return;
    if (!(which ? w.cfg[mi].rvs : w.cfg[mi].fwd).ssc) return;
    k2_ic_cool_row(w, row, which);
}

__global__ void k_kn_lut(KnLut* lut) {
    const int i = threadIdx.x;
    if (i < KN_LUT_N) kn_lut_entry(i, lut->ratio[i], lut->lg2_ratio[i]);
}

// log2 of the smallest / largest observation frequency (code units, without the 1+z shift)
__global__ void k_nu_range(const double* __restrict__ lg2_nu, int n, double* out) {
    __shared__ double s_lo[256], s_hi[256];
    double lo = kInf, hi = -kInf;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        lo = fmin(lo, lg2_nu[i]);
        hi = fmax(hi, lg2_nu[i]);
    }
    s_lo[threadIdx.x] = lo;
    s_hi[threadIdx.x] = hi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            s_lo[threadIdx.x] = fmin(s_lo[threadIdx.x], s_lo[threadIdx.x + o]);
            s_hi[threadIdx.x] = fmax(s_hi[threadIdx.x], s_hi[threadIdx.x + o]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = s_lo[0];
        out[1] = s_hi[0];
    }
}

// EATS row constants of every (model, (phi,theta) row): cos to the line of sight, time coefficient,
// log2 solid angle, representative shock row
__global__ void k_rowgeom(BatchWs w) {
    const int mi = blockIdx.y;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (w.status[mi] & VAG_ST_CAPACITY) return;
    if (q >= w.hdr[mi].n_theta * w.hdr[mi].n_phi_eff) return;
    k_rowgeom_body(w, mi, q);
}

__global__ void k_rowcos(BatchWs w) {
    const int mi = blockIdx.y;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const ModelCfg& cfg = w.cfg[mi];
    if (!(cfg.fwd.ssc || (cfg.has_rvs && cfg.rvs.ssc))) return;
    if (q >= w.hdr[mi].n_theta * w.hdr[mi].n_phi_eff) return;
    k_rowcos_body(w, mi, q);
}
__global__ void k_dop_extrema(BatchWs w) {
    const int mi = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const ModelCfg& cfg = w.cfg[mi];
    if (!(cfg.fwd.ssc || (cfg.has_rvs && cfg.rvs.ssc))) return;
    if (k >= w.hdr[mi].n_t) return;
    k_dop_extrema_body(w, mi, k);
}

// K2b: SSC spectrum tables, one warp per unique cell (both shocks); warps stride over the batch's cells.
// RAGGED: each model's tables are sized by its own data set's band, w.nu_range[2 m .. 2 m + 1] (k_nu_range_sets).  The
// table comes in w rather than as a parameter of its own: an added parameter changes the code of k_ic_spectrum<false>.
template <bool RAGGED>
__global__ void __launch_bounds__(128) k_ic_spectrum(BatchWs w, int n_rows, int n_warps) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const WarpPar par{(int)(threadIdx.x & 31)};
    double* scratch = w.ic_scratch + (size_t)warp * IC_SCRATCH_DOUBLES;
    BatchWs wm = w;  // RAGGED: w with the band of the cell's model
    for (long long g = warp; g < w.n_cells; g += n_warps) {
        // row of global cell g: last row whose first cell is <= g
        int lo = 0, hi = n_rows;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (w.row_cell_off[mid] <= g)
                lo = mid;
            else
                hi = mid;
        }
        const int row = lo;
        const int k = (int)(g - w.row_cell_off[row]);
        const int mi = w.row_model[row];
        const ModelCfg& cfg = w.cfg[mi];
        if constexpr (RAGGED) wm.nu_range = w.nu_range + 2 * (size_t)mi;
        for (int which = 0; which < 2; ++which) {
            if (which && !cfg.has_rvs) continue;
            if (!(which ? cfg.rvs : cfg.fwd).ssc) continue;
            const int st = k2b_ic_spectrum_cell(par, RAGGED ? wm : w, row, k, which, scratch);
            if (st && par.lane == 0) atomicOr(&w.status[mi], st);
        }
    }
}

// observation request pre-pass: log2 of the (unit-scaled) times and frequencies
__global__ void k_prep_obs(const double* __restrict__ t, int n_t, const double* __restrict__ nu, int n_nu,
                           double* lg2_t, double* t_lin, double* lg2_nu, double* nu_lin, double* nu23,
                           int nu_in_code_units) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_t) {
        const double tl = t[i] * unit::sec;
        t_lin[i] = tl;
        lg2_t[i] = log2(tl);
    }
    if (i < n_nu) {
        const double v = nu_in_code_units ? nu[i] : nu[i] * unit::Hz;
        const double l = log2(v);
        lg2_nu[i] = l;
        nu_lin[i] = v;
        nu23[i] = exp2((2. / 3) * l);
    }
}

// Distinct frequencies of a series request (one CTA).  out_n = their number, or EATS_NU_TILE + 1 when there are more
// (or a NaN); band_of[i] = index of point i's frequency in the list; the list is kept as log2 / linear / ^(2/3).
// The list grows in order of first appearance: each round appends the unmatched point of lowest index.
__device__ __forceinline__ void series_bands_cta(const double* __restrict__ lg2_nu, const double* __restrict__ nu_lin,
                                                 const double* __restrict__ nu23, int n, int* band_of, double* b_lg2,
                                                 double* b_lin, double* b_23, int* out_n) {
    __shared__ double s_u[EATS_NU_TILE + 1];
    __shared__ int s_cnt, s_cand;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const double v = i < n ? lg2_nu[i] : 0.0;
        int mine = -1;
        for (;;) {
            const int cnt = s_cnt;
            if (mine < 0)
                for (int q = 0; q < cnt; ++q)
                    if (s_u[q] == v) mine = q;
            __syncthreads();
            if (threadIdx.x == 0) s_cand = 0x7fffffff;
            __syncthreads();
            if (i < n && mine < 0) atomicMin(&s_cand, i);
            __syncthreads();
            const int cand = s_cand;
            if (cand == 0x7fffffff) break;
            if (cnt >= EATS_NU_TILE) {  // a ninth value (or a NaN, which matches nothing): not a banded request
                if (threadIdx.x == 0) *out_n = EATS_NU_TILE + 1;
                return;
            }
            if (threadIdx.x == 0) {
                s_u[cnt] = lg2_nu[cand];
                b_lg2[cnt] = lg2_nu[cand];
                b_lin[cnt] = nu_lin[cand];
                b_23[cnt] = nu23[cand];
                s_cnt = cnt + 1;
            }
            __syncthreads();
        }
        if (i < n) band_of[i] = mine;
        __syncthreads();
    }
    if (threadIdx.x == 0) *out_n = s_cnt;
}
__global__ void __launch_bounds__(1024) k_series_bands(const double* __restrict__ lg2_nu, const double* __restrict__ nu_lin,
                                                        const double* __restrict__ nu23, int n, int* band_of, double* b_lg2,
                                                        double* b_lin, double* b_23, int* out_n) {
    series_bands_cta(lg2_nu, nu_lin, nu23, n, band_of, b_lg2, b_lin, b_23, out_n);
}

// Observer::flux (src/core/observer.h:555-567): band[m][c][j] = sum_i F[m][c][i][j] * w[i]
__global__ void k_band_reduce(const double* __restrict__ F, const double* __restrict__ wgt, double* __restrict__ out,
                              size_t n_mc, int n_nu, int n_t) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_mc * n_t) return;
    const size_t mc = e / n_t;
    const int j = (int)(e - mc * n_t);
    const double* f = F + mc * (size_t)n_nu * n_t + j;
    double s = 0;
    for (int i = 0; i < n_nu; ++i) s += f[(size_t)i * n_t] * wgt[i];
    out[e] = s;
}

// K3.  grid = (model, split, shock).  out[model][comp][n_nu][n_t] (grid) or [model][comp][n] (series)
// MODE 0: synchrotron of shocks without ssc; MODE 1: synchrotron of shocks with ssc (IC-corrected
// spectrum); MODE 2: SSC component (per-cell tables).  blockIdx.z = shock (0 forward, 1 reverse).
#ifndef EATS_MIN_BLOCKS
#define EATS_MIN_BLOCKS 8
#endif
// KIND: the request kind, compiled separately (see eats_phase1)
enum { EATS_GRID = 0, EATS_POINT = 1, EATS_BANDED = 2 };
// MODE 1 (synchrotron with the inverse-Compton correction) carries the IC record of the cell next to the tile state: at
// 64 registers it spilled 120 M local loads per config-4 batch; 5 CTAs / SM (90 registers) hold it without spills.
// RAGGED: the CTA's request is rebased on its model's data set and the model's [VAG_NCOMP][n] (series) or
// [VAG_NCOMP][n_nu][n] (grid) block is written at its output offset.  A grid CTA tiles its own n_nu with the batch's
// nu_tile: a tile is min(nu_tile, n_nu - l0) wide, and as nu_tile = min(EATS_NU_TILE, widest n_nu) >= min(EATS_NU_TILE,
// own n_nu), the tiles are those of the model's own call; nu_tile itself only sets strides (staged tile, accumulators).
template <int MODE, int KIND, bool RAGGED>
__global__ void __launch_bounds__(128, MODE == 1 ? 5 : EATS_MIN_BLOCKS) k_eats(BatchWs w, EatsRequest rq0, double* __restrict__ out, int n_split,
                                                 int row_chunk, int max_n_t, int nu_tile, size_t split_stride, SetsDev sd) {
    extern __shared__ __align__(16) double smem[];
    const int mi = blockIdx.x;
    const int split = blockIdx.y;
    const int which = (int)blockIdx.z + (MODE == 2 ? 2 : 0);  // 0 fwd sync, 1 rvs sync, 2 fwd ssc, 3 rvs ssc
    {
        const ModelCfg& cfg = w.cfg[mi];
        if ((which & 1) && !cfg.has_rvs) return;
        const bool ssc = ((which & 1) ? cfg.rvs : cfg.fwd).ssc != 0;
        if ((MODE == 0) == ssc) return;  // MODE 0 handles the shocks without ssc, MODE 1/2 those with
    }
    if (w.status[mi] & VAG_ST_CAPACITY) return;
    EatsModel M = make_eats_model(w, mi, which);
    M.breach = &w.status[mi];
    {
        // log2_softplus table -> head of the dynamic shared memory (16-byte aligned rows)
        for (int a = threadIdx.x; a < SPL_DOUBLES; a += blockDim.x) smem[a] = w.sp_lut[a];
        M.sp_lut = smem;
    }
    const int n_t = M.h->n_t;
    const int erows = M.h->n_theta * M.h->n_phi_eff;
    constexpr bool series = KIND != EATS_GRID;
    constexpr bool banded = KIND == EATS_BANDED;  // series points read a (node, band) tile staged as in grid mode
    double* acc = smem + SPL_DOUBLES;     // [acc_cols][acc_stride]
    const int acc_stride = rq0.acc_stride;
    const int acc_cols = series ? 1 : nu_tile;
    EatsShared sh = eats_carve(acc + acc_cols * acc_stride, max_n_t, series && !banded, row_chunk, nu_tile);
    EatsRequest rq = rq0;
    if constexpr (RAGGED && series) {
        const int set = sd.set_of[mi];
        const SeriesSet ds = sd.sets[set];
        rq.n_t_obs = rq.n_nu = ds.n;
        rq.lg2_t_obs += ds.off;
        rq.t_obs_lin += ds.off;
        const size_t nu_off = banded ? (size_t)set * EATS_NU_TILE : (size_t)ds.off;  // band table / points
        rq.lg2_nu_obs += nu_off;
        rq.nu_obs_lin += nu_off;
        rq.nu23_obs += nu_off;
        rq.n_bands = banded ? ds.n_nu : 0;
        rq.band_of += ds.off;
    } else if constexpr (RAGGED) {  // grid: the set's times x its frequency nodes, tiled by nu_tile as a call of its own
        const SeriesSet ds = sd.sets[sd.set_of[mi]];
        rq.n_t_obs = ds.n;
        rq.n_nu = ds.n_nu;
        rq.lg2_t_obs += ds.off;
        rq.t_obs_lin += ds.off;
        rq.lg2_nu_obs += ds.nu_off;
        rq.nu_obs_lin += ds.nu_off;
        rq.nu23_obs += ds.nu_off;
    }
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int comp = which == 0 ? VAG_C_FWD_SYNC : which == 1 ? VAG_C_RVS_SYNC : which == 2 ? VAG_C_FWD_SSC : VAG_C_RVS_SSC;
    const size_t comp_sz = series ? (size_t)rq.n_t_obs : (size_t)rq.n_nu * rq.n_t_obs;
    // row-split batches (n_split > 1, small batches): each split owns a slab of `out` (= the partial buffer) and
    // k_sum_splits adds the slabs in split order -- deterministic, unlike an atomicAdd into one cell
    double* dst =
        RAGGED ? out + (size_t)split * split_stride + (size_t)(sd.out_off[mi] - sd.out_off[0]) * VAG_NCOMP + comp * comp_sz
               : out + (size_t)split * split_stride + ((size_t)mi * VAG_NCOMP + comp) * comp_sz;
    const int n_nu_tiles = series ? 1 : (rq.n_nu + nu_tile - 1) / nu_tile;
    const RowGeom* rowg = w.rowgeom + (size_t)mi * w.max_erows;
    // rows per pass: this model's lattice may be shorter than the batch maximum the buffers are sized for
    const int rpp = eats_rows_per_pass(n_t, row_chunk, nthr);
    for (int tile = 0; tile < n_nu_tiles; ++tile) {
        const int l0 = tile * nu_tile;
        const int nl = series ? (banded ? rq.n_bands : 1) : imin(nu_tile, rq.n_nu - l0);
        for (int i0 = 0; i0 < rq.n_t_obs; i0 += EATS_T_BLOCK) {
            rq.i0 = i0;
            rq.ni = imin(EATS_T_BLOCK, rq.n_t_obs - i0);
            // zeroed by the thread that accumulates into and finally reads the column (ii == tid mod nthr): no barrier is
            // needed even when this split has no pass to run (compute-sanitizer racecheck, profiles/r02_sanitize.txt)
            for (int ii = tid; ii < rq.ni; ii += nthr)
                for (int l = 0; l < acc_cols; ++l) acc[l * acc_stride + ii] = 0.0;
            for (int q0 = split * rpp; q0 < erows; q0 += n_split * rpp) {
                const int nrows = imin(rpp, erows - q0);
                sh.rowg = rowg + q0;
                __syncthreads();  // previous pass finished reading the staged rows (and the table is loaded)
                eats_phase1<MODE, KIND == EATS_POINT>(M, rq, sh, nrows, l0, nl, tid, nthr);
                __syncthreads();
                if (banded)
                    eats_phase2_banded(M, rq, sh, nrows, acc, tid, nthr);
                else if (series)
                    eats_phase2_series<MODE>(M, rq, sh, nrows, acc, tid, nthr);
                else
                    eats_phase2_grid(M, rq, sh, nrows, nl, acc, tid, nthr);
            }
            // accumulator columns are thread-owned (ii == tid mod nthr): no barrier needed here
            for (int ii = tid; ii < rq.ni; ii += nthr) {
                for (int l = 0; l < (series ? 1 : nl); ++l) {
                    const double v = flux_scale(M, acc[l * acc_stride + ii]);
                    double* p = series ? (dst + i0 + ii) : (dst + (size_t)(l0 + l) * rq.n_t_obs + i0 + ii);
                    *p = v;
                }
            }
            __syncthreads();
        }
    }
}

// out[e] = sum over the row splits, in split order
__global__ void k_sum_splits(double* __restrict__ out, const double* __restrict__ part, int n_split, size_t elems) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= elems) return;
    double s = 0;
    for (int q = 0; q < n_split; ++q) s += part[(size_t)q * elems + e];
    out[e] = s;
}

// total = sum of the present components (PyFlux::calc_total, pybind/pymodel.cpp:350-364)
__global__ void k_total(double* out, size_t n_models, size_t comp_sz) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_models * comp_sz) return;
    const size_t mi = i / comp_sz, e = i - mi * comp_sz;
    double* o = out + mi * VAG_NCOMP * comp_sz;
    o[e] = o[VAG_C_FWD_SYNC * comp_sz + e] + o[VAG_C_FWD_SSC * comp_sz + e] + o[VAG_C_RVS_SYNC * comp_sz + e] +
           o[VAG_C_RVS_SSC * comp_sz + e];
}

// K4: one warp per model; chi2 over the series total (fitter.py:497-501)
// A model whose ODE exhausted Boost's 500 consecutive step rejections is an exception in the reference
// (max_step_checker.hpp:99-106) that the samplers turn into logL = -inf (samplers.py:63-70): chi2 = +inf here.
// accumulate: add to chi2[] (band terms after the point term, fitter.py:525-531).
// ext (per point) with av (per model): host extinction F e^{-A_V k} shifts the observed value to lnF + A_V k.  The
// explicit intrinsics round the product, then the sum, as numpy does; a contracted FMA would differ in the last bit.
// (the warp of model `warp`: F its total plane, the data its point slice)
__device__ __forceinline__ void chi2_warp(int warp, int lane, const double* __restrict__ F, int n, const double* __restrict__ lnF,
                                          const double* __restrict__ sigma_ln, const double* __restrict__ wgt,
                                          const double* __restrict__ av, const double* __restrict__ ext, double* chi2,
                                          const int* __restrict__ status, int accumulate) {
    double s = 0;
    if (ext) {
        const double a = av[warp];
        for (int i = lane; i < n; i += 32)
            s += chi2_term(__dadd_rn(lnF[i], __dmul_rn(a, ext[i])), F[i], sigma_ln[i], wgt[i]);
    } else {
        for (int i = lane; i < n; i += 32) s += chi2_term(lnF[i], F[i], sigma_ln[i], wgt[i]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
        if (accumulate) s += chi2[warp];
        const bool fatal = status && (status[warp] & VAG_ST_ODE_FAIL500);
        chi2[warp] = (isfinite(s) && !fatal) ? s : kInf;
    }
}
// RAGGED: the warp of model m reads its total plane and its data set's slice of the data (ext: of ext_k)
template <bool RAGGED>
__global__ void k_chi2(const double* __restrict__ flux, size_t n_models, int n, const double* __restrict__ lnF,
                       const double* __restrict__ sigma_ln, const double* __restrict__ wgt,
                       const double* __restrict__ av, const double* __restrict__ ext, double* chi2,
                       const int* __restrict__ status, int accumulate, SetsDev sd) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= (int)n_models) return;
    if constexpr (RAGGED) {
        const SeriesSet s = sd.sets[sd.set_of[warp]];
        const double* F = flux + (size_t)(sd.out_off[warp] - sd.out_off[0]) * VAG_NCOMP;  // total
        chi2_warp(warp, lane, F, s.n, lnF + s.off, sigma_ln + s.off, wgt + s.off, av, ext ? ext + s.off : nullptr, chi2,
                  status, accumulate);
    } else {
        const double* F = flux + (size_t)warp * VAG_NCOMP * n;  // total
        chi2_warp(warp, lane, F, n, lnF, sigma_ln, wgt, av, ext, chi2, status, accumulate);
    }
}

// vag_details_ic: [VAG_IC_DETAIL_PLANES][n_cells] <- IcCell records
__global__ void k_ic_export(const IcCell* __restrict__ ic, size_t n_cells, double* __restrict__ out) {
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells) return;
    const IcCell& e = ic[c];
    const double v[VAG_IC_DETAIL_PLANES] = {e.gamma_m, e.gamma_c, e.gamma_a, e.gamma_M, e.ys.gamma_m_hat, e.ys.gamma_c_hat, e.ys.Y_T};
#pragma unroll
    for (int a = 0; a < VAG_IC_DETAIL_PLANES; ++a) out[(size_t)a * n_cells + c] = v[a];
}

// Work counters of a batch (profiling only): [0] forward-only ODE rows, [1] pair ODE rows, [2] shock-table cells x shocks,
// [3] EATS cells = sum_models shocks n_phi_eff n_theta n_t, [4] EATS rows = sum shocks n_phi_eff n_theta,
// [5] theta-quadrature attempts, [6] phi-quadrature attempts x n_theta, [7] sum n_theta
__global__ void k_work(BatchWs w, double* out) {
    const int mi = blockIdx.x * blockDim.x + threadIdx.x;
    if (mi >= w.n_models) return;
    const GridHeader& h = w.hdr[mi];
    const ModelCfg& c = w.cfg[mi];
    const double S = c.has_rvs ? 2.0 : 1.0;
    atomicAdd(out + (c.has_rvs ? 1 : 0), (double)h.n_reps);
    atomicAdd(out + 2, S * h.n_reps * (double)h.n_t);
    atomicAdd(out + 3, S * h.n_phi_eff * (double)h.n_theta * h.n_t);
    atomicAdd(out + 4, S * h.n_phi_eff * (double)h.n_theta);
    atomicAdd(out + 5, (double)h.quad_attempts_theta);
    atomicAdd(out + 6, (double)h.quad_attempts_phi * h.n_theta);
    atomicAdd(out + 7, (double)h.n_theta);
}

__global__ void k_or_status(int32_t* acc, const int32_t* __restrict__ st, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) acc[i] |= st[i];
}

// models whose grid exceeded the compiled capacity produce NaN, never a silent partial result (CTA / model; RAGGED: the
// model's block of the ragged output)
template <bool RAGGED>
__global__ void k_nan_capacity(BatchWs w, double* out, size_t comp_sz_total, SetsDev sd) {
    const int mi = blockIdx.x;
    if (!(w.status[mi] & VAG_ST_CAPACITY)) return;
    if constexpr (RAGGED) {
        const size_t per_model = VAG_NCOMP * ragged_comp_size(sd, mi);
        double* o = out + (size_t)(sd.out_off[mi] - sd.out_off[0]) * VAG_NCOMP;
        for (size_t i = threadIdx.x; i < per_model; i += blockDim.x) o[i] = NAN;
    } else {
        for (size_t i = threadIdx.x; i < comp_sz_total; i += blockDim.x) out[(size_t)mi * comp_sz_total + i] = NAN;
    }
}

// Self-test of vag_libm.cuh on the device: out[i] = gl::fn(x[i] [, y[i]]) (fn as in vag_selftest_libm, include/vag.h)
__global__ void k_libm_selftest(int fn, const double* __restrict__ x, const double* __restrict__ y, double* __restrict__ out,
                                size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double a = x[i], b = y ? y[i] : 0.0;
        double r = 0;
        switch (fn) {
            case 0: r = gl::exp(a); break;
            case 1: r = gl::exp2(a); break;
            case 2: r = gl::log(a); break;
            case 3: r = gl::log2(a); break;
            case 4: r = gl::log10(a); break;
            case 5: r = gl::pow(a, b); break;
            case 6: r = gl::sin(a); break;
            case 7: r = gl::cos(a); break;
        }
        out[i] = r;
    }
}

// FP64 FMA throughput probe (roofline denominator for the ODE / radiation / EATS kernels, which are
// FP64-pipe or dependent-latency bound; MEASURED_PEAKS.json has no FP64 entry)
__global__ void __launch_bounds__(256) k_fp64_peak(double* sink, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 12345.678) sink[0] = a0;
}

// Planning of a batch whose parameters are on the device (thread / record): ok[i] = vag_params_validate accepts in[i],
// caps[0..1] = max over the accepted records' bounds (zeroed by the caller), and, with run, the records that will run:
// a rejected record is replaced by stand_in, so no kernel downstream meets a set the reference constructors refuse.
__global__ void __launch_bounds__(256) k_plan(const vag_params* __restrict__ in, size_t n, vag_params stand_in,
                                              vag_params* __restrict__ run, int32_t* __restrict__ ok, int* caps) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int ct = 0, cp = 0;
    if (i < n) {
        const bool good = params_check(in[i]) == PR_OK;
        ok[i] = good ? 1 : 0;
        if (good) {
            const Caps c = caps_of(in[i]);
            ct = c.theta;
            cp = c.phi;
        }
        if (run) run[i] = good ? in[i] : stand_in;
    }
    ct = __reduce_max_sync(0xffffffffu, ct);
    cp = __reduce_max_sync(0xffffffffu, cp);
    if ((threadIdx.x & 31) == 0) {
        atomicMax(caps, ct);
        atomicMax(caps + 1, cp);
    }
}

// After a planned run (block / model): a rejected record ran as the stand-in; its result becomes VAG_ST_INVALID,
// chi2 = +inf (the reference raises, its samplers give logL = -inf, samplers.py:63-70) and NaN flux.
__global__ void k_reject(const int32_t* __restrict__ ok, int32_t* status, double* chi2, double* out, size_t per_model) {
    const size_t mi = blockIdx.x;
    if (ok[mi]) return;
    if (threadIdx.x == 0) {
        if (status) status[mi] = VAG_ST_INVALID;
        if (chi2) chi2[mi] = kInf;
    }
    for (size_t i = threadIdx.x; out && i < per_model; i += blockDim.x) out[mi * per_model + i] = NAN;
}

// ---- ragged series requests (see SeriesSet): the kernels that stay apart from their shared-request ones ----------
// k_series_bands_sets shares series_bands_cta with k_series_bands, but runs one CTA per set and reduces over the sets.
// k_nu_range_sets (a warp per model) and k_nu_range (one CTA per batch) compute different things.  k_total_sets (a CTA
// per model) and k_total (a thread per element) have different launch geometries: a fold would change k_total's launch.

// k_series_bands per data set (CTA / set) into sets[].n_nu and the set's band table.  red[0] = max over the sets of
// n_bands, red[1] = min over the sets of floor(3 n / n_bands): the batch is banded when every set passes series_banded
// (see series_banded_sets).  red is preset to {0, INT_MAX} by the caller.
__global__ void __launch_bounds__(256) k_series_bands_sets(const double* __restrict__ lg2_nu, const double* __restrict__ nu_lin,
                                                           const double* __restrict__ nu23, SeriesSet* sets, int* band_of,
                                                           double* b_lg2, double* b_lin, double* b_23, int* red) {
    const int d = blockIdx.x;
    const int off = sets[d].off, n = sets[d].n;
    const size_t b = (size_t)d * EATS_NU_TILE;
    series_bands_cta(lg2_nu + off, nu_lin + off, nu23 + off, n, band_of + off, b_lg2 + b, b_lin + b, b_23 + b,
                     &sets[d].n_nu);
    if (threadIdx.x == 0) {
        const int nb = sets[d].n_nu;
        atomicMax(red, nb);
        atomicMin(red + 1, (int)min(3LL * n / max(nb, 1), (long long)INT_MAX));
    }
}

// k_nu_range per model (warp / model): out[2 m], out[2 m + 1] = log2 of the smallest / largest frequency of its data set
// (GRID: of its slice of the frequency nodes)
template <bool GRID>
__global__ void k_nu_range_sets(const double* __restrict__ lg2_nu, SetsDev sd, int n_models, double* out) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n_models) return;
    const SeriesSet s = sd.sets[sd.set_of[warp]];
    const int off = GRID ? s.nu_off : s.off, n = GRID ? s.n_nu : s.n;
    double lo = kInf, hi = -kInf;
    for (int i = lane; i < n; i += 32) {
        lo = fmin(lo, lg2_nu[off + i]);
        hi = fmax(hi, lg2_nu[off + i]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) {
        out[2 * warp] = lo;
        out[2 * warp + 1] = hi;
    }
}

// k_total on a ragged output (CTA / model)
__global__ void k_total_sets(double* out, SetsDev sd) {
    const int mi = blockIdx.x;
    const size_t cs = ragged_comp_size(sd, mi);
    double* o = out + (size_t)(sd.out_off[mi] - sd.out_off[0]) * VAG_NCOMP;
    for (size_t e = threadIdx.x; e < cs; e += blockDim.x)
        o[e] = o[VAG_C_FWD_SYNC * cs + e] + o[VAG_C_FWD_SSC * cs + e] + o[VAG_C_RVS_SYNC * cs + e] + o[VAG_C_RVS_SSC * cs + e];
}

// ---- band-integrated data in a ragged batch (vag_flux_band_multi, vag_chi2_multi_bands) ----------------------------
// An evaluation is one (model, band): a model of the ragged grid request whose set is the band (its times, its nodes).

// k_band_reduce per evaluation (CTA / evaluation): its [VAG_NCOMP][n_nu][n] grid block (sd.out_off counts from the first
// evaluation of the call) -> [VAG_NCOMP][n] at VAG_NCOMP * red_off[e], with the weights of its node slice, summed in
// k_band_reduce's order
__global__ void k_band_reduce_sets(const double* __restrict__ F, const double* __restrict__ wgt, double* __restrict__ out,
                                   const long long* __restrict__ red_off, SetsDev sd) {
    const int e = blockIdx.x;
    const SeriesSet b = sd.sets[sd.set_of[e]];
    const double* f0 = F + (size_t)sd.out_off[e] * VAG_NCOMP;
    const double* wb = wgt + b.nu_off;
    double* o = out + (size_t)red_off[e] * VAG_NCOMP;
    for (int q = threadIdx.x; q < VAG_NCOMP * b.n; q += blockDim.x) {
        const int c = q / b.n, j = q - c * b.n;
        const double* f = f0 + (size_t)c * b.n_nu * b.n + j;
        double s = 0;
        for (int i = 0; i < b.n_nu; ++i) s += f[(size_t)i * b.n] * wb[i];
        o[q] = s;
    }
}

// Band terms of vag_chi2_multi_bands (warp / model).  Model m starts from its point term (pt_of[m] >= 0: the point pass's
// chi2_pts / st_pts; otherwise 0 and no status) and adds the band terms of its evaluations e0[m] .. e0[m + 1] - 1 in band
// order through chi2_warp with accumulate, each one's fatal test on its own band run's status st_eval[e], as vag_chi2's
// k_chi2 launches do.  status[m] = the OR over the terms.  The band data lnF / sig / wgt sit at the band times' offsets.
__global__ void k_chi2_bands(const double* __restrict__ band, const long long* __restrict__ red_off, SetsDev sd,
                             const double* __restrict__ lnF, const double* __restrict__ sig, const double* __restrict__ wgt,
                             const int* __restrict__ st_eval, const int* __restrict__ e0, const int* __restrict__ pt_of,
                             const double* __restrict__ chi2_pts, const int* __restrict__ st_pts, size_t n_models,
                             double* chi2, int32_t* status) {
    const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (m >= (int)n_models) return;
    const int p = pt_of[m];
    int st = p >= 0 ? st_pts[p] : 0;
    if (lane == 0) chi2[m] = p >= 0 ? chi2_pts[p] : 0.0;  // read back by lane 0 only (chi2_warp)
    for (int e = e0[m]; e < e0[m + 1]; ++e) {
        const SeriesSet b = sd.sets[sd.set_of[e]];
        chi2_warp(0, lane, band + (size_t)red_off[e] * VAG_NCOMP, b.n, lnF + b.off, sig + b.off, wgt + b.off, nullptr,
                  nullptr, chi2 + m, st_eval + e, 1);
        st |= st_eval[e];
    }
    if (lane == 0) status[m] = st;
}

// ---- the gathers of vag_chi2_multi_bands(_dev) ------------------------------------------------------------------
// dst[i] = src[idx[i]]: the parameter record of every entry of the lists, gathered from the records of the models, and
// for the first n_av entries (the point pass's models) their A_V as well: av_dst[i] = av_src[idx[i]]
__global__ void k_gather_params_av(const vag_params* __restrict__ src, const int* __restrict__ idx, size_t n, vag_params* dst,
                                   const double* __restrict__ av_src, size_t n_av, double* av_dst) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = idx[i];
    dst[i] = src[j];
    if (i < n_av) av_dst[i] = av_src[j];
}

// The band data into the concatenated band workspace (CTA / band): plane k of dst (t, lnF_obs, sigma_ln, w; `stride`
// doubles each) receives band b's device array src[4 b + k] at the band's time offset tab[b].off
__global__ void k_gather_bands(const double* const* __restrict__ src, const SeriesSet* __restrict__ tab, size_t stride,
                               double* dst) {
    const int b = blockIdx.x;
    const SeriesSet B = tab[b];
    for (int k = 0; k < 4; ++k) {
        const double* __restrict__ a = src[4 * (size_t)b + k];
        double* d = dst + k * stride + B.off;
        for (int i = threadIdx.x; i < B.n; i += blockDim.x) d[i] = a[i];
    }
}

// ---- posterior-predictive bands (vag_flux_quantiles_multi) --------------------------------------------------------
// The members of every set (CTA / set): of its candidates cand[c0[d] .. c0[d + 1]) -- the models whose dataset_of is d,
// in model order -- those whose status has neither VAG_ST_ODE_FAIL500 (the reference throws) nor VAG_ST_CAPACITY (NaN
// output), kept in order as the element offsets VAG_NCOMP * out_off[m] of their `total` planes in the ragged grid output;
// n_used[d] = their number
__global__ void __launch_bounds__(256) k_quant_members(const int* __restrict__ cand, const int* __restrict__ c0,
                                                       const int32_t* __restrict__ status, const long long* __restrict__ out_off,
                                                       long long* __restrict__ mem_off, long long* __restrict__ n_used) {
    __shared__ int s_warp[8];
    __shared__ int s_count;
    const int d = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int lo = c0[d], hi = c0[d + 1];
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    for (int base = lo; base < hi; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int m = i < hi ? cand[i] : -1;
        const bool keep = m >= 0 && !(status[m] & (VAG_ST_ODE_FAIL500 | VAG_ST_CAPACITY));
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[wid] = __popc(bal);
        __syncthreads();
        int pos = s_count + __popc(bal & ((1u << lane) - 1u));
        for (int w = 0; w < wid; ++w) pos += s_warp[w];
        if (keep) mem_off[lo + pos] = (long long)VAG_NCOMP * out_off[m];
        __syncthreads();
        if (threadIdx.x == 0)
            for (int w = 0; w < 8; ++w) s_count += s_warp[w];
        __syncthreads();
    }
    if (threadIdx.x == 0) n_used[d] = s_count;
}

// numpy.quantile(method="linear") of every (set, column) over the set's members (vag_quantile.cuh), CTA / (set, tile of
// QUANT_COLS consecutive columns of its [n_nu][n_t] grid), a warp / column.  tile0[d]: the first tile of set d, col0[d]:
// its first column among the concatenated columns of all sets; set d's members' offsets start at mem_off[c0[d]].  The
// members' rows of the tile are read coalesced; a set of at most rows_cap members is staged as keys in shared memory
// ([QUANT_COLS][n]) and selected there, a larger one is selected from global memory (L2) in every pass.
// out: set d's [n_q][n_nu][n_t] block at n_q * col0[d].
constexpr int QUANT_COLS = 4;
constexpr size_t QUANT_SMEM_BUDGET = 160 * 1024;  // dynamic shared memory k_quantiles may stage a tile in
__global__ void __launch_bounds__(QUANT_COLS * 32) k_quantiles(const double* __restrict__ F, const long long* __restrict__ mem_off,
                                                             const int* __restrict__ c0, const long long* __restrict__ n_used,
                                                             const long long* __restrict__ tile0,
                                                             const long long* __restrict__ col0, int n_sets,
                                                             const double* __restrict__ q, int n_q, int rows_cap,
                                                             double* __restrict__ out) {
    extern __shared__ uint64_t s_keys[];
    __shared__ unsigned s_hist[QUANT_COLS][QUANT_BINS];
    const long long tile = blockIdx.x;
    int d = 0;  // the last set whose first tile is <= tile (every set has one tile or more)
    for (int hi = n_sets; hi - d > 1;) {
        const int mid = (d + hi) / 2;
        if (tile0[mid] <= tile)
            d = mid;
        else
            hi = mid;
    }
    const long long cols = col0[d + 1] - col0[d], c_first = (tile - tile0[d]) * QUANT_COLS;
    const int n = (int)n_used[d];
    const long long* __restrict__ mo = mem_off + c0[d];
    const int wid = threadIdx.x >> 5;
    const bool staged = n <= rows_cap;
    if (staged) {
        for (int e = threadIdx.x; e < n * QUANT_COLS; e += blockDim.x) {
            const int i = e / QUANT_COLS, k = e - i * QUANT_COLS;
            if (c_first + k < cols) s_keys[(size_t)k * n + i] = quant_key(F[mo[i] + c_first + k]);
        }
        __syncthreads();
    }
    const long long c = c_first + wid;
    if (c >= cols) return;
    const QuantWarp grp{(int)(threadIdx.x & 31)};
    double* o = out + n_q * col0[d] + c;
    if (staged) {
        const uint64_t* ks = s_keys + (size_t)wid * n;
        quant_column(grp, [ks](int i) { return ks[i]; }, n, q, n_q, o, (size_t)cols, s_hist[wid]);
    } else {
        const double* f = F + c;
        quant_column(grp, [f, mo](int i) { return quant_key(f[mo[i]]); }, n, q, n_q, o, (size_t)cols, s_hist[wid]);
    }
}

// ---- exposure averages (vag_flux_density_exposures, vag_chi2_multi_bands_exposures) -------------------------------
// CTA / model, a thread / (component, point): out[c][i] = expo_mean of point i's samples in F (vag_exposure.cuh).  Shared
// request: model m's samples are F[m][VAG_NCOMP][n_s], its points out[m][VAG_NCOMP][n], point i's samples at
// pos[s0[i] .. s0[i + 1]).  RAGGED: model m's samples are its block of the ragged sample request (sx: the sets of samples),
// its points its block of the ragged point output (sd: the sets of points, whose nu_off is the set's first point in s0).
template <bool RAGGED>
__global__ void __launch_bounds__(128) k_expo_average(const double* __restrict__ F, int n_s, int n, const int* __restrict__ s0,
                                                      const int* __restrict__ pos, double* __restrict__ out, SetsDev sx,
                                                      SetsDev sd) {
    const int mi = blockIdx.x;
    const double* f = F + (size_t)mi * VAG_NCOMP * n_s;
    double* o = out + (size_t)mi * VAG_NCOMP * n;
    if constexpr (RAGGED) {
        const int d = sd.set_of[mi];
        const SeriesSet S = sd.sets[d];
        n_s = sx.sets[d].n;
        n = S.n;
        s0 += S.nu_off;
        f = F + (size_t)(sx.out_off[mi] - sx.out_off[0]) * VAG_NCOMP;
        o = out + (size_t)(sd.out_off[mi] - sd.out_off[0]) * VAG_NCOMP;
    }
    for (int q = threadIdx.x; q < VAG_NCOMP * n; q += blockDim.x) {
        const int c = q / n, i = q - c * n;
        const int a = s0[i];
        o[q] = expo_mean(f + (size_t)c * n_s, pos + a, s0[i + 1] - a);
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return fail(VAG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
    } while (0)

// device buffer grown on demand; freed with the context that owns it (vag_destroy makes its device current)
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
};

}  // namespace

struct vag_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    DevBuf model_buf, row_buf, cell_buf, obs_buf, ic_buf, lut_buf, sp_buf, geom_buf, split_buf, work_buf;
    DevBuf io_params, io_status, io_t, io_nu, io_w, io_out, io_sets, io_bands;  // staging of the host-buffer entry points
    DevBuf plan_buf;                // device planning: ok[], the capacities, the records that run
    int* h_totals = nullptr;        // pinned
    char* h_plan = nullptr;         // pinned, grown on demand: the capacities planned on the device, with ok[] ahead of them
    size_t h_plan_cap = 0;
    long long* h_cells = nullptr;   // pinned
    int* h_bands = nullptr;         // pinned [2]: distinct frequencies of the series request in flight (ragged: see k_series_bands_sets)
    int series_mode = 0;            // vag_set_series_mode: 0 auto, 1 per-point spectra always, 2 banded whenever possible
    int grid_lanes = 0;             // vag_set_grid_lanes: 0 by batch size, else k_grid<grid_lanes> for every batch
    int cap_theta = 384, cap_phi = 128;  // vag_set_capacity: what the *_dev entry points run with (host calls size each batch)
    int dbg_max_ode_steps = 0, dbg_max_ode_fails = 0;
    bool profiling = false;
    int out_mode = VAG_OUT_DENSE;
    int total_alias = -1;  // VAG_OUT_PRESENT_ALIAS_TOTAL: component plane the last host call's `total` equals, or -1
    cudaEvent_t ev[8] = {};
    float stage_ms[8] = {};
    double work[8] = {};   // k_work counters of the last profiled pass
    int launches = 0;
    int sm_count = 148;
    // warps of k_ic_spectrum per SM (one warp per cell in flight, 30 KB of scratch each): as many as are resident.  Measured
    // on config 4: 12 / 16 / 20 / 24 / 28 warps per SM -> 75.1 / 68.6 / 65.0 / 61.1 / 58.5 ms per batch (latency-bound, IPC 1.3)
    int ic_warps_per_sm = 16;
};

namespace {

template <class T>
T* carve(char*& p, size_t n) {
    T* r = reinterpret_cast<T*>(p);
    p += ((n * sizeof(T) + 255) / 256) * 256;
    return r;
}
template <class T>
size_t carve_sz(size_t n) {
    return ((n * sizeof(T) + 255) / 256) * 256;
}

// Host arrays packed for one upload, in 256-byte aligned slices (carve's layout); put() returns the slice's byte offset
struct Pack {
    std::vector<char> h;
    template <class T>
    size_t put(const T* p, size_t n) {
        const size_t o = h.size();
        const char* b = reinterpret_cast<const char*>(p);
        if (n) h.insert(h.end(), b, b + sizeof(T) * n);
        h.resize(o + carve_sz<T>(n));
        return o;
    }
    template <class T>
    size_t put(const std::vector<T>& v) {
        return put(v.data(), v.size());
    }
};
template <class T>
T* at(void* base, size_t off) {
    return reinterpret_cast<T*>(static_cast<char*>(base) + off);
}


constexpr size_t EATS_SMEM_BUDGET = 200 * 1024;  // dynamic shared memory k_eats may ask for
// models per pipeline pass: k_rowgeom / k_rowcos / k_dop_extrema index the model with gridDim.y (<= 65535), and the
// per-model workspaces of a pass stay below a few GB; larger batches are processed in consecutive passes
constexpr size_t MAX_MODELS_PER_PASS = 32768;

struct Request {
    bool series;
    const double* d_t;
    const double* d_nu;
    size_t n_t, n_nu;
    bool nu_code_units = false;
    const double *d_lnF = nullptr, *d_sig = nullptr, *d_w = nullptr;  // [n_t] observations of a chi-squared series
    const double* d_ext = nullptr;  // [n_t] extinction per point, or NULL
    const double* d_av = nullptr;   // [n_models] A_V per model of the batch, set with d_ext (run_flux offsets it per pass)
    // A ragged request (every model its own data set; d_t ... d_ext concatenated over the sets; a grid request: d_t and
    // d_nu): the device tables (run_flux slices set_of and out_off per pass), the host prefix sums of the models' output
    // points [n_models + 1], the number of sets, the size of the largest (grid: the most times) and, for a grid request,
    // the most frequency nodes of a model
    const SetsDev* sets = nullptr;
    const long long* h_off = nullptr;
    int n_sets = 0;
    size_t max_set = 0, max_nu = 0;
};

int setup_models(vag_context* ctx, BatchWs& w, const vag_params* d_params, size_t n, Caps caps) {
    w = BatchWs{};
    w.n_models = (int)n;
    w.dbg_max_ode_steps = ctx->dbg_max_ode_steps;
    w.dbg_max_ode_fails = ctx->dbg_max_ode_fails;
    w.cap_theta = caps.theta;
    w.cap_phi = caps.phi;
    w.work_per_model = grid_work_doubles(w.cap_theta, w.cap_phi);
    w.params = d_params;
    w.sp_lut = static_cast<const double*>(ctx->sp_buf.p);
    size_t bytes = carve_sz<ModelCfg>(n) + carve_sz<GridHeader>(n) + carve_sz<double>(n * w.cap_theta) * 2 +
                   carve_sz<double>(n * w.cap_phi) + carve_sz<double>(n * w.work_per_model) +
                   carve_sz<int>(n * w.cap_theta) * 2 + carve_sz<int>(n + 1) + carve_sz<long long>(n + 1) +
                   carve_sz<int>(TOT_N) + carve_sz<int>(n);
    CK(ctx->model_buf.ensure(bytes));
    char* p = static_cast<char*>(ctx->model_buf.p);
    w.cfg = carve<ModelCfg>(p, n);
    w.hdr = carve<GridHeader>(p, n);
    w.theta = carve<double>(p, n * w.cap_theta);
    w.t_dec = carve<double>(p, n * w.cap_theta);
    w.phi = carve<double>(p, n * w.cap_phi);
    w.work = carve<double>(p, n * w.work_per_model);
    w.reps = carve<int>(p, n * w.cap_theta);
    w.rep_of = carve<int>(p, n * w.cap_theta);
    w.row_off = carve<int>(p, n + 1);
    w.cell_off = carve<long long>(p, n + 1);
    w.totals = carve<int>(p, TOT_N);
    w.status = carve<int>(p, n);
    return VAG_OK;
}

int setup_rows(vag_context* ctx, BatchWs& w, int rows, long long cells, bool any_spread) {
    w.n_cells = cells;
    CK(ctx->row_buf.ensure(carve_sz<int>(rows) * 3 + carve_sz<RowDyn>(rows) + carve_sz<long long>(rows + 1)));
    char* p = static_cast<char*>(ctx->row_buf.p);
    w.row_model = carve<int>(p, rows);
    w.row_rep = carve<int>(p, rows);
    w.inj_idx = carve<int>(p, rows);
    w.row_dyn = carve<RowDyn>(p, rows);
    w.row_cell_off = carve<long long>(p, rows + 1);
    const size_t plane = carve_sz<double>((size_t)cells);
    CK(ctx->cell_buf.ensure(plane * (1 + 12 + 2 + (any_spread ? 4 : 0)) + carve_sz<double>((size_t)cells * PH_NCOEF) * 2));
    p = static_cast<char*>(ctx->cell_buf.p);
    w.t_rows = carve<double>(p, (size_t)cells);
    for (int a = 0; a < 6; ++a) w.fwd[a] = carve<double>(p, (size_t)cells);
    for (int a = 0; a < 6; ++a) w.rvs[a] = carve<double>(p, (size_t)cells);
    w.geo_u = carve<double>(p, (size_t)cells);
    w.geo_lg2r2 = carve<double>(p, (size_t)cells);
    w.coef_fwd = carve<double>(p, (size_t)cells * PH_NCOEF);
    w.coef_rvs = carve<double>(p, (size_t)cells * PH_NCOEF);
    w.sh_theta = w.geo_cth = w.geo_sth = w.geo_dcos = nullptr;
    if (any_spread) {
        w.sh_theta = carve<double>(p, (size_t)cells);
        w.geo_cth = carve<double>(p, (size_t)cells);
        w.geo_sth = carve<double>(p, (size_t)cells);
        w.geo_dcos = carve<double>(p, (size_t)cells);
    }
    return VAG_OK;
}

// inverse-Compton workspaces (only when some model of the batch has ssc=True)
int setup_ic(vag_context* ctx, BatchWs& w, size_t n, long long cells, int n_ic_warps, cudaStream_t s) {
    const size_t nc = (size_t)cells;
    const size_t bytes = 2 * (carve_sz<IcCell>(nc) + carve_sz<IcTable>(nc) + carve_sz<double>(nc * IC_CAP_OUT)) +
                         carve_sz<double>(n * w.max_erows) + 2 * carve_sz<double>(n * w.max_n_t) +
                         carve_sz<double>((size_t)n_ic_warps * IC_SCRATCH_DOUBLES);
    CK(ctx->ic_buf.ensure(bytes));
    char* p = static_cast<char*>(ctx->ic_buf.p);
    for (int a = 0; a < 2; ++a) {
        w.ic[a] = carve<IcCell>(p, nc);
        w.ictab_h[a] = carve<IcTable>(p, nc);
        w.ictab[a] = carve<double>(p, nc * IC_CAP_OUT);
    }
    w.rowcos = carve<double>(p, n * w.max_erows);
    w.dop_min = carve<double>(p, n * w.max_n_t);
    w.dop_max = carve<double>(p, n * w.max_n_t);
    w.ic_scratch = carve<double>(p, (size_t)n_ic_warps * IC_SCRATCH_DOUBLES);
    if (!ctx->lut_buf.p) {
        CK(ctx->lut_buf.ensure(sizeof(KnLut)));
        k_kn_lut<<<1, KN_LUT_N, 0, s>>>(static_cast<KnLut*>(ctx->lut_buf.p));
    }
    w.lut = static_cast<const KnLut*>(ctx->lut_buf.p);
    return VAG_OK;
}

void mark(vag_context* ctx, int i, cudaStream_t s) {
    if (ctx->profiling) cudaEventRecord(ctx->ev[i], s);
}

// The kernel variants: the launch sites and vag_create's function attributes take them from here
using GridKernel = void (*)(BatchWs, const double*, int, SetsDev);
using EatsKernel = void (*)(BatchWs, EatsRequest, double*, int, int, int, int, size_t, SetsDev);
constexpr int GRID_LANES[] = {4, 8, 16, 32};
constexpr int EATS_MODES = 3, EATS_KINDS = 3;

// (defined after run_front: the cubin lists the kernel templates in the order the source first names them)
GridKernel grid_kernel(int lanes, bool ragged);
EatsKernel eats_kernel(int mode, int kind, bool ragged);

// Lanes per model of k_grid: the widest group whose launch fits into one wave of resident CTAs (GRID_MIN_BLOCKS CTAs of
// 128 threads per SM).  Narrower groups only pay once a wider launch would need a second wave: the models of one warp
// still diverge outside the quadrature rounds (GroupPar::lockstep), and with fewer than 6 lanes the six stage
// evaluations of an attempt take two passes.  k_grid stage per batch on the bench draw (B200, 1000 W;
// G = 4 / 8 / 16 / 32, ms): 16384 models 0.74 / 0.82 / 1.21 / 1.95, 4096: 0.50 / 0.36 / 0.36 / 0.52,
// 1024: 0.45 / 0.31 / 0.28 / 0.26 (G = 2 was never the fastest: 1.23 ms at 16384 before the lockstep rounds).
int grid_lanes_for(size_t n, int sm_count) {
    const size_t resident_lanes = (size_t)sm_count * GRID_MIN_BLOCKS * 128;
    int g = 32;
    while (g > 4 && n * g > resident_lanes) g >>= 1;
    return g;
}

// grid + dynamics + radiation for a batch; fills w and the totals
// (sets: each model's observation window from its own data set of d_t)
int run_front(vag_context* ctx, BatchWs& w, const vag_params* d_params, size_t n, Caps caps, const double* d_t,
              size_t n_t, cudaStream_t s, int* totals_out, long long* cells_out, const SetsDev* sets = nullptr) {
    int rc = setup_models(ctx, w, d_params, n, caps);
    if (rc) return rc;
    mark(ctx, 0, s);
    const int lanes = ctx->grid_lanes ? ctx->grid_lanes : grid_lanes_for(n, ctx->sm_count);
    grid_kernel(lanes, sets != nullptr)<<<(unsigned)((n * lanes + 127) / 128), 128, 0, s>>>(w, d_t, (int)n_t,
                                                                                          sets ? *sets : SetsDev{});
    k_scan<<<1, 1024, 0, s>>>(w);
    ctx->launches += 2;
    CK(cudaMemcpyAsync(ctx->h_totals, w.totals, sizeof(int) * TOT_N, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(ctx->h_cells, w.cell_off + n, sizeof(long long), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const int rows = ctx->h_totals[TOT_ROWS];
    const long long cells = *ctx->h_cells;
    std::memcpy(totals_out, ctx->h_totals, sizeof(int) * TOT_N);
    *cells_out = cells;
    rc = setup_rows(ctx, w, std::max(rows, 1), std::max<long long>(cells, 1), ctx->h_totals[TOT_ANY_SPREAD] != 0);
    if (rc) return rc;
    w.max_n_t = std::max(ctx->h_totals[TOT_MAX_NT], 1);
    w.max_erows = std::max(ctx->h_totals[TOT_MAX_EROWS], 1);
    CK(ctx->geom_buf.ensure(sizeof(RowGeom) * n * (size_t)w.max_erows));
    w.rowgeom = static_cast<RowGeom*>(ctx->geom_buf.p);
    w.any_ssc = ctx->h_totals[TOT_ANY_SSC];
    if (w.any_ssc) {
        const int n_ic_warps = (int)std::min<long long>(std::max<long long>(cells, 1), (long long)ctx->sm_count * ctx->ic_warps_per_sm);
        rc = setup_ic(ctx, w, n, std::max<long long>(cells, 1), n_ic_warps, s);
        if (rc) return rc;
    }
    if (rows > 0) {
        k_rowmap<<<(unsigned)((n + 63) / 64), 64, 0, s>>>(w);
        k_rowgeom<<<dim3((unsigned)((w.max_erows + 127) / 128), (unsigned)n), 128, 0, s>>>(w);
        k_lattice<<<(unsigned)((rows + 3) / 4), 128, 0, s>>>(w, rows);
        ctx->launches += 2;
        mark(ctx, 1, s);
        {
            // rows per warp: up to one warp per scheduler before warps are filled up
            int lanes = 32;
            // Fewer rows per warp shorten a row (less divergence) but multiply the 255-register CTAs that other batches'
            // kernels have to share the SMs with.  Measured on the config-5 batch (4096 rows; 8 / 16 / 32 rows per warp):
            // one batch alone 1.80 / 1.88 / 2.03 ms, four batches in flight 1.13 / 1.33 / 1.36 M evaluations/s --
            // so warps are thinned only while they stay below two per SM.
            // (512 rows, the share of an 8-GPU ensemble: 1 / 2 / 4 / 8 rows per warp 1.56 / 1.59 / 1.64 / 1.71 ms)
            while (lanes > 1 && (rows + lanes / 2 - 1) / (lanes / 2) <= ctx->sm_count * 2) lanes >>= 1;
            const unsigned nb = (unsigned)((rows + lanes - 1) / lanes);
            if (ctx->h_totals[TOT_ANY_FWD_ONLY]) {
                k_dynamics<false><<<nb, 32, 0, s>>>(w, rows, lanes);
                ctx->launches++;
            }
            if (ctx->h_totals[TOT_ANY_PAIR]) {
                k_dynamics<true><<<nb, 32, 0, s>>>(w, rows, lanes);
                ctx->launches++;
            }
        }
        mark(ctx, 2, s);
        k_radiation<<<(unsigned)rows, 64, 0, s>>>(w);
        ctx->launches += 2;
        if (w.any_ssc) {
            k_ic_cooling<<<dim3((unsigned)((rows + 31) / 32), 2), 32, 0, s>>>(w, rows);
            ctx->launches++;
        }
    } else {
        mark(ctx, 1, s);
        mark(ctx, 2, s);
    }
    mark(ctx, 3, s);
    CK(cudaGetLastError());
    return VAG_OK;
}

GridKernel grid_kernel(int lanes, bool ragged) {
    switch (lanes) {
        case 4: return ragged ? k_grid<4, true> : k_grid<4, false>;
        case 8: return ragged ? k_grid<8, true> : k_grid<8, false>;
        case 16: return ragged ? k_grid<16, true> : k_grid<16, false>;
        default: return ragged ? k_grid<32, true> : k_grid<32, false>;
    }
}

EatsKernel eats_kernel(int mode, int kind, bool ragged) {
    static const EatsKernel k[2][EATS_MODES][EATS_KINDS] = {
        {{k_eats<0, EATS_GRID, false>, k_eats<0, EATS_POINT, false>, k_eats<0, EATS_BANDED, false>},
         {k_eats<1, EATS_GRID, false>, k_eats<1, EATS_POINT, false>, k_eats<1, EATS_BANDED, false>},
         {k_eats<2, EATS_GRID, false>, k_eats<2, EATS_POINT, false>, k_eats<2, EATS_BANDED, false>}},
        {{k_eats<0, EATS_GRID, true>, k_eats<0, EATS_POINT, true>, k_eats<0, EATS_BANDED, true>},
         {k_eats<1, EATS_GRID, true>, k_eats<1, EATS_POINT, true>, k_eats<1, EATS_BANDED, true>},
         {k_eats<2, EATS_GRID, true>, k_eats<2, EATS_POINT, true>, k_eats<2, EATS_BANDED, true>}}};
    return k[ragged][mode][kind];
}

// flux of a batch into d_out [n][VAG_NCOMP][comp]; with d_chi2, also the chi-squared of the series against rq_in's data
int run_flux_pass(vag_context* ctx, const vag_params* d_params, size_t n, Caps caps, const Request& rq_in, double* d_out,
                  int32_t* d_status, double* d_chi2, cudaStream_t s) {
    const size_t n_t = rq_in.n_t, n_nu = rq_in.n_nu;
    const SetsDev* sets = rq_in.sets;
    // observation arrays (a ragged request: one band table per data set, the SSC band of every model)
    const size_t n_tables = sets ? (size_t)rq_in.n_sets : 1, n_ranges = sets ? 2 * n : 0;
    CK(ctx->obs_buf.ensure(sizeof(double) * (2 * n_t + 3 * n_nu + 8 + 3 * EATS_NU_TILE * n_tables + n_ranges) +
                           sizeof(int) * (n_t + 2)));
    double* lg2_t = static_cast<double*>(ctx->obs_buf.p);
    double* t_lin = lg2_t + n_t;
    double* lg2_nu = t_lin + n_t;
    double* nu_lin = lg2_nu + n_nu;
    double* nu23 = nu_lin + n_nu;
    double* nu_range = nu23 + n_nu;
    double* band_lg2 = nu_range + 8;
    double* band_lin = band_lg2 + EATS_NU_TILE * n_tables;
    double* band_23 = band_lin + EATS_NU_TILE * n_tables;
    double* nu_range_of = band_23 + EATS_NU_TILE * n_tables;
    int* band_of = reinterpret_cast<int*>(nu_range_of + n_ranges);
    int* d_n_bands = band_of + n_t;
    {
        const size_t m = std::max(n_t, n_nu);
        k_prep_obs<<<(unsigned)((m + 127) / 128), 128, 0, s>>>(rq_in.d_t, (int)n_t, rq_in.d_nu, (int)n_nu, lg2_t, t_lin,
                                                              lg2_nu, nu_lin, nu23, rq_in.nu_code_units ? 1 : 0);
        ctx->launches++;
    }
    *ctx->h_bands = 0;
    if (rq_in.series && ctx->series_mode != 1) {
        // distinct frequencies of the request; the count reaches the host with run_front's synchronisation
        if (sets) {
            CK(cudaMemsetAsync(d_n_bands, 0, sizeof(int), s));
            CK(cudaMemsetAsync(d_n_bands + 1, 0x7f, sizeof(int), s));
            k_series_bands_sets<<<(unsigned)rq_in.n_sets, 256, 0, s>>>(lg2_nu, nu_lin, nu23, sets->sets, band_of, band_lg2,
                                                                       band_lin, band_23, d_n_bands);
            CK(cudaMemcpyAsync(ctx->h_bands, d_n_bands, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
        } else {
            k_series_bands<<<1, 1024, 0, s>>>(lg2_nu, nu_lin, nu23, (int)n_nu, band_of, band_lg2, band_lin, band_23, d_n_bands);
            CK(cudaMemcpyAsync(ctx->h_bands, d_n_bands, sizeof(int), cudaMemcpyDeviceToHost, s));
        }
        ctx->launches++;
    }
    BatchWs w;
    int totals[TOT_N];
    long long cells = 0;
    int rc = run_front(ctx, w, d_params, n, caps, rq_in.d_t, n_t, s, totals, &cells, sets);
    if (rc) return rc;

    if (w.any_ssc && totals[TOT_ROWS] > 0) {
        // SSC tables: observation band -> per-row line-of-sight cosines -> per-k Doppler extrema -> tables
        // (a ragged request: each model's band is its own data set's, as its shared-request call would see it)
        w.nu_range = sets ? nu_range_of : nu_range;
        if (sets)
            (rq_in.series ? k_nu_range_sets<false> : k_nu_range_sets<true>)<<<(unsigned)((n * 32 + 127) / 128), 128, 0, s>>>(
                lg2_nu, *sets, (int)n, nu_range_of);
        else
            k_nu_range<<<1, 256, 0, s>>>(lg2_nu, (int)n_nu, nu_range);
        k_rowcos<<<dim3((unsigned)((w.max_erows + 127) / 128), (unsigned)n), 128, 0, s>>>(w);
        k_dop_extrema<<<dim3((unsigned)((w.max_n_t + 63) / 64), (unsigned)n), 64, 0, s>>>(w);
        const int n_ic_warps = (int)std::min<long long>(std::max<long long>(cells, 1), (long long)ctx->sm_count * ctx->ic_warps_per_sm);
        const unsigned ic_blocks = (unsigned)((n_ic_warps * 32 + 127) / 128);
        (sets ? k_ic_spectrum<true> : k_ic_spectrum<false>)<<<ic_blocks, 128, 0, s>>>(w, totals[TOT_ROWS], n_ic_warps);
        ctx->launches += 4;
    }
    // points per component plane of a model (shared request), and the elements of the pass's output
    const size_t comp_sz = rq_in.series ? n_t : n_nu * n_t;
    const size_t elems = sets ? (size_t)VAG_NCOMP * (rq_in.h_off[n] - rq_in.h_off[0]) : n * VAG_NCOMP * comp_sz;
    CK(cudaMemsetAsync(d_out, 0, sizeof(double) * elems, s));
    const int max_n_t = std::max(totals[TOT_MAX_NT], 2);
    const int max_erows = std::max(totals[TOT_MAX_EROWS], 1);
    if (totals[TOT_ROWS] > 0) {
        // shared-memory budget -> rows staged per pass
        const size_t budget = EATS_SMEM_BUDGET;
        int row_chunk = EATS_ROW_CHUNK;
        // a ragged request: h_bands = the largest set's distinct frequencies and min floor(3 n / n_bands) over the sets
        const int n_bands_req = rq_in.series ? *ctx->h_bands : 0;
        const bool banded = sets ? ctx->series_mode != 1 && series_banded_sets(n_bands_req, ctx->h_bands[1], max_n_t,
                                                                               ctx->series_mode)
                                 : series_banded(n_bands_req, max_n_t, n_t, ctx->series_mode);
        // (a ragged grid request: the widest node set of the batch; each CTA tiles its own, see k_eats)
        const int nu_tile = rq_in.series ? (banded ? n_bands_req : 1)
                                         : (int)std::min<size_t>(EATS_NU_TILE, sets ? rq_in.max_nu : n_nu);
        const int acc_cols = rq_in.series ? 1 : nu_tile;
        const int acc_n = (int)(sets ? rq_in.max_set : n_t);  // accumulator columns: the longest request of the batch
        auto smem_bytes = [&](int rc_) {
            return sizeof(double) * (acc_cols * eats_acc_stride(acc_n) +
                                     eats_shared_doubles(max_n_t, rq_in.series && !banded, rc_, nu_tile) + SPL_DOUBLES);
        };
        // fewer staged rows per pass while that buys residency: 8 CTAs / SM need <= 27 KB each (227 KB per SM,
        // 1 KB per CTA reserved by the system)
        while (row_chunk > 4 && smem_bytes(row_chunk) > 27 * 1024) --row_chunk;
        while (row_chunk > 1 && smem_bytes(row_chunk) > budget) --row_chunk;
        if (smem_bytes(row_chunk) > budget)
            return fail(VAG_ERR_CAPACITY, "time lattice too long for the EATS shared-memory stage");
        // Row split: a (model, shock) whose rows do not fit one pass is cut into up to `chunks` CTAs, as many as it takes to
        // put ~2 waves of CTAs (8 resident per SM) on the device.  Tophat-on-axis batches of thousands of models need
        // none; a few hundred structured off-axis or SSC models (hundreds of rows each, BASELINE.json configs 2 and 4)
        // would otherwise run as one long CTA per model on a mostly idle device.  The splits write disjoint slabs that
        // k_sum_splits adds in a fixed order (deterministic).
        const int chunks = (max_erows + row_chunk - 1) / row_chunk;
        const int n_shock = totals[TOT_ANY_PAIR] ? 2 : 1;
        const size_t target_ctas = (size_t)ctx->sm_count * EATS_MIN_BLOCKS * 2;
        const size_t have = n * (size_t)n_shock;
        int n_split = (have < target_ctas) ? (int)std::min<size_t>(chunks, (target_ctas + have - 1) / have) : 1;
        const size_t slab_bytes = sizeof(double) * elems;
        while (n_split > 1 && slab_bytes * n_split > ((size_t)1 << 30)) --n_split;  // <= 1 GiB of slabs
        n_split = std::max(n_split, 1);
        const size_t sb = smem_bytes(row_chunk);  // <= EATS_SMEM_BUDGET, the opt-in limit set once in vag_create
        EatsRequest rq{};
        rq.series = rq_in.series ? 1 : 0;
        rq.n_t_obs = (int)n_t;
        rq.n_nu = (int)n_nu;
        rq.lg2_t_obs = lg2_t;
        rq.lg2_nu_obs = banded ? band_lg2 : lg2_nu;
        rq.nu_obs_lin = banded ? band_lin : nu_lin;
        rq.nu23_obs = banded ? band_23 : nu23;
        rq.n_bands = banded ? n_bands_req : 0;
        rq.band_of = band_of;
        rq.t_obs_lin = t_lin;
        rq.acc_stride = eats_acc_stride(acc_n);
        const dim3 eg((unsigned)n, (unsigned)n_split, (unsigned)n_shock);  // no reverse shock in the batch: no z = 1 CTAs
        double* eats_out = d_out;
        if (n_split > 1) {
            CK(ctx->split_buf.ensure(sizeof(double) * elems * n_split));
            eats_out = static_cast<double*>(ctx->split_buf.p);
            CK(cudaMemsetAsync(eats_out, 0, sizeof(double) * elems * n_split, s));
        }
        const int kind = !rq_in.series ? EATS_GRID : banded ? EATS_BANDED : EATS_POINT;
        const int n_modes = w.any_ssc ? EATS_MODES : 1;
        for (int mode = 0; mode < n_modes; ++mode)
            eats_kernel(mode, kind, sets != nullptr)<<<eg, 128, sb, s>>>(w, rq, eats_out, n_split, row_chunk, max_n_t, nu_tile,
                                                                         elems, sets ? *sets : SetsDev{});
        ctx->launches += n_modes;
        if (n_split > 1) {
            k_sum_splits<<<(unsigned)((elems + 255) / 256), 256, 0, s>>>(d_out, eats_out, n_split, elems);
            ctx->launches++;
        }
    }
    mark(ctx, 4, s);
    {
        const size_t tot = n * comp_sz;
        if (sets)
            k_total_sets<<<(unsigned)n, 128, 0, s>>>(d_out, *sets);
        else
            k_total<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(d_out, n, comp_sz);
        ctx->launches++;
        // the SSC lattices can overflow later than the grid (k_ic_spectrum sets the bit after k_scan read the OR):
        // with ssc shocks in the batch the kernel runs unconditionally and tests each model's bit on the device
        if ((totals[TOT_STATUS_OR] & VAG_ST_CAPACITY) || w.any_ssc) {
            (sets ? k_nan_capacity<true> : k_nan_capacity<false>)<<<(unsigned)n, 128, 0, s>>>(w, d_out, VAG_NCOMP * comp_sz,
                                                                                              sets ? *sets : SetsDev{});
            ctx->launches++;
        }
    }
    if (d_chi2) {
        (sets ? k_chi2<true> : k_chi2<false>)<<<(unsigned)((n * 32 + 127) / 128), 128, 0, s>>>(
            d_out, n, (int)n_t, rq_in.d_lnF, rq_in.d_sig, rq_in.d_w, rq_in.d_av, rq_in.d_ext, d_chi2, w.status, 0,
            sets ? *sets : SetsDev{});
        ctx->launches++;
    }
    mark(ctx, 5, s);
    if (d_status) CK(cudaMemcpyAsync(d_status, w.status, sizeof(int) * n, cudaMemcpyDeviceToDevice, s));
    CK(cudaGetLastError());
    if (ctx->profiling) {
        CK(ctx->work_buf.ensure(sizeof(double) * 8));
        CK(cudaMemsetAsync(ctx->work_buf.p, 0, sizeof(double) * 8, s));
        k_work<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(w, static_cast<double*>(ctx->work_buf.p));
        CK(cudaMemcpyAsync(ctx->work, ctx->work_buf.p, sizeof(double) * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (int i = 0; i < 5; ++i) cudaEventElapsedTime(&ctx->stage_ms[i], ctx->ev[i], ctx->ev[i + 1]);
    }
    return VAG_OK;
}

int run_flux(vag_context* ctx, const vag_params* d_params, size_t n, Caps caps, const Request& rq, double* d_out,
             int32_t* d_status, double* d_chi2, cudaStream_t s) {
    ctx->launches = 0;
    const size_t comp_sz = rq.series ? rq.n_t : rq.n_nu * rq.n_t;
    for (size_t lo = 0; lo < n; lo += MAX_MODELS_PER_PASS) {
        const size_t m = std::min(MAX_MODELS_PER_PASS, n - lo);
        Request rq_pass = rq;
        if (rq.d_av) rq_pass.d_av = rq.d_av + lo;
        SetsDev sets_pass{};
        if (rq.sets) {
            sets_pass = SetsDev{rq.sets->set_of + lo, rq.sets->sets, rq.sets->out_off + lo};
            rq_pass.sets = &sets_pass;
            rq_pass.h_off = rq.h_off + lo;
        }
        const size_t out_lo = rq.sets ? (size_t)rq.h_off[lo] * VAG_NCOMP : lo * VAG_NCOMP * comp_sz;
        if (int rc = run_flux_pass(ctx, d_params + lo, m, caps, rq_pass, d_out + out_lo,
                                   d_status ? d_status + lo : nullptr, d_chi2 ? d_chi2 + lo : nullptr, s))
            return rc;
    }
    return VAG_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* vag_last_error(void) { return g_err.c_str(); }
const char* vag_version(void) { return "vegasafterglow_b200 0.1 (sm_100a)"; }

void vag_params_default(vag_params* p) {
    std::memset(p, 0, sizeof(*p));
    p->k_e = p->k_g = 2.0;
    p->duration = 1.0;
    p->theta_w = 0.3;
    p->E_iso_w = 1e50;
    p->Gamma0_w = 50.0;
    p->n0 = INFINITY;
    p->fwd = vag_radiation{0.1, 0.01, 2.3, 1.0, 0, 0};
    p->rvs = vag_radiation{0.1, 0.01, 2.3, 1.0, 0, 0};
    p->axisymmetric = 1;
    p->radiative_fireball = 1;
    p->wind_k_m = 2.0;
}

int vag_params_validate(const vag_params* p) {
    static const char* const rad[4] = {"eps_e must be in (0, 1]", "eps_B must be in (0, 1]", "xi_e must be in (0, 1]",
                                       "p must be > 1"};
    const int r = params_check(*p);
    const char* m = nullptr;
    switch (r) {
        case PR_OK: return VAG_OK;
        case PR_JET_TYPE: m = "jet_type must be one of VAG_JET_* (0..5)"; break;
        case PR_MEDIUM_TYPE: m = "medium_type must be 0 (ISM) or 1 (wind)"; break;
        case PR_THETA_C: m = "theta_c must be in (0, pi/2]"; break;
        case PR_E_ISO: m = "E_iso must be finite and > 0"; break;
        case PR_GAMMA0: m = "Gamma0 must be > 1"; break;
        case PR_DURATION: m = "duration must be finite and > 0"; break;
        case PR_K_EG: m = "k_e and k_g must be finite and > 0"; break;
        case PR_E_ISO_W: m = "E_iso_w must be finite and > 0"; break;
        case PR_GAMMA0_W: m = "Gamma0_w must be > 1"; break;
        case PR_THETA_W: m = "theta_w must be in (0, pi/2]"; break;
        case PR_THETA_W_ORDER:
            return fail(VAG_ERR_INVALID, "theta_w (wing angle) must be greater than theta_c (core angle), got theta_w=" +
                                             std::to_string(p->theta_w) + ", theta_c=" + std::to_string(p->theta_c));
        case PR_SIGMA0: m = "sigma0 must be finite and >= 0"; break;
        case PR_MAG_L0: m = "L0 must be finite and > 0"; break;
        case PR_MAG_T0: m = "t0 must be finite and > 0"; break;
        case PR_MAG_Q: m = "q must be finite and > 0"; break;
        case PR_MAG_WING: m = "PowerLawWing takes no magnetar (pybind/pybind.cpp:220-223)"; break;
        case PR_N_ISM: m = "n_ism must be finite and >= 0"; break;
        case PR_A_STAR: m = "A_star must be finite and > 0"; break;
        case PR_N0: m = "n0 must be > 0 (or +inf for no floor)"; break;
        case PR_K_M: m = "k_m must be finite and > 0"; break;
        case PR_LUMI_DIST: m = "lumi_dist must be finite and > 0"; break;
        case PR_Z: m = "z must be finite and >= 0"; break;
        case PR_THETA_OBS: m = "theta_obs must be in [0, pi]"; break;
        case PR_PHI_OBS: m = "phi_obs must be finite"; break;
        case PR_RTOL: m = "rtol must be in (0, 1)"; break;
        case PR_NONFINITE_RES: m = "resolutions and rtol must be finite"; break;
        default:  // PyRadiation: PR_FWD_* / PR_RVS_*
            return fail(VAG_ERR_INVALID, std::string(r < PR_RVS_EPS_E ? "fwd_rad." : "rvs_rad.") +
                                             rad[(r - PR_FWD_EPS_E) % 4]);
    }
    return fail(VAG_ERR_INVALID, m);
}

int vag_create(int device, vag_context** out) {
    if (!out) return fail(VAG_ERR_INVALID, "out is NULL");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(VAG_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count = 0"));
    if (device < 0 || device >= count) return fail(VAG_ERR_INVALID, "device index out of range");
    CK(cudaSetDevice(device));
    vag_context* c = new vag_context();
    c->device = device;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CK(cudaMallocHost(&c->h_totals, sizeof(int) * TOT_N));
    CK(cudaMallocHost(&c->h_cells, sizeof(long long)));
    CK(cudaMallocHost(&c->h_bands, 2 * sizeof(int)));
    for (auto& ev : c->ev) CK(cudaEventCreate(&ev));
    {
        std::vector<double> lut(SPL_DOUBLES);
        build_softplus_lut(lut.data());
        CK(c->sp_buf.ensure(sizeof(double) * SPL_DOUBLES));
        CK(cudaMemcpy(c->sp_buf.p, lut.data(), sizeof(double) * SPL_DOUBLES, cudaMemcpyHostToDevice));
    }
    {
        // node sequences of find_theta_range (vag_grid.cuh ThetaWalk): plain IEEE running sums, identical on host and
        // device; uploaded once per device
        static std::mutex mu;
        static bool done[256] = {};
        std::lock_guard<std::mutex> lk(mu);
        if (device < 256 && !done[device]) {
            ThetaWalk tw;
            build_theta_walk(tw);
            CK(cudaMemcpyToSymbol(g_theta_walk, &tw, sizeof(tw)));
            done[device] = true;
        }
    }
    // k_grid spills its scratch to local memory: prefer L1.  k_dynamics keeps its dopri5 stage vectors
    // in shared memory (23 KB per 32-row CTA): give it the full carve-out so several CTAs share an SM.
    for (bool ragged : {false, true})
        for (int lanes : GRID_LANES) cudaFuncSetCacheConfig(grid_kernel(lanes, ragged), cudaFuncCachePreferL1);
    cudaFuncSetAttribute(k_dynamics<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    // per-function process state: set once, to the largest request run_flux can make (not per call, where two contexts
    // with different request shapes would race on it)
    for (bool ragged : {false, true})
        for (int mode = 0; mode < EATS_MODES; ++mode)
            for (int kind = 0; kind < EATS_KINDS; ++kind)
                CK(cudaFuncSetAttribute(eats_kernel(mode, kind, ragged), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)EATS_SMEM_BUDGET));
    CK(cudaFuncSetAttribute(k_quantiles, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QUANT_SMEM_BUDGET));
    {
        int blocks = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, k_ic_spectrum<false>, 128, 0) == cudaSuccess && blocks > 0)
            c->ic_warps_per_sm = std::min(blocks, 8) * 4;
    }
    *out = c;
    return VAG_OK;
}

void vag_destroy(vag_context* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->h_totals) cudaFreeHost(c->h_totals);
    if (c->h_cells) cudaFreeHost(c->h_cells);
    if (c->h_bands) cudaFreeHost(c->h_bands);
    if (c->h_plan) cudaFreeHost(c->h_plan);
    for (auto& ev : c->ev)
        if (ev) cudaEventDestroy(ev);
    cudaStreamDestroy(c->stream);
    delete c;  // frees the DevBufs
}

int vag_set_profiling(vag_context* ctx, int enable) {
    ctx->profiling = enable != 0;
    return VAG_OK;
}
int vag_last_stage_ms(vag_context* ctx, float ms[8]) {
    for (int i = 0; i < 8; ++i) ms[i] = ctx->stage_ms[i];
    return VAG_OK;
}
int vag_last_launch_count(vag_context* ctx) { return ctx->launches; }
int vag_last_work(vag_context* ctx, double work[8]) {
    for (int i = 0; i < 8; ++i) work[i] = ctx->work[i];
    return VAG_OK;
}
int vag_synchronize(vag_context* ctx) {
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return VAG_OK;
}
int vag_set_output_mode(vag_context* ctx, int mode) {
    if (mode != VAG_OUT_DENSE && mode != VAG_OUT_PRESENT && mode != VAG_OUT_PRESENT_ALIAS_TOTAL)
        return fail(VAG_ERR_INVALID, "unknown output mode");
    ctx->out_mode = mode;
    return VAG_OK;
}
int vag_last_total_alias(vag_context* ctx) { return ctx ? ctx->total_alias : -1; }
int vag_set_series_mode(vag_context* ctx, int mode) {
    if (mode < 0 || mode > 2) return fail(VAG_ERR_INVALID, "unknown series mode");
    ctx->series_mode = mode;
    return VAG_OK;
}
int vag_set_grid_lanes(vag_context* ctx, int lanes) {
    if (lanes != 0 && lanes != 4 && lanes != 8 && lanes != 16 && lanes != 32)
        return fail(VAG_ERR_INVALID, "grid lanes must be 0, 4, 8, 16 or 32");
    ctx->grid_lanes = lanes;
    return VAG_OK;
}
int vag_set_capacity(vag_context* ctx, int cap_theta, int cap_phi) {
    if (cap_theta < 40 || cap_phi < 2) return fail(VAG_ERR_INVALID, "capacity too small");
    ctx->cap_theta = cap_theta;
    ctx->cap_phi = cap_phi;
    return VAG_OK;
}

int vag_debug_set_ode_limits(vag_context* ctx, int max_steps, int max_fails) {
    if (!ctx) return fail(VAG_ERR_INVALID, "ctx is NULL");
    ctx->dbg_max_ode_steps = max_steps > 0 ? max_steps : 0;
    ctx->dbg_max_ode_fails = max_fails > 0 ? max_fails : 0;
    return VAG_OK;
}

int vag_measure_fp64_peak(vag_context* ctx, double* tflops) {
    CK(cudaSetDevice(ctx->device));
    CK(ctx->io_out.ensure(64));
    const int iters = 1 << 16, blocks = ctx->sm_count * 8, threads = 256;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(a, ctx->stream));
        k_fp64_peak<<<blocks, threads, 0, ctx->stream>>>(static_cast<double*>(ctx->io_out.p), iters);
        CK(cudaEventRecord(b, ctx->stream));
        CK(cudaEventSynchronize(b));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, a, b));
        const double fl = 2.0 * 8 * (double)iters * blocks * threads;
        best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    *tflops = best;
    return VAG_OK;
}

int vag_selftest_libm(vag_context* ctx, int fn, const double* x, const double* y, double* out, size_t n) {
    if (fn < 0 || fn > 7) return fail(VAG_ERR_INVALID, "vag_selftest_libm: fn must be 0..7");
    if ((fn == 5) != (y != nullptr)) return fail(VAG_ERR_INVALID, "vag_selftest_libm: y is required for pow only");
    if (n == 0) return VAG_OK;
    CK(cudaSetDevice(ctx->device));
    CK(ctx->io_out.ensure(3 * n * sizeof(double)));
    double* d_x = static_cast<double*>(ctx->io_out.p);
    double* d_y = d_x + n;
    double* d_o = d_y + n;
    CK(cudaMemcpyAsync(d_x, x, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if (y) CK(cudaMemcpyAsync(d_y, y, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    k_libm_selftest<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(fn, d_x, y ? d_y : nullptr, d_o, n);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d_o, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return VAG_OK;
}

// ---- preparation of the host-buffer entry points ------------------------------------------------------
// validates the parameter sets and uploads them; *caps: the capacities their grids need
static int prepare_params(vag_context* ctx, const vag_params* params, size_t n_models, Caps* caps) {
    if (!ctx) return fail(VAG_ERR_INVALID, "ctx is NULL");
    if (!params && n_models) return fail(VAG_ERR_INVALID, "params is NULL");
    for (size_t i = 0; i < n_models; ++i)
        if (int rc = vag_params_validate(&params[i])) return rc;
    CK(cudaSetDevice(ctx->device));
    *caps = caps_for(params, n_models);
    CK(ctx->io_params.ensure(sizeof(vag_params) * std::max<size_t>(n_models, 1)));
    CK(ctx->io_status.ensure(sizeof(int32_t) * std::max<size_t>(n_models, 1)));
    CK(cudaMemcpyAsync(ctx->io_params.p, params, sizeof(vag_params) * n_models, cudaMemcpyHostToDevice, ctx->stream));
    return VAG_OK;
}

// log10(t_end / t_start) sizes the time lattice: a zero, negative or non-finite epoch has no meaning
static int check_times(const double* t, size_t n_t) {
    if (n_t == 0 || !t) return fail(VAG_ERR_INVALID, "time array must be non-empty");
    for (size_t i = 1; i < n_t; ++i)  // is_ascending, pybind/pybind.h:28
        if (!(t[i - 1] <= t[i])) return fail(VAG_ERR_INVALID, "time array must be in ascending order");
    for (size_t i = 0; i < n_t; ++i)
        if (!finite_pos(t[i])) return fail(VAG_ERR_INVALID, "observation times must be finite and > 0");
    return VAG_OK;
}

// times -> io_t, checked by the caller
static int upload_times(vag_context* ctx, const double* t, size_t n_t) {
    CK(ctx->io_t.ensure(sizeof(double) * n_t));
    CK(cudaMemcpyAsync(ctx->io_t.p, t, sizeof(double) * n_t, cudaMemcpyHostToDevice, ctx->stream));
    return VAG_OK;
}

// times -> io_t, frequencies -> io_nu, checked by the caller
static int upload_request(vag_context* ctx, const double* t, size_t n_t, const double* nu, size_t n_nu) {
    if (int rc = upload_times(ctx, t, n_t)) return rc;
    CK(ctx->io_nu.ensure(sizeof(double) * n_nu));
    CK(cudaMemcpyAsync(ctx->io_nu.p, nu, sizeof(double) * n_nu, cudaMemcpyHostToDevice, ctx->stream));
    return VAG_OK;
}

static int prepare_request(vag_context* ctx, const double* t, size_t n_t, const double* nu, size_t n_nu) {
    if (int rc = check_times(t, n_t)) return rc;
    if (n_nu == 0 || !nu) return fail(VAG_ERR_INVALID, "frequency array must be non-empty");
    for (size_t i = 0; i < n_nu; ++i)
        if (!finite_pos(nu[i])) return fail(VAG_ERR_INVALID, "observation frequencies must be finite and > 0");
    return upload_request(ctx, t, n_t, nu, n_nu);
}

// ---- device-buffer entry points ----------------------------------------------------------------
// makes the context's device current and picks the stream of a _dev call: the caller's, or the context's when NULL
static int dev_stream(vag_context* ctx, void* stream, cudaStream_t* s) {
    CK(cudaSetDevice(ctx->device));
    *s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return VAG_OK;
}

// the caller's buffers and stream, the capacities of vag_set_capacity; with d_chi2 the series flux is scratch
static int flux_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const Request& rq, double* d_out,
                    int32_t* d_status, double* d_chi2, void* stream) {
    if (!ctx) return fail(VAG_ERR_INVALID, "ctx is NULL");
    if (rq.n_t == 0) return fail(VAG_ERR_INVALID, "time array must be non-empty");
    if (rq.n_nu == 0) return fail(VAG_ERR_INVALID, "frequency array must be non-empty");
    cudaStream_t s;
    if (int rc = dev_stream(ctx, stream, &s)) return rc;
    if (d_chi2) {
        CK(ctx->io_out.ensure(sizeof(double) * n_models * VAG_NCOMP * rq.n_t));
        d_out = static_cast<double*>(ctx->io_out.p);
    }
    return run_flux(ctx, d_params, n_models, Caps{ctx->cap_theta, ctx->cap_phi}, rq, d_out, d_status, d_chi2, s);
}

int vag_flux_density_grid_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t,
                              size_t n_t, const double* d_nu, size_t n_nu, double* d_out, int32_t* d_status,
                              void* stream) {
    return flux_dev(ctx, d_params, n_models, Request{false, d_t, d_nu, n_t, n_nu}, d_out, d_status, nullptr, stream);
}

int vag_flux_density_series_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t,
                                const double* d_nu, size_t n, double* d_out, int32_t* d_status, void* stream) {
    return flux_dev(ctx, d_params, n_models, Request{true, d_t, d_nu, n, n}, d_out, d_status, nullptr, stream);
}

int vag_chi2_series_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t,
                        const double* d_nu, const double* d_lnF_obs, const double* d_sigma_ln, const double* d_w,
                        size_t n, double* d_chi2, int32_t* d_status, void* stream) {
    Request rq{true, d_t, d_nu, n, n};
    rq.d_lnF = d_lnF_obs;
    rq.d_sig = d_sigma_ln;
    rq.d_w = d_w;
    return flux_dev(ctx, d_params, n_models, rq, nullptr, d_status, d_chi2, stream);
}

// ---- host-buffer entry points --------------------------------------------------------------------
// device -> host transfer of out[n_models][VAG_NCOMP][comp_sz] from src (NULL: io_out) under the context's output mode
static int copy_out(vag_context* ctx, const vag_params* params, size_t n_models, size_t comp_sz, double* out,
                    cudaStream_t s, const double* src_dev = nullptr) {
    if (!src_dev) src_dev = static_cast<const double*>(ctx->io_out.p);
    const size_t row = sizeof(double) * comp_sz, pitch = row * VAG_NCOMP;
    if (ctx->out_mode == VAG_OUT_DENSE) {
        CK(cudaMemcpyAsync(out, src_dev, pitch * n_models, cudaMemcpyDeviceToHost, s));
        return VAG_OK;
    }
    bool present[VAG_NCOMP] = {true, true, false, false, false};
    for (size_t i = 0; i < n_models; ++i) {
        if (params[i].fwd.ssc) present[VAG_C_FWD_SSC] = true;
        if (params[i].has_rvs) {
            present[VAG_C_RVS_SYNC] = true;
            if (params[i].rvs.ssc) present[VAG_C_RVS_SSC] = true;
        }
    }
    // exactly one emission component in the whole batch: `total` is that component, bit for bit -- do not ship it twice
    ctx->total_alias = -1;
    if (ctx->out_mode == VAG_OUT_PRESENT_ALIAS_TOTAL) {
        int n_present = 0, which = -1;
        for (int c = 1; c < VAG_NCOMP; ++c)
            if (present[c]) {
                ++n_present;
                which = c;
            }
        if (n_present == 1) {
            present[VAG_C_TOTAL] = false;
            ctx->total_alias = which;
        }
    }
    const char* src = reinterpret_cast<const char*>(src_dev);
    char* dst = reinterpret_cast<char*>(out);
    for (int c = 0; c < VAG_NCOMP;) {
        if (!present[c]) {
            ++c;
            continue;
        }
        int c1 = c;
        while (c1 + 1 < VAG_NCOMP && present[c1 + 1]) ++c1;  // adjacent present planes travel together
        CK(cudaMemcpy2DAsync(dst + row * c, pitch, src + row * c, pitch, row * (c1 - c + 1), n_models,
                             cudaMemcpyDeviceToHost, s));
        c = c1 + 1;
    }
    return VAG_OK;
}

static int flux_host(vag_context* ctx, const vag_params* params, size_t n_models, bool series, const double* t,
                     size_t n_t, const double* nu, size_t n_nu, double* out, int32_t* status) {
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (int rc = prepare_request(ctx, t, n_t, nu, n_nu)) return rc;
    if (n_models == 0) return VAG_OK;
    const size_t comp_sz = series ? n_t : n_nu * n_t;
    CK(ctx->io_out.ensure(sizeof(double) * n_models * VAG_NCOMP * comp_sz));
    cudaStream_t s = ctx->stream;
    const Request rq{series, static_cast<double*>(ctx->io_t.p), static_cast<double*>(ctx->io_nu.p), n_t, n_nu};
    if (int rc = run_flux(ctx, static_cast<vag_params*>(ctx->io_params.p), n_models, caps, rq,
                          static_cast<double*>(ctx->io_out.p), static_cast<int32_t*>(ctx->io_status.p), nullptr, s))
        return rc;
    if (int rc = copy_out(ctx, params, n_models, comp_sz, out, s)) return rc;
    if (status) CK(cudaMemcpyAsync(status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

int vag_flux_density_grid(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, size_t n_t,
                          const double* nu, size_t n_nu, double* out, int32_t* status) {
    return flux_host(ctx, params, n_models, false, t, n_t, nu, n_nu, out, status);
}

int vag_flux_density_series(vag_context* ctx, const vag_params* params, size_t n_models, const double* t,
                            const double* nu, size_t n, double* out, int32_t* status) {
    return flux_host(ctx, params, n_models, true, t, n, nu, n, out, status);
}

// Model.flux_density_exposures (pybind/pymodel.cpp:412-496): the samples of every point (vag_exposure.cuh) as one
// shared series request, then k_expo_average; only the averages cross PCIe.  Checks first, in the mirror's order.
int vag_flux_density_exposures(vag_context* ctx, const vag_params* params, size_t n_models, const double* t,
                               const double* nu, const double* expo_time, size_t n, size_t num_points, double* out,
                               int32_t* status) {
    if (!ctx || !out || (n && (!t || !nu || !expo_time))) return fail(VAG_ERR_INVALID, "NULL argument");
    if (num_points < 2) return fail(VAG_ERR_INVALID, "num_points must be at least 2 to sample within each exposure time");
    for (size_t i = 0; i < n; ++i)
        if (!(std::isfinite(expo_time[i]) && expo_time[i] > 0))
            return fail(VAG_ERR_INVALID, "expo_time[" + std::to_string(i) + "] must be finite and > 0, got " +
                                             std::to_string(expo_time[i]));
    if (n == 0) return fail(VAG_ERR_INVALID, "time array must be non-empty");
    if (num_points > (size_t)INT_MAX / n) return fail(VAG_ERR_INVALID, "n * num_points samples must fit in a 32-bit int");
    for (size_t i = 0; i < n; ++i)
        if (!finite_pos(t[i])) return fail(VAG_ERR_INVALID, "observation times must be finite and > 0");
    for (size_t i = 0; i < n; ++i)
        if (!finite_pos(nu[i])) return fail(VAG_ERR_INVALID, "observation frequencies must be finite and > 0");
    ExpoPlan P;
    expo_plan_append(t, nu, expo_time, n, (int)num_points, P);
    const size_t n_s = P.t.size();
    if (int rc = check_times(P.t.data(), n_s)) return rc;  // a sample time that overflowed
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (n_models == 0) return VAG_OK;
    cudaStream_t s = ctx->stream;
    if (int rc = upload_request(ctx, P.t.data(), n_s, P.nu.data(), n_s)) return rc;
    Pack pk;
    const size_t o_s0 = pk.put(P.s0), o_pos = pk.put(P.pos);
    CK(ctx->io_sets.ensure(pk.h.size()));
    CK(cudaMemcpyAsync(ctx->io_sets.p, pk.h.data(), pk.h.size(), cudaMemcpyHostToDevice, s));
    CK(ctx->io_out.ensure(sizeof(double) * n_models * VAG_NCOMP * (n_s + n)));
    double* d_samples = static_cast<double*>(ctx->io_out.p);
    double* d_avg = d_samples + n_models * VAG_NCOMP * n_s;
    const Request rq{true, static_cast<double*>(ctx->io_t.p), static_cast<double*>(ctx->io_nu.p), n_s, n_s};
    if (int rc = run_flux(ctx, static_cast<vag_params*>(ctx->io_params.p), n_models, caps, rq, d_samples,
                          static_cast<int32_t*>(ctx->io_status.p), nullptr, s))
        return rc;
    k_expo_average<false><<<(unsigned)n_models, 128, 0, s>>>(d_samples, (int)n_s, (int)n, at<int>(ctx->io_sets.p, o_s0),
                                                             at<int>(ctx->io_sets.p, o_pos), d_avg, SetsDev{}, SetsDev{});
    ctx->launches++;
    CK(cudaGetLastError());
    if (int rc = copy_out(ctx, params, n_models, n, out, s, d_avg)) return rc;
    if (status) CK(cudaMemcpyAsync(status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

// Frequency grid (code units) and quadrature weights of PyModel::flux (pybind/pymodel.cpp:391-410): xt::logspace of the
// unit-scaled bounds, Boole's rule in ln(nu) with 3/8 / Simpson / trapezoid remainders (src/core/quadrature.h:138-191),
// times the Jacobian nu and the code-unit -> Hz factor, so that sum_i F_nu[cgs](nu_i) w_i is erg cm^-2 s^-1.
struct BandGrid {
    std::vector<double> nu, wgt;
};

static int band_grid(double nu_min, double nu_max, size_t num_nu, BandGrid& g) {
    if (!(nu_min > 0) || !std::isfinite(nu_min)) return fail(VAG_ERR_INVALID, "nu_min must be positive");
    if (!(nu_max > nu_min) || !std::isfinite(nu_max)) return fail(VAG_ERR_INVALID, "nu_max must be greater than nu_min");
    if (num_nu < 2) return fail(VAG_ERR_INVALID, "num_nu must be at least 2");
    std::vector<double>& nu = g.nu;
    std::vector<double>& wgt = g.wgt;
    nu.assign(num_nu, 0.0);
    wgt.assign(num_nu, 0.0);
    const double a = std::log10(nu_min * unit::Hz), b = std::log10(nu_max * unit::Hz);
    const double step = (b - a) / std::fmax(1.0, (double)(num_nu - 1));
    for (size_t i = 0; i < num_nu; ++i) nu[i] = std::pow(10.0, (i == num_nu - 1) ? b : a + step * (double)i);
    const double h = std::log(nu[1] / nu[0]);
    const double cb = 2.0 * h / 45.0;
    size_t j = 0;
    for (; j + 4 < num_nu; j += 4) {
        wgt[j] += cb * 7;
        wgt[j + 1] += cb * 32;
        wgt[j + 2] += cb * 12;
        wgt[j + 3] += cb * 32;
        wgt[j + 4] += cb * 7;
    }
    const size_t remaining = num_nu - 1 - j;
    if (remaining == 3) {
        const double c38 = 3.0 * h / 8.0;
        wgt[j] += c38;
        wgt[j + 1] += c38 * 3;
        wgt[j + 2] += c38 * 3;
        wgt[j + 3] += c38;
    } else if (remaining == 2) {
        const double c13 = h / 3.0;
        wgt[j] += c13;
        wgt[j + 1] += c13 * 4;
        wgt[j + 2] += c13;
    } else if (remaining == 1) {
        wgt[j] += 0.5 * h;
        wgt[j + 1] += 0.5 * h;
    }
    for (size_t i = 0; i < num_nu; ++i) wgt[i] = wgt[i] * nu[i] / unit::Hz;
    return VAG_OK;
}

// Band-integrated flux of a batch whose parameters and times d_t are on the device: grid evaluation on the band's
// frequency nodes g.nu (uploaded to io_nu, the weights to io_w), then the weighted sum over frequency.
// *d_band -> [n_models][VAG_NCOMP][n_t] inside io_out.
static int run_band(vag_context* ctx, const vag_params* d_params, size_t n_models, Caps caps, const double* d_t, size_t n_t,
                    const BandGrid& g, int32_t* d_status, double** d_band, cudaStream_t s) {
    const size_t num_nu = g.nu.size();
    CK(ctx->io_nu.ensure(sizeof(double) * num_nu));
    CK(ctx->io_w.ensure(sizeof(double) * num_nu));
    const size_t grid_elems = n_models * VAG_NCOMP * num_nu * n_t;
    CK(ctx->io_out.ensure(sizeof(double) * (grid_elems + n_models * VAG_NCOMP * n_t)));
    CK(cudaMemcpyAsync(ctx->io_nu.p, g.nu.data(), sizeof(double) * num_nu, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ctx->io_w.p, g.wgt.data(), sizeof(double) * num_nu, cudaMemcpyHostToDevice, s));
    double* d_grid = static_cast<double*>(ctx->io_out.p);
    *d_band = d_grid + grid_elems;
    Request rq{false, d_t, static_cast<double*>(ctx->io_nu.p), n_t, num_nu, true};
    if (int rc = run_flux(ctx, d_params, n_models, caps, rq, d_grid, d_status, nullptr, s)) return rc;
    const size_t n_mc = n_models * VAG_NCOMP;
    k_band_reduce<<<(unsigned)((n_mc * n_t + 255) / 256), 256, 0, s>>>(d_grid, static_cast<double*>(ctx->io_w.p), *d_band,
                                                                     n_mc, (int)num_nu, (int)n_t);
    ctx->launches++;
    CK(cudaGetLastError());
    return VAG_OK;
}

// Replaces PyModel::flux (pybind/pymodel.cpp:391-410): band-integrated flux over [nu_min, nu_max]
int vag_flux_band(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, size_t n_t,
                  double nu_min, double nu_max, size_t num_nu, double* out, int32_t* status) {
    BandGrid g;
    if (int rc = band_grid(nu_min, nu_max, num_nu, g)) return rc;
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (int rc = check_times(t, n_t)) return rc;
    if (int rc = upload_times(ctx, t, n_t)) return rc;
    if (n_models == 0) return VAG_OK;
    cudaStream_t s = ctx->stream;
    double* d_band = nullptr;
    if (int rc = run_band(ctx, static_cast<vag_params*>(ctx->io_params.p), n_models, caps, static_cast<double*>(ctx->io_t.p),
                          n_t, g, static_cast<int32_t*>(ctx->io_status.p), &d_band, s))
        return rc;
    CK(cudaMemcpyAsync(out, d_band, sizeof(double) * n_models * VAG_NCOMP * n_t, cudaMemcpyDeviceToHost, s));
    if (status) CK(cudaMemcpyAsync(status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

// The likelihood's data on the device: the point series (n == 0: none; ext / av both set or both NULL) and the bands
struct Chi2Points {
    const double *t, *nu, *lnF, *sig, *w, *ext, *av;
    size_t n;
};
struct BandTerm {
    const double *t, *lnF, *sig, *w;
    size_t n;
    const BandGrid* g;
};

// The series request of pts (lnF ... av NULL: the flux alone); with sd a ragged one on the n_sets data sets of sd, the
// largest of max_set points, whose models' output points have the host prefix sums h_off
static Request points_request(const Chi2Points& pts, const SetsDev* sd = nullptr, const long long* h_off = nullptr,
                              size_t n_sets = 0, size_t max_set = 0) {
    Request rq{true, pts.t, pts.nu, pts.n, pts.n};
    rq.d_lnF = pts.lnF;
    rq.d_sig = pts.sig;
    rq.d_w = pts.w;
    rq.d_ext = pts.ext;
    rq.d_av = pts.av;
    rq.sets = sd;
    rq.h_off = h_off;
    rq.n_sets = (int)n_sets;
    rq.max_set = max_set;
    return rq;
}

// chi2[n] of a batch whose parameters and data are on the device: the point term (k_chi2 inside run_flux writes chi2),
// then per band Model.flux and an accumulating k_chi2.  The status of every run goes to io_status; with band terms it is
// ORed into d_stat_or, which is then the call's status.  ctx->launches counts every launch of the call.
static int chi2_run(vag_context* ctx, const vag_params* d_params, size_t n_models, Caps caps, const Chi2Points& pts,
                    const BandTerm* bands, size_t n_bands, double* d_chi2, int32_t* d_stat_or, cudaStream_t s) {
    int32_t* d_status = static_cast<int32_t*>(ctx->io_status.p);
    const bool or_status = n_bands > 0;
    const unsigned og = (unsigned)((n_models + 255) / 256), cg = (unsigned)((n_models * 32 + 127) / 128);
    if (or_status) CK(cudaMemsetAsync(d_stat_or, 0, sizeof(int32_t) * n_models, s));
    int launches = 0;
    if (pts.n) {  // the first term: run_flux writes chi2
        CK(ctx->io_out.ensure(sizeof(double) * n_models * VAG_NCOMP * pts.n));
        if (int rc = run_flux(ctx, d_params, n_models, caps, points_request(pts), static_cast<double*>(ctx->io_out.p), d_status,
                              d_chi2, s))
            return rc;
        launches += ctx->launches;
        if (or_status) {
            k_or_status<<<og, 256, 0, s>>>(d_stat_or, d_status, n_models);
            launches++;
        }
    } else {
        CK(cudaMemsetAsync(d_chi2, 0, sizeof(double) * n_models, s));
    }
    for (size_t b = 0; b < n_bands; ++b) {
        const BandTerm& B = bands[b];
        double* d_band = nullptr;
        if (int rc = run_band(ctx, d_params, n_models, caps, B.t, B.n, *B.g, d_status, &d_band, s)) return rc;
        k_chi2<false><<<cg, 128, 0, s>>>(d_band, n_models, (int)B.n, B.lnF, B.sig, B.w, nullptr, nullptr, d_chi2, d_status, 1,
                                         SetsDev{});
        k_or_status<<<og, 256, 0, s>>>(d_stat_or, d_status, n_models);
        launches += ctx->launches + 2;
    }
    ctx->launches = launches;
    CK(cudaGetLastError());
    return VAG_OK;
}

// The rules of every chi-squared entry point for point data and fitted extinction (before any work is enqueued): with
// points all their arrays are set (`arrays`), ext_k and A_V are both set or both NULL, extinction needs points, and ext_k
// in host memory (!device) is finite
static int check_points(size_t n_points, bool arrays, const double* ext_k, const double* A_V, bool device) {
    if (n_points && !arrays) return fail(VAG_ERR_INVALID, "point data arrays must not be NULL when there are points");
    if ((ext_k != nullptr) != (A_V != nullptr)) return fail(VAG_ERR_INVALID, "ext_k and A_V must both be NULL or both be set");
    if (ext_k && n_points == 0) return fail(VAG_ERR_INVALID, "extinction needs point data (no points)");
    for (size_t i = 0; ext_k && !device && i < n_points; ++i)
        if (!std::isfinite(ext_k[i])) return fail(VAG_ERR_INVALID, "extinction coefficients ext_k must be finite");
    return VAG_OK;
}

// The checks of one band (data: lnF_obs / sigma_ln / w too) and its frequency grid; with `device` its arrays are device
// memory, whose values are not read (only t != NULL is checked)
static int check_band(const vag_band_obs& B, size_t b, bool data, BandGrid& g, bool device) {
    const std::string name = "band " + std::to_string(b) + ": ";
    if (B.n == 0) return fail(VAG_ERR_INVALID, name + "empty (n = 0)");
    if (data && (!B.lnF_obs || !B.sigma_ln || !B.w)) return fail(VAG_ERR_INVALID, name + "data arrays must not be NULL");
    if (device) {
        if (!B.t) return fail(VAG_ERR_INVALID, name + "time array must not be NULL");
    } else if (check_times(B.t, B.n)) {
        return fail(VAG_ERR_INVALID, name + g_err);
    }
    if (band_grid(B.nu_min, B.nu_max, B.num_nu, g)) return fail(VAG_ERR_INVALID, name + g_err);
    return VAG_OK;
}

// The checks of vag_chi2_ext and vag_chi2_dev, all before any work is enqueued: the arguments, the point data and
// extinction, and every band with its grid; with `device` the data are device memory, whose values are not read
static int check_chi2_args(vag_context* ctx, const double* chi2, size_t n_points, bool point_ptrs, const double* ext_k,
                           const double* A_V, const vag_band_obs* bands, size_t n_bands, bool device,
                           std::vector<BandGrid>& grids) {
    if (!ctx || !chi2) return fail(VAG_ERR_INVALID, "NULL argument");
    if (n_bands && !bands) return fail(VAG_ERR_INVALID, "bands is NULL");
    if (n_points == 0 && n_bands == 0) return fail(VAG_ERR_INVALID, "no data: n_points and n_bands are both 0");
    if (int rc = check_points(n_points, point_ptrs, ext_k, A_V, device)) return rc;
    grids.resize(n_bands);
    for (size_t b = 0; b < n_bands; ++b)
        if (int rc = check_band(bands[b], b, true, grids[b], device)) return rc;
    return VAG_OK;
}

// Replaces Fitter._evaluate (VegasAfterglow/fitting/fitter.py:503-533) for a batch of parameter sets: the chi-squared of the
// point data (flux_density series) plus one term per band-integrated data set (Model.flux), all in ln-flux space.
// With ext_k / A_V, the observed ln-flux of point i for model m is lnF_obs[i] + A_V[m] ext_k[i] (host extinction).
int vag_chi2_ext(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, const double* nu,
                 const double* lnF_obs, const double* sigma_ln, const double* w, const double* ext_k, size_t n_points,
                 const double* A_V, const vag_band_obs* bands, size_t n_bands, double* chi2, int32_t* status) {
    std::vector<BandGrid> grids;
    if (int rc = check_chi2_args(ctx, chi2, n_points, t && nu && lnF_obs && sigma_ln && w, ext_k, A_V, bands, n_bands, false,
                                 grids))
        return rc;
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (n_points)
        if (int rc = prepare_request(ctx, t, n_points, nu, n_points)) return rc;
    if (n_models == 0) return VAG_OK;
    cudaStream_t s = ctx->stream;
    // one upload: lnF / sigma_ln / w of the points (with extinction ext_k [n_points] and A_V [n_models]) and t / lnF /
    // sigma_ln / w of every band; then room for chi2 and the status OR [n_models]
    const size_t n_ext = ext_k ? n_points : 0;
    Pack pk;
    const size_t o_lnF = pk.put(lnF_obs, n_points), o_sig = pk.put(sigma_ln, n_points), o_w = pk.put(w, n_points),
                 o_ext = pk.put(ext_k, n_ext), o_av = pk.put(A_V, n_ext ? n_models : 0);
    std::vector<size_t> o_band;  // [n_bands][4]
    for (size_t b = 0; b < n_bands; ++b)
        for (const double* a : {bands[b].t, bands[b].lnF_obs, bands[b].sigma_ln, bands[b].w}) o_band.push_back(pk.put(a, bands[b].n));
    const size_t up = pk.h.size(), o_or = up + carve_sz<double>(n_models);
    CK(ctx->io_sets.ensure(o_or + carve_sz<int32_t>(n_models)));
    void* base = ctx->io_sets.p;
    CK(cudaMemcpyAsync(base, pk.h.data(), up, cudaMemcpyHostToDevice, s));
    Chi2Points pts{};
    if (n_points)
        pts = Chi2Points{static_cast<double*>(ctx->io_t.p), static_cast<double*>(ctx->io_nu.p), at<double>(base, o_lnF),
                         at<double>(base, o_sig), at<double>(base, o_w), n_ext ? at<double>(base, o_ext) : nullptr,
                         n_ext ? at<double>(base, o_av) : nullptr, n_points};
    std::vector<BandTerm> terms(n_bands);
    for (size_t b = 0; b < n_bands; ++b) {
        const size_t* o = &o_band[4 * b];
        terms[b] = BandTerm{at<double>(base, o[0]), at<double>(base, o[1]), at<double>(base, o[2]), at<double>(base, o[3]),
                            bands[b].n, &grids[b]};
    }
    double* d_chi2 = at<double>(base, up);
    int32_t* d_stat_or = at<int32_t>(base, o_or);
    if (int rc = chi2_run(ctx, static_cast<vag_params*>(ctx->io_params.p), n_models, caps, pts, terms.data(), n_bands, d_chi2,
                          d_stat_or, s))
        return rc;
    CK(cudaMemcpyAsync(chi2, d_chi2, sizeof(double) * n_models, cudaMemcpyDeviceToHost, s));
    if (status)
        CK(cudaMemcpyAsync(status, n_bands ? d_stat_or : ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost,
                           s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

int vag_chi2(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, const double* nu,
             const double* lnF_obs, const double* sigma_ln, const double* w, size_t n_points, const vag_band_obs* bands,
             size_t n_bands, double* chi2, int32_t* status) {
    return vag_chi2_ext(ctx, params, n_models, t, nu, lnF_obs, sigma_ln, w, nullptr, n_points, nullptr, bands, n_bands,
                        chi2, status);
}

// per-parameter-set validation of a batch: ok[i] = 1 where vag_params_validate accepts params[i] (a sampler masks the
// rejected walkers to logL = -inf the way the reference maps the constructor's exception, samplers.py:63-70)
int vag_params_validate_batch(const vag_params* params, size_t n, int32_t* ok) {
    if ((!params || !ok) && n) return fail(VAG_ERR_INVALID, "NULL argument");
    for (size_t i = 0; i < n; ++i) ok[i] = vag_params_validate(&params[i]) == VAG_OK ? 1 : 0;
    return VAG_OK;
}

int vag_chi2_series(vag_context* ctx, const vag_params* params, size_t n_models, const double* t, const double* nu,
                    const double* lnF_obs, const double* sigma_ln, const double* w, size_t n, double* chi2,
                    int32_t* status) {
    return vag_chi2(ctx, params, n_models, t, nu, lnF_obs, sigma_ln, w, n, nullptr, 0, chi2, status);
}

// ---- ragged series requests: several data sets in one batch --------------------------------------------------------
extern "C++" {  // a template over the set type
static size_t band0_of(const vag_series_set&) { return 0; }
static size_t band0_of(const vag_multi_set& S) { return S.band0; }
static size_t n_bands_of(const vag_series_set&) { return 0; }
static size_t n_bands_of(const vag_multi_set& S) { return S.n_bands; }

// The checks of the ragged calls that concern the data sets (before any work is enqueued): a vag_series_set is the
// vag_multi_set of its points and no band.  With `device` the points are device memory, whose values are not read.  The
// number of models is not limited here: the calls with bands bound it through check_multi_count.
template <class Set>
static int check_multi_sets(size_t n_models, const int32_t* dataset_of, const Set* sets, size_t n_sets, const double* t,
                            const double* nu, size_t n_points, size_t n_bands, bool device = false) {
    if (!sets || n_sets == 0) return fail(VAG_ERR_INVALID, "no data sets: sets is NULL or n_sets is 0");
    if (n_points > (size_t)INT_MAX || n_sets > (size_t)INT_MAX)
        return fail(VAG_ERR_INVALID, "n_points_total and n_sets must fit in a 32-bit int");
    if (n_models && !dataset_of) return fail(VAG_ERR_INVALID, "dataset_of is NULL");
    for (size_t d = 0; d < n_sets; ++d) {
        const std::string name = "data set " + std::to_string(d) + ": ";
        const Set& S = sets[d];
        const size_t band0 = band0_of(S), nb = n_bands_of(S);
        if (S.n == 0 && nb == 0) return fail(VAG_ERR_INVALID, name + "no data: empty (n = 0 and n_bands = 0)");
        if (S.offset > n_points || S.n > n_points - S.offset)
            return fail(VAG_ERR_INVALID, name + "points [" + std::to_string(S.offset) + ", " + std::to_string(S.offset) +
                                             " + " + std::to_string(S.n) + ") lie outside the " + std::to_string(n_points) +
                                             " points");
        if (band0 > n_bands || nb > n_bands - band0)
            return fail(VAG_ERR_INVALID, name + "bands [" + std::to_string(band0) + ", " + std::to_string(band0) + " + " +
                                             std::to_string(nb) + ") lie outside the " + std::to_string(n_bands) + " bands");
        if (S.n == 0 || device) continue;
        if (check_times(t + S.offset, S.n)) return fail(VAG_ERR_INVALID, name + g_err);
        for (size_t i = S.offset; i < S.offset + S.n; ++i)
            if (!finite_pos(nu[i])) return fail(VAG_ERR_INVALID, name + "observation frequencies must be finite and > 0");
    }
    for (size_t m = 0; m < n_models; ++m)
        if (dataset_of[m] < 0 || (size_t)dataset_of[m] >= n_sets)
            return fail(VAG_ERR_INVALID, "model " + std::to_string(m) + ": dataset_of = " + std::to_string(dataset_of[m]) +
                                             " is not a data set index (n_sets = " + std::to_string(n_sets) + ")");
    return VAG_OK;
}
}  // extern "C++"

// The series flux (out != NULL) or the chi-squared (chi2 != NULL) of a ragged request from host buffers, arguments checked
// by the caller: the concatenated points pts (with chi2 their lnF / sig / w [/ ext] and A_V per model in pts.av).  out:
// model m's [VAG_NCOMP][n of its set] block at m's offset, the prefix sum of the sizes of the data sets of models 0 .. m-1.
static int sets_host(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                     const vag_series_set* sets, size_t n_sets, const Chi2Points& pts, double* out, double* chi2,
                     int32_t* status) {
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (n_models == 0) return VAG_OK;
    std::vector<SeriesSet> hs(n_sets);
    size_t max_set = 0;
    for (size_t d = 0; d < n_sets; ++d) {
        hs[d] = SeriesSet{(int)sets[d].offset, (int)sets[d].n, 0, 0};
        max_set = std::max(max_set, sets[d].n);
    }
    std::vector<long long> off(n_models + 1, 0);
    for (size_t m = 0; m < n_models; ++m) off[m + 1] = off[m] + (long long)sets[dataset_of[m]].n;
    const size_t n_out = (size_t)off[n_models] * VAG_NCOMP;
    cudaStream_t s = ctx->stream;
    // one upload: the points (with chi2 their data), the tables; then room for chi2 [n_models]
    const size_t n = pts.n, n_data = chi2 ? n : 0, n_ext = chi2 && pts.ext ? n : 0;
    Pack pk;
    const size_t o_t = pk.put(pts.t, n), o_nu = pk.put(pts.nu, n), o_lnF = pk.put(pts.lnF, n_data),
                 o_sig = pk.put(pts.sig, n_data), o_w = pk.put(pts.w, n_data), o_ext = pk.put(pts.ext, n_ext),
                 o_av = pk.put(pts.av, n_ext ? n_models : 0), o_set_of = pk.put(dataset_of, n_models), o_sets = pk.put(hs),
                 o_off = pk.put(off), up = pk.h.size();
    CK(ctx->io_sets.ensure(up + carve_sz<double>(n_models)));
    void* base = ctx->io_sets.p;
    CK(cudaMemcpyAsync(base, pk.h.data(), up, cudaMemcpyHostToDevice, s));
    auto dev = [&](size_t o, size_t n_up) -> const double* { return n_up ? at<double>(base, o) : nullptr; };
    const Chi2Points d{at<double>(base, o_t), at<double>(base, o_nu), dev(o_lnF, n_data), dev(o_sig, n_data),
                       dev(o_w, n_data), dev(o_ext, n_ext), dev(o_av, n_ext), n};
    const SetsDev sd{at<int>(base, o_set_of), at<SeriesSet>(base, o_sets), at<long long>(base, o_off)};
    double* d_chi2 = chi2 ? at<double>(base, up) : nullptr;
    CK(ctx->io_out.ensure(sizeof(double) * std::max<size_t>(n_out, 1)));
    if (int rc = run_flux(ctx, static_cast<vag_params*>(ctx->io_params.p), n_models, caps,
                          points_request(d, &sd, off.data(), n_sets, max_set), static_cast<double*>(ctx->io_out.p),
                          static_cast<int32_t*>(ctx->io_status.p), d_chi2, s))
        return rc;
    if (out) CK(cudaMemcpyAsync(out, ctx->io_out.p, sizeof(double) * n_out, cudaMemcpyDeviceToHost, s));
    if (chi2) CK(cudaMemcpyAsync(chi2, d_chi2, sizeof(double) * n_models, cudaMemcpyDeviceToHost, s));
    if (status) CK(cudaMemcpyAsync(status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

int vag_flux_density_series_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                                  const vag_series_set* sets, size_t n_sets, const double* t, const double* nu,
                                  size_t n_points_total, double* out, int32_t* status) {
    if (!ctx || !out) return fail(VAG_ERR_INVALID, "NULL argument");
    if (int rc = check_points(n_points_total, t && nu, nullptr, nullptr, false)) return rc;
    if (int rc = check_multi_sets(n_models, dataset_of, sets, n_sets, t, nu, n_points_total, 0)) return rc;
    return sets_host(ctx, params, n_models, dataset_of, sets, n_sets,
                     Chi2Points{t, nu, nullptr, nullptr, nullptr, nullptr, nullptr, n_points_total}, out, nullptr, status);
}

int vag_chi2_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                   const vag_series_set* sets, size_t n_sets, const double* t, const double* nu, const double* lnF_obs,
                   const double* sigma_ln, const double* w, const double* ext_k, size_t n_points_total, const double* A_V,
                   double* chi2, int32_t* status) {
    if (!ctx || !chi2) return fail(VAG_ERR_INVALID, "NULL argument");
    if (int rc = check_points(n_points_total, t && nu && lnF_obs && sigma_ln && w, ext_k, A_V, false)) return rc;
    if (int rc = check_multi_sets(n_models, dataset_of, sets, n_sets, t, nu, n_points_total, 0)) return rc;
    return sets_host(ctx, params, n_models, dataset_of, sets, n_sets,
                     Chi2Points{t, nu, lnF_obs, sigma_ln, w, ext_k, A_V, n_points_total}, nullptr, chi2, status);
}

// ---- band-integrated data in a ragged batch ----------------------------------------------------------------------
// Every band checked, its grid built, and the concatenated times and nodes within a 32-bit int
static int check_bands(const vag_band_obs* bands, size_t n_bands, bool data, std::vector<BandGrid>& grids,
                       bool device = false) {
    grids.resize(n_bands);
    size_t n_t = 0, n_nu = 0;
    for (size_t b = 0; b < n_bands; ++b) {
        if (int rc = check_band(bands[b], b, data, grids[b], device)) return rc;
        n_t += bands[b].n;
        n_nu += bands[b].num_nu;
    }
    if (n_t > (size_t)INT_MAX || n_nu > (size_t)INT_MAX)
        return fail(VAG_ERR_INVALID, "the band times and frequency nodes of all bands must fit in a 32-bit int");
    return VAG_OK;
}

// vag_params_validate with the model named
static int check_models(const vag_params* params, size_t n_models) {
    if (!params && n_models) return fail(VAG_ERR_INVALID, "params is NULL");
    for (size_t m = 0; m < n_models; ++m)
        if (vag_params_validate(&params[m])) return fail(VAG_ERR_INVALID, "model " + std::to_string(m) + ": " + g_err);
    return VAG_OK;
}

// A ragged grid request: evaluation e (record e of the run) on set set_of[e] of `tab`, whose SeriesSet is its slice of
// the concatenated times and of the concatenated frequencies.  put() adds the set table, the evaluations' sets and their
// output offsets to the caller's one upload; bind() points the device table at that upload; run() evaluates them all as
// one request through run_flux (passes of 32768 evaluations), evaluation e's [VAG_NCOMP][n_nu][n] block at element
// VAG_NCOMP * off[e] of d_grid.  The band pass (quadrature nodes in code units) and vag_flux_density_grid_multi /
// vag_flux_quantiles_multi (frequencies in Hz) run through it.
struct GridSets {
    std::vector<long long> off;  // [n_eval + 1] first (time x frequency) point of each evaluation's block
    size_t n_sets = 0, max_n = 0, max_nu = 0, o_tab = 0, o_of = 0, o_off = 0;
    SetsDev sd{};
    void put(Pack& pk, const std::vector<SeriesSet>& tab, const int32_t* set_of, size_t n_eval) {
        n_sets = tab.size();
        off.assign(n_eval + 1, 0);
        for (size_t e = 0; e < n_eval; ++e) {
            const SeriesSet& S = tab[set_of[e]];
            off[e + 1] = off[e] + (long long)S.n * S.n_nu;
            max_n = std::max(max_n, (size_t)S.n);
            max_nu = std::max(max_nu, (size_t)S.n_nu);
        }
        o_tab = pk.put(tab);
        o_of = pk.put(set_of, n_eval);
        o_off = pk.put(off);
    }
    const SetsDev& bind(void* base) {
        sd = SetsDev{at<int>(base, o_of), at<SeriesSet>(base, o_tab), at<long long>(base, o_off)};
        return sd;
    }
    size_t elems() const { return (size_t)off.back() * VAG_NCOMP; }
    int run(vag_context* ctx, const vag_params* d_params, Caps caps, const double* d_t, size_t n_t, const double* d_nu,
            size_t n_nu, bool nu_code_units, double* d_grid, int32_t* d_status, cudaStream_t s) const {
        Request rq{false, d_t, d_nu, n_t, n_nu, nu_code_units};
        rq.sets = &sd;
        rq.h_off = off.data();
        rq.n_sets = (int)n_sets;
        rq.max_set = max_n;
        rq.max_nu = max_nu;
        return run_flux(ctx, d_params, off.size() - 1, caps, rq, d_grid, d_status, nullptr, s);
    }
};

// The band pass: evaluation e evaluates record e of d_params on band band_of[e], all as one ragged grid request
// (GridSets), then k_band_reduce_sets.  Times, frequency nodes (code units) and weights are
// concatenated over the bands, and with `data` lnF_obs / sigma_ln / w at the times' offsets.  Its tables go to io_bands,
// the grid and the band fluxes to io_out.  ctx->launches: run_flux's + 1.  With `device` (implies data) the bands' t /
// lnF_obs / sigma_ln / w are device pointers: the host uploads a table of them with the other tables, and k_gather_bands
// (one more launch) copies the arrays into the concatenated workspace behind that upload.
struct BandPass {
    SetsDev sd;                      // every evaluation: its band, the band table, its grid block's offset
    const long long* red_off;        // [n_eval + 1] first band-flux point of each evaluation
    const double *lnF, *sig, *w;     // with data
    double* red;                     // [VAG_NCOMP * h_red_off[n_eval]] band fluxes
    std::vector<long long> h_red_off;
};
static int band_pass(vag_context* ctx, const vag_params* d_params, size_t n_eval, Caps caps, const int32_t* band_of,
                     const vag_band_obs* bands, size_t n_bands, const std::vector<BandGrid>& grids, bool data,
                     int32_t* d_status, BandPass& bp, cudaStream_t s, bool device = false) {
    std::vector<SeriesSet> tab(n_bands);
    std::vector<double> t, nu, wgt, lnF, sig, w;
    std::vector<const double*> src;  // device: [n_bands][4] t, lnF_obs, sigma_ln, w
    size_t n_t = 0;
    for (size_t b = 0; b < n_bands; ++b) {
        const vag_band_obs& B = bands[b];
        const BandGrid& g = grids[b];
        tab[b] = SeriesSet{(int)n_t, (int)B.n, (int)g.nu.size(), (int)nu.size()};
        n_t += B.n;
        nu.insert(nu.end(), g.nu.begin(), g.nu.end());
        wgt.insert(wgt.end(), g.wgt.begin(), g.wgt.end());
        if (device) {
            src.insert(src.end(), {B.t, B.lnF_obs, B.sigma_ln, B.w});
            continue;
        }
        t.insert(t.end(), B.t, B.t + B.n);
        if (data) {
            lnF.insert(lnF.end(), B.lnF_obs, B.lnF_obs + B.n);
            sig.insert(sig.end(), B.sigma_ln, B.sigma_ln + B.n);
            w.insert(w.end(), B.w, B.w + B.n);
        }
    }
    bp.h_red_off.assign(n_eval + 1, 0);
    for (size_t e = 0; e < n_eval; ++e) bp.h_red_off[e + 1] = bp.h_red_off[e] + tab[band_of[e]].n;
    Pack pk;
    GridSets gs;
    const size_t o_t = pk.put(t), o_nu = pk.put(nu), o_wgt = pk.put(wgt);
    gs.put(pk, tab, band_of, n_eval);
    const size_t o_ro = pk.put(bp.h_red_off), o_lnF = pk.put(lnF), o_sig = pk.put(sig), o_w = pk.put(w), o_src = pk.put(src);
    const size_t up = pk.h.size(), plane = device ? carve_sz<double>(n_t) / sizeof(double) : 0;
    CK(ctx->io_bands.ensure(up + 4 * sizeof(double) * plane));
    void* base = ctx->io_bands.p;
    CK(cudaMemcpyAsync(base, pk.h.data(), up, cudaMemcpyHostToDevice, s));
    bp.sd = gs.bind(base);
    bp.red_off = at<long long>(base, o_ro);
    const double* d_t = at<double>(base, o_t);
    bp.lnF = data ? at<double>(base, o_lnF) : nullptr;
    bp.sig = data ? at<double>(base, o_sig) : nullptr;
    bp.w = data ? at<double>(base, o_w) : nullptr;
    if (device) {
        double* planes = at<double>(base, up);
        k_gather_bands<<<(unsigned)n_bands, 128, 0, s>>>(at<const double*>(base, o_src), bp.sd.sets, plane, planes);
        d_t = planes;
        bp.lnF = planes + plane;
        bp.sig = planes + 2 * plane;
        bp.w = planes + 3 * plane;
    }
    const size_t grid_elems = gs.elems(), red_elems = (size_t)bp.h_red_off[n_eval] * VAG_NCOMP;
    CK(ctx->io_out.ensure(sizeof(double) * (grid_elems + red_elems)));
    double* d_grid = static_cast<double*>(ctx->io_out.p);
    bp.red = d_grid + grid_elems;
    if (int rc = gs.run(ctx, d_params, caps, d_t, n_t, at<double>(base, o_nu), nu.size(), true, d_grid, d_status, s)) return rc;
    k_band_reduce_sets<<<(unsigned)n_eval, 128, 0, s>>>(d_grid, at<double>(base, o_wgt), bp.red, bp.red_off, bp.sd);
    ctx->launches += device ? 2 : 1;  // (k_gather_bands ran before run_flux, which restarts the count)
    CK(cudaGetLastError());
    return VAG_OK;
}

int vag_flux_band_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* band_of,
                        const vag_band_obs* bands, size_t n_bands, double* out, int32_t* status) {
    if (!ctx || !out) return fail(VAG_ERR_INVALID, "NULL argument");
    if (!bands || n_bands == 0) return fail(VAG_ERR_INVALID, "no bands: bands is NULL or n_bands is 0");
    if (n_models && !band_of) return fail(VAG_ERR_INVALID, "band_of is NULL");
    if (n_models > (size_t)INT_MAX) return fail(VAG_ERR_INVALID, "n_models must fit in a 32-bit int");
    std::vector<BandGrid> grids;
    if (int rc = check_bands(bands, n_bands, false, grids)) return rc;
    for (size_t m = 0; m < n_models; ++m)
        if (band_of[m] < 0 || (size_t)band_of[m] >= n_bands)
            return fail(VAG_ERR_INVALID, "model " + std::to_string(m) + ": band_of = " + std::to_string(band_of[m]) +
                                             " is not a band index (n_bands = " + std::to_string(n_bands) + ")");
    if (int rc = check_models(params, n_models)) return rc;
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (n_models == 0) return VAG_OK;
    cudaStream_t s = ctx->stream;
    BandPass bp;
    if (int rc = band_pass(ctx, static_cast<vag_params*>(ctx->io_params.p), n_models, caps, band_of, bands, n_bands, grids,
                           false, static_cast<int32_t*>(ctx->io_status.p), bp, s))
        return rc;
    CK(cudaMemcpyAsync(out, bp.red, sizeof(double) * VAG_NCOMP * bp.h_red_off[n_models], cudaMemcpyDeviceToHost, s));
    if (status) CK(cudaMemcpyAsync(status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

// ---- per-model grid requests and their quantiles across models -----------------------------------------------------
// The checks of vag_flux_density_grid_multi / vag_flux_quantiles_multi, all before any work is enqueued
static int check_grid_multi(const vag_params* params, size_t n_models, const int32_t* dataset_of, const vag_grid_set* sets,
                            size_t n_sets, const double* t, size_t n_t_total, const double* nu, size_t n_nu_total) {
    if (!sets || n_sets == 0) return fail(VAG_ERR_INVALID, "no grid sets: sets is NULL or n_sets is 0");
    if (!t || !nu) return fail(VAG_ERR_INVALID, "t or nu is NULL");
    if (n_t_total > (size_t)INT_MAX || n_nu_total > (size_t)INT_MAX || n_sets > (size_t)INT_MAX ||
        n_models > (size_t)INT_MAX)
        return fail(VAG_ERR_INVALID, "n_t_total, n_nu_total, n_sets and n_models must fit in a 32-bit int");
    if (n_models && !dataset_of) return fail(VAG_ERR_INVALID, "dataset_of is NULL");
    for (size_t d = 0; d < n_sets; ++d) {
        const std::string name = "set " + std::to_string(d) + ": ";
        const vag_grid_set& S = sets[d];
        if (S.n_t == 0) return fail(VAG_ERR_INVALID, name + "no times (n_t = 0)");
        if (S.n_nu == 0) return fail(VAG_ERR_INVALID, name + "no frequencies (n_nu = 0)");
        if (S.t0 > n_t_total || S.n_t > n_t_total - S.t0)
            return fail(VAG_ERR_INVALID, name + "times [" + std::to_string(S.t0) + ", " + std::to_string(S.t0) + " + " +
                                             std::to_string(S.n_t) + ") lie outside the " + std::to_string(n_t_total) + " times");
        if (S.nu0 > n_nu_total || S.n_nu > n_nu_total - S.nu0)
            return fail(VAG_ERR_INVALID, name + "frequencies [" + std::to_string(S.nu0) + ", " + std::to_string(S.nu0) + " + " +
                                             std::to_string(S.n_nu) + ") lie outside the " + std::to_string(n_nu_total) +
                                             " frequencies");
        if (check_times(t + S.t0, S.n_t)) return fail(VAG_ERR_INVALID, name + g_err);
        for (size_t i = S.nu0; i < S.nu0 + S.n_nu; ++i)
            if (!finite_pos(nu[i])) return fail(VAG_ERR_INVALID, name + "observation frequencies must be finite and > 0");
    }
    for (size_t m = 0; m < n_models; ++m)
        if (dataset_of[m] < 0 || (size_t)dataset_of[m] >= n_sets)
            return fail(VAG_ERR_INVALID, "model " + std::to_string(m) + ": dataset_of = " + std::to_string(dataset_of[m]) +
                                             " is not a set index (n_sets = " + std::to_string(n_sets) + ")");
    return check_models(params, n_models);
}

// The grid run of both calls on checked arguments, whose records prepare_params uploaded: pk holds the times, the
// frequencies (Hz) and gs's tables, then whatever the caller packed behind them; one upload of it to io_sets with `room`
// more bytes behind, then the run into io_out (status: io_status).  *base: the upload on the device.
static int grid_multi_run(vag_context* ctx, Caps caps, const Pack& pk, size_t o_t, size_t n_t_total,
                          size_t o_nu, size_t n_nu_total, GridSets& gs, size_t room, void** base, cudaStream_t s) {
    CK(ctx->io_sets.ensure(pk.h.size() + room));
    *base = ctx->io_sets.p;
    CK(cudaMemcpyAsync(*base, pk.h.data(), pk.h.size(), cudaMemcpyHostToDevice, s));
    gs.bind(*base);
    CK(ctx->io_out.ensure(sizeof(double) * std::max<size_t>(gs.elems(), 1)));
    return gs.run(ctx, static_cast<vag_params*>(ctx->io_params.p), caps, at<double>(*base, o_t), n_t_total,
                  at<double>(*base, o_nu), n_nu_total, false, static_cast<double*>(ctx->io_out.p),
                  static_cast<int32_t*>(ctx->io_status.p), s);
}

static std::vector<SeriesSet> grid_table(const vag_grid_set* sets, size_t n_sets) {
    std::vector<SeriesSet> tab(n_sets);
    for (size_t d = 0; d < n_sets; ++d)
        tab[d] = SeriesSet{(int)sets[d].t0, (int)sets[d].n_t, (int)sets[d].n_nu, (int)sets[d].nu0};
    return tab;
}

int vag_flux_density_grid_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                                const vag_grid_set* sets, size_t n_sets, const double* t, size_t n_t_total,
                                const double* nu, size_t n_nu_total, double* out, int32_t* status) {
    if (!ctx || !out) return fail(VAG_ERR_INVALID, "NULL argument");
    if (int rc = check_grid_multi(params, n_models, dataset_of, sets, n_sets, t, n_t_total, nu, n_nu_total)) return rc;
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (n_models == 0) return VAG_OK;
    cudaStream_t s = ctx->stream;
    Pack pk;
    GridSets gs;
    const size_t o_t = pk.put(t, n_t_total), o_nu = pk.put(nu, n_nu_total);
    gs.put(pk, grid_table(sets, n_sets), dataset_of, n_models);
    void* base = nullptr;
    if (int rc = grid_multi_run(ctx, caps, pk, o_t, n_t_total, o_nu, n_nu_total, gs, 0, &base, s)) return rc;
    CK(cudaMemcpyAsync(out, ctx->io_out.p, sizeof(double) * gs.elems(), cudaMemcpyDeviceToHost, s));
    if (status) CK(cudaMemcpyAsync(status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

// The grid run of vag_flux_density_grid_multi, then k_quant_members and k_quantiles on its output in io_out: one upload
// of the request, the run's tables, q and the quantile plan (the models of every set, in model order; every set's first
// tile and first column), with room behind it for the members' offsets, n_used and the bands.
int vag_flux_quantiles_multi(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                             const vag_grid_set* sets, size_t n_sets, const double* t, size_t n_t_total, const double* nu,
                             size_t n_nu_total, const double* q, size_t n_q, double* out, int64_t* n_used,
                             int32_t* status) {
    if (!ctx || !out || !n_used) return fail(VAG_ERR_INVALID, "NULL argument");
    if (n_q == 0 || !q) return fail(VAG_ERR_INVALID, "no quantiles: q is NULL or n_q is 0");
    if (n_q > (size_t)INT_MAX) return fail(VAG_ERR_INVALID, "n_q must fit in a 32-bit int");
    for (size_t j = 0; j < n_q; ++j)
        if (!(q[j] >= 0.0 && q[j] <= 1.0))
            return fail(VAG_ERR_INVALID, "q[" + std::to_string(j) + "] must be finite and in [0, 1]");
    if (int rc = check_grid_multi(params, n_models, dataset_of, sets, n_sets, t, n_t_total, nu, n_nu_total)) return rc;
    std::vector<long long> tile0(n_sets + 1, 0), col0(n_sets + 1, 0);
    for (size_t d = 0; d < n_sets; ++d) {
        const long long cols = (long long)(sets[d].n_t * sets[d].n_nu);
        col0[d + 1] = col0[d] + cols;
        tile0[d + 1] = tile0[d] + (cols + QUANT_COLS - 1) / QUANT_COLS;
    }
    if (tile0[n_sets] > INT_MAX) return fail(VAG_ERR_INVALID, "too many (set, frequency, time) columns for one call");
    const size_t n_out = n_q * (size_t)col0[n_sets];
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (n_models == 0) {  // no set has members
        std::fill(out, out + n_out, NAN);
        std::fill(n_used, n_used + n_sets, 0);
        return VAG_OK;
    }
    std::vector<int> c0(n_sets + 1, 0), cand(n_models);
    for (size_t m = 0; m < n_models; ++m) ++c0[dataset_of[m] + 1];
    int max_cand = 0;
    for (size_t d = 0; d < n_sets; ++d) {
        max_cand = std::max(max_cand, c0[d + 1]);
        c0[d + 1] += c0[d];
    }
    {
        std::vector<int> fill(c0.begin(), c0.end() - 1);
        for (size_t m = 0; m < n_models; ++m) cand[fill[dataset_of[m]]++] = (int)m;
    }
    cudaStream_t s = ctx->stream;
    Pack pk;
    GridSets gs;
    const size_t o_t = pk.put(t, n_t_total), o_nu = pk.put(nu, n_nu_total);
    gs.put(pk, grid_table(sets, n_sets), dataset_of, n_models);
    const size_t o_q = pk.put(q, n_q), o_cand = pk.put(cand), o_c0 = pk.put(c0), o_tile0 = pk.put(tile0),
                 o_col0 = pk.put(col0), up = pk.h.size();
    const size_t o_mem = up, o_used = o_mem + carve_sz<long long>(n_models), o_out = o_used + carve_sz<long long>(n_sets),
                 end = o_out + carve_sz<double>(n_out);
    void* base = nullptr;
    if (int rc = grid_multi_run(ctx, caps, pk, o_t, n_t_total, o_nu, n_nu_total, gs, end - up, &base, s)) return rc;
    const int launches = ctx->launches;
    long long* d_used = at<long long>(base, o_used);
    double* d_out = at<double>(base, o_out);
    k_quant_members<<<(unsigned)n_sets, 256, 0, s>>>(at<int>(base, o_cand), at<int>(base, o_c0),
                                                     static_cast<int32_t*>(ctx->io_status.p), gs.sd.out_off,
                                                     at<long long>(base, o_mem), d_used);
    // members staged in shared memory up to the budget; a larger set selects from global memory
    const int rows_cap = (int)std::min<size_t>((size_t)max_cand, QUANT_SMEM_BUDGET / (QUANT_COLS * sizeof(uint64_t)));
    k_quantiles<<<(unsigned)tile0[n_sets], QUANT_COLS * 32, (size_t)rows_cap * QUANT_COLS * sizeof(uint64_t), s>>>(
        static_cast<double*>(ctx->io_out.p), at<long long>(base, o_mem), at<int>(base, o_c0), d_used,
        at<long long>(base, o_tile0), at<long long>(base, o_col0), (int)n_sets, at<double>(base, o_q), (int)n_q, rows_cap,
        d_out);
    CK(cudaGetLastError());
    ctx->launches = launches + 2;
    CK(cudaMemcpyAsync(out, d_out, sizeof(double) * n_out, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(n_used, d_used, sizeof(int64_t) * n_sets, cudaMemcpyDeviceToHost, s));
    if (status) CK(cudaMemcpyAsync(status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

// The two lists of vag_chi2_multi_bands(_dev), over the models m with ok[m] (every model when ok is NULL): the models whose
// set has points (pt_of[m] = index in the point pass, or -1) and the (model, band) evaluations, model-major; gather = the
// model of every entry of both, the point pass first.  The point pass's data sets are all the sets with points, whether a
// model uses them or not.
struct MultiLists {
    std::vector<int> gather, pt_of, e0, eval_band, pt_set_of;
    std::vector<SeriesSet> pt_sets;
    std::vector<long long> pt_off{0};
    size_t max_set = 0, n_pt = 0, n_eval = 0;
};
static void multi_lists(size_t n_models, const int32_t* dataset_of, const vag_multi_set* sets, size_t n_sets,
                        const int32_t* ok, MultiLists& L) {
    L.pt_of.assign(n_models, -1);
    L.e0.assign(n_models + 1, 0);
    std::vector<int> set_idx(n_sets, -1);  // point-pass index of each set with points
    for (size_t d = 0; d < n_sets; ++d)
        if (sets[d].n) {
            set_idx[d] = (int)L.pt_sets.size();
            L.pt_sets.push_back(SeriesSet{(int)sets[d].offset, (int)sets[d].n, 0, 0});
            L.max_set = std::max(L.max_set, sets[d].n);
        }
    for (size_t m = 0; m < n_models; ++m) {
        const vag_multi_set& S = sets[dataset_of[m]];
        if (!S.n || (ok && !ok[m])) continue;
        L.pt_of[m] = (int)L.gather.size();
        L.gather.push_back((int)m);
        L.pt_set_of.push_back(set_idx[dataset_of[m]]);
        L.pt_off.push_back(L.pt_off.back() + (long long)S.n);
    }
    L.n_pt = L.gather.size();
    for (size_t m = 0; m < n_models; ++m) {
        const vag_multi_set& S = sets[dataset_of[m]];
        for (size_t j = 0; (!ok || ok[m]) && j < S.n_bands; ++j) {
            L.gather.push_back((int)m);
            L.eval_band.push_back((int)(S.band0 + j));
        }
        L.e0[m + 1] = (int)L.eval_band.size();
    }
    L.n_eval = L.eval_band.size();
}

// The entries of both lists over all models within a 32-bit int (sets and dataset_of checked)
static int check_multi_count(size_t n_models, const int32_t* dataset_of, const vag_multi_set* sets) {
    size_t n = 0;
    for (size_t m = 0; m < n_models; ++m) {
        const vag_multi_set& S = sets[dataset_of[m]];
        n += S.n_bands + (S.n ? 1 : 0);
        if (n > (size_t)INT_MAX) return fail(VAG_ERR_INVALID, "the (model, band) evaluations must fit in a 32-bit int");
    }
    return VAG_OK;
}

// The exposures of vag_chi2_multi_bands_exposures (checked): the samples of every set with points, in L.pt_sets' order
// (vag_exposure.cuh, with the set's num_expo), whose nu_off becomes the set's first point in the plan; the point pass's
// sets of samples and its models' blocks of samples.
struct MultiExpo {
    ExpoPlan plan;
    std::vector<SeriesSet> sets;    // [sets with points] slices of the concatenated samples
    std::vector<long long> off{0};  // [n_pt + 1] first sample of each point model's block
    size_t max_set = 0;
};
static void multi_expo(const vag_multi_set* sets, size_t n_sets, const double* t, const double* nu, const double* expo_time,
                       const int32_t* num_expo, MultiLists& L, MultiExpo& X) {
    for (size_t d = 0, q = 0; d < n_sets; ++d) {
        const vag_multi_set& S = sets[d];
        if (!S.n) continue;
        const size_t first = X.plan.t.size();
        L.pt_sets[q++].nu_off = (int)(X.plan.s0.size() - 1);
        expo_plan_append(t + S.offset, nu + S.offset, expo_time + S.offset, S.n, num_expo[d], X.plan);
        X.sets.push_back(SeriesSet{(int)first, (int)(X.plan.t.size() - first), 0, 0});
        X.max_set = std::max(X.max_set, X.plan.t.size() - first);
    }
    for (size_t i = 0; i < L.n_pt; ++i) X.off.push_back(X.off.back() + X.sets[L.pt_set_of[i]].n);
}

// L's tables and the intermediate results on the device
struct MultiDev {
    const int *pt_of, *e0;
    SetsDev pt_sd;              // the point pass: its models' data sets, the sets, the output offsets
    double* chi2_pts;           // [n_pt]
    int32_t *st_pts, *st_eval;  // [n_pt], [n_eval]
    SetsDev pt_sx;              // with exposures: the point pass over the samples (pt_sd: its averages)
    const int *s0, *pos;        // with exposures: the plan (MultiExpo)
};

// Steps 1, 2 (with 3) and 4 below on the records d_rec gathered for L (the point models', then the evaluations'): the point
// pass on pts (pts.av: the A_V of each point model), the band pass (device: its data are device pointers), and
// k_chi2_bands over all n_models.  With exposures X, the point pass runs on the samples (pts.t / pts.nu), k_expo_average
// averages them and k_chi2 compares the averages with the points' data.  *launches: the launches of the three.
static int multi_passes(vag_context* ctx, const vag_params* d_rec, const MultiLists& L, Caps caps, const Chi2Points& pts,
                        const MultiDev& tb, const vag_band_obs* bands, size_t n_bands, const std::vector<BandGrid>& grids,
                        bool device, size_t n_models, double* d_chi2, int32_t* d_status, cudaStream_t s, int* launches,
                        const MultiExpo* X = nullptr) {
    *launches = 0;
    if (L.n_pt && !X) {
        CK(ctx->io_out.ensure(sizeof(double) * VAG_NCOMP * (size_t)L.pt_off[L.n_pt]));
        if (int rc = run_flux(ctx, d_rec, L.n_pt, caps, points_request(pts, &tb.pt_sd, L.pt_off.data(), L.pt_sets.size(),
                                                                       L.max_set),
                              static_cast<double*>(ctx->io_out.p), tb.st_pts, tb.chi2_pts, s))
            return rc;
        *launches += ctx->launches;
    } else if (L.n_pt) {
        const size_t n_samples = (size_t)X->off[L.n_pt];
        CK(ctx->io_out.ensure(sizeof(double) * VAG_NCOMP * (n_samples + (size_t)L.pt_off[L.n_pt])));
        double* d_samples = static_cast<double*>(ctx->io_out.p);
        double* d_avg = d_samples + VAG_NCOMP * n_samples;
        const Chi2Points flux{pts.t, pts.nu, nullptr, nullptr, nullptr, nullptr, nullptr, X->plan.t.size()};
        if (int rc = run_flux(ctx, d_rec, L.n_pt, caps, points_request(flux, &tb.pt_sx, X->off.data(), X->sets.size(),
                                                                       X->max_set),
                              d_samples, tb.st_pts, nullptr, s))
            return rc;
        k_expo_average<true><<<(unsigned)L.n_pt, 128, 0, s>>>(d_samples, 0, 0, tb.s0, tb.pos, d_avg, tb.pt_sx, tb.pt_sd);
        k_chi2<true><<<(unsigned)((L.n_pt * 32 + 127) / 128), 128, 0, s>>>(d_avg, L.n_pt, 0, pts.lnF, pts.sig, pts.w, pts.av,
                                                                           pts.ext, tb.chi2_pts, tb.st_pts, 0, tb.pt_sd);
        *launches += ctx->launches + 2;
    }
    BandPass bp{};
    if (L.n_eval) {
        if (int rc = band_pass(ctx, d_rec + L.n_pt, L.n_eval, caps, L.eval_band.data(), bands, n_bands, grids, true,
                               tb.st_eval, bp, s, device))
            return rc;
        *launches += ctx->launches;
    }
    k_chi2_bands<<<(unsigned)((n_models * 32 + 127) / 128), 128, 0, s>>>(bp.red, bp.red_off, bp.sd, bp.lnF, bp.sig, bp.w,
                                                                         tb.st_eval, tb.e0, tb.pt_of, tb.chi2_pts, tb.st_pts,
                                                                         n_models, d_chi2, d_status);
    *launches += 1;
    CK(cudaGetLastError());
    return VAG_OK;
}

// The body of vag_chi2_multi_bands(_dev) on the lists L of the models that run and their records d_params[n_models] on
// the device: one upload of the lists and the point pass's tables -- and, from host memory (`host`), of the points pts and
// A_V[n_models] -- then room for the gathered records, the point models' A_V and the results.  k_gather_params_av gathers
// the records of both lists and the A_V, and multi_passes runs steps 1 to 4.  chi2 / status [n_models]: device outputs,
// or NULL to place them in io_sets.  With exposures X (host only) the uploaded t / nu are X's samples, with X's tables.
// *launches: k_gather_params_av's and multi_passes'.
static int multi_chi2(vag_context* ctx, const vag_params* d_params, size_t n_models, const MultiLists& L, Caps caps,
                      Chi2Points pts, const double* A_V, bool host, const vag_band_obs* bands, size_t n_bands,
                      const std::vector<BandGrid>& grids, double*& chi2, int32_t*& status, cudaStream_t s, int* launches,
                      const MultiExpo* X = nullptr) {
    const size_t n_pt = L.n_pt, n_eval = L.n_eval, n_up = host && n_pt ? pts.n : 0, n_av = A_V ? n_pt : 0;
    const size_t n_tnu = X ? (n_up ? X->plan.t.size() : 0) : n_up;
    Pack pk;
    const size_t o_gather = pk.put(L.gather), o_pt_of = pk.put(L.pt_of), o_e0 = pk.put(L.e0), o_sets = pk.put(L.pt_sets),
                 o_set_of = pk.put(L.pt_set_of), o_off = pk.put(L.pt_off),
                 o_t = pk.put(X ? X->plan.t.data() : pts.t, n_tnu), o_nu = pk.put(X ? X->plan.nu.data() : pts.nu, n_tnu),
                 o_lnF = pk.put(pts.lnF, n_up), o_sig = pk.put(pts.sig, n_up), o_w = pk.put(pts.w, n_up),
                 o_ext = pk.put(pts.ext, pts.ext ? n_up : 0), o_A_V = pk.put(A_V, host && A_V ? n_models : 0);
    size_t o_sx = 0, o_offx = 0, o_s0 = 0, o_pos = 0;
    if (X) {
        o_sx = pk.put(X->sets);
        o_offx = pk.put(X->off);
        o_s0 = pk.put(X->plan.s0);
        o_pos = pk.put(X->plan.pos);
    }
    const size_t up = pk.h.size(), o_rec = up, o_av = o_rec + carve_sz<vag_params>(n_pt + n_eval),
                 o_chi2_pts = o_av + carve_sz<double>(n_av), o_st_pts = o_chi2_pts + carve_sz<double>(n_pt),
                 o_st_eval = o_st_pts + carve_sz<int>(n_pt), o_chi2 = o_st_eval + carve_sz<int>(n_eval),
                 o_status = o_chi2 + (chi2 ? 0 : carve_sz<double>(n_models)),
                 end = o_status + (status ? 0 : carve_sz<int>(n_models));
    CK(ctx->io_sets.ensure(end));
    void* base = ctx->io_sets.p;
    CK(cudaMemcpyAsync(base, pk.h.data(), up, cudaMemcpyHostToDevice, s));
    if (host)
        pts = Chi2Points{at<double>(base, o_t), at<double>(base, o_nu), at<double>(base, o_lnF), at<double>(base, o_sig),
                         at<double>(base, o_w), pts.ext ? at<double>(base, o_ext) : nullptr, nullptr, pts.n};
    pts.av = A_V ? at<double>(base, o_av) : nullptr;
    if (!chi2) chi2 = at<double>(base, o_chi2);
    if (!status) status = at<int32_t>(base, o_status);
    vag_params* d_rec = at<vag_params>(base, o_rec);
    k_gather_params_av<<<(unsigned)((n_pt + n_eval + 127) / 128), 128, 0, s>>>(
        d_params, at<int>(base, o_gather), n_pt + n_eval, d_rec, host && A_V ? at<double>(base, o_A_V) : A_V, n_av, at<double>(base, o_av));
    MultiDev tb{at<int>(base, o_pt_of), at<int>(base, o_e0),
                SetsDev{at<int>(base, o_set_of), at<SeriesSet>(base, o_sets), at<long long>(base, o_off)},
                at<double>(base, o_chi2_pts), at<int32_t>(base, o_st_pts), at<int32_t>(base, o_st_eval), SetsDev{},
                nullptr, nullptr};
    if (X) {
        tb.pt_sx = SetsDev{tb.pt_sd.set_of, at<SeriesSet>(base, o_sx), at<long long>(base, o_offx)};
        tb.s0 = at<int>(base, o_s0);
        tb.pos = at<int>(base, o_pos);
    }
    if (int rc = multi_passes(ctx, d_rec, L, caps, pts, tb, bands, n_bands, grids, !host, n_models, chi2, status, s, launches,
                              X))
        return rc;
    *launches += 1;  // k_gather_params_av
    return VAG_OK;
}

// The exposure checks of vag_chi2_multi_bands_exposures, after those of vag_chi2_multi_bands: every expo_time finite and
// >= 0, num_expo >= 2 for every set with points of which one has an exposure, every sample time finite, the samples
// within a 32-bit int
static int check_multi_expo(const vag_multi_set* sets, size_t n_sets, const double* t, size_t n_points_total,
                            const double* expo_time, const int32_t* num_expo) {
    if (n_points_total && !expo_time) return fail(VAG_ERR_INVALID, "expo_time is NULL");
    if (!num_expo) return fail(VAG_ERR_INVALID, "num_expo is NULL");
    for (size_t i = 0; i < n_points_total; ++i)
        if (!(std::isfinite(expo_time[i]) && expo_time[i] >= 0))
            return fail(VAG_ERR_INVALID, "point " + std::to_string(i) + ": expo_time = " + std::to_string(expo_time[i]) +
                                             " must be finite and >= 0");
    size_t total = 0;
    for (size_t d = 0; d < n_sets; ++d) {
        const vag_multi_set& S = sets[d];
        const std::string name = "data set " + std::to_string(d) + ": ";
        size_t n_exp = 0;
        for (size_t i = S.offset; i < S.offset + S.n; ++i) n_exp += expo_time[i] > 0;
        if (n_exp && num_expo[d] < 2)
            return fail(VAG_ERR_INVALID, name + "num_expo = " + std::to_string(num_expo[d]) +
                                             " must be at least 2 (the set has exposures)");
        for (size_t i = S.offset; i < S.offset + S.n; ++i) {  // the last sample, the latest of the point's
            if (!(expo_time[i] > 0)) continue;
            volatile double step = (double)(num_expo[d] - 1) * (expo_time[i] / (double)(num_expo[d] - 1));
            if (!std::isfinite(t[i] + step))
                return fail(VAG_ERR_INVALID, name + "point " + std::to_string(i) + ": its last sample time is not finite");
        }
        total += S.n + n_exp * (size_t)(n_exp ? num_expo[d] - 1 : 0);
        if (total > (size_t)INT_MAX) return fail(VAG_ERR_INVALID, "the samples of all data sets must fit in a 32-bit int");
    }
    return VAG_OK;
}

// 1. the ragged point pass over the models whose set has points (vag_chi2_multi's, on those models and the sets with
// points; with exposures on their samples, then averaged), 2. the band pass over every (model, band) evaluation,
// model-major, 3. its reduction, 4. k_chi2_bands, through multi_chi2 on the records uploaded by prepare_params
static int multi_bands_host(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                            const vag_multi_set* sets, size_t n_sets, const double* t, const double* nu, const double* lnF_obs,
                            const double* sigma_ln, const double* w, const double* ext_k, size_t n_points_total,
                            const double* A_V, bool exposures, const double* expo_time, const int32_t* num_expo,
                            const vag_band_obs* bands, size_t n_bands_total, double* chi2, int32_t* status) {
    if (!ctx || !chi2) return fail(VAG_ERR_INVALID, "NULL argument");
    if (n_bands_total && !bands) return fail(VAG_ERR_INVALID, "bands is NULL");
    if (int rc = check_points(n_points_total, t && nu && lnF_obs && sigma_ln && w, ext_k, A_V, false)) return rc;
    if (int rc = check_multi_sets(n_models, dataset_of, sets, n_sets, t, nu, n_points_total, n_bands_total)) return rc;
    std::vector<BandGrid> grids;
    if (int rc = check_bands(bands, n_bands_total, true, grids)) return rc;
    if (int rc = check_models(params, n_models)) return rc;
    if (int rc = check_multi_count(n_models, dataset_of, sets)) return rc;
    if (exposures)
        if (int rc = check_multi_expo(sets, n_sets, t, n_points_total, expo_time, num_expo)) return rc;
    MultiLists L;
    multi_lists(n_models, dataset_of, sets, n_sets, nullptr, L);
    MultiExpo X;
    if (exposures) multi_expo(sets, n_sets, t, nu, expo_time, num_expo, L, X);
    Caps caps;
    if (int rc = prepare_params(ctx, params, n_models, &caps)) return rc;
    if (n_models == 0) return VAG_OK;
    cudaStream_t s = ctx->stream;
    double* d_chi2 = nullptr;
    int32_t* d_status = nullptr;
    int launches = 0;
    if (int rc = multi_chi2(ctx, static_cast<vag_params*>(ctx->io_params.p), n_models, L, caps,
                            Chi2Points{t, nu, lnF_obs, sigma_ln, w, ext_k, nullptr, n_points_total}, A_V, true, bands,
                            n_bands_total, grids, d_chi2, d_status, s, &launches, exposures ? &X : nullptr))
        return rc;
    ctx->launches = launches;
    CK(cudaMemcpyAsync(chi2, d_chi2, sizeof(double) * n_models, cudaMemcpyDeviceToHost, s));
    if (status) CK(cudaMemcpyAsync(status, d_status, sizeof(int32_t) * n_models, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

int vag_chi2_multi_bands(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                         const vag_multi_set* sets, size_t n_sets, const double* t, const double* nu, const double* lnF_obs,
                         const double* sigma_ln, const double* w, const double* ext_k, size_t n_points_total,
                         const double* A_V, const vag_band_obs* bands, size_t n_bands_total, double* chi2, int32_t* status) {
    return multi_bands_host(ctx, params, n_models, dataset_of, sets, n_sets, t, nu, lnF_obs, sigma_ln, w, ext_k,
                            n_points_total, A_V, false, nullptr, nullptr, bands, n_bands_total, chi2, status);
}

int vag_chi2_multi_bands_exposures(vag_context* ctx, const vag_params* params, size_t n_models, const int32_t* dataset_of,
                                   const vag_multi_set* sets, size_t n_sets, const double* t, const double* nu,
                                   const double* lnF_obs, const double* sigma_ln, const double* w, const double* ext_k,
                                   size_t n_points_total, const double* A_V, const double* expo_time,
                                   const int32_t* num_expo, const vag_band_obs* bands, size_t n_bands_total, double* chi2,
                                   int32_t* status) {
    return multi_bands_host(ctx, params, n_models, dataset_of, sets, n_sets, t, nu, lnF_obs, sigma_ln, w, ext_k,
                            n_points_total, A_V, true, expo_time, num_expo, bands, n_bands_total, chi2, status);
}

// ---- device-buffer entry points that plan on the device --------------------------------------------------------
// The record that runs in place of a rejected one: an on-axis tophat in ISM (one ODE row, one phi row) with coarse theta
// and time resolutions, so that its theta grid and time lattice stay below those of the batch's real models, which size
// the EATS stage of the whole batch
static vag_params stand_in_params() {
    vag_params p;
    vag_params_default(&p);
    p.jet_type = VAG_JET_TOPHAT;
    p.theta_c = 0.1;
    p.E_iso = 1e52;
    p.Gamma0 = 100.0;
    p.medium_type = VAG_MEDIUM_ISM;
    p.n_ism = 1.0;
    p.lumi_dist = 1e28;
    p.theta_resol = 0.05;
    p.t_resol = 2.0;
    return p;
}

// k_plan over the n device records d_params and the capacities of the accepted ones on the host (caps_for's floor
// included), because setup_models sizes the workspaces on the host.  In plan_buf ok[] (unless the caller's d_ok takes it)
// and the two capacities sit back to back, so one D2H into the pinned h_plan (grown on demand) -- of the capacities, or
// with `host_ok` of ok[] and the capacities -- and one synchronisation of s bring them back.  With `stand_ins` the records
// that run follow (P.run: a rejected one replaced by stand_in_params()), and the capacities cover the stand-in too.
struct Plan {
    const int32_t* ok;       // device ok[]
    const int32_t* h_ok;     // host_ok: ok[] on the host, until the context's next plan
    const vag_params* run;   // stand_ins: the records that run
    Caps caps;
};
static int plan(vag_context* ctx, const vag_params* d_params, size_t n, int32_t* d_ok, bool stand_ins, bool host_ok,
                cudaStream_t s, Plan* P) {
    const size_t ok_bytes = d_ok ? 0 : carve_sz<int32_t>(n), caps_at = ok_bytes, run_at = caps_at + carve_sz<int>(2);
    const size_t back = host_ok ? ok_bytes : 0, bytes = back + sizeof(int) * 2;  // h_plan: [ok[]] capacities
    CK(ctx->plan_buf.ensure(run_at + (stand_ins ? carve_sz<vag_params>(n) : 0)));
    if (bytes > ctx->h_plan_cap) {
        if (ctx->h_plan) cudaFreeHost(ctx->h_plan);
        ctx->h_plan = nullptr;
        ctx->h_plan_cap = 0;
        const size_t want = bytes + bytes / 4;
        CK(cudaMallocHost(&ctx->h_plan, want));
        ctx->h_plan_cap = want;
    }
    void* base = ctx->plan_buf.p;
    int32_t* ok = d_ok ? d_ok : at<int32_t>(base, 0);
    int* d_caps = at<int>(base, caps_at);
    vag_params* run = stand_ins ? at<vag_params>(base, run_at) : nullptr;
    CK(cudaMemsetAsync(d_caps, 0, sizeof(int) * 2, s));
    k_plan<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_params, n, stand_in_params(), run, ok, d_caps);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(ctx->h_plan, at<char>(base, caps_at - back), bytes, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const int* hc = at<int>(ctx->h_plan, back);
    P->caps = Caps{std::max(64, hc[0]), std::max(8, hc[1])};
    if (stand_ins) {
        const Caps sc = caps_of(stand_in_params());
        P->caps = Caps{std::max(P->caps.theta, sc.theta), std::max(P->caps.phi, sc.phi)};
    }
    P->ok = ok;
    P->h_ok = host_ok ? reinterpret_cast<const int32_t*>(ctx->h_plan) : nullptr;
    P->run = run;
    return VAG_OK;
}

int vag_params_validate_batch_dev(vag_context* ctx, const vag_params* d_params, size_t n, int32_t* d_ok, int caps[2],
                                  void* stream) {
    if (!ctx || !caps || (n && (!d_params || !d_ok))) return fail(VAG_ERR_INVALID, "NULL argument");
    ctx->launches = 0;
    if (n == 0) {
        caps[0] = 64;
        caps[1] = 8;
        return VAG_OK;
    }
    cudaStream_t s;
    if (int rc = dev_stream(ctx, stream, &s)) return rc;
    Plan P;
    if (int rc = plan(ctx, d_params, n, d_ok, false, false, s, &P)) return rc;
    ctx->launches = 1;
    caps[0] = P.caps.theta;
    caps[1] = P.caps.phi;
    return VAG_OK;
}

int vag_flux_band_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t, size_t n_t,
                      double nu_min, double nu_max, size_t num_nu, double* d_out, int32_t* d_status, void* stream) {
    if (!ctx || !d_out || (n_models && !d_params)) return fail(VAG_ERR_INVALID, "NULL argument");
    BandGrid g;
    if (int rc = band_grid(nu_min, nu_max, num_nu, g)) return rc;
    if (n_t == 0 || !d_t) return fail(VAG_ERR_INVALID, "time array must be non-empty");
    if (n_models == 0) return VAG_OK;
    cudaStream_t s;
    if (int rc = dev_stream(ctx, stream, &s)) return rc;
    Plan P;
    if (int rc = plan(ctx, d_params, n_models, nullptr, true, false, s, &P)) return rc;
    CK(ctx->io_status.ensure(sizeof(int32_t) * n_models));
    double* d_band = nullptr;
    if (int rc = run_band(ctx, P.run, n_models, P.caps, d_t, n_t, g, static_cast<int32_t*>(ctx->io_status.p), &d_band, s))
        return rc;
    const size_t per_model = VAG_NCOMP * n_t;
    CK(cudaMemcpyAsync(d_out, d_band, sizeof(double) * n_models * per_model, cudaMemcpyDeviceToDevice, s));
    if (d_status)
        CK(cudaMemcpyAsync(d_status, ctx->io_status.p, sizeof(int32_t) * n_models, cudaMemcpyDeviceToDevice, s));
    k_reject<<<(unsigned)n_models, 128, 0, s>>>(P.ok, d_status, nullptr, d_out, per_model);
    ctx->launches += 2;  // k_plan, k_reject
    CK(cudaGetLastError());
    return VAG_OK;
}

int vag_chi2_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const double* d_t, const double* d_nu,
                 const double* d_lnF_obs, const double* d_sigma_ln, const double* d_w, const double* d_ext_k, size_t n_points,
                 const double* d_A_V, const vag_band_obs* bands, size_t n_bands, double* d_chi2, int32_t* d_status,
                 void* stream) {
    std::vector<BandGrid> grids;
    if (int rc = check_chi2_args(ctx, d_chi2, n_points, d_t && d_nu && d_lnF_obs && d_sigma_ln && d_w, d_ext_k, d_A_V,
                                 bands, n_bands, true, grids))
        return rc;
    if (n_models && !d_params) return fail(VAG_ERR_INVALID, "params is NULL");
    if (n_models == 0) return VAG_OK;
    cudaStream_t s;
    if (int rc = dev_stream(ctx, stream, &s)) return rc;
    Plan P;
    if (int rc = plan(ctx, d_params, n_models, nullptr, true, false, s, &P)) return rc;
    CK(ctx->io_status.ensure(sizeof(int32_t) * n_models));
    CK(ctx->io_sets.ensure(sizeof(int32_t) * n_models));  // status OR of the band terms
    int32_t* d_stat_or = static_cast<int32_t*>(ctx->io_sets.p);
    const Chi2Points pts{d_t, d_nu, d_lnF_obs, d_sigma_ln, d_w, d_ext_k, d_A_V, n_points};
    std::vector<BandTerm> terms(n_bands);
    for (size_t b = 0; b < n_bands; ++b)
        terms[b] = BandTerm{bands[b].t, bands[b].lnF_obs, bands[b].sigma_ln, bands[b].w, bands[b].n, &grids[b]};
    if (int rc = chi2_run(ctx, P.run, n_models, P.caps, pts, terms.data(), n_bands, d_chi2, d_stat_or, s)) return rc;
    if (d_status)
        CK(cudaMemcpyAsync(d_status, n_bands ? d_stat_or : ctx->io_status.p, sizeof(int32_t) * n_models,
                           cudaMemcpyDeviceToDevice, s));
    k_reject<<<(unsigned)n_models, 128, 0, s>>>(P.ok, d_status, d_chi2, nullptr, 0);
    ctx->launches += 2;  // k_plan, k_reject
    CK(cudaGetLastError());
    return VAG_OK;
}

// vag_chi2_multi_bands on device buffers, planned on the device: k_plan, then the lists of the accepted models alone
// (multi_lists with ok[]), multi_chi2 on device data (the band data gathered on the device by k_gather_bands), and
// k_reject for the rejected models
int vag_chi2_multi_bands_dev(vag_context* ctx, const vag_params* d_params, size_t n_models, const int32_t* dataset_of,
                             const vag_multi_set* sets, size_t n_sets, const double* d_t, const double* d_nu,
                             const double* d_lnF_obs, const double* d_sigma_ln, const double* d_w, const double* d_ext_k,
                             size_t n_points_total, const double* d_A_V, const vag_band_obs* bands, size_t n_bands_total,
                             double* d_chi2, int32_t* d_status, void* stream) {
    if (!ctx || (n_models && !d_chi2)) return fail(VAG_ERR_INVALID, "NULL argument");
    if (n_models && !d_params) return fail(VAG_ERR_INVALID, "params is NULL");
    if (n_bands_total && !bands) return fail(VAG_ERR_INVALID, "bands is NULL");
    if (int rc = check_points(n_points_total, d_t && d_nu && d_lnF_obs && d_sigma_ln && d_w, d_ext_k, d_A_V, true)) return rc;
    if (int rc = check_multi_sets(n_models, dataset_of, sets, n_sets, d_t, d_nu, n_points_total, n_bands_total, true))
        return rc;
    std::vector<BandGrid> grids;
    if (int rc = check_bands(bands, n_bands_total, true, grids, true)) return rc;
    if (int rc = check_multi_count(n_models, dataset_of, sets)) return rc;
    if (n_models == 0) return VAG_OK;
    cudaStream_t s;
    if (int rc = dev_stream(ctx, stream, &s)) return rc;
    Plan P;
    if (int rc = plan(ctx, d_params, n_models, nullptr, false, true, s, &P)) return rc;
    MultiLists L;
    multi_lists(n_models, dataset_of, sets, n_sets, P.h_ok, L);
    int launches = 0;
    double* chi2 = d_chi2;
    int32_t* status = d_status;  // NULL: scratch for k_chi2_bands
    if (L.n_pt + L.n_eval)
        if (int rc = multi_chi2(ctx, d_params, n_models, L, P.caps,
                                Chi2Points{d_t, d_nu, d_lnF_obs, d_sigma_ln, d_w, d_ext_k, nullptr, n_points_total}, d_A_V,
                                false, bands, n_bands_total, grids, chi2, status, s, &launches))
            return rc;
    // k_chi2_bands gave the rejected models (no point term, no band) chi2 = 0 and status 0; k_reject overwrites them
    k_reject<<<(unsigned)n_models, 128, 0, s>>>(P.ok, d_status, d_chi2, nullptr, 0);
    ctx->launches = launches + 2;  // k_plan, k_reject
    CK(cudaGetLastError());
    return VAG_OK;
}

// ---- introspection ---------------------------------------------------------------------------------
// one parameter set through grid, dynamics and radiation over [t_min, t_max]
static int details_front(vag_context* ctx, const vag_params* p, double t_min, double t_max, BatchWs& w, long long* cells) {
    Caps caps;
    if (int rc = prepare_params(ctx, p, 1, &caps)) return rc;
    const double tt[2] = {t_min, t_max};
    CK(ctx->io_t.ensure(sizeof(tt)));
    CK(cudaMemcpyAsync(ctx->io_t.p, tt, sizeof(tt), cudaMemcpyHostToDevice, ctx->stream));
    int totals[TOT_N];
    ctx->launches = 0;
    return run_front(ctx, w, static_cast<vag_params*>(ctx->io_params.p), 1, caps, static_cast<double*>(ctx->io_t.p), 2,
                     ctx->stream, totals, cells);
}

int vag_details(vag_context* ctx, const vag_params* p, double t_min, double t_max, vag_grid_info* info, double* theta,
                double* phi, int32_t* reps, double* t_rows, double* fwd_shock, double* rvs_shock, int32_t* inj_idx) {
    if (!ctx || !p) return fail(VAG_ERR_INVALID, "NULL argument");
    BatchWs w;
    long long cells = 0;
    if (int rc = details_front(ctx, p, t_min, t_max, w, &cells)) return rc;
    cudaStream_t s = ctx->stream;
    GridHeader h;
    int st = 0;
    CK(cudaMemcpyAsync(&h, w.hdr, sizeof(h), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&st, w.status, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (info) {
        info->n_phi = h.n_phi;
        info->n_theta = h.n_theta;
        info->n_t = h.n_t;
        info->n_reps = h.n_reps;
        info->symmetry = h.symmetry;
        info->phi_mirrored = h.phi_mirrored;
        info->n_phi_eff = h.n_phi_eff;
        info->status = st;
    }
    const size_t nc = (size_t)h.n_reps * h.n_t;
    // theta and the theta index of every ODE row (the representatives of the symmetry groups, or r % n_theta for a
    // rows3d model) serve the output arrays and the theta plane of the shock tables
    std::vector<double> th(h.n_theta);
    std::vector<int32_t> rep(h.n_reps);
    CK(cudaMemcpyAsync(th.data(), w.theta, sizeof(double) * h.n_theta, cudaMemcpyDeviceToHost, s));
    if (!h.rows3d) CK(cudaMemcpyAsync(rep.data(), w.reps, sizeof(int) * h.n_reps, cudaMemcpyDeviceToHost, s));
    if (phi) CK(cudaMemcpyAsync(phi, w.phi, sizeof(double) * h.n_phi, cudaMemcpyDeviceToHost, s));
    if (t_rows) CK(cudaMemcpyAsync(t_rows, w.t_rows, sizeof(double) * nc, cudaMemcpyDeviceToHost, s));
    if (inj_idx) CK(cudaMemcpyAsync(inj_idx, w.inj_idx, sizeof(int) * h.n_reps, cudaMemcpyDeviceToHost, s));
    auto dump = [&](double* const* pl, double* o) -> int {
        const int map[7] = {0, 1, -1, 2, 3, 4, 5};
        for (int a = 0; a < 7; ++a)
            if (map[a] >= 0) CK(cudaMemcpyAsync(o + (size_t)a * nc, pl[map[a]], sizeof(double) * nc, cudaMemcpyDeviceToHost, s));
        return VAG_OK;
    };
    if (fwd_shock)
        if (int rc = dump(w.fwd, fwd_shock)) return rc;
    if (rvs_shock && p->has_rvs)
        if (int rc = dump(w.rvs, rvs_shock)) return rc;
    CK(cudaStreamSynchronize(s));
    if (h.rows3d)
        for (int r = 0; r < h.n_reps; ++r) rep[r] = r % h.n_theta;
    if (theta) std::copy(th.begin(), th.end(), theta);
    if (reps) std::copy(rep.begin(), rep.end(), reps);
    auto fill_theta = [&](double* o) {
        for (int r = 0; r < h.n_reps; ++r)
            for (int k = 0; k < h.n_t; ++k) o[(2 * (size_t)h.n_reps + r) * h.n_t + k] = th[rep[r]];
    };
    if (fwd_shock) fill_theta(fwd_shock);
    if (fwd_shock && w.sh_theta) {  // spreading model: Shock::theta varies along k
        CK(cudaMemcpyAsync(fwd_shock + 2 * nc, w.sh_theta, sizeof(double) * nc, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    if (rvs_shock && p->has_rvs) fill_theta(rvs_shock);
    return VAG_OK;
}

int vag_details_photons(vag_context* ctx, const vag_params* p, double t_min, double t_max, double* fwd, double* rvs) {
    if (!ctx || !p || !fwd) return fail(VAG_ERR_INVALID, "NULL argument");
    BatchWs w;
    long long cells = 0;
    if (int rc = details_front(ctx, p, t_min, t_max, w, &cells)) return rc;
    cudaStream_t s = ctx->stream;
    const int planes[6] = {PH_LOG2_NU_M, PH_LOG2_NU_C, PH_LOG2_NU_A, PH_LOG2_NU_M_MAX, PH_LOG2_I_MAX, PH_INV_NU_M_MAX};
    const size_t nc = (size_t)cells;
    for (int a = 0; a < 6; ++a) {
        CK(cudaMemcpyAsync(fwd + a * nc, w.coef_fwd + (size_t)planes[a] * nc, sizeof(double) * nc, cudaMemcpyDeviceToHost, s));
        if (rvs && p->has_rvs)
            CK(cudaMemcpyAsync(rvs + a * nc, w.coef_rvs + (size_t)planes[a] * nc, sizeof(double) * nc, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    return VAG_OK;
}

// Electron / inverse-Compton bookkeeping of the shocks with ssc=True (after KN_cooling / Thomson_cooling), per unique cell
int vag_details_ic(vag_context* ctx, const vag_params* p, double t_min, double t_max, double* fwd, double* rvs) {
    if (!ctx || !p || !fwd) return fail(VAG_ERR_INVALID, "NULL argument");
    BatchWs w;
    long long cells = 0;
    if (int rc = details_front(ctx, p, t_min, t_max, w, &cells)) return rc;
    cudaStream_t s = ctx->stream;
    const size_t nc = (size_t)cells;
    CK(ctx->io_out.ensure(sizeof(double) * VAG_IC_DETAIL_PLANES * std::max<size_t>(nc, 1)));
    double* d_out = static_cast<double*>(ctx->io_out.p);
    for (int which = 0; which < 2; ++which) {
        double* dst = which ? rvs : fwd;
        if (which && !(rvs && p->has_rvs)) continue;
        const bool ssc = (which ? p->rvs.ssc : p->fwd.ssc) != 0;
        if (ssc && w.any_ssc && nc > 0) {
            k_ic_export<<<(unsigned)((nc + 127) / 128), 128, 0, s>>>(w.ic[which], nc, d_out);
            CK(cudaMemcpyAsync(dst, d_out, sizeof(double) * VAG_IC_DETAIL_PLANES * nc, cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
        } else {
            std::memset(dst, 0, sizeof(double) * VAG_IC_DETAIL_PLANES * nc);
        }
    }
    CK(cudaGetLastError());
    return VAG_OK;
}

}  // extern "C"
