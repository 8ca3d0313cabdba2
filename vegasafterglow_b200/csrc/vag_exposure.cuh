// vag_exposure.cuh -- exposure-averaged flux densities: the rule of the reference's Model.flux_density_exposures
// (pybind/pymodel.cpp:412-496), shared by vag_flux_density_exposures and vag_chi2_multi_bands_exposures.
//
// Point i with exposure e_i > 0 is sampled k times over its exposure: dt = e_i / (k - 1), t_j = t_i + j dt for
// j = 0 .. k-1, the product and the sum rounded separately (numpy's t[:, None] + j * dt[:, None]).  A point with e_i = 0
// is one sample at t_i.  All samples of a request are sorted stably by time -- ties by point index, then by j -- and
// evaluated as one series.  A point's value is the flux of its samples added to 0.0 in sorted order, divided by their
// number (np.add.at, then / k).  The stable sort keeps the samples of one point in j order, since t_i + j dt does not
// decrease with j.
//
// The plan (samples and the map from points to their sorted positions) is built on the host; the averaging body runs in
// k_expo_average on the device and in the host tests, so both run the same operations.
#pragma once

#include <algorithm>
#include <cstddef>
#include <numeric>
#include <vector>

#include "vag_common.cuh"

namespace vag {

// The samples of the sets appended so far.  t / nu: each set's series request, ascending in t, the sets one after the
// other.  Point p (counting the points of every appended set, in order) has its samples at pos[s0[p] .. s0[p + 1]) of
// its set's request, in j order.
struct ExpoPlan {
    std::vector<double> t, nu;
    std::vector<int> s0{0}, pos;
};

// Appends the samples of the n points (t, nu, e) of one set, k samples for a point with e > 0 (k >= 2), one for e == 0.
// The caller bounds the number of samples.
inline void expo_plan_append(const double* t, const double* nu, const double* e, size_t n, int k, ExpoPlan& P) {
    std::vector<double> ts;  // in (point, j) order
    std::vector<int> of;
    for (size_t i = 0; i < n; ++i) {
        if (e[i] > 0) {
            const double dt = e[i] / (double)(k - 1);
            for (int j = 0; j < k; ++j) {
                volatile double step = (double)j * dt;  // rounded before the sum: no contraction into an FMA
                ts.push_back(t[i] + step);
                of.push_back((int)i);
            }
        } else {
            ts.push_back(t[i]);
            of.push_back((int)i);
        }
    }
    std::vector<int> order(ts.size()), rank(ts.size());
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return ts[a] < ts[b]; });
    for (size_t r = 0; r < order.size(); ++r) {
        rank[order[r]] = (int)r;
        P.t.push_back(ts[order[r]]);
        P.nu.push_back(nu[of[order[r]]]);
    }
    for (size_t q = 0; q < ts.size(); ++q) {
        P.pos.push_back(rank[q]);
        if (q + 1 == ts.size() || of[q + 1] != of[q]) P.s0.push_back((int)P.pos.size());
    }
}

// The average of one point: its k samples' flux f[pos[0]], ..., f[pos[k - 1]] added to 0.0 in this order, divided by k
VAG_HD double expo_mean(const double* f, const int* pos, int k) {
    double s = 0.0;
#if defined(__CUDA_ARCH__)
    for (int j = 0; j < k; ++j) s = __dadd_rn(s, f[pos[j]]);
    return __ddiv_rn(s, (double)k);
#else
    for (int j = 0; j < k; ++j) s += f[pos[j]];
    return s / (double)k;
#endif
}

}  // namespace vag
