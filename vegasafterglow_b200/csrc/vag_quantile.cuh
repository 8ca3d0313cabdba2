// vag_quantile.cuh -- exact quantiles of a column of doubles: numpy.quantile(x, q, method="linear") bit for bit (the sign
// of a zero aside), by selection of the two order statistics that numpy interpolates between.
//
// numpy 2.3 (_quantile, _get_indexes, _lerp in numpy/lib/_function_base_impl.py): h = (n - 1) q, lo = floor(h),
// hi = min(lo + 1, n - 1), g = h - lo; with a = x_(lo) and b = x_(hi) of the sorted column the result is
// a + (b - a) g, or b - (b - a) (1 - g) when g >= 0.5, each operation rounded on its own.  A column holding a NaN gives NaN.
// (Where h >= n - 1 numpy takes a = b = x_(n-1) with g = h + 1, which gives the same value for every finite x_(n-1);
// an infinite one gives NaN either way, as b - a is NaN.)
//
// Selection is an MSB radix select over the order-preserving uint64 image of the doubles: 8 passes of 8 bits, each a
// 256-bin histogram of the keys that share the prefix found so far, so the result is the exact order statistic whatever
// the order of the column (deterministic).  x_(lo + 1) then takes one more pass: it is x_(lo) when more than lo + 1 keys
// are <= x_(lo)'s, else the smallest key above it.  The functions take the cooperating group as a template argument:
// QuantWarp (a warp, device) or QuantSeq (one thread, the host tests), so the device and the host run the same body.
#pragma once

#include <cstdint>
#include <cstring>

#include "vag_common.cuh"

namespace vag {

// order-preserving image: a < b (as doubles, -0 < +0) <=> key(a) < key(b); NaNs land outside [key(-inf), key(+inf)]
VAG_HD uint64_t quant_key(double x) {
#if defined(__CUDA_ARCH__)
    const uint64_t u = (uint64_t)__double_as_longlong(x);
#else
    uint64_t u;
    std::memcpy(&u, &x, sizeof u);
#endif
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
VAG_HD double quant_val(uint64_t k) {
    const uint64_t u = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double x;
    std::memcpy(&x, &u, sizeof x);
    return x;
#endif
}

// the two order statistics of q among n > 0 values and the weight between them (numpy's linear method)
struct QuantRanks {
    long long lo, hi;
    double g;
};
VAG_HD QuantRanks quant_ranks(long long n, double q) {
    const double h = (double)(n - 1) * q;
    const double f = floor(h);
    const long long lo = (long long)f;
    return QuantRanks{lo, lo + 1 < n ? lo + 1 : n - 1, h - f};
}

// numpy's _lerp, every operation rounded (no contraction into an FMA)
VAG_HD double quant_lerp(double a, double b, double g) {
#if defined(__CUDA_ARCH__)
    const double d = __dsub_rn(b, a);
    return g >= 0.5 ? __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(d, g));
#else
    volatile double d = b - a;  // volatile: the host compiler may not fuse the product into the sum either
    volatile double p = g >= 0.5 ? d * (1.0 - g) : d * g;
    return g >= 0.5 ? b - p : a + p;
#endif
}

// One host thread as the group (the CPU tests)
struct QuantSeq {
    static constexpr int lane = 0, width = 1;
    void sync() const {}
    void inc(unsigned* c) const { ++*c; }
    unsigned excl_scan(unsigned v, unsigned* total) const {
        *total = v;
        return 0;
    }
    int owner(bool) const { return 0; }
    template <class T>
    T bcast(T v, int) const {
        return v;
    }
    bool any(bool v) const { return v; }
    unsigned long long sum(unsigned long long v) const { return v; }
    unsigned long long min(unsigned long long v) const { return v; }
};
#if defined(__CUDACC__)
// One warp: keys strided over the lanes, histogram increments as shared-memory atomics
struct QuantWarp {
    int lane;
    static constexpr int width = 32;
    __device__ __forceinline__ void sync() const { __syncwarp(); }
    __device__ __forceinline__ void inc(unsigned* c) const { atomicAdd(c, 1u); }
    __device__ __forceinline__ unsigned excl_scan(unsigned v, unsigned* total) const {
        unsigned s = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned u = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += u;
        }
        *total = __shfl_sync(0xffffffffu, s, 31);
        return s - v;
    }
    __device__ __forceinline__ int owner(bool mine) const { return __ffs(__ballot_sync(0xffffffffu, mine)) - 1; }
    template <class T>
    __device__ __forceinline__ T bcast(T v, int src) const {
        return __shfl_sync(0xffffffffu, v, src);
    }
    __device__ __forceinline__ bool any(bool v) const { return __any_sync(0xffffffffu, v); }
    __device__ __forceinline__ unsigned long long sum(unsigned long long v) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    }
    __device__ __forceinline__ unsigned long long min(unsigned long long v) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o);
            v = u < v ? u : v;
        }
        return v;
    }
};
#endif

constexpr int QUANT_BINS = 256;

// Key of rank r (0-based, r < n) among the keys key(0 .. n-1); hist: QUANT_BINS counters of the group's own
template <class G, class K>
VAG_HD uint64_t quant_select(const G& grp, const K& key, int n, long long r, unsigned* hist) {
    constexpr int per_lane = QUANT_BINS / G::width;
    uint64_t prefix = 0, mask = 0;
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int b = grp.lane; b < QUANT_BINS; b += G::width) hist[b] = 0;
        grp.sync();
        for (int i = grp.lane; i < n; i += G::width) {
            const uint64_t k = key(i);
            if ((k & mask) == prefix) grp.inc(&hist[(k >> shift) & 0xff]);
        }
        grp.sync();
        // the bin that holds rank r: every lane sums its own run of bins, the scan finds the run, its lane the bin
        unsigned own = 0, total = 0;
        for (int b = 0; b < per_lane; ++b) own += hist[grp.lane * per_lane + b];
        const unsigned below = grp.excl_scan(own, &total);
        const int src = grp.owner(below <= r && r < (long long)below + own);
        int bin = 0;
        unsigned before = below;
        if (grp.lane == src) {
            bin = grp.lane * per_lane;
            while (before + hist[bin] <= r) before += hist[bin++];
        }
        bin = grp.bcast(bin, src);
        before = grp.bcast(before, src);
        grp.sync();  // every lane has read the histogram before the next pass clears it
        r -= before;
        prefix |= (uint64_t)bin << shift;
        mask |= (uint64_t)0xff << shift;
    }
    return prefix;
}

// out[j * out_stride] = numpy.quantile(column, q[j], method="linear") for j < n_q, the column being the n values whose
// keys are key(0 .. n-1); NaN for every j when n == 0 or a value is NaN.  Written by lane 0.
template <class G, class K>
VAG_HD void quant_column(const G& grp, const K& key, int n, const double* q, int n_q, double* out, size_t out_stride,
                         unsigned* hist) {
    bool nan = n == 0;
    for (int i = grp.lane; i < n; i += G::width) nan |= isnan(quant_val(key(i)));
    if (grp.any(nan)) {
        if (grp.lane == 0)
            for (int j = 0; j < n_q; ++j) out[j * out_stride] = NAN;
        return;
    }
    for (int j = 0; j < n_q; ++j) {
        const QuantRanks R = quant_ranks(n, q[j]);
        const uint64_t a = quant_select(grp, key, n, R.lo, hist);
        uint64_t b = a;
        if (R.hi != R.lo) {
            unsigned long long le = 0, above = ~0ull;
            for (int i = grp.lane; i < n; i += G::width) {
                const uint64_t k = key(i);
                le += k <= a;
                if (k > a && k < above) above = k;
            }
            le = grp.sum(le);
            above = grp.min(above);
            b = (long long)le >= R.hi + 1 ? a : above;
        }
        if (grp.lane == 0) out[j * out_stride] = quant_lerp(quant_val(a), quant_val(b), R.g);
    }
}

}  // namespace vag
