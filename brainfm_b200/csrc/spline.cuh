// Spline helpers shared by the resampling kernels (interpol.cu) and the fused chain's cubic zoom back (gen.cu):
// the bound folding, the B-spline weights and the per-line recursive prefilter of torch-interpol 0.2.3.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace bfm {

// ---- Python-style integer helpers ----------------------------------------------------------------
__device__ __forceinline__ int64_t pymod(int64_t a, int64_t n) {
    int64_t r = a % n;
    return r < 0 ? r + n : r;
}
__device__ __forceinline__ int64_t floordiv(int64_t a, int64_t n) {
    int64_t q = a / n;
    return (a % n != 0 && ((a < 0) != (n < 0))) ? q - 1 : q;
}

// Bound.index (bounds.py:30-60) in the integer type I: int64_t for arbitrary coordinates, int where the caller
// keeps |i| < 2^30 (32-bit modulo inline instead of the 64-bit division subroutine)
template <typename I>
__device__ __forceinline__ int bound_index_t(int type, I i, int n) {
    using U = typename std::make_unsigned<I>::type;
    // every bound maps an in-range index to itself: the 64-bit modulo arithmetic below (~100 instructions per call,
    // six calls per voxel of a linear pull) only runs for the taps that actually leave the volume
    if ((U)i < (U)n) return (int)i;
    auto pm = [](I a, I m) { const I r = a % m; return r < 0 ? r + m : r; };
    switch (type) {
        case 0: case 1: return (int)(i < 0 ? 0 : (i > n - 1 ? n - 1 : i));
        case 3: case 5: {
            const I n2 = 2 * (I)n;
            i = i < 0 ? n2 - 1 - pm(-i - 1, n2) : pm(i, n2);
            return (int)(i >= n ? n2 - 1 - i : i);
        }
        case 2: {
            if (n == 1) return 0;
            const I n2 = 2 * ((I)n - 1);
            i = pm(i < 0 ? -i : i, n2);
            return (int)(i >= n ? n2 - i : i);
        }
        case 4: {
            const I n2 = 2 * ((I)n + 1);
            i = i < 0 ? -i - 2 : i;
            i = pm(i, n2);
            i = i > n ? n2 - 2 - i : i;
            if (i == -1) i = 0;
            if (i == n) i = n - 1;
            return (int)i;
        }
        case 6: return (int)pm(i, n);
        default: return (int)i;
    }
}
__device__ __forceinline__ int bound_index(int type, int64_t i, int n) { return bound_index_t<int64_t>(type, i, n); }
// Bound.transform (bounds.py:62-89): sign applied to the gathered value (1 when the reference returns None)
__device__ __forceinline__ int bound_sign(int type, int64_t i, int n) {
    switch (type) {
        case 4: {
            if (n == 1) return 1;
            const int64_t n2 = 2 * ((int64_t)n + 1);
            i = i < 0 ? -i + (n - 1) : i;
            i = pymod(i, n2);
            int x = (i == 0) ? 0 : 1;
            if (pymod(i, n + 1) == n) x = 0;
            i = floordiv(i, n + 1);
            return pymod(i, 2) > 0 ? -x : x;
        }
        case 5: {
            if ((uint64_t)i < (uint64_t)n) return 1;
            i = i < 0 ? n - 1 - i : i;
            i = floordiv(i, n);
            return pymod(i, 2) > 0 ? -1 : 1;
        }
        case 0: return (i < 0 || i >= n) ? 0 : 1;
        default: return 1;
    }
}

// Spline.fastweight (splines.py:30-79)
template <typename T>
__device__ __forceinline__ T spline_weight(int order, T x) {
    x = x < 0 ? -x : x;
    switch (order) {
        case 0: return T(1);
        case 1: return T(1) - x;
        case 2: return x < T(0.5) ? T(0.75) - x * x : T(0.5) * (T(1.5) - x) * (T(1.5) - x);
        case 3: return x < T(1) ? (x * x * (x - T(2)) * T(3) + T(4)) / T(6) : (T(2) - x) * (T(2) - x) * (T(2) - x) / T(6);
        case 4: {
            if (x < T(0.5)) { T a = x * x; return a * (a * T(0.25) - T(0.625)) + T(115.) / T(192.); }
            if (x < T(1.5)) return x * (x * (x * (T(5) - x) / T(6) - T(1.25)) + T(5.) / T(24.)) + T(55.) / T(96.);
            T a = x - T(2.5); a = a * a; return a * a / T(24);
        }
        case 5: {
            if (x < T(1)) { T a = x * x; return a * (a * (T(0.25) - x / T(12)) - T(0.5)) + T(0.55); }
            if (x < T(2)) return x * (x * (x * (x * (x / T(24) - T(0.375)) + T(1.25)) - T(1.75)) + T(0.625)) + T(0.425);
            T a = T(3) - x; T a2 = a * a; return a2 * a2 * a / T(120);
        }
        case 6: {
            if (x < T(0.5)) { T a = x * x; return a * (a * (T(7.) / T(48.) - a / T(36)) - T(77.) / T(192.)) + T(5887.) / T(11520.); }
            if (x < T(1.5)) return x * (x * (x * (x * (x * (x / T(48) - T(7.) / T(48.)) + T(0.328125)) - T(35.) / T(288.)) - T(91.) / T(256.)) - T(7.) / T(768.)) + T(7861.) / T(15360.);
            if (x < T(2.5)) return x * (x * (x * (x * (x * (T(7.) / T(60.) - x / T(120)) - T(0.65625)) + T(133.) / T(72.)) - T(2.5703125)) + T(1267.) / T(960.)) + T(1379.) / T(7680.);
            T a = x - T(3.5); T a2 = a * a; return a2 * a2 * a2 / T(720);
        }
        default: {  // 7
            if (x < T(1)) { T a = x * x; return a * (a * (a * (x / T(144) - T(1.) / T(36.)) + T(1.) / T(9.)) - T(1.) / T(3.)) + T(151.) / T(315.); }
            if (x < T(2)) return x * (x * (x * (x * (x * (x * (T(0.05) - x / T(240)) - T(7.) / T(30.)) + T(0.5)) - T(7.) / T(18.)) - T(0.1)) - T(7.) / T(90.)) + T(103.) / T(210.);
            if (x < T(3)) return x * (x * (x * (x * (x * (x * (x / T(720) - T(1.) / T(36.)) + T(7.) / T(30.)) - T(19.) / T(18.)) + T(49.) / T(18.)) - T(23.) / T(6.)) + T(217.) / T(90.)) - T(139.) / T(630.);
            T a = T(4) - x; T a2 = a * a; T a4 = a2 * a2; return a4 * a2 * a / T(5040);
        }
    }
}

// ---- prefilter: one thread per line ------------------------------------------------------------------
struct FilterArgs {
    int64_t outer, inner;   // tensor viewed as (outer, n, inner); line stride = inner
    int n;
    int bound;              // 0 zero,1 replicate,2 dct1,3 dct2,6 dft
    int npoles;
    double poles[3];
};

// One line of the recursive prefilter, in place; element i of the line lives at c[i * st].
// Entry e of the filter_line weight table `wt` (float32): per pole k, at k*(2n+2), the dct2 initial-value weights
// A[i] = pole^i + pole^(2n-1-i) (n entries), then the dft powers P[j] = pole^j (n+2 entries).
__device__ __forceinline__ float filter_weight(const FilterArgs &a, int e) {
    const int n = a.n;
    const int k = e / (2 * n + 2), r = e - k * (2 * n + 2);
    const double pole = a.poles[k];
    // |pole|^j rounds to (+-)0 in float32 beyond j = cut: skip the float64 pow there (same value, the sign of a
    // zero does not reach the sums)
    const int cut = (int)ceil(-151.0 / log2(fabs(pole)));
    auto powf_ = [&](int j) { return j > cut ? 0.f : (float)pow(pole, (double)j); };
    float v = 0.f;
    if (r < n) {
        if (a.bound == 1 || a.bound == 3) v = powf_(r) + powf_(2 * n - 1 - r);
    } else if (a.bound == 6) {
        v = powf_(r - n);
    }
    return v;
}

// ST: the stride type (int where the caller keeps every element offset of the line below 2^31).
template <typename T, typename ST = int64_t>
__device__ __forceinline__ void filter_line(T *c, const ST st, const FilterArgs &a, const T *wt = nullptr) {
    // wt (optional): per pole k, at wt + k*(2n+2): the dct2 initial-value weights A[i] = (T)pole^i + (T)pole^(2n-1-i)
    // (n entries) followed by the powers P[j] = (T)pole^j (n+2 entries) -- the same expressions as below, evaluated
    // once per block instead of once per line (they do not depend on the line).
    const int n = a.n;
    {
        double gain = 1.0;
        for (int k = 0; k < a.npoles; ++k) gain *= (1.0 - a.poles[k]) * (1.0 - 1.0 / a.poles[k]);
        const T tg = (T)gain;
        for (int i = 0; i < n; ++i) c[i * st] *= tg;                         // coeff.py:265-266
        for (int k = 0; k < a.npoles; ++k) {
            const double pole = a.poles[k];
            const T tp = (T)pole;
            const int max_iter0 = (int)ceil(-30.0 / log(fabs(pole)));
            // ---- initial value (coeff.py:69-177)
            T init;
            if (a.bound == 0 || a.bound == 2) {                               // dct1
                if (max_iter0 < n) {
                    T s = 0, pw = tp;
                    for (int i = 1; i < max_iter0; ++i) { s += c[i * st] * pw; pw *= tp; }
                    init = s + c[0];
                } else {
                    const double polen = pow(pole, (double)(n - 1));
                    T s = 0, pw = tp;
                    for (int i = 1; i < n - 1; ++i) {
                        s += c[i * st] * (pw + (T)(polen * polen) / pw);
                        pw *= tp;
                    }
                    init = s + (c[0] + (T)polen * c[(int64_t)(n - 1) * st]);
                    const double pl = pow(pole, (double)(n - 1));
                    init = init / (T)(1.0 - pl * pl);
                }
            } else if (a.bound == 1 || a.bound == 3) {                        // dct2
                const double polen = pow(pole, (double)n);
                const double pole_last = polen * (1.0 + 1.0 / (pole + polen * polen));
                T s = 0;
                if (wt) {
                    const T *A = wt + (int64_t)k * (2 * n + 2);
                    for (int i = 1; i < n - 1; ++i) s += c[i * st] * A[i];
                } else {
                    for (int i = 1; i < n - 1; ++i)
                        s += c[i * st] * ((T)pow(pole, (double)i) + (T)pow(pole, (double)(2 * n - 1 - i)));
                }
                T v = s + (c[0] + (T)pole_last * c[(int64_t)(n - 1) * st]);
                v = v * (T)(pole / (1.0 - polen * polen));
                init = v + c[0];
            } else {                                                          // dft
                const int mi = max_iter0 < n ? max_iter0 : n;
                T s = 0;
                const T *P = wt ? wt + (int64_t)k * (2 * n + 2) + n : nullptr;
                for (int i = 1; i < mi; ++i) s += c[(int64_t)(n - i) * st] * (P ? P[i] : (T)pow(pole, (double)i));
                init = (s + c[0]) / (T)(1.0 - pow(pole, (double)mi));
            }
            c[0] = init;
            {   // causal recursion, previous value carried in a register                    coeff.py:272-273
                T prev = init;
#pragma unroll 8
                for (int i = 1; i < n; ++i) { prev = fma(tp, prev, c[i * st]); c[i * st] = prev; }
            }
            // ---- final value (coeff.py:181-224)
            T fin;
            const ST l = (ST)(n - 1) * st;
            if (a.bound == 0 || a.bound == 2) fin = (tp * c[l - st] + c[l]) * (T)(pole / (pole * pole - 1.0));
            else if (a.bound == 1 || a.bound == 3) fin = c[l] * (T)(pole / (pole - 1.0));
            else {
                const int mi = max_iter0 < n ? max_iter0 : n;
                T s = 0;
                const T *P = wt ? wt + (int64_t)k * (2 * n + 2) + n : nullptr;
                for (int i = 0; i < mi - 1; ++i) s += c[i * st] * (P ? P[i + 2] : (T)pow(pole, (double)(i + 2)));
                fin = (s + tp * c[l]) / (T)(pow(pole, (double)mi) - 1.0);
            }
            c[l] = fin;
            {   // anticausal recursion                                                      coeff.py:277-278
                T nxt = fin;
#pragma unroll 8
                for (int i = n - 2; i >= 0; --i) { nxt = (nxt - c[i * st]) * tp; c[i * st] = nxt; }
            }
        }
    }
}

}  // namespace bfm
