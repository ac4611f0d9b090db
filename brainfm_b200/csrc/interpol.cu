// Spline resampling kernels behind brainfm_b200.interpol (utils/interpol of the reference = torch-interpol 0.2.3).
//   pull / push / count / grad : utils/interpol/nd.py:81-288, iso0.py:24-100, iso1.py:29-387 (forward semantics)
//   bounds                     : utils/interpol/bounds.py:30-89
//   spline weights             : utils/interpol/splines.py:30-160 (orders 0..7)
//   in-bounds mask             : utils/interpol/jit_utils.py:242-255
//   prefilter                  : utils/interpol/coeff.py:35-281
// One thread per sampled point; every channel of the point is processed by that thread so the (order+1)^3 node
// indices / weights are computed once.  Always 3-D: the Python layer pads lower-dimensional problems with
// singleton axes (order 0, coordinate 0).
#include "spline.cuh"

namespace bfm {

// Spline.fastgrad (splines.py:90-147): derivative of the weight wrt the distance
template <typename T>
__device__ __forceinline__ T spline_grad(int order, T xs) {
    if (order == 0) return T(0);
    const T sgn = xs > 0 ? T(1) : (xs < 0 ? T(-1) : T(0));
    const T x = xs < 0 ? -xs : xs;
    T g;
    switch (order) {
        case 1: g = T(1); break;
        case 2: g = x < T(0.5) ? T(-2) * x : x - T(1.5); break;
        case 3: g = x < T(1) ? x * (x * T(1.5) - T(2)) : T(-0.5) * (T(2) - x) * (T(2) - x); break;
        case 4:
            if (x < T(0.5)) g = x * (x * x - T(1.25));
            else if (x < T(1.5)) g = x * (x * (x * (T(-2.) / T(3.)) + T(2.5)) - T(2.5)) + T(5.) / T(24.);
            else { T a = T(2) * x - T(5); g = a * a * a / T(48); }
            break;
        case 5:
            if (x < T(1)) g = x * (x * (x * (x * (T(-5.) / T(12.)) + T(1))) - T(1));
            else if (x < T(2)) g = x * (x * (x * (x * (T(5.) / T(24.)) - T(1.5)) + T(3.75)) - T(3.5)) + T(0.625);
            else { T a = x - T(3); a = a * a; g = a * a / T(-24); }
            break;
        case 6:
            if (x < T(0.5)) { T a = x * x; g = x * (a * (T(7.) / T(12.)) - a * a / T(6) - T(77.) / T(96.)); }
            else if (x < T(1.5)) g = x * (x * (x * (x * (x * T(0.125) - T(35.) / T(48.)) + T(1.3125)) - T(35.) / T(96.)) - T(0.7109375)) - T(7.) / T(768.);
            else if (x < T(2.5)) g = x * (x * (x * (x * (x / T(-20) + T(7.) / T(12.)) - T(2.625)) + T(133.) / T(24.)) - T(5.140625)) + T(1267.) / T(960.);
            else { T a = T(2) * x - T(7); T a2 = a * a; g = a2 * a2 * a / T(3840); }
            break;
        default:
            if (x < T(1)) { T a = x * x; g = x * (a * (a * (x * (T(7.) / T(144.)) - T(1.) / T(6.)) + T(4.) / T(9.)) - T(2.) / T(3.)); }
            else if (x < T(2)) g = x * (x * (x * (x * (x * (x * (T(-7.) / T(240.)) + T(3.) / T(10.)) - T(7.) / T(6.)) + T(2)) - T(7.) / T(6.)) - T(1.) / T(5.)) - T(7.) / T(90.);
            else if (x < T(3)) g = x * (x * (x * (x * (x * (x * (T(7.) / T(720.)) - T(1.) / T(6.)) + T(7.) / T(6.)) - T(38.) / T(9.)) + T(49.) / T(6.)) - T(23.) / T(3.)) + T(217.) / T(90.);
            else { T a = x - T(4); T a2 = a * a; g = a2 * a2 * a2 / T(-720); }
            break;
    }
    return g * sgn;
}

// Spline.fasthess (splines.py:149-195): second derivative of the weight wrt the distance (even in x)
template <typename T>
__device__ __forceinline__ T spline_hess(int order, T xs) {
    if (order <= 1) return T(0);
    const T x = xs < 0 ? -xs : xs;
    switch (order) {
        case 2: return x < T(0.5) ? T(-2) : T(1);
        case 3: return x < T(1) ? T(3) * x - T(2) : T(2) - x;
        case 4:
            if (x < T(0.5)) return T(3) * x * x - T(1.25);
            if (x < T(1.5)) return x * (T(-2) * x + T(5)) - T(2.5);
            { T a = T(2) * x - T(5); return a * a / T(8); }
        case 5:
            if (x < T(1)) { T a = x * x; return -a * (x * (T(5.) / T(3.)) - T(3)) - T(1); }
            if (x < T(2)) return x * (x * (x * (T(5.) / T(6.)) - T(9.) / T(2.)) + T(15.) / T(2.)) - T(7.) / T(2.);
            return T(9.) / T(2.) - x * (x * (x / T(6) - T(3.) / T(2.)) + T(9.) / T(2.));
        case 6:
            if (x < T(0.5)) { T a = x * x; return -a * (a * (T(5.) / T(6.)) - T(7.) / T(4.)) - T(77.) / T(96.); }
            if (x < T(1.5)) return x * (x * (x * (x * (T(5.) / T(8.)) - T(35.) / T(12.)) + T(63.) / T(16.)) - T(35.) / T(48.)) - T(91.) / T(128.);
            if (x < T(2.5)) return -(x * (x * (x * (x / T(4) - T(7.) / T(3.)) + T(63.) / T(8.)) - T(133.) / T(12.)) + T(329.) / T(64.));
            return x * (x * (x * (x / T(24) - T(7.) / T(12.)) + T(49.) / T(16.)) - T(343.) / T(48.)) + T(2401.) / T(384.);
        default:
            if (x < T(1)) { T a = x * x; return a * (a * (x * (T(7.) / T(24.)) - T(5.) / T(6.)) + T(4.) / T(3.)) - T(2.) / T(3.); }
            if (x < T(2)) return -(x * (x * (x * (x * (x * (T(7.) / T(40.)) - T(3.) / T(2.)) + T(14.) / T(3.)) - T(6)) + T(7.) / T(3.)) + T(1.) / T(5.));
            if (x < T(3)) return x * (x * (x * (x * (x * (T(7.) / T(120.)) - T(5.) / T(6.)) + T(14.) / T(3.)) - T(38.) / T(3.)) + T(49.) / T(3.)) - T(23.) / T(3.);
            return -(x * (x * (x * (x * (x / T(120) - T(1.) / T(6.)) + T(4.) / T(3.)) - T(16.) / T(3.)) + T(32.) / T(3.)) - T(128.) / T(15.));
    }
}

struct InterpolArgs {
    int ishape[3];
    int order[3];
    int bound[3];
    int extrapolate;
    int iso;          // 1: every order is 0 => torch.round (half to even) instead of floor(g+0.5) (iso0.py:10-15)
                      // 2: every order is 1 => iso1 gradients (+v1 - v0, iso1.py:269-387); the generic nd path
                      //    uses sign(dist) for order-1 axes (splines.py:90-97), kept as in the reference
    int B, C, Bi, Bg; // output batch, channels, input batch (1 or B), grid batch (1 or B)
    int64_t P;        // points per batch element
};

// MODE_PUSHGRAD / MODE_HESSDOT: the two halves of grid_grad's backward pass (pushpull.py:303-325):
//   PUSHGRAD  inp = incoming gradient (B, C, P, 3) -> out (B, C, *ishape) += sum_d inp_d * d/dg_d(weights)    (nd.py:292-365)
//   HESSDOT   inp = image, gout = incoming gradient (B, C, P, 3) -> out (B, P, 3):
//             out_e = sum_c sum_d gout[c, d] * d2/(dg_d dg_e) pull(inp_c)                         (nd.py:368-465, contracted)
enum { MODE_PULL = 0, MODE_PUSH = 1, MODE_GRAD = 2, MODE_PUSHGRAD = 3, MODE_HESSDOT = 4 };

template <typename T, int MAXN, int MODE>
__global__ void __launch_bounds__(128) k_interpol(const T *__restrict__ inp, const T *__restrict__ grid,
                                                   T *__restrict__ out, const InterpolArgs a,
                                                   const T *__restrict__ gout = nullptr) {
    const int64_t total = (int64_t)a.B * a.P;
    const int64_t vol = (int64_t)a.ishape[0] * a.ishape[1] * a.ishape[2];
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(q / a.P);
        const int64_t p = q - (int64_t)b * a.P;
        const T *g = grid + ((int64_t)(a.Bg == 1 ? 0 : b) * a.P + p) * 3;
        int idx[3][MAXN];
        T w[3][MAXN], gw[3][MAXN], hw[3][MAXN];
        bool inb = true;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const T x = g[d];
            const int n = a.ishape[d], o = a.order[d];
            if (a.extrapolate != 1) {
                const T thr = a.extrapolate == 2 ? T(0.55) : T(0.05);
                inb = inb && (x > -thr) && (x < T(n - 1) + thr);
            }
            T f0;
            if (o == 0 && a.iso == 1) f0 = rint(x);
            else f0 = floor(x - T(o - 1) / T(2));
            const T dist0 = x - f0;
            const int64_t i0 = (int64_t)f0;
#pragma unroll
            for (int k = 0; k < MAXN; ++k) {
                if (k <= o) {
                    const int sg = bound_sign(a.bound[d], i0 + k, n);
                    idx[d][k] = bound_index(a.bound[d], i0 + k, n);
                    const T dist = dist0 - T(k);
                    w[d][k] = (o == 0 ? T(1) : spline_weight<T>(o, dist)) * T(sg);
                    if (MODE == MODE_GRAD || MODE == MODE_PUSHGRAD || MODE == MODE_HESSDOT)
                        gw[d][k] = (a.iso == 2 ? (k == 0 ? T(-1) : T(1)) : spline_grad<T>(o, dist)) * T(sg);
                    if (MODE == MODE_HESSDOT) hw[d][k] = a.iso == 2 ? T(0) : spline_hess<T>(o, dist) * T(sg);
                }
            }
        }
        const T m = inb ? T(1) : T(0);
        if (MODE == MODE_PULL || MODE == MODE_GRAD) {
            for (int c = 0; c < a.C; ++c) {
                const T *src = inp + ((int64_t)(a.Bi == 1 ? 0 : b) * a.C + c) * vol;
                T acc = 0, a0 = 0, a1 = 0, a2 = 0;
                for (int kx = 0; kx <= a.order[0]; ++kx)
                    for (int ky = 0; ky <= a.order[1]; ++ky)
                        for (int kz = 0; kz <= a.order[2]; ++kz) {
                            const T v = src[((int64_t)idx[0][kx] * a.ishape[1] + idx[1][ky]) * a.ishape[2] + idx[2][kz]];
                            if (MODE == MODE_PULL) acc += v * w[0][kx] * w[1][ky] * w[2][kz];
                            else {
                                a0 += v * gw[0][kx] * w[1][ky] * w[2][kz];
                                a1 += v * w[0][kx] * gw[1][ky] * w[2][kz];
                                a2 += v * w[0][kx] * w[1][ky] * gw[2][kz];
                            }
                        }
                if (MODE == MODE_PULL) out[((int64_t)b * a.C + c) * a.P + p] = acc * m;
                else {
                    T *o3 = out + (((int64_t)b * a.C + c) * a.P + p) * 3;
                    o3[0] = a0 * m; o3[1] = a1 * m; o3[2] = a2 * m;
                }
            }
        } else if (MODE == MODE_PUSHGRAD) {
            for (int c = 0; c < a.C; ++c) {
                const T *g3 = inp + (((int64_t)(a.Bi == 1 ? 0 : b) * a.C + c) * a.P + p) * 3;
                const T g0 = g3[0] * m, g1 = g3[1] * m, g2 = g3[2] * m;
                T *dst = out + ((int64_t)b * a.C + c) * vol;
                for (int kx = 0; kx <= a.order[0]; ++kx)
                    for (int ky = 0; ky <= a.order[1]; ++ky)
                        for (int kz = 0; kz <= a.order[2]; ++kz)
                            atomicAdd(dst + ((int64_t)idx[0][kx] * a.ishape[1] + idx[1][ky]) * a.ishape[2] + idx[2][kz],
                                      g0 * gw[0][kx] * w[1][ky] * w[2][kz] + g1 * w[0][kx] * gw[1][ky] * w[2][kz] +
                                          g2 * w[0][kx] * w[1][ky] * gw[2][kz]);
            }
        } else if (MODE == MODE_HESSDOT) {
            T o0 = 0, o1 = 0, o2 = 0;
            for (int c = 0; c < a.C; ++c) {
                const T *src = inp + ((int64_t)(a.Bi == 1 ? 0 : b) * a.C + c) * vol;
                T h00 = 0, h11 = 0, h22 = 0, h01 = 0, h02 = 0, h12 = 0;
                for (int kx = 0; kx <= a.order[0]; ++kx)
                    for (int ky = 0; ky <= a.order[1]; ++ky)
                        for (int kz = 0; kz <= a.order[2]; ++kz) {
                            const T v = src[((int64_t)idx[0][kx] * a.ishape[1] + idx[1][ky]) * a.ishape[2] + idx[2][kz]];
                            h00 += v * hw[0][kx] * w[1][ky] * w[2][kz];
                            h11 += v * w[0][kx] * hw[1][ky] * w[2][kz];
                            h22 += v * w[0][kx] * w[1][ky] * hw[2][kz];
                            h01 += v * gw[0][kx] * gw[1][ky] * w[2][kz];
                            h02 += v * gw[0][kx] * w[1][ky] * gw[2][kz];
                            h12 += v * w[0][kx] * gw[1][ky] * gw[2][kz];
                        }
                const T *g3 = gout + (((int64_t)b * a.C + c) * a.P + p) * 3;
                const T g0 = g3[0], g1 = g3[1], g2 = g3[2];
                o0 += g0 * h00 + g1 * h01 + g2 * h02;
                o1 += g0 * h01 + g1 * h11 + g2 * h12;
                o2 += g0 * h02 + g1 * h12 + g2 * h22;
            }
            T *o3 = out + ((int64_t)b * a.P + p) * 3;
            o3[0] = o0 * m; o3[1] = o1 * m; o3[2] = o2 * m;
        } else {  // push / count (inp == nullptr => ones)
            for (int c = 0; c < a.C; ++c) {
                const T v0 = (inp ? inp[((int64_t)(a.Bi == 1 ? 0 : b) * a.C + c) * a.P + p] : T(1)) * m;
                T *dst = out + ((int64_t)b * a.C + c) * vol;
                for (int kx = 0; kx <= a.order[0]; ++kx)
                    for (int ky = 0; ky <= a.order[1]; ++ky)
                        for (int kz = 0; kz <= a.order[2]; ++kz)
                            atomicAdd(dst + ((int64_t)idx[0][kx] * a.ishape[1] + idx[1][ky]) * a.ishape[2] + idx[2][kz],
                                      v0 * w[0][kx] * w[1][ky] * w[2][kz]);
            }
        }
    }
}


// ---- fast pull: float32, one spline order on every axis (linear or cubic), compile-time unrolled -----------
// Same arithmetic as k_interpol (node indices, bound signs, weights from the same helpers); what changes is the
// memory side: 32-bit element offsets premultiplied by the input strides, so that channels-last inputs (a permuted
// view, e.g. a displacement field) are read in place, with ONE 128-bit load per tap for 4 channels of unit stride;
// weights of a tap are combined once and reused by every channel.
struct PullFastArgs {
    int ishape[3];
    int bound[3];
    int extrapolate;
    int B, C;
    int64_t sB, gB;       // input / grid batch strides (elements); 0 when broadcast
    int sC, sX, sY, sZ;   // input element strides inside one batch element
    int64_t P;
    int out_chlast;       // 0: out (B, C, P);  1: out (B, P, C) (the memory format follows a channels-last input)
};

template <int ORDER, int CV>
__global__ void __launch_bounds__(256) k_pull_fast(const float *__restrict__ inp, const float *__restrict__ grid,
                                                   float *__restrict__ out, const PullFastArgs a) {
    constexpr int NK = ORDER + 1;
    const int64_t total = (int64_t)a.B * a.P;
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= total) return;
    const int b = (int)(q / a.P);
    const int64_t p = q - (int64_t)b * a.P;
    const float *g = grid + (int64_t)b * a.gB + p * 3;
    int off[3][NK];
    float w[3][NK];
    bool inb = true;
    const int strides[3] = {a.sX, a.sY, a.sZ};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float x = __ldg(g + d);
        const int n = a.ishape[d];
        if (a.extrapolate != 1) {
            const float thr = a.extrapolate == 2 ? 0.55f : 0.05f;
            inb = inb && (x > -thr) && (x < float(n - 1) + thr);
        }
        const float f0 = floorf(x - float(ORDER - 1) / 2.f);
        const float dist0 = x - f0;
        const int64_t i0 = (int64_t)f0;
#pragma unroll
        for (int k = 0; k < NK; ++k) {
            const int sg = bound_sign(a.bound[d], i0 + k, n);
            off[d][k] = bound_index(a.bound[d], i0 + k, n) * strides[d];
            w[d][k] = spline_weight<float>(ORDER, dist0 - float(k)) * float(sg);
        }
    }
    const float m = inb ? 1.f : 0.f;
    const float *src = inp + (int64_t)b * a.sB;
    const int64_t oC = a.out_chlast ? 1 : a.P;
    float *dst = out + (int64_t)b * a.C * a.P + (a.out_chlast ? p * a.C : p);
    if (CV >= 2) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int kx = 0; kx < NK; ++kx)
#pragma unroll
            for (int ky = 0; ky < NK; ++ky) {
                const int oxy = off[0][kx] + off[1][ky];
                const float wxy = w[0][kx] * w[1][ky];
#pragma unroll
                for (int kz = 0; kz < NK; ++kz) {
                    const float ww = wxy * w[2][kz];
                    const float *t = src + oxy + off[2][kz];
                    if (CV == 4) {
                        const float4 v = __ldg((const float4 *)t);
                        acc[0] = fmaf(v.x, ww, acc[0]); acc[1] = fmaf(v.y, ww, acc[1]);
                        acc[2] = fmaf(v.z, ww, acc[2]); acc[3] = fmaf(v.w, ww, acc[3]);
                    } else if (CV == 2) {
                        const float2 v = __ldg((const float2 *)t);
                        acc[0] = fmaf(v.x, ww, acc[0]); acc[1] = fmaf(v.y, ww, acc[1]);
                    } else {
                        acc[0] = fmaf(__ldg(t), ww, acc[0]); acc[1] = fmaf(__ldg(t + 1), ww, acc[1]);
                        acc[2] = fmaf(__ldg(t + 2), ww, acc[2]);
                    }
                }
            }
        if (CV == 4 && a.out_chlast) {
            *(float4 *)dst = make_float4(acc[0] * m, acc[1] * m, acc[2] * m, acc[3] * m);
        } else {
#pragma unroll
            for (int c = 0; c < CV; ++c) dst[c * oC] = acc[c] * m;
        }
    } else {
        for (int c = 0; c < a.C; ++c) {
            const float *sc = src + (int64_t)c * a.sC;
            float acc = 0.f;
#pragma unroll
            for (int kx = 0; kx < NK; ++kx)
#pragma unroll
                for (int ky = 0; ky < NK; ++ky) {
                    const int oxy = off[0][kx] + off[1][ky];
                    const float wxy = w[0][kx] * w[1][ky];
#pragma unroll
                    for (int kz = 0; kz < NK; ++kz) acc = fmaf(__ldg(sc + oxy + off[2][kz]), wxy * w[2][kz], acc);
                }
            dst[c * oC] = acc * m;
        }
    }
}

// One scaling-and-squaring step of a displacement field, fused: out = disp + pull(disp, identity + disp) with linear
// interpolation (SURVEY K13; the composition `disp += grid_pull(disp, add_identity_grid(disp))` of BASELINE configs[2]).
// disp, out: (B, X, Y, Z, 3) float32.  Same operations in the same order as k_add_identity followed by
// k_pull_fast<1, 3> and the final add -- identical bits -- but the grid and the pulled field never exist in HBM:
// 24 bytes per voxel and step instead of ~100.
// CS = floats per voxel record: 3 (the caller's layout) or 4 ({d0, d1, d2, 0}: one 128-bit load per trilinear tap
// instead of three 32-bit loads whose 12-byte stride spreads a warp's request over 3-4 cache lines -- 93 -> ~40 L1
// wavefronts per 32 voxels; bfm_exp_velocity keeps the field in this layout between its steps).
template <int CS>
__global__ void __launch_bounds__(256) k_compose_linear3(const float *__restrict__ disp, float *__restrict__ out,
                                                         const PullFastArgs a) {
    const int64_t total = (int64_t)a.B * a.P;
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= total) return;
    const int b = (int)(q / a.P);
    const int64_t p = q - (int64_t)b * a.P;
    const int X = a.ishape[0], Y = a.ishape[1], Z = a.ishape[2];
    const int z = (int)(p % Z);
    const int64_t r = p / Z;
    const int y = (int)(r % Y);
    const int x = (int)(r / Y);
    (void)X;
    float d0, d1, d2;
    if (CS == 4) {
        const float4 v = __ldg((const float4 *)disp + q);
        d0 = v.x; d1 = v.y; d2 = v.z;
    } else {
        const float *dp = disp + q * 3;
        d0 = __ldg(dp); d1 = __ldg(dp + 1); d2 = __ldg(dp + 2);
    }
    const float g[3] = {d0 + (float)x, d1 + (float)y, d2 + (float)z};
    int off[3][2];
    float w[3][2];
    bool inb = true;
    const int strides[3] = {Y * Z * CS, Z * CS, CS};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float xx = g[d];
        const int n = a.ishape[d];
        if (a.extrapolate != 1) {
            const float thr = a.extrapolate == 2 ? 0.55f : 0.05f;
            inb = inb && (xx > -thr) && (xx < float(n - 1) + thr);
        }
        const float f0 = floorf(xx);
        const float dist0 = xx - f0;
        const int64_t i0 = (int64_t)f0;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int sg = bound_sign(a.bound[d], i0 + k, n);
            off[d][k] = bound_index(a.bound[d], i0 + k, n) * strides[d];
            w[d][k] = spline_weight<float>(1, dist0 - float(k)) * float(sg);
        }
    }
    const float m = inb ? 1.f : 0.f;
    const float *src = disp + (int64_t)b * a.P * CS;
    float acc[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int kx = 0; kx < 2; ++kx)
#pragma unroll
        for (int ky = 0; ky < 2; ++ky) {
            const int oxy = off[0][kx] + off[1][ky];
            const float wxy = w[0][kx] * w[1][ky];
#pragma unroll
            for (int kz = 0; kz < 2; ++kz) {
                const float ww = wxy * w[2][kz];
                const float *t = src + oxy + off[2][kz];
                if (CS == 4) {
                    const float4 v = __ldg((const float4 *)t);
                    acc[0] = fmaf(v.x, ww, acc[0]); acc[1] = fmaf(v.y, ww, acc[1]); acc[2] = fmaf(v.z, ww, acc[2]);
                } else {
                    acc[0] = fmaf(__ldg(t), ww, acc[0]); acc[1] = fmaf(__ldg(t + 1), ww, acc[1]);
                    acc[2] = fmaf(__ldg(t + 2), ww, acc[2]);
                }
            }
        }
    if (CS == 4) {
        ((float4 *)out)[q] = make_float4(d0 + acc[0] * m, d1 + acc[1] * m, d2 + acc[2] * m, 0.f);
    } else {
        float *o = out + q * 3;
        o[0] = d0 + acc[0] * m; o[1] = d1 + acc[1] * m; o[2] = d2 + acc[2] * m;
    }
}

// (n, 3) * scale -> (n, 4) records {x, y, z, 0} and back
__global__ void __launch_bounds__(256) k_pack34(const float *__restrict__ src, float4 *__restrict__ dst, int64_t n, float scale) {
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n) return;
    const float *p = src + q * 3;
    dst[q] = make_float4(__ldg(p) * scale, __ldg(p + 1) * scale, __ldg(p + 2) * scale, 0.f);
}
__global__ void __launch_bounds__(256) k_unpack43(const float4 *__restrict__ src, float *__restrict__ dst, int64_t n) {
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n) return;
    const float4 v = __ldg(src + q);
    float *p = dst + q * 3;
    p[0] = v.x; p[1] = v.y; p[2] = v.z;
}

// out = disp + identity grid, (B, X, Y, Z, 3) float32 (add_identity_grid, utils/interpol/api.py:480-521)
__global__ void __launch_bounds__(256) k_add_identity(const float *__restrict__ disp, float *__restrict__ out, int B,
                                                      int X, int Y, int Z) {
    const int64_t total = (int64_t)B * X * Y * Z;
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= total) return;
    const int z = (int)(q % Z);
    const int64_t r = q / Z;
    const int y = (int)(r % Y);
    const int x = (int)((r / Y) % X);
    const float *d = disp + q * 3;
    float *o = out + q * 3;
    o[0] = __ldg(d) + (float)x;
    o[1] = __ldg(d + 1) + (float)y;
    o[2] = __ldg(d + 2) + (float)z;
}


template <typename T>
__global__ void k_spline_filter(T *__restrict__ data, const FilterArgs a) {
    const int64_t lines = a.outer * a.inner;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < lines; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = q / a.inner, in = q - o * a.inner;
        filter_line<T>(data + o * (int64_t)a.n * a.inner + in, a.inner, a);
    }
}

// Tiled float32 prefilter: a block stages L whole lines in shared memory with coalesced 1-pass loads, every thread
// runs the recursion of its own line there (bank-conflict free: pitch L for strided lines, an odd pitch for
// contiguous ones), and the tile is written back once -- one HBM read and one write per element and axis instead
// of the four strided sweeps of the thread-per-line kernel.
__device__ __forceinline__ int pitch_or_n(bool contig, int pitch, int n) { return contig ? pitch : n; }

template <bool CONTIG>
__global__ void __launch_bounds__(128) k_spline_filter_tile(float *__restrict__ data, const FilterArgs a, int L,
                                                            int pitch) {
    extern __shared__ float tile[];
    const int n = a.n, tid = threadIdx.x;
    float *wt = tile + (size_t)L * pitch_or_n(CONTIG, pitch, n);
    for (int e = tid; e < a.npoles * (2 * n + 2); e += blockDim.x) wt[e] = filter_weight(a, e);
    // The element loops keep 8 independent global loads in flight per thread (one load per iteration left the stage
    // long-scoreboard bound: 8.8-12 stalled warps per issue, 0.8 TB/s; profiles/r2_ncu_prefilter_summary.csv) and index
    // with shifts (L == 32) / carry arithmetic instead of divisions.
    constexpr int kU = 8;
    if (CONTIG) {                      // inner == 1: lines [q0, q0+L) are one contiguous run of L*n floats
        const int64_t q0 = (int64_t)blockIdx.x * L;
        const int nl = (int)min((int64_t)L, a.outer - q0);
        float *base = data + q0 * n;
        const int total = nl * n;
        const int dr = blockDim.x / n, dc = blockDim.x - dr * n;
        {
            int row = tid / n, col = tid - row * n;
            for (int e0 = tid; e0 < total; e0 += kU * blockDim.x) {
                float v[kU];
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int e = e0 + u * blockDim.x;
                    v[u] = e < total ? __ldg(base + e) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    if (e0 + u * (int)blockDim.x < total) tile[row * pitch + col] = v[u];
                    row += dr; col += dc;
                    if (col >= n) { col -= n; ++row; }
                }
            }
        }
        __syncthreads();
        if (tid < nl) filter_line<float>(tile + tid * pitch, 1, a, wt);
        __syncthreads();
        {
            int row = tid / n, col = tid - row * n;
            for (int e = tid; e < total; e += blockDim.x) {
                base[e] = tile[row * pitch + col];
                row += dr; col += dc;
                if (col >= n) { col -= n; ++row; }
            }
        }
    } else {                           // lines (o, in0 .. in0+L): element i of line t at data[o*n*inner + i*inner + in0 + t]
        const int64_t per_o = (a.inner + L - 1) / L;
        const int64_t o = blockIdx.x / per_o, in0 = (blockIdx.x % per_o) * L;
        const int nl = (int)min((int64_t)L, a.inner - in0);
        float *base = data + o * (int64_t)n * a.inner + in0;
        const int t = tid & 31, i0 = tid >> 5, di = blockDim.x >> 5;        // L == 32 (host): one row per warp and step
        if (t < nl) {
            const float *src = base + t;
            for (int i = i0; i < n; i += kU * di) {
                float v[kU];
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int ii = i + u * di;
                    v[u] = ii < n ? __ldg(src + (int64_t)ii * a.inner) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int ii = i + u * di;
                    if (ii < n) tile[ii * 32 + t] = v[u];
                }
            }
        }
        __syncthreads();
        if (tid < nl) filter_line<float>(tile + tid, L, a, wt);
        __syncthreads();
        if (t < nl) {
            float *dst = base + t;
            for (int i = i0; i < n; i += di) dst[(int64_t)i * a.inner] = tile[i * 32 + t];
        }
    }
}

template <typename T>
static int launch_interpol(int mode, const void *inp, const void *grid, void *out, const InterpolArgs &a, cudaStream_t s,
                           const void *gout = nullptr) {
    const int maxo = a.order[0] > a.order[1] ? (a.order[0] > a.order[2] ? a.order[0] : a.order[2])
                                             : (a.order[1] > a.order[2] ? a.order[1] : a.order[2]);
    const int64_t total = (int64_t)a.B * a.P;
    int64_t gsz = (total + 127) / 128;
    if (gsz > 148 * 64) gsz = 148 * 64;
    if (gsz < 1) gsz = 1;
    const T *ip = (const T *)inp, *gp = (const T *)grid;
    T *op = (T *)out;
#define BFM_GO(MAXN)                                                                                     \
    do {                                                                                                 \
        if (mode == MODE_PULL) k_interpol<T, MAXN, MODE_PULL><<<(unsigned)gsz, 128, 0, s>>>(ip, gp, op, a);    \
        else if (mode == MODE_PUSH) k_interpol<T, MAXN, MODE_PUSH><<<(unsigned)gsz, 128, 0, s>>>(ip, gp, op, a); \
        else if (mode == MODE_PUSHGRAD) k_interpol<T, MAXN, MODE_PUSHGRAD><<<(unsigned)gsz, 128, 0, s>>>(ip, gp, op, a); \
        else if (mode == MODE_HESSDOT) k_interpol<T, MAXN, MODE_HESSDOT><<<(unsigned)gsz, 128, 0, s>>>(ip, gp, op, a, (const T *)gout); \
        else k_interpol<T, MAXN, MODE_GRAD><<<(unsigned)gsz, 128, 0, s>>>(ip, gp, op, a);                      \
    } while (0)
    if (maxo <= 1) BFM_GO(2);
    else if (maxo <= 3) BFM_GO(4);
    else BFM_GO(8);
#undef BFM_GO
    return check_launch("bfm_interpol");
}
}  // namespace bfm

using namespace bfm;

extern "C" {

int bfm_interpol(int mode, int is_double, const void *inp, const void *grid, void *out, const int *ishape,
                 const int *order, const int *bound, int extrapolate, int iso, int B, int C, int Bi, int Bg,
                 int64_t P, void *stream) {
    BFM_REQUIRE(grid && out && ishape && order && bound, "bfm_interpol: null pointer");
    BFM_REQUIRE(mode >= 0 && mode <= 2, "bfm_interpol: mode must be 0 (pull), 1 (push/count), 2 (grad)");
    BFM_REQUIRE(inp || mode == MODE_PUSH, "bfm_interpol: input required");
    BFM_REQUIRE(B > 0 && C > 0 && P >= 0 && (Bi == 1 || Bi == B) && (Bg == 1 || Bg == B), "bfm_interpol: bad batch");
    InterpolArgs a;
    BFM_REQUIRE(iso >= 0 && iso <= 2, "bfm_interpol: iso must be 0, 1 or 2");
    for (int d = 0; d < 3; ++d) {
        if (ishape[d] <= 0) return fail(BFM_E_INVALID, "%s", "bfm_interpol: non-positive shape");
        if (order[d] < 0 || order[d] > 7) return fail(BFM_E_INVALID, "%s", "bfm_interpol: order must be 0..7");
        if (bound[d] < 0 || bound[d] > 6) return fail(BFM_E_INVALID, "%s", "bfm_interpol: bound must be 0..6");
        a.ishape[d] = ishape[d]; a.order[d] = order[d]; a.bound[d] = bound[d];
    }
    BFM_REQUIRE(extrapolate >= 0 && extrapolate <= 2, "bfm_interpol: extrapolate must be 0, 1 or 2");
    a.extrapolate = extrapolate; a.iso = iso;
    a.B = B; a.C = C; a.Bi = Bi; a.Bg = Bg; a.P = P;
    if (P == 0) return BFM_OK;
    return is_double ? launch_interpol<double>(mode, inp, grid, out, a, (cudaStream_t)stream)
                     : launch_interpol<float>(mode, inp, grid, out, a, (cudaStream_t)stream);
}

int bfm_interpol_grad_backward(int is_double, const void *gout, const void *inp, const void *grid, void *grad_inp,
                               void *grad_grid, const int *ishape, const int *order, const int *bound, int extrapolate,
                               int iso, int B, int C, int64_t P, void *stream) {
    BFM_REQUIRE(gout && inp && grid && ishape && order && bound, "bfm_interpol_grad_backward: null pointer");
    BFM_REQUIRE(B > 0 && C > 0 && P >= 0, "bfm_interpol_grad_backward: bad batch");
    BFM_REQUIRE(iso >= 0 && iso <= 2 && extrapolate >= 0 && extrapolate <= 2, "bfm_interpol_grad_backward: bad option");
    InterpolArgs a;
    for (int d = 0; d < 3; ++d) {
        if (ishape[d] <= 0) return fail(BFM_E_INVALID, "%s", "bfm_interpol_grad_backward: non-positive shape");
        if (order[d] < 0 || order[d] > 7) return fail(BFM_E_INVALID, "%s", "bfm_interpol_grad_backward: order must be 0..7");
        if (bound[d] < 0 || bound[d] > 6) return fail(BFM_E_INVALID, "%s", "bfm_interpol_grad_backward: bound must be 0..6");
        a.ishape[d] = ishape[d]; a.order[d] = order[d]; a.bound[d] = bound[d];
    }
    a.extrapolate = extrapolate; a.iso = iso;
    a.B = B; a.C = C; a.Bi = B; a.Bg = B; a.P = P;
    if (P == 0) return BFM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = BFM_OK;
    if (grad_inp)
        rc = is_double ? launch_interpol<double>(MODE_PUSHGRAD, gout, grid, grad_inp, a, st)
                       : launch_interpol<float>(MODE_PUSHGRAD, gout, grid, grad_inp, a, st);
    if (rc == BFM_OK && grad_grid)
        rc = is_double ? launch_interpol<double>(MODE_HESSDOT, inp, grid, grad_grid, a, st, gout)
                       : launch_interpol<float>(MODE_HESSDOT, inp, grid, grad_grid, a, st, gout);
    return rc;
}

int bfm_interpol_pull_fast(const float *inp, const int64_t *istride, const float *grid, int64_t grid_bstride,
                           float *out, int out_chlast, const int *ishape, int order, const int *bound, int extrapolate,
                           int B, int C, int64_t P, void *stream) {
    BFM_REQUIRE(inp && istride && grid && out && ishape && bound, "bfm_interpol_pull_fast: null pointer");
    BFM_REQUIRE(B > 0 && C > 0 && P >= 0, "bfm_interpol_pull_fast: bad batch");
    BFM_REQUIRE(extrapolate >= 0 && extrapolate <= 2, "bfm_interpol_pull_fast: extrapolate must be 0, 1 or 2");
    if (order != 1 && order != 3) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_interpol_pull_fast: order must be 1 or 3");
    PullFastArgs a;
    int64_t span = 0;
    for (int d = 0; d < 3; ++d) {
        if (ishape[d] <= 0) return fail(BFM_E_INVALID, "%s", "bfm_interpol_pull_fast: non-positive shape");
        if (bound[d] < 0 || bound[d] > 6) return fail(BFM_E_INVALID, "%s", "bfm_interpol_pull_fast: bound must be 0..6");
        if (istride[2 + d] < 0) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_interpol_pull_fast: negative stride");
        a.ishape[d] = ishape[d]; a.bound[d] = bound[d];
        span += (int64_t)(ishape[d] - 1) * istride[2 + d];
    }
    if (istride[0] < 0 || istride[1] < 0) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_interpol_pull_fast: negative stride");
    span += (int64_t)(C - 1) * istride[1];
    if (span >= (1LL << 31)) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_interpol_pull_fast: batch element too large");
    a.extrapolate = extrapolate; a.B = B; a.C = C; a.P = P;
    a.sB = istride[0]; a.sC = (int)istride[1]; a.sX = (int)istride[2]; a.sY = (int)istride[3]; a.sZ = (int)istride[4];
    a.gB = grid_bstride;
    a.out_chlast = out_chlast ? 1 : 0;
    if (a.out_chlast && C == 4 && ((uintptr_t)out % 16) != 0)
        return fail(BFM_E_INVALID, "%s", "bfm_interpol_pull_fast: channels-last output must be 16-byte aligned");
    if (P == 0) return BFM_OK;
    const int64_t total = (int64_t)B * P;
    const int64_t nblocks = (total + 255) / 256;
    if (nblocks >= (1LL << 31)) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_interpol_pull_fast: too many points");
    cudaStream_t s = (cudaStream_t)stream;
    int cv = 0;
    if (a.sC == 1 && C == 3) cv = 3;
    if (a.sC == 1 && C == 4 && ((uintptr_t)inp % 16) == 0 && a.sX % 4 == 0 && a.sY % 4 == 0 && a.sZ % 4 == 0 &&
        a.sB % 4 == 0)
        cv = 4;
    if (a.sC == 1 && C == 2 && ((uintptr_t)inp % 8) == 0 && a.sX % 2 == 0 && a.sY % 2 == 0 && a.sZ % 2 == 0 &&
        a.sB % 2 == 0)
        cv = 2;
#define BFM_PF(O)                                                                                   \
    do {                                                                                            \
        if (cv == 4) k_pull_fast<O, 4><<<(unsigned)nblocks, 256, 0, s>>>(inp, grid, out, a);        \
        else if (cv == 3) k_pull_fast<O, 3><<<(unsigned)nblocks, 256, 0, s>>>(inp, grid, out, a);   \
        else if (cv == 2) k_pull_fast<O, 2><<<(unsigned)nblocks, 256, 0, s>>>(inp, grid, out, a);   \
        else k_pull_fast<O, 0><<<(unsigned)nblocks, 256, 0, s>>>(inp, grid, out, a);                \
    } while (0)
    if (order == 1) BFM_PF(1);
    else BFM_PF(3);
#undef BFM_PF
    return check_launch("bfm_interpol_pull_fast");
}

int bfm_compose_step(const float *disp, float *out, int B, int X, int Y, int Z, const int *bound, int extrapolate,
                     void *stream) {
    BFM_REQUIRE(disp && out && bound && disp != out && B > 0 && X > 0 && Y > 0 && Z > 0, "bfm_compose_step: bad argument");
    BFM_REQUIRE(extrapolate >= 0 && extrapolate <= 2, "bfm_compose_step: extrapolate must be 0, 1 or 2");
    PullFastArgs a;
    a.ishape[0] = X; a.ishape[1] = Y; a.ishape[2] = Z;
    for (int d = 0; d < 3; ++d) {
        if (bound[d] < 0 || bound[d] > 6) return fail(BFM_E_INVALID, "%s", "bfm_compose_step: bound must be 0..6");
        a.bound[d] = bound[d];
    }
    a.extrapolate = extrapolate; a.B = B; a.C = 3; a.P = (int64_t)X * Y * Z;
    if (a.P * 3 >= (1LL << 31)) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_compose_step: field too large for 32-bit offsets");
    a.sB = a.P * 3; a.sC = 1; a.sX = Y * Z * 3; a.sY = Z * 3; a.sZ = 3; a.gB = 0; a.out_chlast = 1;
    const int64_t nblocks = ((int64_t)B * a.P + 255) / 256;
    if (nblocks >= (1LL << 31)) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_compose_step: too many points");
    k_compose_linear3<3><<<(unsigned)nblocks, 256, 0, (cudaStream_t)stream>>>(disp, out, a);
    return check_launch("bfm_compose_step");
}

int bfm_exp_velocity(const float *svf, float *out, int B, int X, int Y, int Z, int steps, const int *bound,
                     int extrapolate, float *scratch, void *stream) {
    BFM_REQUIRE(svf && out && bound && scratch && B > 0 && X > 0 && Y > 0 && Z > 0 && steps >= 0 && steps < 31,
                "bfm_exp_velocity: bad argument");
    BFM_REQUIRE(extrapolate >= 0 && extrapolate <= 2, "bfm_exp_velocity: extrapolate must be 0, 1 or 2");
    BFM_REQUIRE(((uintptr_t)scratch % 16) == 0, "bfm_exp_velocity: scratch must be 16-byte aligned");
    PullFastArgs a;
    a.ishape[0] = X; a.ishape[1] = Y; a.ishape[2] = Z;
    for (int d = 0; d < 3; ++d) {
        if (bound[d] < 0 || bound[d] > 6) return fail(BFM_E_INVALID, "%s", "bfm_exp_velocity: bound must be 0..6");
        a.bound[d] = bound[d];
    }
    a.extrapolate = extrapolate; a.B = B; a.C = 3; a.P = (int64_t)X * Y * Z;
    if (a.P * 4 >= (1LL << 31)) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_exp_velocity: field too large for 32-bit offsets");
    a.sB = a.P * 4; a.sC = 1; a.sX = Y * Z * 4; a.sY = Z * 4; a.sZ = 4; a.gB = 0; a.out_chlast = 1;
    const int64_t n = (int64_t)B * a.P;
    const int64_t nblocks = (n + 255) / 256;
    if (nblocks >= (1LL << 31)) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_exp_velocity: too many points");
    cudaStream_t st = (cudaStream_t)stream;
    float *cur = scratch, *nxt = scratch + n * 4;
    float scale = 1.f;
    for (int q = 0; q < steps; ++q) scale *= 0.5f;                      // svf / 2**steps, exact
    k_pack34<<<(unsigned)nblocks, 256, 0, st>>>(svf, (float4 *)cur, n, scale);
    for (int q = 0; q < steps; ++q) {
        k_compose_linear3<4><<<(unsigned)nblocks, 256, 0, st>>>(cur, nxt, a);
        float *t = cur; cur = nxt; nxt = t;
    }
    k_unpack43<<<(unsigned)nblocks, 256, 0, st>>>((const float4 *)cur, out, n);
    g_launches.fetch_add(steps + 1);
    return check_launch("bfm_exp_velocity");
}

int bfm_add_identity_grid(const float *disp, float *out, int B, int X, int Y, int Z, void *stream) {
    BFM_REQUIRE(disp && out && B > 0 && X > 0 && Y > 0 && Z > 0, "bfm_add_identity_grid: bad argument");
    const int64_t total = (int64_t)B * X * Y * Z;
    const int64_t nblocks = (total + 255) / 256;
    if (nblocks >= (1LL << 31)) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_add_identity_grid: too many points");
    k_add_identity<<<(unsigned)nblocks, 256, 0, (cudaStream_t)stream>>>(disp, out, B, X, Y, Z);
    return check_launch("bfm_add_identity_grid");
}

int bfm_spline_filter(void *data, int is_double, int64_t outer, int n, int64_t inner, int bound, const double *poles_host,
                      int npoles, void *stream) {
    BFM_REQUIRE(data && outer > 0 && n > 0 && inner > 0, "bfm_spline_filter: bad argument");
    BFM_REQUIRE(npoles >= 0 && npoles <= 3, "bfm_spline_filter: at most 3 poles (order <= 7)");
    if (!(bound == 0 || bound == 1 || bound == 2 || bound == 3 || bound == 6))
        return fail(BFM_E_UNSUPPORTED, "%s", "bfm_spline_filter: only zero/replicate/dct1/dct2/dft are implemented");
    if (n == 1 || npoles == 0) return BFM_OK;
    FilterArgs a;
    a.outer = outer; a.inner = inner; a.n = n; a.bound = bound; a.npoles = npoles;
    for (int k = 0; k < 3; ++k) a.poles[k] = k < npoles ? poles_host[k] : 0.0;
    const int64_t lines = outer * inner;
    if (!is_double) {
        // tiled path: L whole lines per block in shared memory (<= 160 KB), L a multiple of 32
        const bool contig = inner == 1;
        const int pitch = contig ? (n | 1) : 0;
        // 32 lines per block: several blocks per SM overlap their load / recursion / store phases
        const int64_t wt_bytes = (int64_t)npoles * (2 * n + 2) * 4;
        int L = (int64_t)32 * (contig ? pitch : n) * 4 + wt_bytes <= 160 * 1024 ? 32 : 0;
        const int64_t nblocks = contig ? (outer + L - 1) / (L > 0 ? L : 1) : outer * ((inner + L - 1) / (L > 0 ? L : 1));
        if (L >= 32 && lines >= 32 && nblocks < (1LL << 31)) {
            const size_t smem = (size_t)L * (contig ? pitch : n) * 4 + (size_t)wt_bytes;
            static bool attr_done = false;
            if (!attr_done) {
                cudaFuncSetAttribute(k_spline_filter_tile<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
                cudaFuncSetAttribute(k_spline_filter_tile<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
                attr_done = true;
            }
            if (contig) k_spline_filter_tile<true><<<(unsigned)nblocks, 128, smem, (cudaStream_t)stream>>>((float *)data, a, L, pitch);
            else k_spline_filter_tile<false><<<(unsigned)nblocks, 128, smem, (cudaStream_t)stream>>>((float *)data, a, L, L);
            return check_launch("bfm_spline_filter");
        }
    }
    int64_t gsz = (lines + 127) / 128;
    if (gsz > 148 * 32) gsz = 148 * 32;
    if (is_double) k_spline_filter<double><<<(unsigned)gsz, 128, 0, (cudaStream_t)stream>>>((double *)data, a);
    else k_spline_filter<float><<<(unsigned)gsz, 128, 0, (cudaStream_t)stream>>>((float *)data, a);
    return check_launch("bfm_spline_filter");
}

}  // extern "C"
