// Fused, batched synthesis chain: BaseGen.generate_sample + augment_sample with the stock steps
// (Generator/datasets.py:306-428).  One launch per stage covers the whole batch (blockIdx.y = sample).
//
//   bbox     deform_grid (datasets.py:264-303): bounding box of the deformed grid.  The coordinate field is
//            multilinear between the nodes of the small random grid, so its extrema sit on the voxels next to
//            node boundaries: only those candidates are evaluated (~10^4 instead of 4*10^6 voxels).  The
//            result is accepted only when floor/ceil cannot be changed by the fp32 evaluation error; otherwise
//            (and for SVF-integrated fields) the full scan runs -- the integers are always exact.
//   gmm      mus[Gr] + sigmas[Gr]*eps, clamp (datasets.py:364-372) over the bbox crop -> syn
//   warp     coordinates -> trilinear gather of syn -> mix -> clamp -> gamma -> bias field
//            (utils.py:140-192, datasets.py:379-411, utils.py:568-589) -> i_bf, bflog_out
//   resample blur o downsample as banded per-axis maps + noise (utils.py:83-94, 591-609, 633-638)
//   finish   myzoom_torch (or, with bspline_zooming, the cubic B-spline resize) back to the grid, global max,
//            normalise, flip (datasets.py:337-352)
//
// Every kernel is instruction-issue bound on B200 (see profiles/), so the code is organised to minimise
// instructions per voxel: the sample descriptor is staged in shared memory, loop invariants live in registers,
// a warp owns several rows so per-k table entries are loaded once, element indices are 32-bit.
#include "spline.cuh"

namespace bfm {

constexpr float kBoxDelta = 1e-3f;   // bound on |computed - exact| source coordinate (see DESIGN.md)

// Pair mode (bfm_gen_sample.syn_pair_ok): the GMM stage writes float2 {synthetic, aux_src[0]} per source voxel and
// k_gen_warp_pk gathers both volumes with one 64-bit load per trilinear tap.
constexpr int kPkNodes = 48;         // z nodes (+1 duplicate of the last) of a small grid that fit k_gen_warp_pk
__host__ __device__ __forceinline__ bool use_pairs(const bfm_gen_sample &s) {
    return s.syn_pair_ok && s.n_aux == 1 && !s.mix[0] && !s.real_input && !(s.d.src[2] & 3) && !s.d.F_full &&
           (!s.d.fsmall || s.d.fs[2] < kPkNodes) && (!s.bfsmall || s.bs[2] < kPkNodes);
}

// Undegraded resolution class (resolution == thickness == the training resolution: identity band, new_size == size):
// the banded pass is a copy and the zoom back is the identity (weights exactly 1 and 0), so those samples take
// k_gen_identity -- noise + clamp straight from i_bf into `out` -- instead of the band and upsample kernels.
__host__ __device__ __forceinline__ bool is_identity_sample(const bfm_gen_sample &s) {
    return s.n_band == 1 && s.band[0].T == 1 && s.band[0].build == 0 && s.x_count == 0 &&
           s.new_size[0] == s.d.size[0] && s.new_size[1] == s.d.size[1] && s.new_size[2] == s.d.size[2] &&
           ((s.d.size[1] * s.d.size[2]) & 3) == 0;
}

// Cubic zoom back (zoom_order == 3, the generator's bspline_zooming): prefilter + cubic pull in the finish stage.  The
// undegraded class keeps k_gen_identity: at integer nodes the cubic pull of the prefiltered coefficients reproduces
// its input up to rounding.
__host__ __device__ __forceinline__ bool cubic_zoom(const bfm_gen_sample &s) {
    return s.zoom_order == 3 && !is_identity_sample(s);
}

__device__ __forceinline__ void stage_desc(bfm_gen_sample *dst, const bfm_gen_sample *src) {
    const int n = (int)(sizeof(bfm_gen_sample) / 4);
    const uint32_t *s = (const uint32_t *)src;
    uint32_t *d = (uint32_t *)dst;
    for (int q = threadIdx.x; q < n; q += blockDim.x) d[q] = __ldg(s + q);
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------- bbox
// Samples of one item (BrainIDGen: several contrasts, one deformation) share ONE bounding box: the box is computed
// by the first of them only -- the in-place float -> int conversions of decide / finish must run exactly once.
__device__ __forceinline__ bool bbox_follower(const bfm_gen_sample *__restrict__ S, int b) {
    return b > 0 && S[b].bbox == S[b - 1].bbox;
}

__global__ void k_gen_bbox_init(const bfm_gen_sample *__restrict__ S) {
    int *bb = S[blockIdx.x].bbox;
    if (!bbox_follower(S, blockIdx.x)) {
        if (threadIdx.x < 3) bb[threadIdx.x] = 0x7f7fffff;
        else if (threadIdx.x < 6) bb[threadIdx.x] = 0;
        else if (threadIdx.x == 6) bb[6] = 1;               // 1 = full scan still required
    }
    if (threadIdx.x == 7) {
        // chain values are >= 0 after the noise clamp and the linear zoom keeps them so: the raw bits order them.  The
        // cubic zoom overshoots below 0 next to clamped zeros: order-preserving encoding from -inf (k_gen_cubic_zoom).
        if (cubic_zoom(S[blockIdx.x])) *(int *)S[blockIdx.x].maxval = f2ord(-INFINITY);
        else *S[blockIdx.x].maxval = 0.f;
    }
    if (threadIdx.x >= 8 && threadIdx.x < 8 + 2 * S[blockIdx.x].n_aux) {
        const int q = threadIdx.x - 8;
        S[blockIdx.x].aux_mm[q] = (q & 1) ? f2ord(-INFINITY) : f2ord(INFINITY);
    }
}

// ---------------------------------------------------------------------------------------------- plan
// Banded map of one axis = (zero-padded Gaussian correlation, utils.py:74-94) followed by (masked 2-tap linear
// sampling at the float64 np.arange positions, utils.py:595-605), built on the device: one block per
// (pass, sample).  Same construction as brainfm_b200.plan.band_host (which the op-level API still uses).
__device__ __forceinline__ void build_band(int n_in, int n_out, int T, double sigma, int *start, float *w) {
    __shared__ float g[64];
    __shared__ float gsum;
    const int half = (T - 2) / 2, L = 2 * half + 1;
    if (L > 64) return;                                    // rejected on the host
    if (sigma > 0.0) {
        // make_gaussian_kernel: float32 tensor ops, the python-float sigma enters as a float32 scalar
        const float sg = (float)sigma;
        for (int t = threadIdx.x; t < L; t += blockDim.x) {
            const float q = __fdiv_rn((float)(t - half), sg);
            g[t] = expf(-__fmul_rn(__fmul_rn(q, q), 0.5f));
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double acc = 0.0;
            for (int t = 0; t < L; ++t) acc += (double)g[t];
            gsum = (float)acc;
        }
        __syncthreads();
        for (int t = threadIdx.x; t < L; t += blockDim.x) g[t] = __fdiv_rn(g[t], gsum);
    } else if (threadIdx.x == 0) {
        g[0] = 1.f;
    }
    __syncthreads();
    // np.arange(delta, delta + n_out/f, 1/f)[:n_out] in float64: start + i*((start+step) - start)
    const double f = (double)n_out / (double)n_in;
    const double delta = (1.0 - f) / (2.0 * f), step = 1.0 / f;
    const double dd = (delta + step) - delta;
    for (int o = threadIdx.x; o < n_out; o += blockDim.x) {
        const float v = (float)(delta + (double)o * dd);
        const bool ok = (v > 0.f) && (v <= (float)(n_in - 1));
        const float fx = floorf(v);
        const int lo = (int)fx, hi = min(lo + 1, n_in - 1);
        const float wh = __fsub_rn(v, fx), wl = __fsub_rn(1.f, wh);
        start[o] = lo - half;
        float *wr = w + (size_t)o * T;
        const bool shift = hi != lo;
        for (int t = 0; t < T; ++t) {
            double acc = 0.0;
            if (ok) {
                if (t < L) acc += (double)wl * (double)g[t];
                if (shift) { if (t >= 1) acc += (double)wh * (double)g[t - 1]; }
                else if (t < L) acc += (double)wh * (double)g[t];
            }
            wr[t] = (float)acc;
        }
    }
}

__global__ void __launch_bounds__(128) k_gen_plan(const bfm_gen_sample *__restrict__ S) {
    const bfm_gen_sample &s = S[blockIdx.y];
    const int pass = blockIdx.x;
    if (pass >= s.n_band) return;
    const bfm_band &b = s.band[pass];
    if (!b.build) return;
    build_band(b.n_in, b.n_out, b.T, b.sigma, const_cast<int *>(b.start), const_cast<float *>(b.w));
}

// Small random grids of the native planner (gen_small): std * N(0,1), Philox streams 2 (deformation) and 3 (bias).
__global__ void __launch_bounds__(256) k_gen_small(const bfm_gen_sample *__restrict__ S) {
    const bfm_gen_sample &s = S[blockIdx.y];
    const int which = blockIdx.z;                       // 0: deformation grid, 1: bias grid
    if (!(s.gen_small & (1 << which))) return;
    float *dst = const_cast<float *>(which == 0 ? s.d.fsmall : s.bfsmall);
    if (!dst) return;
    const int n = which == 0 ? s.d.fs[0] * s.d.fs[1] * s.d.fs[2] * 3 : s.bs[0] * s.bs[1] * s.bs[2];
    const float std = which == 0 ? s.fs_std : s.bf_std;
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; 4 * g < n; g += gridDim.x * blockDim.x) {
        const float4 e = philox_normal4(s.seed, 2u + which, (uint64_t)g);
        const float v[4] = {e.x, e.y, e.z, e.w};
        for (int q = 0; q < 4; ++q)
            if (4 * g + q < n) dst[4 * g + q] = std * v[q];
    }
}

__global__ void __launch_bounds__(128) k_band_build(int n_in, int n_out, int T, double sigma, int *start, float *w) {
    build_band(n_in, n_out, T, sigma, start, w);
}

// all three zoom passes for one voxel -- same operations as the row-wise evaluation
__device__ __forceinline__ void field_direct(const bfm_deform &d, int i, int j, int k, float &f0, float &f1, float &f2) {
    const bfm_zoom_tab &t = d.ftab;
    const int n1 = d.fs[1], n2 = d.fs[2];
    const int x0 = t.lo[0][i], x1 = t.hi[0][i], y0 = t.lo[1][j], y1 = t.hi[1][j], z0 = t.lo[2][k], z1 = t.hi[2][k];
    const float wx0 = t.wl[0][i], wx1 = t.wh[0][i], wy0 = t.wl[1][j], wy1 = t.wh[1][j], wz0 = t.wl[2][k], wz1 = t.wh[2][k];
    float out[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        auto at = [&](int x, int y, int z) { return __ldg(d.fsmall + ((x * n1 + y) * n2 + z) * 3 + c); };
        const float a0 = lerp_rn(wx0, at(x0, y0, z0), wx1, at(x1, y0, z0));
        const float b0 = lerp_rn(wx0, at(x0, y1, z0), wx1, at(x1, y1, z0));
        const float a1 = lerp_rn(wx0, at(x0, y0, z1), wx1, at(x1, y0, z1));
        const float b1 = lerp_rn(wx0, at(x0, y1, z1), wx1, at(x1, y1, z1));
        const float c0 = lerp_rn(wy0, a0, wy1, b0);
        const float c1 = lerp_rn(wy0, a1, wy1, b1);
        out[c] = lerp_rn(wz0, c0, wz1, c1);
    }
    f0 = out[0]; f1 = d.photo ? 0.f : out[1]; f2 = out[2];
}

__device__ __forceinline__ void block_minmax_atomic(float lo[3], float hi[3], int *bb_bits) {
    __shared__ float red[32][6];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        lo[a] = warp_min(lo[a]);
        hi[a] = warp_max(hi[a]);
    }
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            red[warp][a] = lo[a];
            red[warp][3 + a] = hi[a];
        }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float v = red[0][threadIdx.x];
        for (int w = 1; w < nw; ++w) v = threadIdx.x < 3 ? fminf(v, red[w][threadIdx.x]) : fmaxf(v, red[w][threadIdx.x]);
        // coordinates are >= 0 after the clamp: the raw bit pattern is order preserving
        if (threadIdx.x < 3) atomicMin(bb_bits + threadIdx.x, __float_as_int(v));
        else atomicMax(bb_bits + threadIdx.x, __float_as_int(v));
    }
}

__global__ void __launch_bounds__(256) k_gen_bbox_cand(const bfm_gen_sample *__restrict__ S) {
    __shared__ bfm_gen_sample sd;
    if (bbox_follower(S, blockIdx.y)) return;
    stage_desc(&sd, S + blockIdx.y);
    const bfm_deform &d = sd.d;
    if (d.F_full || d.ncand[0] <= 0) return;                // no structure to exploit: full scan
    const int n0 = d.ncand[0], n1 = d.ncand[1], n2 = d.ncand[2];
    const int total = n0 * n1 * n2;
    if ((int)(blockIdx.x * blockDim.x) >= total) return;
    const DefRegs g = load_def(d);
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {0.f, 0.f, 0.f};
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < total) {
        const int c = p % n2, b = (p / n2) % n1, a = p / (n1 * n2);
        const int i = __ldg(d.cand[0] + a), j = __ldg(d.cand[1] + b), k = __ldg(d.cand[2] + c);
        float x1 = __fsub_rn((float)i, g.ctr0), y1 = __fsub_rn((float)j, g.ctr1), z1 = __fsub_rn((float)k, g.ctr2);
        if (d.fsmall) {
            float f0, f1, f2;
            field_direct(d, i, j, k, f0, f1, f2);
            x1 = __fadd_rn(x1, f0); y1 = __fadd_rn(y1, f1); z1 = __fadd_rn(z1, f2);
        }
        float px, py, pz;
        affine_clamp(g, x1, y1, z1, px, py, pz);
        lo[0] = hi[0] = px; lo[1] = hi[1] = py; lo[2] = hi[2] = pz;
    }
    block_minmax_atomic(lo, hi, sd.bbox);
}

__global__ void k_gen_bbox_decide(const bfm_gen_sample *__restrict__ S) {
    if (bbox_follower(S, blockIdx.x)) return;
    const bfm_gen_sample &s = S[blockIdx.x];
    int *bb = s.bbox;
    __shared__ int ambiguous;
    if (threadIdx.x == 0) ambiguous = (s.d.F_full || s.d.ncand[0] <= 0) ? 1 : 0;
    __syncthreads();
    int result = 0;
    if (threadIdx.x < 6) {
        const int a = threadIdx.x % 3;
        const float v = __int_as_float(bb[threadIdx.x]);
        bool exact;
        if (threadIdx.x < 3) {
            // true minimum over all voxels lies in [v - 2*delta, v] and is >= 0
            exact = (v == 0.f) || (floorf(v - 2.f * kBoxDelta) == floorf(v));
            result = (int)floorf(v);
        } else {
            exact = (v == (float)(s.d.src[a] - 1)) || (ceilf(v + 2.f * kBoxDelta) == ceilf(v));
            result = 1 + (int)ceilf(v);
        }
        if (!exact) atomicOr(&ambiguous, 1);
    }
    __syncthreads();
    if (threadIdx.x < 6) bb[threadIdx.x] = ambiguous ? (threadIdx.x < 3 ? 0x7f7fffff : 0) : result;
    if (threadIdx.x == 6) bb[6] = ambiguous;
}

__global__ void __launch_bounds__(kRowWarps * 32) k_gen_bbox_full(const bfm_gen_sample *__restrict__ S, int fstride) {
    extern __shared__ float smem[];
    __shared__ bfm_gen_sample sd;
    if (bbox_follower(S, blockIdx.y)) return;
    if (S[blockIdx.y].bbox[6] == 0) return;                  // candidate result was provably exact
    stage_desc(&sd, S + blockIdx.y);
    const bfm_deform &d = sd.d;
    const DefRegs g = load_def(d);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *smF = smem + warp * kRowsPerWarp * fstride;
    const int n_rows = g.s0 * g.s1;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {0.f, 0.f, 0.f};
    // persistent blocks (the scan is rarely needed: an early exit must not cost a launch of thousands of blocks)
    for (int chunk = blockIdx.x; chunk * kRowWarps * kRowsPerWarp < n_rows; chunk += gridDim.x) {
        const int row0 = (chunk * kRowWarps + warp) * kRowsPerWarp;
        if (row0 < n_rows) {
            deform_rows<kRowsPerWarp>(d, g, smF, row0, n_rows, lane, [](int) {},
                                      [&](int, int, int, int, int, float px, float py, float pz) {
                                          lo[0] = fminf(lo[0], px); hi[0] = fmaxf(hi[0], px);
                                          lo[1] = fminf(lo[1], py); hi[1] = fmaxf(hi[1], py);
                                          lo[2] = fminf(lo[2], pz); hi[2] = fmaxf(hi[2], pz);
                                      });
        }
        __syncwarp();
    }
    block_minmax_atomic(lo, hi, sd.bbox);
}

// Slab mode: source x range of the owned output planes [x_begin, x_begin + x_count) -> gmm_xr (see bfm.h).
// init: {+inf bits, 0}; scan: persistent blocks over the slab's rows; finish: floor(min), 1 + ceil(max).
__global__ void k_gen_slab_xr_init(const bfm_gen_sample *__restrict__ S) {
    const bfm_gen_sample &s = S[blockIdx.x];
    if (s.gmm_xr && s.x_count > 0 && threadIdx.x < 2) s.gmm_xr[threadIdx.x] = threadIdx.x ? 0 : 0x7f7fffff;
}

// Candidate form (same argument as k_gen_bbox_cand): between two kinks of the zoom weights the clamped source coordinate
// is affine in the voxel index, so over the slab [c0, c1) x all j x all k its extrema sit on the candidate voxels with
// i in (candidates of axis 0 inside the slab) + {c0, c1 - 1}: ~10^4 evaluations instead of the slab's voxels.  The
// range only has to be a superset, so k_gen_slab_xr_finish widens it by the evaluation-error bound instead of
// falling back to a scan.  SVF-integrated fields / missing candidate lists take the scan (k_gen_slab_xr).
__global__ void __launch_bounds__(256) k_gen_slab_xr_cand(const bfm_gen_sample *__restrict__ S) {
    __shared__ bfm_gen_sample sd;
    __shared__ float red[8][2];
    {
        const bfm_gen_sample &s0 = S[blockIdx.y];
        if (!s0.gmm_xr || s0.x_count <= 0 || s0.d.F_full || s0.d.ncand[0] <= 0) return;
        const int total0 = (s0.d.ncand[0] + 2) * s0.d.ncand[1] * s0.d.ncand[2];
        if ((int)(blockIdx.x * blockDim.x) >= total0) return;
    }
    stage_desc(&sd, S + blockIdx.y);
    const bfm_deform &d = sd.d;
    const int n0 = d.ncand[0] + 2, n1 = d.ncand[1], n2 = d.ncand[2];
    const int total = n0 * n1 * n2;
    const DefRegs g = load_def(d);
    const int c0 = sd.x_begin, c1 = sd.x_begin + sd.x_count;
    float lo = INFINITY, hi = 0.f;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < total) {
        const int c = p % n2, b = (p / n2) % n1, a = p / (n1 * n2);
        const int i = a < n0 - 2 ? __ldg(d.cand[0] + a) : (a == n0 - 2 ? c0 : c1 - 1);
        if (i >= c0 && i < c1) {
            const int j = __ldg(d.cand[1] + b), k = __ldg(d.cand[2] + c);
            float x1 = __fsub_rn((float)i, g.ctr0), y1 = __fsub_rn((float)j, g.ctr1), z1 = __fsub_rn((float)k, g.ctr2);
            if (d.fsmall) {
                float f0, f1, f2;
                field_direct(d, i, j, k, f0, f1, f2);
                x1 = __fadd_rn(x1, f0); y1 = __fadd_rn(y1, f1); z1 = __fadd_rn(z1, f2);
            }
            float px, py, pz;
            affine_clamp(g, x1, y1, z1, px, py, pz);
            lo = hi = px;
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    lo = warp_min(lo); hi = warp_max(hi);
    if (lane == 0) { red[warp][0] = lo; red[warp][1] = hi; }
    __syncthreads();
    if (threadIdx.x < 2) {
        float v = red[0][threadIdx.x];
        for (int w = 1; w < nw; ++w) v = threadIdx.x ? fmaxf(v, red[w][1]) : fminf(v, red[w][0]);
        if (threadIdx.x) atomicMax(sd.gmm_xr + 1, __float_as_int(v));
        else atomicMin(sd.gmm_xr, __float_as_int(v));
    }
}

__global__ void __launch_bounds__(kRowWarps * 32) k_gen_slab_xr(const bfm_gen_sample *__restrict__ S, int fstride) {
    extern __shared__ float smem[];
    __shared__ bfm_gen_sample sd;
    __shared__ float red[32][2];
    {
        const bfm_gen_sample &s0 = S[blockIdx.y];
        if (!s0.gmm_xr || s0.x_count <= 0) return;
        if (!s0.d.F_full && s0.d.ncand[0] > 0) return;          // k_gen_slab_xr_cand covers it
    }
    stage_desc(&sd, S + blockIdx.y);
    const bfm_deform &d = sd.d;
    const DefRegs g = load_def(d);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    float *smF = smem + warp * kRowsPerWarp * fstride;
    const int first = sd.x_begin * g.s1, n_rows = (sd.x_begin + sd.x_count) * g.s1;
    float lo = INFINITY, hi = 0.f;
    for (int chunk = blockIdx.x; first + chunk * kRowWarps * kRowsPerWarp < n_rows; chunk += gridDim.x) {
        const int row0 = first + (chunk * kRowWarps + warp) * kRowsPerWarp;
        if (row0 < n_rows) {
            deform_rows<kRowsPerWarp>(d, g, smF, row0, n_rows, lane, [](int) {},
                                      [&](int, int, int, int, int, float px, float, float) {
                                          lo = fminf(lo, px); hi = fmaxf(hi, px);
                                      });
        }
        __syncwarp();
    }
    lo = warp_min(lo); hi = warp_max(hi);
    if (lane == 0) { red[warp][0] = lo; red[warp][1] = hi; }
    __syncthreads();
    if (threadIdx.x < 2) {
        float v = red[0][threadIdx.x];
        for (int w = 1; w < nw; ++w) v = threadIdx.x ? fmaxf(v, red[w][1]) : fminf(v, red[w][0]);
        if (threadIdx.x) atomicMax(sd.gmm_xr + 1, __float_as_int(v));      // coordinates >= 0: bit order == float order
        else atomicMin(sd.gmm_xr, __float_as_int(v));
    }
}

__global__ void k_gen_slab_xr_finish(const bfm_gen_sample *__restrict__ S) {
    const bfm_gen_sample &s = S[blockIdx.x];
    if (!s.gmm_xr || s.x_count <= 0) return;
    // 2 * kBoxDelta: bound on |candidate extremum - true extremum| (DESIGN.md, bounding box); a superset is harmless
    if (threadIdx.x == 0) s.gmm_xr[0] = max(0, (int)floorf(__int_as_float(s.gmm_xr[0]) - 2.f * kBoxDelta));
    else if (threadIdx.x == 1) s.gmm_xr[1] = 1 + (int)ceilf(__int_as_float(s.gmm_xr[1]) + 2.f * kBoxDelta);
}

__global__ void k_gen_bbox_finish(const bfm_gen_sample *__restrict__ S) {
    if (bbox_follower(S, blockIdx.x)) return;
    int *bb = S[blockIdx.x].bbox;
    if (bb[6] == 0) return;
    __syncthreads();
    // lo = floor(min), hi = 1 + ceil(max)   (datasets.py:288-293)
    if (threadIdx.x < 3) bb[threadIdx.x] = (int)floorf(__int_as_float(bb[threadIdx.x]));
    else if (threadIdx.x < 6) bb[threadIdx.x] = 1 + (int)ceilf(__int_as_float(bb[threadIdx.x]));
}

// ---------------------------------------------------------------------------------------------- gmm
// One thread = 4 consecutive source voxels along z (one 32-bit label load, one 128-bit store).
__device__ __forceinline__ int label_index(float g) {
    if (g == 77.f) g = 2.f;                       // datasets.py:366
    int r = __float2int_rn(g);                    // torch.round: half to even
    return min(max(r, 0), 255);
}

// Vector path (n2 % 4 == 0): block = one x plane of the crop (blockIdx.y) and one of gridDim.x tiles of its rows;
// the 512-entry mean/std table is loaded once per block and the threads walk the (row, z-group) items of the tile
// with carry arithmetic (no division in the loop).  Only the handful of descriptor fields the stage needs is read.
__global__ void __launch_bounds__(256) k_gen_gmm_planes(const bfm_gen_sample *__restrict__ S) {
    __shared__ float lut[512];
    const bfm_gen_sample *sp = S + blockIdx.z;
    const int n0 = sp->d.src[0], n1 = sp->d.src[1], n2 = sp->d.src[2];
    if ((n2 & 3) || sp->real_input) return;                        // handled by k_gen_gmm / nothing to synthesise
    const int *bb = sp->bbox;
    const int b0 = bb[0], b1 = bb[1], b2 = bb[2], e0 = bb[3], e1 = bb[4], e2 = bb[5];
    const int x = b0 + blockIdx.y;
    if (x >= e0 || x >= n0) return;
    if (sp->gmm_xr && sp->x_count > 0 && (x < sp->gmm_xr[0] || x >= sp->gmm_xr[1])) return;   // slab mode: reachable planes
    // rows of this tile
    const int rows = e1 - b1, per = (rows + gridDim.x - 1) / gridDim.x;
    const int ya = b1 + blockIdx.x * per, yb = min(ya + per, e1);
    if (ya >= yb) return;
    const float *mu = sp->mu, *sigma = sp->sigma;
    for (int q = threadIdx.x; q < 512; q += blockDim.x) lut[q] = q < 256 ? __ldg(mu + q) : __ldg(sigma + q - 256);
    __syncthreads();
    const int zg0 = b2 >> 2, wz = ((e2 + 3) >> 2) - zg0;           // z groups touched by the crop
    if (wz <= 0) return;
    const int items = (yb - ya) * wz;
    const int dy = blockDim.x / wz, dz = blockDim.x - dy * wz;      // one step of blockDim.x items
    int y = ya + threadIdx.x / wz, zg = zg0 + threadIdx.x % wz;
    const float *__restrict__ eps = sp->eps_gmm;
    const void *labels = sp->labels;
    const int is_u8 = sp->label_is_u8;
    const uint64_t seed = sp->seed;
    float *__restrict__ syn = sp->syn;
    const float *__restrict__ pair_src = use_pairs(*sp) ? sp->aux_src[0] : nullptr;
    const int c1 = e1 - b1, c2 = e2 - b2;
    for (int f = threadIdx.x; f < items; f += blockDim.x) {
        const int z = zg << 2;
        const int p0 = (x * n1 + y) * n2 + z;
        float ev[4];
        if (!eps) {
            const float4 e = philox_normal4(seed, 0u, (uint64_t)(p0 >> 2));
            ev[0] = e.x; ev[1] = e.y; ev[2] = e.z; ev[3] = e.w;
        } else {
            const float *er = eps + ((x - b0) * c1 + (y - b1)) * c2 - b2;
#pragma unroll
            for (int q = 0; q < 4; ++q) ev[q] = (z + q >= b2 && z + q < e2) ? __ldg(er + z + q) : 0.f;
        }
        int lab[4];
        if (is_u8) {
            const uint32_t w = __ldg((const uint32_t *)((const uint8_t *)labels + p0));
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int l = (w >> (8 * q)) & 0xff;
                lab[q] = (l == 77) ? 2 : l;
            }
        } else {
            const float4 v = __ldg((const float4 *)((const float *)labels + p0));
            lab[0] = label_index(v.x); lab[1] = label_index(v.y); lab[2] = label_index(v.z); lab[3] = label_index(v.w);
        }
        float o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float v = __fadd_rn(lut[lab[q]], __fmul_rn(lut[256 + lab[q]], ev[q]));
            o[q] = v < 0.f ? 0.f : v;
        }
        // positions just outside the crop are never gathered with a non-zero weight; writing them keeps the
        // store 128-bit (the values are finite, which is all the warp kernel's always-read hi taps need)
        if (pair_src) {                  // pair mode: {synthetic, real-image target} per voxel
            const float4 t = __ldg((const float4 *)(pair_src + p0));
            float4 *dst = (float4 *)(syn + 2 * (size_t)p0);
            dst[0] = make_float4(o[0], t.x, o[1], t.y);
            dst[1] = make_float4(o[2], t.z, o[3], t.w);
        } else {
            *(float4 *)(syn + p0) = make_float4(o[0], o[1], o[2], o[3]);
        }
        y += dy; zg += dz;
        if (zg >= zg0 + wz) { zg -= wz; ++y; }
    }
}

__global__ void __launch_bounds__(256) k_gen_gmm(const bfm_gen_sample *__restrict__ S) {
    __shared__ bfm_gen_sample sd;
    __shared__ float lut[512];
    stage_desc(&sd, S + blockIdx.y);
    const bfm_gen_sample &s = sd;
    const int n0 = s.d.src[0], n1 = s.d.src[1], n2 = s.d.src[2];
    if ((n2 & 3) == 0 || s.real_input) return;       // handled by k_gen_gmm_planes / nothing to synthesise
    const int total = n0 * n1 * n2;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int blk0 = blockIdx.x * blockDim.x * 4;
    if (blk0 >= total) return;
    {   // whole block outside the crop slab along x?  (blocks cover contiguous flat ranges)
        const int xa = blk0 / (n1 * n2), xb = min(blk0 + (int)blockDim.x * 4 - 1, total - 1) / (n1 * n2);
        if (xb < s.bbox[0] || xa >= s.bbox[3]) return;
        if (s.gmm_xr && s.x_count > 0 && (xb < s.gmm_xr[0] || xa >= s.gmm_xr[1])) return;      // slab mode
    }
    for (int q = threadIdx.x; q < 512; q += blockDim.x) lut[q] = q < 256 ? __ldg(s.mu + q) : __ldg(s.sigma + q - 256);
    __syncthreads();
    const int p0 = g * 4;
    if (p0 >= total) return;
    const int b0 = s.bbox[0], b1 = s.bbox[1], b2 = s.bbox[2], e0 = s.bbox[3], e1 = s.bbox[4], e2 = s.bbox[5];
    const int z = p0 % n2, y = (p0 / n2) % n1, x = p0 / (n1 * n2);
    const bool vec = ((n2 & 3) == 0);
    if (vec && (x < b0 || x >= e0 || y < b1 || y >= e1 || z + 3 < b2 || z >= e2)) return;
    const int c1 = e1 - b1, c2 = e2 - b2;
    float ev[4] = {0.f, 0.f, 0.f, 0.f};
    if (!s.eps_gmm) {
        const float4 e = philox_normal4(s.seed, 0u, (uint64_t)g);
        ev[0] = e.x; ev[1] = e.y; ev[2] = e.z; ev[3] = e.w;
    }
    int lab[4];
    if (vec && s.label_is_u8) {
        const uint32_t w = __ldg((const uint32_t *)((const uint8_t *)s.labels + p0));
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int l = (w >> (8 * q)) & 0xff;
            lab[q] = (l == 77) ? 2 : l;
        }
    } else if (vec) {
        const float4 f = __ldg((const float4 *)((const float *)s.labels + p0));
        lab[0] = label_index(f.x); lab[1] = label_index(f.y); lab[2] = label_index(f.z); lab[3] = label_index(f.w);
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int p = p0 + q;
            if (p >= total) { lab[q] = 0; continue; }
            if (s.label_is_u8) {
                const int l = ((const uint8_t *)s.labels)[p];
                lab[q] = (l == 77) ? 2 : l;
            } else {
                lab[q] = label_index(((const float *)s.labels)[p]);
            }
        }
    }
    float outv[4];
    bool inside[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int p = p0 + q;
        int zz = z + q, yy = y, xx = x;
        if (!vec && zz >= n2) {               // group straddles a row end (only when n2 % 4 != 0)
            zz = p % n2; yy = (p / n2) % n1; xx = p / (n1 * n2);
        }
        inside[q] = p < total && xx >= b0 && xx < e0 && yy >= b1 && yy < e1 && zz >= b2 && zz < e2;
        float ee = ev[q];
        if (s.eps_gmm && inside[q]) ee = __ldg(s.eps_gmm + ((xx - b0) * c1 + (yy - b1)) * c2 + (zz - b2));
        const float v = __fadd_rn(lut[lab[q]], __fmul_rn(lut[256 + lab[q]], ee));
        outv[q] = v < 0.f ? 0.f : v;
    }
    if (vec) {
        // positions just outside the crop are never gathered; writing them keeps the store 128-bit
        *(float4 *)(s.syn + p0) = make_float4(outv[0], outv[1], outv[2], outv[3]);
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (inside[q]) s.syn[p0 + q] = outv[q];
    }
}

// ---------------------------------------------------------------------------------------------- warp
// pow / exp forms: ex2.approx(gamma * lg2.approx(x)) and ex2.approx(x*log2e); relative error ~1e-6, inside the
// 1e-5 parity tolerance (the reference's own CPU and CUDA pow differ at that level).
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_pow(float x, float g) { return ex2_approx(g * lg2_approx(x)); }

// Thread = one z index k, persistent over the rows (i, j0..j1) of its block: everything that depends only on k
// (third-pass zoom entries of the deformation and bias grids, centred coordinate) lives in registers for the
// whole block; everything that depends only on i (first zoom pass over the small grids) is evaluated once per
// block into shared memory; everything that depends only on (i, j) (second pass) once per row, kWR rows per
// barrier, double buffered.  A voxel then costs the third pass + affine + 8 (+8 per real-image target) gathers.
//
// Gathers always read the (lo, lo+1) pair per axis: when lo is the last index of the crop the coordinate sits
// exactly on it, the hi weight is 0 and hi = min(lo+1, n-1) (utils.py:148-149) contributes nothing; the buffers
// carry tail padding and only finite values so that 0 * neighbour == 0.
// The coordinate path keeps the reference's separately rounded operations (bit-exact coordinates); the
// interpolation of VALUES uses a + w*(b-a) with one FMA per lerp (<= 1 ulp from the reference's w0*a + w1*b).
#ifndef WARP_ROWS
#define WARP_ROWS 4
#endif
constexpr int kWR = WARP_ROWS;    // rows per barrier
#ifndef WARP_PIPE
#define WARP_PIPE 2
#endif
constexpr int kWP = WARP_PIPE;    // rows whose gathers are in flight together (divides kWR)
constexpr int kT2 = 128;          // floats per second-pass row: 3*fs[2] + bs[2] <= kT2
#ifndef WARP_MINB
#define WARP_MINB 4
#endif

struct WarpShared {
    bfm_gen_sample sd;
    float t2[2][kWR][kT2];
    float red[8][2 * BFM_MAX_AUX];
};

// FIELD: 0 = affine only, 1 = small random grid zoomed on the fly, 2 = full-resolution (SVF-integrated) field
template <int NAUX, bool MIX, int FIELD>
__device__ __forceinline__ void warp_rows(WarpShared &sh, float *t1F, float *t1B, int rpb) {
    const bfm_gen_sample &s = sh.sd;
    const bfm_deform &d = s.d;
    const DefRegs g = load_def(d);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
    const int i = (s.x_count > 0 ? s.x_begin : 0) + blockIdx.y;
    const int j0 = blockIdx.x * rpb, j1 = min(j0 + rpb, g.s1);
    const float *__restrict__ bfsmall = s.bfsmall;
    const int fw = FIELD == 1 ? d.fs[2] * 3 : 0;      // floats per row of the deformation small grid
    const int bw = bfsmall ? s.bs[2] : 0;
    // ---- first zoom pass (axis 0) at this i: t1F[y][z*3+c], t1B[y][z]                 utils.py:239-240
    if (FIELD == 1) {
        const int lo = __ldg(d.ftab.lo[0] + i), hi = __ldg(d.ftab.hi[0] + i);
        const float wl = __ldg(d.ftab.wl[0] + i), wh = __ldg(d.ftab.wh[0] + i);
        const int n = d.fs[1] * fw;
        const float *a = g.fsmall + lo * n, *b = g.fsmall + hi * n;
        for (int q = tid; q < n; q += blockDim.x) t1F[q] = lerp_rn(wl, __ldg(a + q), wh, __ldg(b + q));
    }
    if (bw) {
        const int lo = __ldg(s.btab.lo[0] + i), hi = __ldg(s.btab.hi[0] + i);
        const float wl = __ldg(s.btab.wl[0] + i), wh = __ldg(s.btab.wh[0] + i);
        const int n = s.bs[1] * bw;
        const float *a = bfsmall + lo * n, *b = bfsmall + hi * n;
        for (int q = tid; q < n; q += blockDim.x) t1B[q] = lerp_rn(wl, __ldg(a + q), wh, __ldg(b + q));
    }
    __syncthreads();
    // ---- second pass (axis 1) for kWR rows starting at jj into buffer `buf`           utils.py:241-243
    auto ypass = [&](int jj, int buf) {
        for (int r = warp; r < kWR; r += nwarps) {
            const int j = min(jj + r, g.s1 - 1);
            float *row = sh.t2[buf][r];
            if (FIELD == 1) {
                const int lo = __ldg(d.ftab.lo[1] + j) * fw, hi = __ldg(d.ftab.hi[1] + j) * fw;
                const float wl = __ldg(d.ftab.wl[1] + j), wh = __ldg(d.ftab.wh[1] + j);
                for (int q = lane; q < fw; q += 32) row[q] = lerp_rn(wl, t1F[lo + q], wh, t1F[hi + q]);
            }
            if (bw) {
                const int lo = __ldg(s.btab.lo[1] + j) * bw, hi = __ldg(s.btab.hi[1] + j) * bw;
                const float wl = __ldg(s.btab.wl[1] + j), wh = __ldg(s.btab.wh[1] + j);
                for (int q = lane; q < bw; q += 32) row[fw + q] = lerp_rn(wl, t1B[lo + q], wh, t1B[hi + q]);
            }
        }
    };
    const BoxRegs box = load_box(s.bbox, d.src[1], d.src[2]);
    const int origin = box.b0 * box.n1n2 + box.b1 * box.n2 + box.b2;
    const float *__restrict__ syn = s.syn;
    const float *__restrict__ mix0 = s.mix[0], *__restrict__ mix1 = s.mix[1], *__restrict__ mix2 = s.mix[2];
    const float mw0 = s.mixw[0], mw1 = s.mixw[1], mw2 = s.mixw[2], mw3 = s.mixw[3];
    const float gamma = s.gamma;
    const int real_in = s.real_input;
    float *__restrict__ i_bf = s.i_bf;
    float *__restrict__ bfl = bw ? s.bflog_out : nullptr;
    const float *__restrict__ asrc[NAUX > 0 ? NAUX : 1];
    float *__restrict__ araw[NAUX > 0 ? NAUX : 1];
    float amin[NAUX > 0 ? NAUX : 1], amax[NAUX > 0 ? NAUX : 1];
#pragma unroll
    for (int c = 0; c < NAUX; ++c) { asrc[c] = s.aux_src[c]; araw[c] = s.aux_raw[c]; amin[c] = INFINITY; amax[c] = -INFINITY; }
    const float xc = __fsub_rn((float)i, g.ctr0);
    const int plane_in = i * g.s1, plane_out = (s.flip ? g.s0 - 1 - i : i) * g.s1;
    const bool photo = g.photo != 0;

    for (int k0 = 0; k0 < g.s2; k0 += blockDim.x) {
        const int k = k0 + tid;
        const bool kv = k < g.s2;
        const int kk = kv ? k : g.s2 - 1;
        // ---- everything that only depends on k
        int zlo = 0, zhi = 0, blo = 0, bhi = 0;
        float zwl = 0.f, zwh = 0.f, bwl = 0.f, bwh = 0.f;
        if (FIELD == 1) {
            zlo = __ldg(d.ftab.lo[2] + kk) * 3; zhi = __ldg(d.ftab.hi[2] + kk) * 3;
            zwl = __ldg(d.ftab.wl[2] + kk); zwh = __ldg(d.ftab.wh[2] + kk);
        }
        if (bw) {
            blo = fw + __ldg(s.btab.lo[2] + kk); bhi = fw + __ldg(s.btab.hi[2] + kk);
            bwl = __ldg(s.btab.wl[2] + kk); bwh = __ldg(s.btab.wh[2] + kk);
        }
        const float zc = __fsub_rn((float)kk, g.ctr2);
        int buf = 0;
        ypass(j0, 0);
        __syncthreads();
        for (int jj = j0; jj < j1; jj += kWR) {
            if (jj + kWR < j1) ypass(jj + kWR, buf ^ 1);
            const float *rows = &sh.t2[buf][0][0];
            const float *rzlo = rows + zlo, *rzhi = rows + zhi, *rblo = rows + blo, *rbhi = rows + bhi;
            int p = (plane_in + jj) * g.s2 + kk;                   // element index of (i, jj, k)
            int po = (plane_out + jj) * g.s2 + kk;
            // kWP rows at a time: coordinates and addresses of all of them, then ALL their gathers (8 per row and
            // volume) back to back, then the arithmetic -- the loads of several rows overlap each other's latency
#pragma unroll
            for (int r0 = 0; r0 < kWR; r0 += kWP) {
                if (jj + r0 >= j1) break;
                int e00[kWP];
                float ax[kWP], ay[kWP], az[kWP];
                bool ok[kWP];
#pragma unroll
                for (int q = 0; q < kWP; ++q) {
                    const int r = r0 + q, j = jj + r;
                    float x1 = xc, y1 = __fsub_rn((float)j, g.ctr1), z1 = zc;
                    if (FIELD == 2) {
                        const float *f = g.F_full + (int64_t)(p + r * g.s2) * 3;
                        x1 = __fadd_rn(x1, __ldg(f)); y1 = __fadd_rn(y1, __ldg(f + 1)); z1 = __fadd_rn(z1, __ldg(f + 2));
                    } else if (FIELD == 1) {                                 // third pass (axis 2), utils.py:244-246
                        const float f0 = lerp_rn(zwl, rzlo[r * kT2], zwh, rzhi[r * kT2]);
                        const float f1 = photo ? 0.f : lerp_rn(zwl, rzlo[r * kT2 + 1], zwh, rzhi[r * kT2 + 1]);
                        const float f2 = lerp_rn(zwl, rzlo[r * kT2 + 2], zwh, rzhi[r * kT2 + 2]);
                        x1 = __fadd_rn(x1, f0); y1 = __fadd_rn(y1, f1); z1 = __fadd_rn(z1, f2);
                    }
                    float px, py, pz;
                    affine_clamp(g, x1, y1, z1, px, py, pz);
                    // ---- trilinear taps relative to the crop (fast_3D_interp_torch, utils.py:140-192)
                    const float rx = __fsub_rn(px, box.l0), ry = __fsub_rn(py, box.l1), rz = __fsub_rn(pz, box.l2);
                    ok[q] = (rx > 0.f) & (ry > 0.f) & (rz > 0.f) & (rx <= box.h0) & (ry <= box.h1) & (rz <= box.h2) &
                            (j < j1);
                    const int ix = __float2int_rd(rx), iy = __float2int_rd(ry), iz = __float2int_rd(rz);
                    ax[q] = __fsub_rn(rx, (float)ix); ay[q] = __fsub_rn(ry, (float)iy); az[q] = __fsub_rn(rz, (float)iz);
                    e00[q] = ok[q] ? origin + ix * box.n1n2 + iy * box.n2 + iz : origin;
                }
                float tap[NAUX + 1][kWP][8];
#pragma unroll
                for (int c = 0; c <= NAUX; ++c) {
                    const float *__restrict__ X = c == 0 ? syn : asrc[c > 0 ? c - 1 : 0];
#pragma unroll
                    for (int q = 0; q < kWP; ++q) {
                        const float *b00 = X + e00[q], *b10 = b00 + box.n1n2, *b01 = b00 + box.n2, *b11 = b10 + box.n2;
                        tap[c][q][0] = __ldg(b00); tap[c][q][1] = __ldg(b00 + 1);
                        tap[c][q][2] = __ldg(b10); tap[c][q][3] = __ldg(b10 + 1);
                        tap[c][q][4] = __ldg(b01); tap[c][q][5] = __ldg(b01 + 1);
                        tap[c][q][6] = __ldg(b11); tap[c][q][7] = __ldg(b11 + 1);
                    }
                }
#pragma unroll
                for (int q = 0; q < kWP; ++q) {
                    const int r = r0 + q, j = jj + r;
                    const int pr = p + r * g.s2;
                    auto interp = [&](const float *t) {      // t: 000 001 100 101 010 011 110 111
                        const float c00 = fmaf(ax[q], t[2] - t[0], t[0]), c01 = fmaf(ax[q], t[3] - t[1], t[1]);
                        const float c10 = fmaf(ax[q], t[6] - t[4], t[4]), c11 = fmaf(ax[q], t[7] - t[5], t[5]);
                        const float c0 = fmaf(ay[q], c10 - c00, c00), c1 = fmaf(ay[q], c11 - c01, c01);
                        const float v = fmaf(az[q], c1 - c0, c0);
                        return ok[q] ? v : 0.f;
                    };
                    float v = interp(tap[0][q]);
                    if (MIX) {                                        // datasets.py:379-388
                        v = __fadd_rn(__fmul_rn(mw0, v), __fmul_rn(mw1, mix0[pr]));
                        if (mix1) v = __fadd_rn(v, __fmul_rn(mw2, mix1[pr]));
                        if (mix2) v = __fadd_rn(v, __fmul_rn(mw3, mix2[pr]));
                    }
                    if (real_in == 0) v = fmaxf(v, 0.f);              // datasets.py:411 (synthetic images only)
                    else if (real_in == 2) v = fminf(fmaxf(v, 0.f), 80.f);   // CT window (datasets.py:318-319)
                    // gamma: 300 * (I/300) ** gamma                  utils.py:568-572
                    v = 300.f * fast_pow(v * (1.f / 300.f), gamma);
                    // bias field: I * exp(zoom(BFsmall))             utils.py:574-589
                    float bl = 0.f;
                    if (bw) {
                        bl = lerp_rn(bwl, rblo[r * kT2], bwh, rbhi[r * kT2]);
                        v *= ex2_approx(bl * 1.4426950408889634f);
                    }
                    const bool wr = kv && j < j1;
                    if (wr) {
                        i_bf[pr] = v;
                        if (bfl) bfl[po + r * g.s2] = bl;
                    }
#pragma unroll
                    for (int c = 0; c < NAUX; ++c) {                  // read_and_deform_image: raw warp + min/max
                        const float a = interp(tap[c + 1][q]);
                        if (wr) {
                            araw[c][pr] = a;
                            amin[c] = fminf(amin[c], a);
                            amax[c] = fmaxf(amax[c], a);
                        }
                    }
                }
            }
            __syncthreads();
            buf ^= 1;
        }
    }
    if (NAUX > 0) {
#pragma unroll
        for (int c = 0; c < NAUX; ++c) {
            const float lo = warp_min(amin[c]), hi = warp_max(amax[c]);
            if (lane == 0) { sh.red[warp][2 * c] = lo; sh.red[warp][2 * c + 1] = hi; }
        }
        __syncthreads();
        if (tid < 2 * NAUX) {
            float v = sh.red[0][tid];
            for (int w = 1; w < nwarps; ++w) v = (tid & 1) ? fmaxf(v, sh.red[w][tid]) : fminf(v, sh.red[w][tid]);
            if (tid & 1) atomicMax(s.aux_mm + tid, f2ord(v));
            else atomicMin(s.aux_mm + tid, f2ord(v));
        }
    }
}

template <int NAUX, bool MIX>
__global__ void __launch_bounds__(256, WARP_MINB) k_gen_warp(const bfm_gen_sample *__restrict__ S, int rpb, int t1f_cap) {
    extern __shared__ float smem[];
    __shared__ WarpShared sh;
    {   // each instantiation handles the samples of its own kind
        const bfm_gen_sample *sp = S + blockIdx.z;
        if ((sp->mix[0] != nullptr) != MIX || sp->n_aux != NAUX || use_pairs(*sp)) return;
        const int nx = sp->x_count > 0 ? sp->x_count : sp->d.size[0];
        if ((int)blockIdx.y >= nx || (int)blockIdx.x * rpb >= sp->d.size[1]) return;
    }
    stage_desc(&sh.sd, S + blockIdx.z);
    float *t1F = smem, *t1B = smem + t1f_cap;
    if (sh.sd.d.F_full) warp_rows<NAUX, MIX, 2>(sh, t1F, t1B, rpb);
    else if (sh.sd.d.fsmall) warp_rows<NAUX, MIX, 1>(sh, t1F, t1B, rpb);
    else warp_rows<NAUX, MIX, 0>(sh, t1F, t1B, rpb);
}


// ---------------------------------------------------------------------------------------------- warp, pair mode
// Same arithmetic as warp_rows<1, false, FIELD> for the common sample kind (synthetic input + one real-image target, no
// mixing), reorganised around what the ncu captures of k_gen_warp<1,0> showed (83 % of the L1 data-pipe wavefront
// peak, 220 instructions per voxel):
//   * the GMM stage leaves {synthetic, target} float2 PAIRS per source voxel, so a trilinear tap is ONE 64-bit load for
//     both volumes (8 load requests per voxel instead of 16), and the loaded register pair is directly the operand of
//     the packed f32x2 lerps (14 FFMA2/FADD2 per voxel instead of 28 scalar FFMA/FADD);
//   * a thread evaluates TWO rows (j, j+1) at a time and carries their coordinates as f32x2 pairs: the third zoom pass
//     and the affine map are 27 packed instructions per row pair instead of 54 scalar ones.  The reference's separately
//     rounded `w0*a + w1*b` is FMUL2, FMUL2, FFMA2(x, one, y) -- `one` is an opaque 1.0f kernel parameter because ptxas
//     contracts mul.rn.f32x2 + add.rn.f32x2 into a single FFMA2 (tools/micro/f32x2.cu) -- so coordinates stay bit-exact;
//   * second-pass rows are stored node-major with the two rows of a pair interleaved and the last node duplicated
//     (hi == lo + 1 always): the third pass reads 2 x (LDS.128 + LDS.64) per row pair instead of 12 LDS.32, the bias
//     field 2 LDS.64 instead of 4 LDS.32;
//   * the per-sample affine constants come through the kernel parameters (constant bank -> uniform registers, used as
//     broadcast operands of the packed instructions).
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float a, float b) { u64 r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float2 upk2(u64 v) { float2 o; asm("mov.b64 {%0,%1}, %2;" : "=f"(o.x), "=f"(o.y) : "l"(v)); return o; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ u64 f2u(float2 v) { return pk2(v.x, v.y); }

struct PkSample { float A[9], c2[3], ctr[3], gamma; };
constexpr int kPkBatch = 16;
struct PkParams {
    PkSample s[kPkBatch];
    float one;          // 1.0f, opaque to ptxas
    int base;           // first sample of this launch
};

struct PkShared {
    bfm_gen_sample sd;
    alignas(16) float f2[2][kWR / 2][kPkNodes][8];    // node-major: {c0 r0, c0 r1, c1 r0, c1 r1, c2 r0, c2 r1, -, -}
    alignas(16) float b2[2][kWR / 2][kPkNodes][2];    // {r0, r1}
    float red[8][2];
};

template <int FIELD>
__device__ __forceinline__ void warp_rows_pk(PkShared &sh, float *t1F, float *t1B, int rpb, const PkSample &c,
                                             const float one) {
    const bfm_gen_sample &s = sh.sd;
    const bfm_deform &d = s.d;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
    const int s0 = d.size[0], s1 = d.size[1], s2 = d.size[2];
    const int i = (s.x_count > 0 ? s.x_begin : 0) + blockIdx.y;
    const int j0 = blockIdx.x * rpb, j1 = min(j0 + rpb, s1);
    const float *__restrict__ bfsmall = s.bfsmall;
    const int nf = FIELD == 1 ? d.fs[2] : 0, fw = nf * 3;
    const int nb = bfsmall ? s.bs[2] : 0;
    // ---- first zoom pass (axis 0) at this i: t1F[y][z*3+c], t1B[y][z]                 utils.py:239-240
    if (FIELD == 1) {
        const int lo = __ldg(d.ftab.lo[0] + i), hi = __ldg(d.ftab.hi[0] + i);
        const float wl = __ldg(d.ftab.wl[0] + i), wh = __ldg(d.ftab.wh[0] + i);
        const int n = d.fs[1] * fw;
        const float *a = d.fsmall + lo * n, *b = d.fsmall + hi * n;
        for (int q = tid; q < n; q += blockDim.x) t1F[q] = lerp_rn(wl, __ldg(a + q), wh, __ldg(b + q));
    }
    if (nb) {
        const int lo = __ldg(s.btab.lo[0] + i), hi = __ldg(s.btab.hi[0] + i);
        const float wl = __ldg(s.btab.wl[0] + i), wh = __ldg(s.btab.wh[0] + i);
        const int n = s.bs[1] * nb;
        const float *a = bfsmall + lo * n, *b = bfsmall + hi * n;
        for (int q = tid; q < n; q += blockDim.x) t1B[q] = lerp_rn(wl, __ldg(a + q), wh, __ldg(b + q));
    }
    __syncthreads();
    const bool photo = d.photo != 0;
    // ---- second pass (axis 1) for kWR rows starting at jj into buffer `buf`           utils.py:241-243
    auto ypass = [&](int jj, int buf) {
        for (int r = warp; r < kWR; r += nwarps) {
            const int j = min(jj + r, s1 - 1);
            if (FIELD == 1) {
                const int lo = __ldg(d.ftab.lo[1] + j) * fw, hi = __ldg(d.ftab.hi[1] + j) * fw;
                const float wl = __ldg(d.ftab.wl[1] + j), wh = __ldg(d.ftab.wh[1] + j);
                float *dst = &sh.f2[buf][r >> 1][0][r & 1];
                for (int q = lane; q < fw + 3; q += 32) {             // node nf duplicates node nf - 1
                    const int node = q / 3, ch = q - node * 3, src = min(node, nf - 1) * 3 + ch;
                    const float v = lerp_rn(wl, t1F[lo + src], wh, t1F[hi + src]);
                    dst[node * 8 + ch * 2] = (photo && ch == 1) ? 0.f : v;       // datasets.py:211-212
                }
            }
            if (nb) {
                const int lo = __ldg(s.btab.lo[1] + j) * nb, hi = __ldg(s.btab.hi[1] + j) * nb;
                const float wl = __ldg(s.btab.wl[1] + j), wh = __ldg(s.btab.wh[1] + j);
                float *dst = &sh.b2[buf][r >> 1][0][r & 1];
                for (int q = lane; q <= nb; q += 32) {
                    const int src = min(q, nb - 1);
                    dst[q * 2] = lerp_rn(wl, t1B[lo + src], wh, t1B[hi + src]);
                }
            }
        }
    };
    const BoxRegs box = load_box(s.bbox, d.src[1], d.src[2]);
    const int origin = box.b0 * box.n1n2 + box.b1 * box.n2 + box.b2;
    const float2 *__restrict__ syn2 = (const float2 *)s.syn;
    const float gamma = c.gamma;
    float *__restrict__ i_bf = s.i_bf;
    float *__restrict__ bfl = nb ? s.bflog_out : nullptr;
    float *__restrict__ araw = s.aux_raw[0];
    float amin = INFINITY, amax = -INFINITY;
    const float mx = (float)(d.src[0] - 1), my = (float)(d.src[1] - 1), mz = (float)(d.src[2] - 1);
    const u64 ONE = pk2(one, one);
    const float xc = __fsub_rn((float)i, c.ctr[0]);
    const u64 XC = pk2(xc, xc);
    const u64 NL0 = pk2(-box.l0, -box.l0), NL1 = pk2(-box.l1, -box.l1), NL2 = pk2(-box.l2, -box.l2);
    const int plane_in = i * s1, plane_out = (s.flip ? s0 - 1 - i : i) * s1;

    for (int k0 = 0; k0 < s2; k0 += blockDim.x) {
        const int k = k0 + tid;
        const bool kv = k < s2;
        const int kk = kv ? k : s2 - 1;
        // ---- everything that only depends on k
        int zlo = 0, blo = 0;
        u64 ZWL = 0, ZWH = 0, BWL = 0, BWH = 0;
        if (FIELD == 1) {
            zlo = __ldg(d.ftab.lo[2] + kk);
            const float wl = __ldg(d.ftab.wl[2] + kk), wh = __ldg(d.ftab.wh[2] + kk);
            ZWL = pk2(wl, wl); ZWH = pk2(wh, wh);
        }
        if (nb) {
            blo = __ldg(s.btab.lo[2] + kk);
            const float wl = __ldg(s.btab.wl[2] + kk), wh = __ldg(s.btab.wh[2] + kk);
            BWL = pk2(wl, wl); BWH = pk2(wh, wh);
        }
        const float zc = __fsub_rn((float)kk, c.ctr[2]);
        const u64 ZC = pk2(zc, zc);
        int buf = 0;
        ypass(j0, 0);
        __syncthreads();
        for (int jj = j0; jj < j1; jj += kWR) {
            if (jj + kWR < j1) ypass(jj + kWR, buf ^ 1);
#pragma unroll
            for (int rp = 0; rp < kWR / 2; ++rp) {
                const int j = jj + 2 * rp;
                if (j >= j1) break;
                // ---- coordinates of rows j and j + 1 as f32x2 pairs
                u64 X1 = XC, Y1 = pk2(__fsub_rn((float)j, c.ctr[1]), __fsub_rn((float)(j + 1), c.ctr[1])), Z1 = ZC;
                if (FIELD == 1) {                                    // third pass (axis 2), utils.py:244-246
                    const float4 *fn = (const float4 *)&sh.f2[buf][rp][zlo][0];
                    const float4 l01 = fn[0], h01 = fn[2];
                    const float2 l2 = *(const float2 *)(fn + 1), h2 = *(const float2 *)(fn + 3);
                    const u64 F0 = fma2(mul2(ZWH, pk2(h01.x, h01.y)), ONE, mul2(ZWL, pk2(l01.x, l01.y)));
                    const u64 F1 = fma2(mul2(ZWH, pk2(h01.z, h01.w)), ONE, mul2(ZWL, pk2(l01.z, l01.w)));
                    const u64 F2 = fma2(mul2(ZWH, f2u(h2)), ONE, mul2(ZWL, f2u(l2)));
                    X1 = add2(X1, F0); Y1 = add2(Y1, F1); Z1 = add2(Z1, F2);
                }
                // ((A0*x + A1*y) + A2*z) + c, every product and sum separately rounded (datasets.py:276-278)
                auto affine = [&](const float a0, const float a1, const float a2, const float cc) {
                    const u64 m0 = mul2(pk2(a0, a0), X1), m1 = mul2(pk2(a1, a1), Y1), m2 = mul2(pk2(a2, a2), Z1);
                    return add2(fma2(m2, ONE, fma2(m1, ONE, m0)), pk2(cc, cc));
                };
                const float2 px = upk2(affine(c.A[0], c.A[1], c.A[2], c.c2[0]));
                const float2 py = upk2(affine(c.A[3], c.A[4], c.A[5], c.c2[1]));
                const float2 pz = upk2(affine(c.A[6], c.A[7], c.A[8], c.c2[2]));
                auto clampf = [](float v, float hi) { v = v < 0.f ? 0.f : v; return v > hi ? hi : v; };   // :279-284
                const float2 rx = upk2(add2(pk2(clampf(px.x, mx), clampf(px.y, mx)), NL0));
                const float2 ry = upk2(add2(pk2(clampf(py.x, my), clampf(py.y, my)), NL1));
                const float2 rz = upk2(add2(pk2(clampf(pz.x, mz), clampf(pz.y, mz)), NL2));
                // ---- trilinear taps relative to the crop (fast_3D_interp_torch, utils.py:140-192)
                const float rxa[2] = {rx.x, rx.y}, rya[2] = {ry.x, ry.y}, rza[2] = {rz.x, rz.y};
                int e00[2];
                float ax[2], ay[2], az[2];
                bool ok[2];
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    ok[q] = (rxa[q] > 0.f) & (rya[q] > 0.f) & (rza[q] > 0.f) & (rxa[q] <= box.h0) & (rya[q] <= box.h1) &
                            (rza[q] <= box.h2) & (j + q < j1);
                    const int ix = __float2int_rd(rxa[q]), iy = __float2int_rd(rya[q]), iz = __float2int_rd(rza[q]);
                    ax[q] = __fsub_rn(rxa[q], (float)ix); ay[q] = __fsub_rn(rya[q], (float)iy);
                    az[q] = __fsub_rn(rza[q], (float)iz);
                    e00[q] = ok[q] ? origin + ix * box.n1n2 + iy * box.n2 + iz : origin;
                }
                u64 tap[2][8];                          // {synthetic, target} at 000 001 100 101 010 011 110 111
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const float2 *b00 = syn2 + e00[q], *b10 = b00 + box.n1n2, *b01 = b00 + box.n2, *b11 = b10 + box.n2;
                    tap[q][0] = f2u(__ldg(b00)); tap[q][1] = f2u(__ldg(b00 + 1));
                    tap[q][2] = f2u(__ldg(b10)); tap[q][3] = f2u(__ldg(b10 + 1));
                    tap[q][4] = f2u(__ldg(b01)); tap[q][5] = f2u(__ldg(b01 + 1));
                    tap[q][6] = f2u(__ldg(b11)); tap[q][7] = f2u(__ldg(b11 + 1));
                }
                // bias field rows of the pair                        utils.py:574-589
                float2 bl = make_float2(0.f, 0.f);
                if (nb) {
                    const float2 *bn = (const float2 *)&sh.b2[buf][rp][blo][0];
                    bl = upk2(fma2(mul2(BWH, f2u(bn[1])), ONE, mul2(BWL, f2u(bn[0]))));
                }
                const float bla[2] = {bl.x, bl.y};
                const int pr0 = (plane_in + j) * s2 + kk, po0 = (plane_out + j) * s2 + kk;
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const u64 *t = tap[q];
                    const u64 AX = pk2(ax[q], ax[q]), AY = pk2(ay[q], ay[q]), AZ = pk2(az[q], az[q]);
                    const u64 c00 = fma2(AX, sub2(t[2], t[0]), t[0]), c01 = fma2(AX, sub2(t[3], t[1]), t[1]);
                    const u64 c10 = fma2(AX, sub2(t[6], t[4]), t[4]), c11 = fma2(AX, sub2(t[7], t[5]), t[5]);
                    const u64 c0 = fma2(AY, sub2(c10, c00), c00), c1 = fma2(AY, sub2(c11, c01), c01);
                    const float2 vv = upk2(fma2(AZ, sub2(c1, c0), c0));
                    float v = ok[q] ? vv.x : 0.f;
                    const float a = ok[q] ? vv.y : 0.f;
                    v = fmaxf(v, 0.f);                                // datasets.py:411
                    v = 300.f * fast_pow(v * (1.f / 300.f), gamma);   // utils.py:568-572
                    if (nb) v *= ex2_approx(bla[q] * 1.4426950408889634f);
                    if (kv && j + q < j1) {
                        i_bf[pr0 + q * s2] = v;
                        if (bfl) bfl[po0 + q * s2] = bla[q];
                        araw[pr0 + q * s2] = a;                       // read_and_deform_image: raw warp + min/max
                        amin = fminf(amin, a);
                        amax = fmaxf(amax, a);
                    }
                }
            }
            __syncthreads();
            buf ^= 1;
        }
    }
    {
        const float lo = warp_min(amin), hi = warp_max(amax);
        if (lane == 0) { sh.red[warp][0] = lo; sh.red[warp][1] = hi; }
        __syncthreads();
        if (tid < 2) {
            float v = sh.red[0][tid];
            for (int w = 1; w < nwarps; ++w) v = (tid & 1) ? fmaxf(v, sh.red[w][tid]) : fminf(v, sh.red[w][tid]);
            if (tid & 1) atomicMax(s.aux_mm + tid, f2ord(v));
            else atomicMin(s.aux_mm + tid, f2ord(v));
        }
    }
}

#ifndef WARP_PK_MINB
#define WARP_PK_MINB 4
#endif
__global__ void __launch_bounds__(256, WARP_PK_MINB)
k_gen_warp_pk(const bfm_gen_sample *__restrict__ S, const __grid_constant__ PkParams P, int rpb, int t1f_cap) {
    extern __shared__ float smem[];
    __shared__ PkShared sh;
    const int b = P.base + blockIdx.z;
    {
        const bfm_gen_sample *sp = S + b;
        if (!use_pairs(*sp)) return;
        const int nx = sp->x_count > 0 ? sp->x_count : sp->d.size[0];
        if ((int)blockIdx.y >= nx || (int)blockIdx.x * rpb >= sp->d.size[1]) return;
    }
    stage_desc(&sh.sd, S + b);
    float *t1F = smem, *t1B = smem + t1f_cap;
    if (sh.sd.d.fsmall) warp_rows_pk<1>(sh, t1F, t1B, rpb, P.s[blockIdx.z], P.one);
    else warp_rows_pk<0>(sh, t1F, t1B, rpb, P.s[blockIdx.z], P.one);
}

// ---------------------------------------------------------------------------------------------- resample
// One banded pass.  Axis 0/1: a thread owns VEC consecutive z outputs (128-bit loads when VEC == 4); the tap
// weight is uniform across the warp.  Axis 2: a thread owns one output, taps are contiguous.
#ifndef BAND_UNROLL
#define BAND_UNROLL 4
#endif
constexpr int kBandUnroll = BAND_UNROLL;
template <int VEC>
__global__ void __launch_bounds__(256) k_gen_band(const bfm_gen_sample *__restrict__ S, int pass, int zk_cap) {
    // persistent blocks: a few hundred per sample, each thread walks its outputs with carry arithmetic; only
    // the descriptor fields this pass needs are read (no 936-byte staging per block)
    const bfm_gen_sample &s = S[blockIdx.y];
    const int n_band = s.n_band;
    if (pass >= n_band || is_identity_sample(s)) return;
    int sh0 = s.d.size[0], sh1 = s.d.size[1], sh2 = s.d.size[2];
    for (int q = 0; q < pass; ++q) {
        const int ax = s.band[q].axis, no = s.band[q].n_out;
        if (ax == 0) sh0 = no; else if (ax == 1) sh1 = no; else sh2 = no;
    }
    const bfm_band &b = s.band[pass];
    const int axis = b.axis, T = b.T;
    const int o0 = axis == 0 ? b.n_out : sh0, o1 = axis == 1 ? b.n_out : sh1, o2 = axis == 2 ? b.n_out : sh2;
    if (VEC == 4 && (axis == 2 || (sh2 & 3))) return;        // handled by the scalar instantiation / k_gen_band_z
    if (VEC == 1 && !(axis == 2 || (sh2 & 3))) return;
    if (VEC == 1 && axis == 2 && zk_cap > 0 &&
        ((b.n_out * ((T | 1) + 1) + 8 * (sh2 + b.n_out + 4)) * 4 <= zk_cap)) return;   // k_gen_band_z takes it
    const bool last = (pass == n_band - 1);
    const float *__restrict__ in = pass == 0 ? s.i_bf : s.tmp[(pass - 1) & 1];
    float *__restrict__ out = last ? s.lowres : s.tmp[pass & 1];
    const int stride = axis == 0 ? sh1 * sh2 : axis == 1 ? sh2 : 1;
    const int n_in = axis == 0 ? sh0 : axis == 1 ? sh1 : sh2;
    const int o2v = o2 / VEC;
    const int total = o0 * o1 * o2v;
    const int zf0 = s.zero_first[0], zf1 = s.zero_first[1], zf2 = s.zero_first[2];
    const float nstd = s.noise_std;
    const float *__restrict__ eps = s.eps_noise;
    const uint64_t seed = s.seed;
    const int *__restrict__ bstart = b.start;
    const float *__restrict__ bw = b.w;
    // (i, j, kv) of this thread's first output and of one grid-stride step
    const int step = gridDim.x * blockDim.x;
    const int p_first = blockIdx.x * blockDim.x + threadIdx.x;
    int kv = p_first % o2v, j = (p_first / o2v) % o1, i = p_first / (o1 * o2v);
    const int dk = step % o2v, dj = (step / o2v) % o1, di = step / (o1 * o2v);
    for (int p = p_first; p < total; p += step) {
        const int k = kv * VEC;
        const int q = axis == 0 ? i : axis == 1 ? j : k;
        const int st = __ldg(bstart + q);
        const int base = axis == 0 ? (st * sh1 + j) * sh2 + k : axis == 1 ? (i * sh1 + st) * sh2 + k : (i * sh1 + j) * sh2 + st;
        const float *__restrict__ wr = bw + q * T;
        const int t0 = max(0, -st), t1 = min(T, n_in - st);
        float acc[VEC];
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
        const float *__restrict__ src = in + base;
#pragma unroll kBandUnroll
        for (int t = t0; t < t1; ++t) {
            const float w = __ldg(wr + t);
            if (VEC == 4) {
                const float4 x = __ldg((const float4 *)(src + t * stride));
                acc[0] = fmaf(w, x.x, acc[0]); acc[1] = fmaf(w, x.y, acc[1]);
                acc[2] = fmaf(w, x.z, acc[2]); acc[3] = fmaf(w, x.w, acc[3]);
            } else {
                acc[0] = fmaf(w, __ldg(src + t * stride), acc[0]);
            }
        }
        const int op = (i * o1 + j) * o2 + k;
        if (last) {
            float4 e4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!eps && VEC == 4) e4 = philox_normal4(seed, 1u, (uint64_t)(op >> 2));   // o2 % 4 == 0 here
            const float ev[4] = {e4.x, e4.y, e4.z, e4.w};
#pragma unroll
            for (int c = 0; c < VEC; ++c) {
                if ((zf0 && i == 0) || (zf1 && j == 0) || (zf2 && k + c == 0)) acc[c] = 0.f;
                float e;
                if (eps) e = __ldg(eps + op + c);
                else if (VEC == 4) e = ev[c];
                else {
                    const float4 g4 = philox_normal4(seed, 1u, (uint64_t)(op >> 2));
                    const int r = op & 3;
                    e = r == 0 ? g4.x : r == 1 ? g4.y : r == 2 ? g4.z : g4.w;
                }
                acc[c] = __fadd_rn(acc[c], __fmul_rn(nstd, e));      // utils.py:635-636
                acc[c] = acc[c] < 0.f ? 0.f : acc[c];
            }
        }
        if (VEC == 4) *(float4 *)(out + op) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        else out[op] = acc[0];
        kv += dk; j += dj; i += di;
        if (kv >= o2v) { kv -= o2v; ++j; }
        if (j >= o1) { j -= o1; ++i; }
    }
}


// Axis-2 (z, contiguous) banded pass.  A warp owns one input row at a time: the row is staged in shared memory with
// coalesced loads, the band table of the pass (starts + weights, odd pitch => conflict-free) is staged once per
// persistent block, lane l computes outputs l, l+32, ... from shared memory.  Same tap order and the same
// counter-based noise mapping (group = output index >> 2) as k_gen_band<1>: results are bit-identical to it.
__global__ void __launch_bounds__(256) k_gen_band_z(const bfm_gen_sample *__restrict__ S, int pass, int smem_cap) {
    extern __shared__ float zsm[];
    const bfm_gen_sample &s = S[blockIdx.y];
    const int n_band = s.n_band;
    if (pass >= n_band || is_identity_sample(s)) return;
    const bfm_band &b = s.band[pass];
    if (b.axis != 2) return;
    int sh0 = s.d.size[0], sh1 = s.d.size[1], sh2 = s.d.size[2];
    for (int q = 0; q < pass; ++q) {
        const int ax = s.band[q].axis, no = s.band[q].n_out;
        if (ax == 0) sh0 = no; else if (ax == 1) sh1 = no; else sh2 = no;
    }
    const int T = b.T, Tp = T | 1, n_out = b.n_out, n_in = sh2;
    const int nwarps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // shared layout: weights [n_out][Tp] | starts [n_out] | per warp: row [n_in] + noise [n_out + 4]
    float *wsm = zsm;
    int *ssm = (int *)(wsm + n_out * Tp);
    float *rows = (float *)(ssm + n_out);
    const int per_warp = n_in + n_out + 4;
    if ((n_out * (Tp + 1) + nwarps * per_warp) * 4 > smem_cap) return;      // the host routes this sample to k_gen_band<1>
    const bool last = (pass == n_band - 1);
    const float *__restrict__ in = pass == 0 ? s.i_bf : s.tmp[(pass - 1) & 1];
    float *__restrict__ out = last ? s.lowres : s.tmp[pass & 1];
    for (int q = threadIdx.x; q < n_out * T; q += blockDim.x) {
        const int o = q / T, t = q - o * T;
        wsm[o * Tp + t] = __ldg(b.w + q);
    }
    for (int q = threadIdx.x; q < n_out; q += blockDim.x) ssm[q] = __ldg(b.start + q);
    __syncthreads();
    float *row = rows + warp * per_warp, *nz = row + n_in;
    const int zf0 = s.zero_first[0], zf1 = s.zero_first[1], zf2 = s.zero_first[2];
    const float nstd = s.noise_std;
    const float *__restrict__ eps = s.eps_noise;
    const uint64_t seed = s.seed;
    const int n_rows = sh0 * sh1;
    // the next row of this warp travels in registers while the current one is being consumed from shared memory
    constexpr int kPre = 8;                                  // rows up to 32 * kPre floats are prefetched
    const bool prefetch = n_in <= 32 * kPre;
    float pre[kPre];
    const int rstep = gridDim.x * nwarps;
    auto fetch = [&](int r) {
        const float *__restrict__ src = in + (size_t)r * n_in;
#pragma unroll
        for (int u = 0; u < kPre; ++u) {
            const int q = lane + 32 * u;
            pre[u] = (r < n_rows && q < n_in) ? __ldg(src + q) : 0.f;
        }
    };
    const int r_first = blockIdx.x * nwarps + warp;
    if (prefetch) fetch(r_first);
    for (int r = r_first; r < n_rows; r += rstep) {
        if (prefetch) {
#pragma unroll
            for (int u = 0; u < kPre; ++u) {
                const int q = lane + 32 * u;
                if (q < n_in) row[q] = pre[u];
            }
            fetch(r + rstep);
        } else {
            const float *__restrict__ src = in + (size_t)r * n_in;
            for (int q = lane; q < n_in; q += 32) row[q] = __ldg(src + q);
        }
        const int op0 = r * n_out;
        if (last && !eps) {                      // noise of outputs [op0, op0 + n_out): Philox groups of four
            const int g0 = op0 >> 2, g1 = (op0 + n_out - 1) >> 2;
            for (int g = g0 + lane; g <= g1; g += 32) {
                const float4 e = philox_normal4(seed, 1u, (uint64_t)g);
                const float ev[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int o = 4 * g + c - op0;
                    if (o >= 0 && o < n_out) nz[o] = ev[c];
                }
            }
        }
        __syncwarp();
        const int i = r / sh1, j = r - i * sh1;
        for (int k = lane; k < n_out; k += 32) {
            const int st = ssm[k];
            const int t0 = max(0, -st), t1 = min(T, n_in - st);
            const float *wr = wsm + k * Tp, *x = row + st;
            float acc = 0.f;
            for (int t = t0; t < t1; ++t) acc = fmaf(wr[t], x[t], acc);
            if (last) {
                if ((zf0 && i == 0) || (zf1 && j == 0) || (zf2 && k == 0)) acc = 0.f;
                const float e = eps ? __ldg(eps + op0 + k) : nz[k];
                acc = __fadd_rn(acc, __fmul_rn(nstd, e));                 // utils.py:635-636
                acc = acc < 0.f ? 0.f : acc;
            }
            out[op0 + k] = acc;
        }
        __syncwarp();
    }
}


// out (unnormalised, at its flipped position) = max(0, i_bf + noise_std * eps) with the strict `>0` masks, plus the
// global maximum: what k_gen_band_z (identity band) followed by k_gen_upsample (identity zoom) produce, in one pass.
// Same operations, same counter-based noise (group = voxel index >> 2): bit-identical to the two-kernel form.
__global__ void __launch_bounds__(256) k_gen_identity(const bfm_gen_sample *__restrict__ S) {
    __shared__ float red[8];
    const bfm_gen_sample &s = S[blockIdx.z];
    if (!is_identity_sample(s)) return;
    const int s0 = s.d.size[0], s1 = s.d.size[1], s2 = s.d.size[2], plane = s1 * s2;
    const int i = blockIdx.y;
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    float hi = 0.f;
    if (i < s0 && q < plane) {
        const int io = s.flip ? s0 - 1 - i : i;
        const int op = i * plane + q;                       // voxel index on the (low-res == training) grid
        const float4 x = __ldg((const float4 *)(s.i_bf + op));
        float v[4] = {x.x, x.y, x.z, x.w};
        float e[4];
        if (s.eps_noise) {
            const float4 t = __ldg((const float4 *)(s.eps_noise + op));
            e[0] = t.x; e[1] = t.y; e[2] = t.z; e[3] = t.w;
        } else {
            const float4 t = philox_normal4(s.seed, 1u, (uint64_t)(op >> 2));
            e[0] = t.x; e[1] = t.y; e[2] = t.z; e[3] = t.w;
        }
        const int j = q / s2, k = q - j * s2;               // s2 % 4 == 0 is not required: recompute per element
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int jc = (q + c) / s2, kc = (q + c) - jc * s2;
            if ((s.zero_first[0] && i == 0) || (s.zero_first[1] && jc == 0) || (s.zero_first[2] && kc == 0)) v[c] = 0.f;
            v[c] = __fadd_rn(v[c], __fmul_rn(s.noise_std, e[c]));
            v[c] = v[c] < 0.f ? 0.f : v[c];
            hi = fmaxf(hi, v[c]);
        }
        (void)j; (void)k;
        *(float4 *)(s.out + (size_t)io * plane + q) = make_float4(v[0], v[1], v[2], v[3]);
    }
    hi = warp_max(hi);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = hi;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) hi = fmaxf(hi, red[w]);
        atomicMax((int *)s.maxval, __float_as_int(hi));
    }
}

// ---------------------------------------------------------------------------------------------- finish
// myzoom_torch(lowres, 1/factors) back to the training grid (datasets.py:337-340), in the same persistent-k
// layout as the warp kernel: block = (i, kUR rows j), thread = k.  The first zoom pass (axis 0) of the low-res
// rows this block touches is evaluated once per block into shared memory, the second (axis 1) once per output
// row (kWR rows per barrier, double buffered), so a voxel costs one 2-tap lerp from shared memory.  The kernel
// stores the UNNORMALISED value at its final (flipped) position and reduces the global maximum;
// k_gen_normalize then applies I / max(I) (datasets.py:342-343) and finishes the real-image targets.
#ifndef UPS_ROWS
#define UPS_ROWS 32
#endif
#ifndef UPS_MINB
#define UPS_MINB 8
#endif
constexpr int kUR = UPS_ROWS;     // output rows per block

// myzoom_torch(lowres, 1/factors): three sequential 2-tap passes (axis 0, 1, 2), each `wl*a + wh*b` separately rounded.
// Block = (x plane i, kUR output rows), thread = k.  The first pass (axis 0) of the low-res rows under the block's
// output rows is evaluated once per block into shared memory (t1[y'][z']); a voxel then evaluates the second pass at
// its two z taps and the third pass itself: 4 shared loads + 9 flops, no barrier in the row loop.  (v1 shared the
// second pass through double-buffered row buffers: the y pass + its barriers cost more instructions per voxel than
// the duplicated lerps -- 62 -> ~30 warp instructions per 32 voxels, profiles/r2_ncu_rest_summary.csv.)
__global__ void __launch_bounds__(160, UPS_MINB) k_gen_upsample(const bfm_gen_sample *__restrict__ S, int lz_cap, int ny_cap) {
    extern __shared__ float smem[];
    __shared__ float red[8];
    __shared__ int ylo_s[kUR], yhi_s[kUR];
    __shared__ float ywl_s[kUR], ywh_s[kUR];
    const bfm_gen_sample &s = S[blockIdx.z];
    const int s0 = s.d.size[0], s1 = s.d.size[1], s2 = s.d.size[2];
    if ((int)blockIdx.y >= s0 || (int)blockIdx.x * kUR >= s1) return;
    if (is_identity_sample(s)) return;                  // k_gen_identity (resample stage) already wrote `out`
    if (cubic_zoom(s)) return;                          // k_gen_cubic_zoom
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
    const int ly = s.new_size[1], lz = s.new_size[2];
    const int i = blockIdx.y, j0 = blockIdx.x * kUR, j1 = min(j0 + kUR, s1);
    float *t1 = smem;                                   // [ny][lz]   first pass at this i
    const bfm_zoom_tab &u = s.utab;
    // low-res rows needed by output rows j0..j1-1 (the tables are monotone in j)
    const int y0 = __ldg(u.lo[1] + j0), y1 = __ldg(u.hi[1] + j1 - 1);
    const int ny = y1 - y0 + 1;
    {
        const int lo = __ldg(u.lo[0] + i), hi = __ldg(u.hi[0] + i);
        const float wl = __ldg(u.wl[0] + i), wh = __ldg(u.wh[0] + i);
        const float *a = s.lowres + ((size_t)lo * ly + y0) * lz, *b = s.lowres + ((size_t)hi * ly + y0) * lz;
        const int n = ny * lz;                          // rows y0..y1 are contiguous in the low-res volume
        if ((lz & 3) == 0) {                            // 128-bit loads: both row blocks start on a multiple of lz
            const float4 *a4 = (const float4 *)a, *b4 = (const float4 *)b;
            float4 *t4 = (float4 *)t1;
            for (int q = tid; q < (n >> 2); q += blockDim.x) {
                const float4 x = __ldg(a4 + q), y = __ldg(b4 + q);
                t4[q] = make_float4(lerp_rn(wl, x.x, wh, y.x), lerp_rn(wl, x.y, wh, y.y), lerp_rn(wl, x.z, wh, y.z),
                                    lerp_rn(wl, x.w, wh, y.w));
            }
        } else {
            for (int q = tid; q < n; q += blockDim.x) t1[q] = lerp_rn(wl, __ldg(a + q), wh, __ldg(b + q));
        }
    }
    if (tid < j1 - j0) {
        const int j = j0 + tid;
        ylo_s[tid] = (__ldg(u.lo[1] + j) - y0) * lz; yhi_s[tid] = (__ldg(u.hi[1] + j) - y0) * lz;
        ywl_s[tid] = __ldg(u.wl[1] + j); ywh_s[tid] = __ldg(u.wh[1] + j);
    }
    __syncthreads();
    float *__restrict__ outp = s.out;
    const int plane_out = (s.flip ? s0 - 1 - i : i) * s1;
    float hi = 0.f;
    for (int k = tid; k < s2; k += blockDim.x) {
        const int zlo = __ldg(u.lo[2] + k), zhi = __ldg(u.hi[2] + k);
        const float zwl = __ldg(u.wl[2] + k), zwh = __ldg(u.wh[2] + k);
        float *__restrict__ o = outp + (size_t)(plane_out + j0) * s2 + k;
#pragma unroll 4
        for (int r = 0; r < j1 - j0; ++r) {
            const float *a = t1 + ylo_s[r], *b = t1 + yhi_s[r];
            const float wl = ywl_s[r], wh = ywh_s[r];
            const float vl = lerp_rn(wl, a[zlo], wh, b[zlo]), vh = lerp_rn(wl, a[zhi], wh, b[zhi]);
            const float v = lerp_rn(zwl, vl, zwh, vh);
            o[(size_t)r * s2] = v;
            hi = fmaxf(hi, v);
        }
    }
    hi = warp_max(hi);
    if (lane == 0) red[warp] = hi;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < nwarps; ++w) hi = fmaxf(hi, red[w]);
        atomicMax((int *)s.maxval, __float_as_int(hi));               // values >= 0: bit order == float order
    }
}

// ---------------------------------------------------------------------------------------------- cubic zoom back
// bspline_zooming (datasets.py:337-338): interpol.resize(I, shape=size, anchor='edge', interpolation=3, bound='dct2',
// prefilter=True) of `lowres` back to the training grid.  Three prefilter launches (one per axis, in place on
// `lowres`, which is dead after this stage), then k_gen_cubic_zoom.  blockIdx.z = sample throughout.
constexpr int kCubicLines = 32;   // lines per block of the tiled z prefilter

// the prefilter of one axis of length n: cubic B-spline (one pole, sqrt(3) - 2), dct2 boundary -- the arguments
// brainfm_b200.interpol.spline_coeff passes to bfm_spline_filter
__device__ __forceinline__ FilterArgs cubic_filter_args(int n) {
    FilterArgs a;
    a.outer = 1; a.inner = 1; a.n = n; a.bound = 3; a.npoles = 1;
    a.poles[0] = sqrt(3.0) - 2.0; a.poles[1] = a.poles[2] = 0.0;
    return a;
}

// Sample coordinate of output o of an edge-anchored resize from n_in to n_out (interpol resize, anchor='edge':
// torch.arange(n_out) * scale + 0.5 * (scale - 1) with scale = n_in / n_out): a float32 product and a float32 sum,
// the Python floats rounded to float32 first.
__device__ __forceinline__ float edge_coord(int o, int n_in, int n_out) {
    const double scale = (double)n_in / (double)n_out;
    return __fadd_rn(__fmul_rn((float)o, (float)scale), (float)(0.5 * (scale - 1.0)));
}

// The 4 taps of a cubic pull at x with dct2 folding: k_pull_fast's node indices and weights (the dct2 sign is 1).
__device__ __forceinline__ void cubic_taps(float x, int n, int idx[4], float w[4]) {
    const float f0 = floorf(x - 1.f);
    const float dist0 = x - f0;
    const int i0 = (int)f0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        idx[k] = bound_index_t<int>(3, i0 + k, n);
        w[k] = spline_weight<float>(3, dist0 - float(k));
    }
}

// Prefilter along x (AXIS 0) or y (AXIS 1): one thread per line, adjacent threads on adjacent lines (adjacent z, so
// every step of the recursion is a coalesced access); filter_line of bfm_spline_filter, with its dct2 weight table
// in shared memory.  A length-1 line is its own coefficient (bfm_spline_filter returns before any launch then).
template <int AXIS>
__global__ void __launch_bounds__(256) k_gen_prefilter(const bfm_gen_sample *__restrict__ S) {
    extern __shared__ float wt[];
    const bfm_gen_sample &s = S[blockIdx.z];
    if (!cubic_zoom(s)) return;
    const int l0 = s.new_size[0], l1 = s.new_size[1], l2 = s.new_size[2];
    const int n = AXIS == 0 ? l0 : l1;
    const int lines = AXIS == 0 ? l1 * l2 : l0 * l2;
    if (n == 1 || (int)(blockIdx.x * blockDim.x) >= lines) return;
    const FilterArgs a = cubic_filter_args(n);
    for (int e = threadIdx.x; e < n; e += blockDim.x) wt[e] = filter_weight(a, e);
    __syncthreads();
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= lines) return;
    const int x = AXIS == 0 ? 0 : q / l2, z = q - x * l2;     // AXIS 0: q = y * l2 + z
    filter_line<float, int>(s.lowres + (size_t)x * l1 * l2 + z, AXIS == 0 ? l1 * l2 : l2, a, wt);
}

// Prefilter along z: the lines are contiguous, so a block stages kCubicLines of them in shared memory with coalesced
// loads (128-bit when the line length is a multiple of 4), one thread per line runs the recursion there (odd pitch:
// conflict free) and the tile is written back once -- k_spline_filter_tile<true> batched over descriptors.
__global__ void __launch_bounds__(128) k_gen_prefilter_z(const bfm_gen_sample *__restrict__ S) {
    extern __shared__ float tile[];
    const bfm_gen_sample &s = S[blockIdx.z];
    if (!cubic_zoom(s)) return;
    const int n = s.new_size[2], rows = s.new_size[0] * s.new_size[1];
    const int r0 = blockIdx.x * kCubicLines;
    if (n == 1 || r0 >= rows) return;
    const int tid = threadIdx.x, pitch = n | 1, nl = min(kCubicLines, rows - r0), total = nl * n;
    float *wt = tile + kCubicLines * pitch;
    const FilterArgs a = cubic_filter_args(n);
    for (int e = tid; e < n; e += blockDim.x) wt[e] = filter_weight(a, e);
    float *base = s.lowres + (size_t)r0 * n;
    if ((n & 3) == 0) {                                 // rows start on multiples of 4 floats of a 16-byte aligned base
        for (int e = 4 * tid; e < total; e += 4 * blockDim.x) {
            const float4 v = *(const float4 *)(base + e);
            const int row = e / n;
            float *t = tile + row * pitch + (e - row * n);
            t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w;
        }
    } else {
        for (int e = tid; e < total; e += blockDim.x) {
            const int row = e / n;
            tile[row * pitch + (e - row * n)] = base[e];
        }
    }
    __syncthreads();
    if (tid < nl) filter_line<float, int>(tile + tid * pitch, 1, a, wt);
    __syncthreads();
    if ((n & 3) == 0) {
        for (int e = 4 * tid; e < total; e += 4 * blockDim.x) {
            const int row = e / n;
            const float *t = tile + row * pitch + (e - row * n);
            *(float4 *)(base + e) = make_float4(t[0], t[1], t[2], t[3]);
        }
    } else {
        for (int e = tid; e < total; e += blockDim.x) {
            const int row = e / n;
            base[e] = tile[row * pitch + (e - row * n)];
        }
    }
}

// Cubic pull of the prefiltered `lowres` at the edge-anchored coordinates, evaluated separably in k_gen_upsample's
// layout: block = (x plane i, kUR output rows), thread = k.  The axis-0 pass (4 taps along x) of the low-res rows
// under the block's rows goes to shared memory (t1), then the axis-1 pass of each output row (t2), then 4 taps along
// z per voxel.  The reference sums the 64 taps of a voxel in one loop; the separable sums round in another order
// (float32 differences of a few ulp).  Stores the UNNORMALISED value at its final (flipped) position and reduces the
// maximum with the order-preserving encoding: the cubic output can be negative.
// ny_cap: low-res rows of t1 the host sized the shared memory for (>= the rows any block touches).
__global__ void __launch_bounds__(160) k_gen_cubic_zoom(const bfm_gen_sample *__restrict__ S, int ny_cap) {
    extern __shared__ float smem[];
    __shared__ float red[8];
    __shared__ int yi_s[kUR][4];
    __shared__ float yw_s[kUR][4];
    const bfm_gen_sample &s = S[blockIdx.z];
    const int s0 = s.d.size[0], s1 = s.d.size[1], s2 = s.d.size[2];
    if ((int)blockIdx.y >= s0 || (int)blockIdx.x * kUR >= s1) return;
    if (!cubic_zoom(s)) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
    const int lx = s.new_size[0], ly = s.new_size[1], lz = s.new_size[2];
    const int i = blockIdx.y, j0 = blockIdx.x * kUR, nr = min(kUR, s1 - j0);
    // low-res rows under output rows j0 .. j0+nr-1: the first node of a row is monotone in j, and dct2 folds the
    // taps of the edge rows back inside [max(0, first node of j0), min(ly - 1, first node of the last row + 3)]
    const int y0 = max(0, (int)floorf(edge_coord(j0, ly, s1) - 1.f));
    const int y1 = min(ly - 1, (int)floorf(edge_coord(j0 + nr - 1, ly, s1) - 1.f) + 3);
    const int ny = y1 - y0 + 1;
    float *t1 = smem;                                   // [ny_cap][lz]: axis-0 pass at this i
    float *t2 = smem + (size_t)ny_cap * lz;             // [kUR][lz]:    axis-1 pass of the block's rows
    {
        int xi[4];
        float xw[4];
        cubic_taps(edge_coord(i, lx, s0), lx, xi, xw);
        const float *src[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) src[t] = s.lowres + ((size_t)xi[t] * ly + y0) * lz;
        const int n = ny * lz;                          // rows y0..y1 are contiguous in the low-res volume
        if ((lz & 3) == 0) {                            // 128-bit loads: every row block starts on a multiple of lz
            float4 *t4 = (float4 *)t1;
            for (int q = tid; q < (n >> 2); q += blockDim.x) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const float4 v = __ldg((const float4 *)src[t] + q);
                    acc.x = fmaf(v.x, xw[t], acc.x); acc.y = fmaf(v.y, xw[t], acc.y);
                    acc.z = fmaf(v.z, xw[t], acc.z); acc.w = fmaf(v.w, xw[t], acc.w);
                }
                t4[q] = acc;
            }
        } else {
            for (int q = tid; q < n; q += blockDim.x) {
                float acc = 0.f;
#pragma unroll
                for (int t = 0; t < 4; ++t) acc = fmaf(__ldg(src[t] + q), xw[t], acc);
                t1[q] = acc;
            }
        }
    }
    if (tid < nr) {
        int yi[4];
        float yw[4];
        cubic_taps(edge_coord(j0 + tid, ly, s1), ly, yi, yw);
#pragma unroll
        for (int t = 0; t < 4; ++t) { yi_s[tid][t] = (yi[t] - y0) * lz; yw_s[tid][t] = yw[t]; }
    }
    __syncthreads();
    for (int r = 0; r < nr; ++r) {
        const int a0 = yi_s[r][0], a1 = yi_s[r][1], a2 = yi_s[r][2], a3 = yi_s[r][3];
        const float w0 = yw_s[r][0], w1 = yw_s[r][1], w2 = yw_s[r][2], w3 = yw_s[r][3];
        for (int z = tid; z < lz; z += blockDim.x) {
            float acc = fmaf(t1[a0 + z], w0, 0.f);
            acc = fmaf(t1[a1 + z], w1, acc);
            acc = fmaf(t1[a2 + z], w2, acc);
            t2[r * lz + z] = fmaf(t1[a3 + z], w3, acc);
        }
    }
    __syncthreads();
    const int plane_out = (s.flip ? s0 - 1 - i : i) * s1;
    float hi = -INFINITY;
    for (int k = tid; k < s2; k += blockDim.x) {
        int zi[4];
        float zw[4];
        cubic_taps(edge_coord(k, lz, s2), lz, zi, zw);
        float *__restrict__ o = s.out + (size_t)(plane_out + j0) * s2 + k;
#pragma unroll 4
        for (int r = 0; r < nr; ++r) {
            const float *t = t2 + r * lz;
            float acc = fmaf(t[zi[0]], zw[0], 0.f);
            acc = fmaf(t[zi[1]], zw[1], acc);
            acc = fmaf(t[zi[2]], zw[2], acc);
            acc = fmaf(t[zi[3]], zw[3], acc);
            o[(size_t)r * s2] = acc;
            hi = fmaxf(hi, acc);
        }
    }
    hi = warp_max(hi);
    if (lane == 0) red[warp] = hi;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < nwarps; ++w) hi = fmaxf(hi, red[w]);
        atomicMax((int *)s.maxval, f2ord(hi));
    }
}

// edge_coord for o = 0 .. n_out-1 (bfm_gen_zoom_coords)
__global__ void k_gen_zoom_coords(int n_in, int n_out, float *out) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o < n_out) out[o] = edge_coord(o, n_in, n_out);
}

// I / max(I), optional high_res_residual (datasets.py:342-347) and the real-image targets'
// `Idef -= min; Idef /= max; flip` (utils.py:326-329).  One thread = VEC consecutive z voxels of one x plane.
template <int VEC>
__global__ void __launch_bounds__(256) k_gen_normalize(const bfm_gen_sample *__restrict__ S) {
    const bfm_gen_sample &s = S[blockIdx.z];
    const int s0 = s.d.size[0], plane = s.d.size[1] * s.d.size[2];
    if ((VEC == 4) != ((plane & 3) == 0)) return;
    const int i = blockIdx.y;
    if (i >= s0) return;
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (q >= plane) return;
    const int io = s.flip ? s0 - 1 - i : i;
    const size_t pin = (size_t)i * plane + q, pout = (size_t)io * plane + q;
    // I / max(I) as a multiplication by the correctly rounded reciprocal: <= 1 ulp from the division
    const float rmx = __frcp_rn(cubic_zoom(s) ? ord2f(*(const int *)s.maxval) : *s.maxval);
    float y[VEC];
    if (VEC == 4) {
        const float4 v = *(const float4 *)(s.out + pout);
        y[0] = v.x * rmx; y[1] = v.y * rmx; y[2] = v.z * rmx; y[VEC - 1] = v.w * rmx;
        *(float4 *)(s.out + pout) = make_float4(y[0], y[1], y[2], y[VEC - 1]);
    } else {
        y[0] = s.out[pout] * rmx;
        s.out[pout] = y[0];
    }
    if (s.residual) {
#pragma unroll
        for (int c = 0; c < VEC; ++c) s.residual[pout + c] = __fsub_rn(__ldg(s.i_bf + pin + c) * rmx, y[c]);
    }
    for (int a = 0; a < s.n_aux; ++a) {
        const float mn = ord2f(s.aux_mm[2 * a]), rg = __fsub_rn(ord2f(s.aux_mm[2 * a + 1]), mn);
        const float *__restrict__ raw = s.aux_raw[a] + pin;
        float *__restrict__ o = s.aux_out[a] + pout;
        if (VEC == 4) {
            const float4 v = __ldg((const float4 *)raw);
            *(float4 *)o = make_float4(__fdiv_rn(__fsub_rn(v.x, mn), rg), __fdiv_rn(__fsub_rn(v.y, mn), rg),
                                       __fdiv_rn(__fsub_rn(v.z, mn), rg), __fdiv_rn(__fsub_rn(v.w, mn), rg));
        } else {
            o[0] = __fdiv_rn(__fsub_rn(__ldg(raw), mn), rg);
        }
    }
}

static inline bool misaligned(const void *p, uintptr_t bytes) { return ((uintptr_t)p & (bytes - 1)) != 0; }

static int check_batch(const bfm_gen_sample *h, const bfm_gen_sample *d, int B) {
    if (!h || !d || B <= 0) return fail(BFM_E_INVALID, "%s", "bfm_gen: null descriptors or empty batch");
    for (int b = 0; b < B; ++b) {
        const bfm_gen_sample &s = h[b];
        for (int a = 0; a < 3; ++a)
            if (s.d.size[a] <= 0 || s.d.src[a] <= 0 || s.new_size[a] <= 0)
                return fail(BFM_E_INVALID, "%s", "bfm_gen: non-positive size");
        if ((int64_t)s.d.src[0] * s.d.src[1] * s.d.src[2] >= (1LL << 31) ||
            (int64_t)s.d.size[0] * s.d.size[1] * s.d.size[2] >= (1LL << 31))
            return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen: volumes of 2^31 voxels or more are not supported");
        if (s.d.fsmall && (s.d.fs[2] > kMaxSmallZ || s.d.fs[2] <= 0))
            return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen: deformation small grid too deep");
        if (s.bfsmall && (s.bs[2] > kMaxSmallZ || s.bs[2] <= 0))
            return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen: bias small grid too deep");
        if (!s.syn || !s.bbox || !s.i_bf || !s.lowres || !s.maxval || !s.out ||
            (!s.real_input && (!s.labels || !s.mu || !s.sigma)))
            return fail(BFM_E_INVALID, "%s", "bfm_gen: null buffer");
        if (s.real_input && s.mix[0])
            return fail(BFM_E_INVALID, "%s", "bfm_gen: real-image inputs are not mixed");
        if (s.n_band < 1 || s.n_band > 3) return fail(BFM_E_INVALID, "%s", "bfm_gen: n_band must be 1..3");
        if (s.zoom_order != 0 && s.zoom_order != 3) return fail(BFM_E_INVALID, "%s", "bfm_gen: zoom_order must be 0 or 3");
        if (s.d.size[0] != h[0].d.size[0] || s.d.size[1] != h[0].d.size[1] || s.d.size[2] != h[0].d.size[2])
            return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen: all samples of a batch share the output size");
        // The kernels take 128-bit accesses without looking at the pointers: on the scratch whenever the low-res
        // shape allows (k_gen_band<4>, k_gen_upsample), on the outputs whenever the output plane is a multiple of 4.
        if (misaligned(s.i_bf, 16) || misaligned(s.tmp[0], 16) || misaligned(s.tmp[1], 16) ||
            misaligned(s.lowres, 16) || misaligned(s.syn, 8))
            return fail(BFM_E_INVALID, "%s", "bfm_gen: misaligned scratch (i_bf, tmp, lowres: 16 bytes; syn: 8)");
        if ((((int64_t)s.d.size[1] * s.d.size[2]) & 3) == 0) {
            bool bad = misaligned(s.out, 16) || misaligned(s.bflog_out, 16) || misaligned(s.residual, 16);
            for (int a = 0; a < s.n_aux && a < BFM_MAX_AUX; ++a)
                bad |= misaligned(s.aux_out[a], 16) || misaligned(s.aux_raw[a], 16);
            if (bad) return fail(BFM_E_INVALID, "%s", "bfm_gen: misaligned output (16 bytes when size[1]*size[2] % 4 == 0)");
        }
    }
    return BFM_OK;
}

static inline unsigned rows_grid(const bfm_gen_sample *h) {
    const int64_t rows = (int64_t)h[0].d.size[0] * h[0].d.size[1];
    const int per_block = kRowWarps * kRowsPerWarp;
    return (unsigned)((rows + per_block - 1) / per_block);
}
static inline int max_fstride(const bfm_gen_sample *h, int B) {
    int m = 0;
    for (int b = 0; b < B; ++b)
        if (h[b].d.fsmall && !h[b].d.F_full) m = h[b].d.fs[2] * 3 > m ? h[b].d.fs[2] * 3 : m;
    return m;
}
static inline int max_bstride(const bfm_gen_sample *h, int B) {
    int m = 0;
    for (int b = 0; b < B; ++b)
        if (h[b].bfsmall) m = h[b].bs[2] > m ? h[b].bs[2] : m;
    return m;
}
}  // namespace bfm

using namespace bfm;

extern "C" {

int bfm_gen_bbox(const bfm_gen_sample *h, const bfm_gen_sample *d, int B, void *stream) {
    int rc = check_batch(h, d, B);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    int64_t most = 0;
    for (int b = 0; b < B; ++b) {
        const int64_t n = (int64_t)h[b].d.ncand[0] * h[b].d.ncand[1] * h[b].d.ncand[2];
        if (n >= (1LL << 30)) return fail(BFM_E_INVALID, "%s", "bfm_gen_bbox: too many candidate voxels");
        most = n > most ? n : most;
    }
    k_gen_bbox_init<<<B, 32, 0, s>>>(d);
    if (most > 0) k_gen_bbox_cand<<<dim3((unsigned)((most + 255) / 256), B), 256, 0, s>>>(d);
    k_gen_bbox_decide<<<B, 32, 0, s>>>(d);
    const int fstride = max_fstride(h, B);
    const size_t smem = (size_t)kRowWarps * kRowsPerWarp * fstride * sizeof(float);
    const unsigned full_blocks = min(rows_grid(h), (unsigned)max(8, (4 * 148 + B - 1) / B));
    k_gen_bbox_full<<<dim3(full_blocks, B), kRowWarps * 32, smem, s>>>(d, fstride);
    k_gen_bbox_finish<<<B, 32, 0, s>>>(d);
    g_launches.fetch_add(most > 0 ? 4 : 3);
    bool slab_scan = false, slab_cand = false;
    int64_t most_slab = 0;
    for (int b = 0; b < B; ++b) {
        if (!h[b].gmm_xr || h[b].x_count <= 0) continue;
        if (!h[b].d.F_full && h[b].d.ncand[0] > 0) {
            slab_cand = true;
            most_slab = max(most_slab, (int64_t)(h[b].d.ncand[0] + 2) * h[b].d.ncand[1] * h[b].d.ncand[2]);
        } else {
            slab_scan = true;
        }
    }
    if (slab_scan || slab_cand) {
        k_gen_slab_xr_init<<<B, 32, 0, s>>>(d);
        if (slab_cand) k_gen_slab_xr_cand<<<dim3((unsigned)((most_slab + 255) / 256), B), 256, 0, s>>>(d);
        if (slab_scan) k_gen_slab_xr<<<dim3(full_blocks, B), kRowWarps * 32, smem, s>>>(d, fstride);
        k_gen_slab_xr_finish<<<B, 32, 0, s>>>(d);
        g_launches.fetch_add(2 + (slab_cand ? 1 : 0) + (slab_scan ? 1 : 0) - 1);
    }
    return check_launch("bfm_gen_bbox");
}

int bfm_gen_gmm(const bfm_gen_sample *h, const bfm_gen_sample *d, int B, void *stream) {
    int rc = check_batch(h, d, B);
    if (rc) return rc;
    int64_t flat_groups = 0, plane_groups = 0;
    int max_n0 = 0;
    for (int b = 0; b < B; ++b) {
        if (h[b].real_input) continue;
        const int *n = h[b].d.src;
        if (n[2] & 3) {
            const int64_t g = ((int64_t)n[0] * n[1] * n[2] + 3) / 4;
            flat_groups = g > flat_groups ? g : flat_groups;
        } else {
            const int64_t g = (int64_t)n[1] * (n[2] / 4);
            plane_groups = g > plane_groups ? g : plane_groups;
            max_n0 = n[0] > max_n0 ? n[0] : max_n0;
        }
    }
    if (plane_groups > 0) {
        if (max_n0 > 65535 || B > 65535) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_gmm: grid too large");
        // blockIdx.y walks the x planes of the crop (<= src[0]); a few row tiles per plane when the batch is small
        // and enough blocks for ~2 waves of 148 SMs x 8 resident blocks: with one block per plane a batch of 8 x 160
        // planes is 1.08 waves (a nearly empty second wave).  Measured per sample: 1 tile 13.8 us, 2: 12.6, 4: 13.1,
        // 8: 14.4 (the 512-entry table is staged per block).
        const int64_t want = (2LL * 148 * 8 + (int64_t)max_n0 * B - 1) / ((int64_t)max_n0 * B);
        const int tiles = (int)min((int64_t)8, max((int64_t)1, want));
        k_gen_gmm_planes<<<dim3(tiles, max_n0, B), 256, 0, (cudaStream_t)stream>>>(d);
        rc = check_launch("bfm_gen_gmm");
        if (rc) return rc;
    }
    if (flat_groups > 0) {
        k_gen_gmm<<<dim3((unsigned)((flat_groups + 255) / 256), B), 256, 0, (cudaStream_t)stream>>>(d);
        rc = check_launch("bfm_gen_gmm");
    }
    return rc;
}

int bfm_band_build(int n_in, int n_out, double sigma, int T, int *start, float *w, void *stream) {
    if (n_in <= 0 || n_out <= 0 || !start || !w || T < 2 || T > 64 || (T & 1) ||
        T != 2 * (sigma > 0 ? (int)ceil(3 * sigma) : 0) + 2)
        return fail(BFM_E_INVALID, "%s", "bfm_band_build: T must equal 2*ceil(3*sigma)+2 and be <= 64");
    k_band_build<<<1, 128, 0, (cudaStream_t)stream>>>(n_in, n_out, T, sigma, start, w);
    return check_launch("bfm_band_build");
}

int bfm_gen_plan(const bfm_gen_sample *h, const bfm_gen_sample *d, int B, void *stream) {
    int rc = check_batch(h, d, B);
    if (rc) return rc;
    bool any = false, small = false;
    for (int b = 0; b < B; ++b) {
        if (h[b].gen_small) small = true;
        for (int p = 0; p < h[b].n_band; ++p) {
            const bfm_band &bd = h[b].band[p];
            if (!bd.build) continue;
            any = true;
            if (bd.T < 2 || bd.T > 65 || (bd.T & 1) || !bd.start || !bd.w || bd.n_in <= 0 || bd.n_out <= 0)
                return fail(BFM_E_INVALID, "%s", "bfm_gen_plan: bad band descriptor (T must be even, 2..64)");
        }
    }
    if (small) {
        k_gen_small<<<dim3(4, B, 2), 256, 0, (cudaStream_t)stream>>>(d);
        rc = check_launch("bfm_gen_plan");
        if (rc) return rc;
    }
    if (!any) return BFM_OK;
    k_gen_plan<<<dim3(3, B), 128, 0, (cudaStream_t)stream>>>(d);
    return check_launch("bfm_gen_plan");
}

int bfm_gen_warp(const bfm_gen_sample *h, const bfm_gen_sample *d, int B, void *stream) {
    int rc = check_batch(h, d, B);
    if (rc) return rc;
    int t1f = 0, t1b = 0, wf = 0, wb = 0, s0 = 0, s1 = 0, s2 = 0;
    bool kinds[BFM_MAX_AUX + 2] = {false, false, false, false, false};      // n_aux 0..3, then MIX
    bool any_pk = false;                                                    // pair mode (k_gen_warp_pk)
    for (int b = 0; b < B; ++b) {
        const bfm_gen_sample &s = h[b];
        if (s.n_aux < 0 || s.n_aux > BFM_MAX_AUX || (s.mix[0] && s.n_aux))
            return fail(BFM_E_INVALID, "%s", "bfm_gen_warp: n_aux must be 0..3 and 0 when mixing");
        for (int c = 0; c < s.n_aux; ++c)
            if (!s.aux_src[c] || !s.aux_raw[c] || !s.aux_out[c] || !s.aux_mm)
                return fail(BFM_E_INVALID, "%s", "bfm_gen_warp: null real-image target buffer");
        if (use_pairs(s)) any_pk = true;
        else kinds[s.mix[0] ? BFM_MAX_AUX + 1 : s.n_aux] = true;
        if (s.d.fsmall && !s.d.F_full) {
            t1f = max(t1f, s.d.fs[1] * s.d.fs[2] * 3);
            wf = max(wf, s.d.fs[2] * 3);
        }
        if (s.bfsmall) {
            t1b = max(t1b, s.bs[1] * s.bs[2]);
            wb = max(wb, s.bs[2]);
        }
        if (s.x_count < 0 || s.x_begin < 0 || (s.x_count > 0 && s.x_begin + s.x_count > s.d.size[0]))
            return fail(BFM_E_INVALID, "%s", "bfm_gen_warp: slab outside the grid");
        s0 = max(s0, s.x_count > 0 ? s.x_count : s.d.size[0]);
        s1 = max(s1, s.d.size[1]); s2 = max(s2, s.d.size[2]);
    }
    const size_t smem = (size_t)(t1f + t1b) * sizeof(float);
    if (wf + wb > kT2 || smem > 160 * 1024)
        return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_warp: small grids too large for shared memory");
    const int threads = min(256, (s2 + 31) / 32 * 32);
    // rows per block: a multiple of kWR, small enough for >= ~4 waves of blocks
    int rpb = s1;
    while (rpb > 8 * kWR && (int64_t)B * s0 * ((s1 + rpb - 1) / rpb) < 4 * 148 * 4) rpb = (rpb / 2 + kWR - 1) / kWR * kWR;
    if (rpb > 32) rpb = 32;
    const dim3 grid((s1 + rpb - 1) / rpb, s0, B);
    if (s0 > 65535 || B > 65535) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_warp: grid too large");
    cudaStream_t st = (cudaStream_t)stream;
#define BFM_LAUNCH_WARP(IDX, NA, M)                                                                            \
    if (kinds[IDX]) {                                                                                          \
        if (smem > 40 * 1024)                                                                                  \
            cudaFuncSetAttribute(k_gen_warp<NA, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
        k_gen_warp<NA, M><<<grid, threads, smem, st>>>(d, rpb, t1f);                                \
        rc = check_launch("bfm_gen_warp");                                                                     \
        if (rc) return rc;                                                                                     \
    }
    BFM_LAUNCH_WARP(0, 0, false)
    BFM_LAUNCH_WARP(1, 1, false)
    BFM_LAUNCH_WARP(2, 2, false)
    BFM_LAUNCH_WARP(3, 3, false)
    BFM_LAUNCH_WARP(4, 0, true)
#undef BFM_LAUNCH_WARP
    if (any_pk) {
        if (smem > 40 * 1024)
            cudaFuncSetAttribute(k_gen_warp_pk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        for (int base = 0; base < B; base += kPkBatch) {
            const int nb = min(kPkBatch, B - base);
            PkParams P;
            bool any = false;
            for (int q = 0; q < nb; ++q) {
                const bfm_gen_sample &sm = h[base + q];
                any |= use_pairs(sm);
                for (int a = 0; a < 9; ++a) P.s[q].A[a] = sm.d.A[a];
                for (int a = 0; a < 3; ++a) { P.s[q].c2[a] = sm.d.c2[a]; P.s[q].ctr[a] = sm.d.ctr[a]; }
                P.s[q].gamma = sm.gamma;
            }
            if (!any) continue;
            P.one = 1.0f;
            P.base = base;
            k_gen_warp_pk<<<dim3(grid.x, grid.y, nb), threads, smem, st>>>(d, P, rpb, t1f);
            rc = check_launch("bfm_gen_warp");
            if (rc) return rc;
        }
    }
    return BFM_OK;
}

int bfm_gen_resample(const bfm_gen_sample *h, const bfm_gen_sample *d, int B, void *stream) {
    int rc = check_batch(h, d, B);
    if (rc) return rc;
    int maxp = 0;
    for (int b = 0; b < B; ++b) maxp = h[b].n_band > maxp ? h[b].n_band : maxp;
    // persistent blocks: ~16 per SM over the whole batch
    constexpr int kBandBlocksPerSM = 16;
    const int64_t band_blocks = max((int64_t)8, (int64_t)((int64_t)kBandBlocksPerSM * 148 + B - 1) / B);
    const int zk_cap = 96 * 1024;          // shared memory of k_gen_band_z (2 blocks per SM)
    static bool attr_done = false;
    if (!attr_done) {
        cudaFuncSetAttribute(k_gen_band_z, cudaFuncAttributeMaxDynamicSharedMemorySize, zk_cap);
        attr_done = true;
    }
    {
        int64_t plane = 0;
        int s0 = 0;
        for (int b = 0; b < B; ++b)
            if (is_identity_sample(h[b])) {
                plane = max(plane, (int64_t)h[b].d.size[1] * h[b].d.size[2]);
                s0 = max(s0, h[b].d.size[0]);
            }
        if (plane > 0) {
            if (s0 > 65535 || B > 65535) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_resample: grid too large");
            k_gen_identity<<<dim3((unsigned)((plane / 4 + 255) / 256), s0, B), 256, 0, (cudaStream_t)stream>>>(d);
            int rc2 = check_launch("bfm_gen_resample");
            if (rc2) return rc2;
        }
    }
    for (int pass = 0; pass < maxp; ++pass) {
        int64_t most4 = 0, most1 = 0, rows_z = 0;
        int smem_z = 0;
        for (int b = 0; b < B; ++b) {
            if (pass >= h[b].n_band || is_identity_sample(h[b])) continue;
            int sh[3] = {h[b].d.size[0], h[b].d.size[1], h[b].d.size[2]};
            for (int q = 0; q < pass; ++q) sh[h[b].band[q].axis] = h[b].band[q].n_out;
            const bfm_band &bd = h[b].band[pass];
            const int axis = bd.axis;
            const bool scalar = axis == 2 || (sh[2] & 3);
            const int need_z = (bd.n_out * ((bd.T | 1) + 1) + 8 * (sh[2] + bd.n_out + 4)) * 4;
            if (axis == 2 && need_z <= zk_cap) {
                rows_z = max(rows_z, (int64_t)sh[0] * sh[1]);
                smem_z = max(smem_z, need_z);
                continue;
            }
            sh[axis] = bd.n_out;
            const int64_t n = (int64_t)sh[0] * sh[1] * sh[2];
            if (scalar) most1 = n > most1 ? n : most1;
            else most4 = n / 4 > most4 ? n / 4 : most4;
        }
        if (most4 > 0) {
            k_gen_band<4><<<dim3((unsigned)min((most4 + 255) / 256, band_blocks), B), 256, 0, (cudaStream_t)stream>>>(d, pass, zk_cap);
            int rc2 = check_launch("bfm_gen_resample");
            if (rc2) return rc2;
        }
        if (most1 > 0) {
            k_gen_band<1><<<dim3((unsigned)min((most1 + 255) / 256, band_blocks), B), 256, 0, (cudaStream_t)stream>>>(d, pass, zk_cap);
            int rc2 = check_launch("bfm_gen_resample");
            if (rc2) return rc2;
        }
        if (rows_z > 0) {
            // persistent blocks: as many per SM as the shared memory allows (at most 8 = full occupancy)
            const int per_sm = (int)max((int64_t)1, min((int64_t)8, (int64_t)(200 * 1024) / max(smem_z, 1)));
            const int64_t zb = max((int64_t)4, (int64_t)(per_sm * 148 + B - 1) / B);
            k_gen_band_z<<<dim3((unsigned)min((rows_z + 7) / 8, zb), B), 256, smem_z, (cudaStream_t)stream>>>(d, pass, zk_cap);
            int rc2 = check_launch("bfm_gen_resample");
            if (rc2) return rc2;
        }
    }
    return BFM_OK;
}

int bfm_gen_finish(const bfm_gen_sample *h, const bfm_gen_sample *d, int B, void *stream) {
    int rc = check_batch(h, d, B);
    if (rc) return rc;
    int lz = 1, ny = 1, s0 = 0, s1 = 0, s2 = 0;
    bool vec = false, scalar = false, linear = false;
    int c_lz = 0, c_ny = 1, c_n0 = 1, c_n1 = 1;          // cubic zoom: line lengths and low-res rows under kUR rows
    int64_t c_lines0 = 0, c_lines1 = 0, c_rows2 = 0;     // lines of the x, y and z prefilter
    for (int b = 0; b < B; ++b) {
        const bfm_gen_sample &s = h[b];
        if (cubic_zoom(s)) {
            const int *l = s.new_size;
            c_lz = max(c_lz, l[2]); c_n0 = max(c_n0, l[0]); c_n1 = max(c_n1, l[1]);
            c_lines0 = max(c_lines0, (int64_t)l[1] * l[2]);
            c_lines1 = max(c_lines1, (int64_t)l[0] * l[2]);
            c_rows2 = max(c_rows2, (int64_t)l[0] * l[1]);
            // the first nodes of kUR consecutive rows span <= kUR * ly / s1 + 1 low-res rows (+1 for the float32
            // coordinates), plus 3 more taps; checked exhaustively for ly, s1 <= 320
            c_ny = max(c_ny, min(l[1], (int)((int64_t)kUR * l[1] / s.d.size[1]) + 8));
        } else {
            linear = true;
        }
        lz = max(lz, s.new_size[2]);
        // low-res rows under kUR output rows: at most kUR * ly / s1 + 2 (and never more than ly)
        const int rows = min(s.new_size[1], (int)((int64_t)kUR * s.new_size[1] / s.d.size[1]) + 3);
        ny = max(ny, rows);
        s0 = max(s0, s.d.size[0]); s1 = max(s1, s.d.size[1]); s2 = max(s2, s.d.size[2]);
        if (((int64_t)s.d.size[1] * s.d.size[2]) & 3) scalar = true; else vec = true;
    }
    const size_t smem = (size_t)ny * lz * sizeof(float);
    if (smem > 200 * 1024) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_finish: low-res rows too long for shared memory");
    if (s0 > 65535 || B > 65535) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_finish: grid too large");
    cudaStream_t st = (cudaStream_t)stream;
    const int threads = min(160, (s2 + 31) / 32 * 32);
    const int64_t plane = (int64_t)s1 * s2;
    if (c_lz > 0) {
        const size_t smem_z = ((size_t)kCubicLines * (c_lz | 1) + c_lz) * sizeof(float);
        const size_t smem_c = (size_t)(c_ny + kUR) * c_lz * sizeof(float);
        if (smem_z > 200 * 1024 || smem_c > 200 * 1024 || (c_n0 > c_n1 ? c_n0 : c_n1) > 12 * 1024)
            return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_finish: low-res volume too large for the cubic zoom");
        if (c_lines0 > (1LL << 30) || c_lines1 > (1LL << 30) || c_rows2 > (1LL << 30))
            return fail(BFM_E_UNSUPPORTED, "%s", "bfm_gen_finish: grid too large");
        // without the opt-in, static + dynamic shared memory must fit 48 KB (k_gen_cubic_zoom has ~1 KB static):
        // opt in from 40 KB, as k_gen_upsample does
        if (smem_z > 40 * 1024)
            cudaFuncSetAttribute(k_gen_prefilter_z, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_z);
        if (smem_c > 40 * 1024)
            cudaFuncSetAttribute(k_gen_cubic_zoom, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c);
        k_gen_prefilter<0><<<dim3((unsigned)((c_lines0 + 255) / 256), 1, B), 256, c_n0 * sizeof(float), st>>>(d);
        if ((rc = check_launch("bfm_gen_finish"))) return rc;
        k_gen_prefilter<1><<<dim3((unsigned)((c_lines1 + 255) / 256), 1, B), 256, c_n1 * sizeof(float), st>>>(d);
        if ((rc = check_launch("bfm_gen_finish"))) return rc;
        k_gen_prefilter_z<<<dim3((unsigned)((c_rows2 + kCubicLines - 1) / kCubicLines), 1, B), 128, smem_z, st>>>(d);
        if ((rc = check_launch("bfm_gen_finish"))) return rc;
        k_gen_cubic_zoom<<<dim3((s1 + kUR - 1) / kUR, s0, B), threads, smem_c, st>>>(d, c_ny);
        if ((rc = check_launch("bfm_gen_finish"))) return rc;
    }
    if (linear) {
        if (smem > 40 * 1024)
            cudaFuncSetAttribute(k_gen_upsample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k_gen_upsample<<<dim3((s1 + kUR - 1) / kUR, s0, B), threads, smem, st>>>(d, lz, ny);
        rc = check_launch("bfm_gen_finish");
        if (rc) return rc;
    }
    if (vec) {
        k_gen_normalize<4><<<dim3((unsigned)((plane / 4 + 255) / 256), s0, B), 256, 0, st>>>(d);
        rc = check_launch("bfm_gen_finish");
        if (rc) return rc;
    }
    if (scalar) {
        k_gen_normalize<1><<<dim3((unsigned)((plane + 255) / 256), s0, B), 256, 0, st>>>(d);
        rc = check_launch("bfm_gen_finish");
    }
    return rc;
}

int bfm_gen_zoom_coords(int n_in, int n_out, float *out_dev, void *stream) {
    if (n_in <= 0 || n_out <= 0 || !out_dev) return fail(BFM_E_INVALID, "%s", "bfm_gen_zoom_coords: bad argument");
    k_gen_zoom_coords<<<(n_out + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n_in, n_out, out_dev);
    return check_launch("bfm_gen_zoom_coords");
}

int bfm_gen_run(const bfm_gen_sample *h, const bfm_gen_sample *d, int B, void *stream) {
    int rc;
    if ((rc = bfm_gen_plan(h, d, B, stream))) return rc;
    if ((rc = bfm_gen_bbox(h, d, B, stream))) return rc;
    if ((rc = bfm_gen_gmm(h, d, B, stream))) return rc;
    if ((rc = bfm_gen_warp(h, d, B, stream))) return rc;
    if ((rc = bfm_gen_resample(h, d, B, stream))) return rc;
    return bfm_gen_finish(h, d, B, stream);
}

}  // extern "C"
