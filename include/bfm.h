/*
 * libbfm -- C ABI of the B200 (sm_100a) synthetic-data generator kernels.
 *
 * Drop-in boundary for the hot path of jhuldr/BrainFM's on-the-fly generator.  The reference is
 * pure Python/PyTorch and has no FFI of its own (SURVEY.md 8b); each entry point below replaces the
 * ATen op-chain of the reference function cited next to it and is bound from Python with ctypes
 * (brainfm_b200/_lib.py; the binding a reference maintainer would add is shown in INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller allocates all outputs; no ownership is transferred; no global state;
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered and asynchronous;
 *   - return value: 0 = OK, negative = BFM_E_*; bfm_last_error() gives a thread-local message;
 *   - volumes are row-major (X,Y,Z[,C]) with Z (or C) contiguous, like the reference's tensors.
 */
#ifndef BFM_H_
#define BFM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BFM_OK 0
#define BFM_E_INVALID (-1)      /* bad argument (null pointer, non-positive size, unknown enum) */
#define BFM_E_UNSUPPORTED (-2)  /* valid in the reference but not implemented here */
#define BFM_E_CUDA (-3)         /* CUDA runtime error; see bfm_last_error() */

#define BFM_ABI_VERSION 8

int bfm_abi_version(void);
const char *bfm_last_error(void);
/* number of kernels launched by this library in the calling process since load (bench.py gpu_launches) */
uint64_t bfm_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Op-level entry points (one reference function each)
 * ---------------------------------------------------------------------------------------------- */

/* fast_3D_interp_torch(X, II, JJ, KK, 'linear', default)            Generator/utils.py:140-192
 * X: (nx,ny,nz,C) f32 channels-last; I,J,K: n coordinates; out: (n,C).
 * Points failing  I>0 & J>0 & K>0 & I<=nx-1 & J<=ny-1 & K<=nz-1  get default_value.
 * If default_dev != NULL the default is read from that device scalar (the 'max' mode). */
int bfm_trilerp_pull(const float *X, int nx, int ny, int nz, int C,
                     const float *I, const float *J, const float *K, int64_t n,
                     float default_value, const float *default_dev, float *out, void *stream);

/* fast_3D_interp_torch(X, II, JJ, KK, 'nearest')                    Generator/utils.py:124-138
 * elem_size 1, 4 or 8 bytes per channel value; round-half-even then clamp; bit-exact gather. */
int bfm_nearest_pull(const void *X, int elem_size, int nx, int ny, int nz, int C,
                     const float *I, const float *J, const float *K, int64_t n, void *out, void *stream);

/* myzoom_torch(X, factor)                                            Generator/utils.py:200-257
 * X: (a,b,c,C) -> out (A,B,Cc,C).  lo/hi/wl/wh: per-axis index/weight tables built by the caller with
 * the reference's own float32 arange expressions (lengths A, B, Cc).  Evaluated in the reference's
 * pass order (axis 0, 1, 2) with separately rounded mul/add => bit-exact. */
int bfm_zoom_linear(const float *X, int a, int b, int c, int C,
                    const int *lo0, const int *hi0, const float *wl0, const float *wh0, int A,
                    const int *lo1, const int *hi1, const float *wl1, const float *wh1, int B,
                    const int *lo2, const int *hi2, const float *wl2, const float *wh2, int Cc,
                    float *out, void *stream);

/* gaussian_blur_3d: ONE axis of the separable zero-padded correlation   Generator/utils.py:83-94
 * in/out: (nx,ny,nz) f32; taps: (2*half+1) normalised weights (device). */
int bfm_blur_axis(const float *in, float *out, int nx, int ny, int nz, int axis,
                  const float *taps, int half, void *stream);

/* Banded linear map along one axis: out[i'] = sum_t w[i'*T+t] * in[start[i']+t] (taps outside
 * [0,n) are skipped).  Used for blur o trilinear-downsample (resample_resolution,
 * Generator/utils.py:591-609) with optional fused add_noise (utils.py:633-638) epilogue:
 * out = max(0, out + noise_std*eps)  when noise_std >= 0 (eps == NULL => Philox(seed)). */
int bfm_band_axis(const float *in, float *out, const int *in_shape, int axis, int n_out,
                  const int *start, const float *w, int T,
                  float noise_std, const float *eps, uint64_t seed, void *stream);

/* dst (device) <- src_pinned (page-locked HOST memory, device-accessible under unified addressing), copied by a
 * kernel instead of the copy engine: the plan arena of a batch (a few KB per sample) must not wait behind bulk
 * uploads queued on the copy engine.  Addresses and nbytes: multiples of 16. */
int bfm_upload_pinned(void *dst, const void *src_pinned, int64_t nbytes, void *stream);

/* Label-map / image ingestion (SURVEY 8f-1): dst (float32, n elements) = nan_to_num(src * slope + inter), src in its
 * stored dtype -- 0 uint8, 1 int16, 2 int32, 3 float32, 4 int8 -- so that a volume crosses PCIe in its on-disk width
 * and is widened on the device.  Replaces `nib.load().get_fdata()` scaling + `.astype(float)` + torch.nan_to_num
 * (Generator/utils.py:279, 304-305) + the float32 host->device copy. */
int bfm_ingest_volume(float *dst, const void *src, int src_dtype, int64_t n, float slope, float inter, void *stream);

/* The volume-sized N(0,1) fields of the chain (`torch.randn` of Generator/datasets.py:371 and utils.py:635) come from
 * an in-kernel counter-based generator: Philox4x32-10 keyed on the per-sample `seed`, counter = (group index,
 * stream), Box-Muller on the four 32-bit outputs; element e of a field is component e % 4 of group e / 4.  Streams:
 * 0 GMM noise (indexed by the absolute SOURCE voxel), 1 acquisition noise (absolute low-res voxel), 2 / 3 the small
 * deformation / bias grids.  This entry point writes out[0..n) = that sequence starting at group first_group, so that
 * the distribution the kernels draw from can be tested on its own. */
int bfm_philox_normal(float *out, int64_t n, uint64_t seed, uint32_t stream_id, uint64_t first_group, void *stream);

/* add_noise (Generator/utils.py:633-638) on a PART of a volume: x[i] = max(0, x[i] + noise_std * eps[first_element + i])
 * with eps the stream-`stream_id` sequence of bfm_philox_normal.  Slab mode (one volume cut across GPUs) passes the
 * absolute low-res index of its first voxel, so the assembled volume does not depend on the decomposition. */
int bfm_add_noise_at(float *x, int64_t n, float noise_std, uint64_t seed, uint32_t stream_id, int64_t first_element,
                     void *stream);

/* x = nan_to_num(x) in place (torch.nan_to_num, Generator/utils.py:305): applied once when a real-image volume
 * enters the device cache instead of at every crop read. */
int bfm_sanitize_f32(float *x, int64_t n, void *stream);

/* The banded map of one axis of resample_resolution (Gaussian slice-profile blur, then masked 2-tap linear
 * sampling at the acquisition grid), built on the device: start[n_out], w[n_out*T], T = 2*ceil(3*sigma)+2 <= 64.
 * make_gaussian_kernel Generator/utils.py:74-81; sample positions utils.py:595-605 */
int bfm_band_build(int n_in, int n_out, double sigma, int T, int *start, float *w, void *stream);

/* global min / max of a float volume (device results, 2 floats: min, max)  torch.min/torch.max */
int bfm_minmax(const float *x, int64_t n, float *minmax_dev, void *stream);

/* out = (x - sub[0]) / div[0], optionally flipped along axis 0; sub/div are device scalars (NULL => 0 / 1).
 * read_and_deform_image normalisation + flip                            Generator/utils.py:326-329 */
int bfm_shift_scale_flip(const float *x, float *out, int nx, int64_t plane,
                         const float *sub_dev, const float *div_dev, float post_scale, int flip, void *stream);

/* deform_grid                                                         Generator/datasets.py:264-303
 * Pass 1 (coords_out == NULL): reduces the clamped source coordinates of every output voxel to the
 *   bounding box bbox_dev[6] = {lo0,lo1,lo2, hi0,hi1,hi2} (ints, hi exclusive = 1+ceil(max)).
 * Pass 2 (coords_out != NULL): writes bbox-relative coordinates xx2,yy2,zz2 as 3 planes (3,sx,sy,sz).
 * F is evaluated on the fly from Fsmall (fs0,fs1,fs2,3) through the myzoom tables; Fsmall == NULL
 * means no nonlinear field.  F_full (optional, (sx,sy,sz,3)) overrides Fsmall (SVF-integrated field). */
typedef struct bfm_zoom_tab {
    const int *lo[3];
    const int *hi[3];
    const float *wl[3];
    const float *wh[3];
} bfm_zoom_tab;

typedef struct bfm_deform {
    int size[3];        /* output grid */
    int src[3];         /* source volume shape */
    float A[9];         /* row-major affine (float32 like the reference tensor) */
    float c2[3];
    float ctr[3];       /* (size-1)/2 in float32 */
    const float *fsmall; /* (fs0,fs1,fs2,3) or NULL */
    int fs[3];
    int photo;          /* zero F[...,1] (datasets.py:211-212) */
    bfm_zoom_tab ftab;
    const float *F_full; /* optional full-resolution field (size,3) */
    /* voxels next to the node boundaries of the small grid, per axis (sorted, device); the bounding box of
       the fused chain is evaluated on their product first (bfm_gen_bbox).  ncand[0] == 0: always full scan. */
    const int *cand[3];
    int ncand[3];
} bfm_deform;

int bfm_deform_grid(const bfm_deform *d_host, int *bbox_dev, float *coords_out, void *stream);

/* read_and_deform (+ wrappers): trilinear warp of a full source volume through the deformation,
 * reading only inside the bbox crop                                    Generator/utils.py:296-321
 * value = nan_to_num(src) -> (v - mean)/scale.  default: 0, or the crop maximum when default_max != 0.
 * minmax_out_dev (optional, 2 floats): min and max of the warped volume, reduced in the same kernel
 * (read_and_deform_image's `Idef -= min; Idef /= max`, utils.py:326-327). */
int bfm_warp_volume(const bfm_deform *d_host, const int *bbox_dev, const float *src,
                    float mean, float scale, int default_max, float *scratch_max_dev,
                    float *out, float *minmax_out_dev, void *stream);

/* read_and_deform_segmentation                                        Generator/utils.py:394-424
 * labels: int32 source volume; lut: int32[lut_n]; out: (n_classes, size) f32 one-hot, channel-first,
 * flipped along axis 0 and channel-permuted by vflip (int32[n_classes]) when flip != 0.
 * label_out (optional): (size) int32 warped class index (unflipped). */
int bfm_label_warp_onehot(const bfm_deform *d_host, const int *bbox_dev, const int32_t *labels,
                          const int32_t *lut, int lut_n, int n_classes, const int32_t *vflip, int flip,
                          float *onehot_out, int32_t *label_out, void *stream);

/* random_nonlinear_transform SVF integration step                     Generator/datasets.py:214-223
 * out = Fin + trilerp(Fin, id + Fin)  for a (sx,sy,sz,3) field. */
int bfm_svf_step(const float *Fin, float *Fout, int sx, int sy, int sz, void *stream);
/* The whole integration: out = F * scale, then n_steps bfm_svf_step compositions, with the field kept as 16-byte
 * {f0, f1, f2, 0} records between the steps (one 128-bit load per tap; identical arithmetic).  F, out: (sx,sy,sz,3)
 * float32; scratch: 2 * sx*sy*sz*4 floats, 16-byte aligned.              Generator/datasets.py:214-223 */
int bfm_svf_integrate(const float *F, float *out, int sx, int sy, int sz, int n_steps, float scale, float *scratch,
                      void *stream);

/* ------------------------------------------------------------------------------------------------
 * Fused batched synthesis chain:  BaseGen.generate_sample + augment_sample with the stock steps
 * ['gamma','bias_field','resample','noise']                       Generator/datasets.py:306-428
 * One descriptor per sample (device-visible array); every launch covers the whole batch.
 * ---------------------------------------------------------------------------------------------- */
typedef struct bfm_band {
    const int *start;   /* n_out */
    const float *w;     /* n_out * T */
    int T;              /* 2*ceil(3*sigma) + 2 */
    int n_in, n_out;
    int axis;
    /* build != 0: start/w point to uninitialised device scratch that bfm_gen_plan fills on the GPU from
       (n_in, n_out, sigma) with the reference's expressions (make_gaussian_kernel utils.py:74-81, float64
       np.arange sample positions utils.py:595-605); build == 0: the caller supplies the tables. */
    int build;
    double sigma;
} bfm_band;

#define BFM_MAX_AUX 3

typedef struct bfm_gen_sample {
    bfm_deform d;
    /* labels -> GMM image */
    const void *labels;     /* full source volume */
    int label_is_u8;        /* 1: uint8, 0: float32 (G==77 -> 2, round-half-even) */
    const float *mu;        /* 256 */
    const float *sigma;     /* 256 */
    const float *eps_gmm;   /* injected N(0,1) draws shaped like the bbox crop, or NULL => Philox */
    uint64_t seed;          /* Philox key (per sample) */
    float *syn;             /* scratch, source-volume sized + src[1]*src[2]+src[2]+1 floats of tail padding;
                               must only ever hold finite values (zero it once, then let bfm_gen_gmm write it) */
    int *bbox;              /* 6 ints (device) */
    /* optional mixing with real modalities (datasets.py:379-388): I = v0*I + v[m]*mix[m] */
    const float *mix[3];
    float mixw[4];
    /* gamma + bias field */
    float gamma;            /* exp(gamma_std*n), rounded to float32 like the reference pow */
    const float *bfsmall;   /* (bs0,bs1,bs2) */
    int bs[3];
    bfm_zoom_tab btab;
    float *i_bf;            /* (size) high_res image after bias */
    float *bflog_out;       /* (size) flipped if flip, or NULL */
    int flip;
    /* resolution degradation: up to 3 banded passes, executed in the given order */
    bfm_band band[3];
    int n_band;             /* n_band == 1 with band[0].T == 1, build == 0 and new_size == size denotes the undegraded
                               class (identity band, identity zoom): bfm_gen_resample then writes `out` directly */
    int zero_first[3];      /* strict `>0` mask of identity axes (SURVEY 3.3 item 2) */
    float noise_std;
    const float *eps_noise; /* injected, low-res shaped, or NULL => Philox */
    float *tmp[2];          /* ping-pong scratch, each >= prod(size) floats */
    float *lowres;          /* (new_size), 16-byte aligned */
    int new_size[3];
    /* back to the training grid + normalise */
    bfm_zoom_tab utab;      /* tables of myzoom_torch(lowres, 1/factors), lengths size[d] */
    float *maxval;          /* device scalar */
    float *out;             /* (size) 'input', flipped if flip */
    float *residual;        /* optional 'high_res_residual' */
    /* Real-image targets that share the deformation (read_and_deform_image, Generator/utils.py:324-343):
       warped by the same gather as the synthetic image, then `Idef -= min; Idef /= max` and the flip are
       applied by bfm_gen_finish.  aux_src: full source volumes (f32, finite -- nan_to_num applied when the
       volume is cached -- and followed by >= src[1]*src[2]+src[2]+1 readable floats); aux_raw: (size) scratch;
       aux_out: (size) result; aux_mm: 2*n_aux ints of device scratch.  n_aux must be 0 when mix[0] != NULL
       (the mixing step needs the normalised targets before the warp). */
    int n_aux;
    const float *aux_src[BFM_MAX_AUX];
    float *aux_raw[BFM_MAX_AUX];
    float *aux_out[BFM_MAX_AUX];
    int *aux_mm;
    /* Slab mode (one volume cut into x-slabs of the output grid, one per GPU): bfm_gen_warp only evaluates the
       output planes [x_begin, x_begin + x_count); x_count == 0 means the whole grid.  i_bf, bflog_out and
       aux_raw keep their whole-volume indexing: the caller passes pointers biased by -x_begin planes (the
       flipped plane for bflog_out) so that only the owned planes have to exist. */
    int x_begin, x_count;
    /* Small random grids drawn on the device (native planner, bfm_plan_batch): bfm_gen_plan fills d.fsmall with
       fs_std * N(0,1) when gen_small & 1 (Philox stream 2 of `seed`; random_nonlinear_transform,
       Generator/datasets.py:209) and bfsmall with bf_std * N(0,1) when gen_small & 2 (stream 3; add_bias_field,
       Generator/utils.py:584) -- the pointers must then address writable device scratch. */
    int gen_small;
    float fs_std, bf_std;
    /* Real-image input (BaseGen.augment_sample with input_mode T1 / T2 / FLAIR, Generator/datasets.py:306-316): `syn`
       is the real source volume itself (f32, finite, followed by >= src[1]*src[2]+src[2]+1 readable floats, never
       written), the GMM stage is skipped (labels / mu / sigma may be NULL) and the warped value is NOT clamped at 0
       before the gamma transform.  2 = CT input: the warped value is clamped to [0, 80] (datasets.py:318-319) and
       there is no bias field (bfsmall == NULL, Generator/utils.py:575-577). */
    int real_input;
    /* Pair mode.  syn_pair_ok != 0: `syn` has room for TWICE the floats (2 * (source volume + tail padding), zeroed
       once by the caller; tail padding >= src[1]*src[2]+src[2]+1 pairs, as for the unpaired path).  For samples with
       exactly one real-image target, no mixing, a synthetic input, src[2] % 4 == 0 and no full-resolution field,
       bfm_gen_gmm then writes {synthetic value, aux_src[0] value} PAIRS (float2 per source voxel) and bfm_gen_warp gathers both volumes with one 64-bit load per trilinear tap
       (k_gen_warp_pk: half the load requests of the two-volume gather, packed f32x2 arithmetic).  Results are
       identical to the unpaired path. */
    int syn_pair_ok;
    /* Zoom back to the training grid (bfm_gen_finish; Generator/datasets.py:337-340).  0: myzoom_torch, the linear
       zoom through `utab`.  3: the generator's `bspline_zooming`, i.e. interpol.resize(I, shape=size, anchor='edge',
       interpolation=3, bound='dct2', prefilter=True): the dct2 cubic B-spline prefilter runs in place on `lowres`
       (dead after the finish stage), then a cubic pull at the edge-anchored coordinates; `utab` is not read.  The
       undegraded class keeps its direct path (see n_band).  Any other value: BFM_E_INVALID. */
    int zoom_order;
    /* Slab mode, optional: 2 ints of device scratch.  With x_count > 0, bfm_gen_bbox also reduces the source x range
       [gmm_xr[0], gmm_xr[1]) that the OWNED output planes gather from (same clamped coordinates as the bounding box,
       floor(min) .. 1 + ceil(max)), and bfm_gen_gmm only synthesises those planes of the crop: the bounding box --
       the origin of the crop-relative coordinates -- stays the whole volume's, so results do not depend on the
       decomposition, but a rank no longer runs the GMM stage over the whole replicated label map.  NULL: whole crop. */
    int *gmm_xr;
} bfm_gen_sample;

/* Each stage launches over samples [0,B).  `s_dev` is the device copy of the descriptor array,
 * `s_host` the host copy (grid sizing and argument checks only).
 * Alignment (the kernels take 128-bit accesses without testing the pointers; every stage returns BFM_E_INVALID
 * when one of these fails): i_bf, tmp[0], tmp[1] and lowres 16-byte aligned, syn 8-byte aligned, and when
 * size[1]*size[2] % 4 == 0 also out, bflog_out, residual, aux_out[*] and aux_raw[*].  Per-sample scratch slots
 * therefore advance by prod(size) rounded up to a multiple of 4 floats. */
/* bfm_gen_plan: builds the banded blur-o-downsample tables flagged `build` on the device (no host work, no
 * host->device traffic for them); must precede bfm_gen_resample. */
int bfm_gen_plan(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int B, void *stream);
int bfm_gen_bbox(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int B, void *stream);
int bfm_gen_gmm(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int B, void *stream);
int bfm_gen_warp(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int B, void *stream);
int bfm_gen_resample(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int B, void *stream);
int bfm_gen_finish(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int B, void *stream);
/* Test hook, not part of the generator API: the sample coordinates of the cubic zoom back (zoom_order 3) along one
 * axis, n_in -> n_out: out_dev[o] = o * (n_in/n_out) + 0.5 * (n_in/n_out - 1), evaluated on the device in float32 by
 * the same device function bfm_gen_finish uses, so that the parity tests can pin them bit for bit. */
int bfm_gen_zoom_coords(int n_in, int n_out, float *out_dev, void *stream);
/* all six stages back to back */
int bfm_gen_run(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int B, void *stream);

/* Segmentation target of the fused chain (read_and_deform_segmentation, Generator/utils.py:394-424, with
 * deform_one_hots off): one job per ITEM, all jobs in one launch.  A job warps its class map through the deformation,
 * bounding box and flip of descriptor s_dev[sample] (nearest, round-half-even, clamped to the crop: the arithmetic of
 * bfm_label_warp_onehot) and writes the (n_classes, size) float32 one-hot, flipped along axis 0 with output channel c
 * holding input channel vflip_host[c] when the descriptor's flip is set.  Must run after bfm_gen_bbox and before the
 * descriptors' arena slot is reused.
 *   cls: the class map of the item's segmentation, lut applied (labels < 0 or >= lut_n -> 0), uint8, source shape;
 *   out: 16-byte aligned.  n_classes 1..64, vflip_host[c] in [0, n_classes); all jobs share the output size. */
typedef struct bfm_gen_seg {
    int sample;             /* index into the descriptor array */
    const uint8_t *cls;
    float *out;
} bfm_gen_seg;
int bfm_gen_segmentation(const bfm_gen_sample *s_host, const bfm_gen_sample *s_dev, int n_desc, const bfm_gen_seg *jobs,
                         int n_jobs, int n_classes, const int32_t *vflip_host, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Native host planner: every per-sample scalar draw and all the scalar set-up arithmetic of
 * BaseGen.__getitem__ / BrainIDGen.__getitem__ for synthetic inputs with the stock augmentation chain, in the
 * reference's draw order, filled straight into bfm_gen_sample descriptors (HOST code, no Python per sample):
 *   read_input draw                      Generator/datasets.py:572
 *   get_setup_params, resolution_sampler Generator/datasets.py:466-493, Generator/utils.py:34-57
 *   random_affine_transform              Generator/datasets.py:187-201, make_affine_matrix utils.py:102-116
 *   random_nonlinear_transform (sizes)   Generator/datasets.py:203-212
 *   get_contrast                         Generator/datasets.py:430-464
 *   gamma / bias / resample / noise set-up  Generator/utils.py:568-572, 574-585, 591-609, 633-635
 * Draw source: replay == NULL: an in-library Philox4x32-10 stream keyed on (seed, sample counter) -- same
 * distributions as the reference's numpy/torch draws, not the same streams; the small random grids are then
 * drawn on the device (gen_small).  replay != NULL: the draws are read, in the reference's order, from a flat
 * array of doubles (scalars, then every element of array-shaped draws; the parity tests feed the oracle's
 * log) and the small grids are written into the pinned arena by the host.
 * ---------------------------------------------------------------------------------------------- */
typedef struct bfm_zoom_axis {      /* device-resident myzoom_torch tables of one axis, one (n_in -> n_out) pair */
    const int *lo, *hi;
    const float *wl, *wh;
    const int *cand;                /* bounding-box candidate voxels of this zoom (forward tables only) */
    int ncand;
    int valid;                      /* round(n_in * factor) == n_out */
} bfm_zoom_axis;

typedef struct bfm_plan_aug {       /* parameter ranges of one sample of an item (generator + overrides) */
    double gamma_std, bf_scale_min, bf_scale_max, bf_std_min, bf_std_max, noise_std_min, noise_std_max;
} bfm_plan_aug;

#define BFM_PLAN_MAX_SAMPLES 16

typedef struct bfm_plan_cfg {
    int size[3];
    double res[3];                  /* res_training_data */
    int low_res_only, nonlinear_transform;
    double photo_prob, pathology_prob, random_shape_prob, flip_prob;
    double max_rotation, max_shear, max_scaling;
    double nonlin_scale_min, nonlin_scale_max, nonlin_std_max;
    double ct_prob, mix_synth_prob;
    int8_t ct_group[256];           /* -1, or 0..3 = darker, dark, bright, brighter (constants.py) */
    int n_samples;                  /* samples per item: 1 (BaseGen) or all_samples (BrainIDGen) */
    int bspline_zooming;            /* != 0: every descriptor gets zoom_order = 3 (cubic zoom back); draws nothing */
    bfm_plan_aug aug[BFM_PLAN_MAX_SAMPLES];        /* synthetic inputs (generator + [mild|severe] + synth_image_generator) */
    bfm_plan_aug aug_real[BFM_PLAN_MAX_SAMPLES];   /* real-image inputs (... + real_image_generator) */
    /* directories indexed by n_in = 0..size[a]: fwd = zoom by size/n_in (small grids -> training grid),
       inv = zoom by 1/(n_in/size) (low-res grid -> training grid) */
    const bfm_zoom_axis *fwd[3];
    const bfm_zoom_axis *inv[3];
    const int *ends[3];             /* device {0, size[a]-1}: candidates of an axis without nonlinear field */
    const int *ident_start;         /* device arange(size[2]) and ones(size[2]): identity band */
    const float *ident_w;
} bfm_plan_cfg;

typedef struct bfm_plan_item {
    const void *labels;             /* device, full source volume */
    int label_is_u8;
    int src[3];
    int n_aux;                      /* real-image targets riding on the gather of the item's FIRST sample */
    const float *aux_src[BFM_MAX_AUX];
    float *aux_out[BFM_MAX_AUX];
    float *aux_raw[BFM_MAX_AUX];
    /* replay mode only: injected volume-sized normal fields of each sample (device) */
    const float *eps_gmm[BFM_PLAN_MAX_SAMPLES];
    const float *eps_noise[BFM_PLAN_MAX_SAMPLES];
    /* read_input (Generator/datasets.py:563-588): the input is the first of T1, T2, FLAIR, CT with u < input_prob[m]
       whose volume exists, else synthetic.  real_vol[m]: device volume of T1 / T2 / FLAIR with the source shape
       (f32, finite, padded like aux_src) or NULL when the subject does not have it; ct_vol likewise for CT
       (window [0, 80], no bias field, no bias_field_log output). */
    double input_prob[4];
    const float *real_vol[3];
    const float *ct_vol;
} bfm_plan_item;

typedef struct bfm_plan_out {       /* per SAMPLE buffers (device), caller allocated */
    float *out, *bflog_out, *residual;
    float *syn, *i_bf, *tmp[2], *lowres;
    int64_t syn_pair_ok;            /* see bfm_gen_sample.syn_pair_ok */
} bfm_plan_out;

typedef struct bfm_plan_info {      /* what the host needs to know about a planned ITEM */
    int input_mode;                 /* 0 synth, 1 T1, 2 T2, 3 FLAIR, 4 CT */
    int photo_mode, flip;
    double spac, resolution[3], thickness[3], scaling_factor_distances;
    float A[9], c2[3];
    int fs[3];
    int new_size[BFM_PLAN_MAX_SAMPLES][3];
} bfm_plan_info;

/* Plans n_items items = n_items * cfg->n_samples samples.  descs_host[n]: sample descriptors (item-major), written
 * in place and mirrored into the arena; outs[n]: per-sample buffers.  The arena is one pinned host buffer and its
 * device twin (same layout): on return *arena_used is the end of the reservations and *upload_bytes the length of
 * the host-written prefix that has to reach the device (bfm_upload_pinned) before bfm_gen_run;
 * *descs_dev = device address of the descriptor array.  replay/n_replay: see above (NULL/0 = native draws);
 * *replay_used returns the number of doubles consumed. */
int bfm_plan_batch(const bfm_plan_cfg *cfg, int n_items, const bfm_plan_item *items, const bfm_plan_out *outs,
                   uint64_t seed, uint64_t counter, void *arena_host, void *arena_dev, int64_t arena_capacity,
                   int64_t *arena_used, int64_t *upload_bytes, bfm_gen_sample *descs_host, void **descs_dev,
                   bfm_plan_info *info, const double *replay, int64_t n_replay, int64_t *replay_used);

/* Base pointers of a batch's buffers, per-sample strides implied: out / bflog_out / residual advance by N = prod(size)
 * floats per sample and aux_out by N per fused real-image target, in item order; the scratch advances by
 * Npad = (N + 3) & ~3 floats (i_bf, lowres: Npad per sample, tmp: 2 * Npad, aux_raw: Npad per target) so that every
 * slot keeps the 16-byte alignment of its base; syn by syn_stride. */
typedef struct bfm_step_bufs {
    float *out, *bflog_out, *residual;
    float *syn;
    int64_t syn_stride;
    float *i_bf, *tmp, *lowres;
    float *aux_out, *aux_raw;
    int64_t pair_ok;
} bfm_step_bufs;

/* Lays the buffers of `bufs` out per sample: fills outs[0 .. n_items * cfg->n_samples) and items[n].aux_out / aux_raw
 * of every fused real-image target, in item order (what bfm_plan_batch takes).  Refuses a null out / syn / i_bf / tmp /
 * lowres, and a null aux_out / aux_raw when an item has such a target. */
int bfm_plan_layout(const bfm_plan_cfg *cfg, int n_items, bfm_plan_item *items, const bfm_step_bufs *bufs,
                    bfm_plan_out *outs);

/* bfm_plan_layout + bfm_plan_batch (native draws) + bfm_upload_pinned of the host-written arena prefix + bfm_gen_run:
 * ONE call per batch.  items[n].aux_out / aux_raw are filled in.  arena_used_in: bytes of
 * the arena already reserved; *arena_used_out: after planning. */
int bfm_plan_run(const bfm_plan_cfg *cfg, int n_items, bfm_plan_item *items, const bfm_step_bufs *bufs, uint64_t seed,
                 uint64_t counter, void *arena_host, void *arena_dev, int64_t arena_capacity, int64_t arena_used_in,
                 int64_t *arena_used_out, bfm_gen_sample *descs_host, void **descs_dev, bfm_plan_info *info, void *stream);

/* ------------------------------------------------------------------------------------------------
 * utils/interpol (vendored torch-interpol 0.2.3): spline resampling, forward semantics
 * ---------------------------------------------------------------------------------------------- */

/* grid_pull / grid_push / grid_count / grid_grad                     utils/interpol/nd.py:81-288,
 *                                                                    iso0.py:24-100, iso1.py:29-387
 * Always 3-D (pad lower dimensions with singleton axes, order 0, coordinate 0).
 * mode 0 pull: inp (Bi,C,X,Y,Z), grid (Bg,P,3) -> out (B,C,P)
 * mode 1 push: inp (Bi,C,P) or NULL (= count), grid (Bg,P,3) -> out (B,C,X,Y,Z), PRE-ZEROED by the caller
 * mode 2 grad: like pull, out (B,C,P,3)
 * order[d] 0..7 (splines.py:30-160), bound[d] 0..6 = zero, replicate, dct1, dct2, dst1, dst2, dft
 * (bounds.py:8-89), extrapolate 0 no / 1 yes / 2 hist (jit_utils.py:242-255).  Bi, Bg in {1, B}.
 * iso: 1 when every (real) axis has order 0 (nearest = round-half-even, iso0.py:10-15), 2 when every axis has
 * order 1 (iso1 gradient convention), 0 otherwise (generic nd path) -- the reference's own dispatch
 * (pushpull.py:35-233). */
int bfm_interpol(int mode, int is_double, const void *inp, const void *grid, void *out, const int *ishape,
                 const int *order, const int *bound, int extrapolate, int iso, int B, int C, int Bi, int Bg,
                 int64_t P, void *stream);

/* Backward pass of grid_grad                                            utils/interpol/autograd.py:216-243,
 *                                                                      pushpull.py:303-325, nd.py:292-465
 * gout: incoming gradient (B, C, P, 3); inp (B, C, X, Y, Z); grid (B, P, 3) -- all with the full batch.
 * grad_inp (optional, (B, C, X, Y, Z), PRE-ZEROED): push of gout with the first-derivative weights (grid_pushgrad).
 * grad_grid (optional, (B, P, 3)): sum over channels and d of gout[..., d] * Hessian[..., d, :] (grid_hess contracted
 * with gout), second-derivative weights Spline.fasthess (splines.py:149-195); zero Hessian diagonal for order <= 1. */
int bfm_interpol_grad_backward(int is_double, const void *gout, const void *inp, const void *grid, void *grad_inp,
                               void *grad_grid, const int *ishape, const int *order, const int *bound, int extrapolate,
                               int iso, int B, int C, int64_t P, void *stream);

/* grid_pull fast path: float32, the same spline order (1 = linear, 3 = cubic) on all three axes.
 * inp is addressed through element strides istride[5] = (batch, channel, x, y, z) -- a channels-last view (e.g. a
 * permuted displacement field) is read in place; a zero batch stride broadcasts.  grid (B or 1, P, 3) with batch
 * stride grid_bstride elements; out (B, C, P) contiguous, or (B, P, C) when out_chlast != 0.  Same node indices, bound signs and spline weights as
 * bfm_interpol (utils/interpol/nd.py:81-150); per tap the three weights are multiplied first.  One batch element
 * of the input must span fewer than 2^31 elements. */
int bfm_interpol_pull_fast(const float *inp, const int64_t *istride, const float *grid, int64_t grid_bstride,
                           float *out, int out_chlast, const int *ishape, int order, const int *bound, int extrapolate,
                           int B, int C, int64_t P, void *stream);

/* add_identity_grid for 3-D float32 fields: out = disp + voxel index, (B, X, Y, Z, 3) contiguous
 * utils/interpol/api.py:480-521 */
int bfm_add_identity_grid(const float *disp, float *out, int B, int X, int Y, int Z, void *stream);

/* One scaling-and-squaring step of a 3-D displacement field (SURVEY K13): out = disp + grid_pull(disp, disp + identity)
 * with linear interpolation, (B, X, Y, Z, 3) float32, out != disp.  Bit-identical to bfm_add_identity_grid +
 * bfm_interpol_pull_fast(order 1) + add (utils/interpol/api.py:480-521, nd.py:81-150), without materialising the grid
 * or the pulled field. */
int bfm_compose_step(const float *disp, float *out, int B, int X, int Y, int Z, const int *bound, int extrapolate,
                     void *stream);
/* Scaling and squaring: out = displacement of exp(svf): disp = svf / 2**steps, then `steps` bfm_compose_step
 * compositions, with the field kept as 16-byte {x, y, z, 0} records between the steps (one 128-bit load per tap).
 * svf, out: (B, X, Y, Z, 3) float32; scratch: 2 * B*X*Y*Z*4 floats, 16-byte aligned.  Bit-identical to the step-wise
 * form.                                                       BASELINE configs[2]; Generator/datasets.py:214-223 */
int bfm_exp_velocity(const float *svf, float *out, int B, int X, int Y, int Z, int steps, const int *bound,
                     int extrapolate, float *scratch, void *stream);

/* spline_coeff: in-place recursive prefilter along one axis of a tensor viewed as (outer, n, inner)
 * utils/interpol/coeff.py:35-316.  bound: 0 zero (=dct1), 1 replicate (=dct2), 2 dct1, 3 dct2, 6 dft. */
int bfm_spline_filter(void *data, int is_double, int64_t outer, int n, int64_t inner, int bound,
                      const double *poles_host, int npoles, void *stream);

/* ------------------------------------------------------------------------------------------------
 * ShapeID: Perlin shapes, curl velocity, advection PDE, Runge-Kutta building blocks
 * ---------------------------------------------------------------------------------------------- */

/* generate_perlin_noise_3d                                           ShapeID/perlin3d.py:15-90
 * grad: (res0+1, res1+1, res2+1, 3) float64 unit gradients (tileable copies applied by the caller);
 * out: (shape) float64, bit-exact with the numpy reference. */
int bfm_perlin3d(const double *grad, const int *shape, const int *res, double *out, void *stream);
/* mask = noise >= thr; noise *= mask                                 ShapeID/perlin3d.py:86-90 */
int bfm_threshold_mask(double *noise, double *mask, int64_t n, double thr, void *stream);
/* gradient_c (mode 0) / gradient_f (1) / gradient_b (2) of a 3-D volume -> (shape, 3) float32
 * ShapeID/misc.py:198-259, ShapeID/DiffEqs/pde.py:13-183 */
int bfm_gradient3d(const void *X, int is_double, const int *shape, int mode, const float *spacing, float *out,
                   void *stream);
/* stream_3D * V_multiplier                                           ShapeID/misc.py:66-80, perlin3d.py:149-156 */
int bfm_curl3d(const void *A, const void *B, const void *C, int is_double, const int *shape, float multiplier,
               float *Vx, float *Vy, float *Vz, void *stream);
/* AdvDiffPDE.forward for perf_pattern 'adv', V_type 'vector_div_free' ShapeID/DiffEqs/pde.py:588-640, 301-328, 499-509
 * neumann != 0: replicate-pad the interior before differencing (set_BC). */
int bfm_advect_rhs(const void *C, int is_double, const float *Vx, const float *Vy, const float *Vz, const int *shape,
                   int neumann, const float *spacing, float *out, void *stream);
/* AdvDiffPDE.forward, diffusion part, D_type 'constant' (D == NULL, D_const) or 'scalar' (D: (shape) float32 field)
 * ShapeID/DiffEqs/pde.py:331-353, 551-559, 623-639.  accumulate != 0: out += rhs (perf_pattern 'adv_diff': call
 * bfm_advect_rhs first). */
int bfm_diffuse_rhs(const void *C, int is_double, const float *D, float D_const, const int *shape, int neumann,
                    const float *spacing, int accumulate, float *out, void *stream);

/* out = y0 + sum_j coef[j]*k[j] (float32 partial sums, state precision for the final add); y0 == NULL: out = sum
 * _runge_kutta_step / _scaled_dot_product                            ShapeID/DiffEqs/rk_common.py:22-61, misc.py:22-25 */
int bfm_rk_combine(const void *y0, int is_double, const float *const *k_host, const float *coef_host, int n_terms,
                   int64_t n, void *out, int out_is_double, void *stream);
/* result_dev[0] = sum((err / (atol + rtol*max(|y0|,|y1|)))^2)         ShapeID/DiffEqs/misc.py:146-157 */
int bfm_rk_error_sum(const float *err, const void *y0, const void *y1, int is_double, int64_t n, double rtol,
                     double atol, double *result_dev, void *stream);

/* bfm_rk_combine(NULL, ...) + bfm_rk_error_sum in one pass: the error estimate err = sum_j coef[j]*k[j] is formed in
 * registers and never written.  err_scratch (n floats) is only used when the inputs are not 16-byte aligned or n is
 * not a multiple of 4 (two-kernel form); may be NULL otherwise. */
int bfm_rk_error_fused(const float *const *k_host, const float *coef_host, int n_terms, const void *y0, const void *y1,
                       int is_double, int64_t n, double rtol, double atol, float *err_scratch, double *result_dev,
                       void *stream);

/* Dense output of dopri5 for a float64 state with float32 stages: the quartic through y0, y1, y_mid, f0, f1 at
 * x = (t - t0) / (t1 - t0), evaluated with the reference's tensor expressions and dtype promotions in ONE pass.
 * ShapeID/DiffEqs/interp.py:5-65 */
int bfm_dopri5_interp(const double *y0, const double *y1, const double *y_mid, const float *f0, const float *f1,
                      double dt, double x, int64_t n, double *out, void *stream);

/* ---- pathology branch of generate_sample / augment_sample (op-level) ------------------------------------------- */
/* SYN = clamp(mus[round(G)] + sigmas[round(G)] * eps, 0) over the crop bbox = {x1,y1,z1,x2,y2,z2} of the label volume
 * (label 77 -> 2); eps: (crop) float32 draws or NULL (counter-based field keyed on the absolute source voxel).
 * Generator/datasets.py:364-372 */
int bfm_gmm_crop(const void *labels, int label_is_u8, const int *src, const int *bbox, const float *mu,
                 const float *sigma, const float *eps, uint64_t seed, float *out, void *stream);
/* cerebral = SYN * (Gr != 0); sums_dev[0..3] = sum(SYN | white matter), #white, sum(SYN | grey), #grey
 * Generator/datasets.py:391-398 */
int bfm_pathol_cerebral(const float *syn, const void *labels, int label_is_u8, const int *src, const int *bbox,
                        float *cerebral, double *sums_dev, void *stream);
/* p[c == 0] = 0 (p float32 or float64)                                Generator/datasets.py:399-400 */
int bfm_zero_where_zero(void *p, int p_is_double, const float *c, int64_t n, void *stream);
/* sums_dev[0] = sum(I * P), sums_dev[1] = sum(P)                       Generator/datasets.py:500 */
int bfm_masked_mean(const float *I, const void *P, int p_is_double, int64_t n, double *sums_dev, void *stream);
/* I += Pprob * (mus[round(P)] + sigmas[round(P)] * eps); I[I < 0] = 0 with the reference's dtype promotions (float64
 * P / Pprob: product and sum in float64, one rounding to float32)      Generator/datasets.py:509-513 */
int bfm_encode_pathology(float *I, const void *P, const void *Pprob, int p_is_double, const float *mus,
                         const float *sigmas, int n_tab, const float *eps, uint64_t seed, int64_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BFM_H_ */
