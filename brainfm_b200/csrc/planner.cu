// Native host planner (include/bfm.h "Native host planner"): the per-sample scalar draws and set-up arithmetic
// of BaseGen / BrainIDGen for synthetic inputs with the stock augmentation chain, written straight into
// bfm_gen_sample descriptors.  HOST code: one call plans a whole batch in a few microseconds per sample, where
// the Python planner (brainfm_b200/Generator/datasets.py: _prologue_host, _plan_synth, _build_descs) spends
// ~250 us per sample.  Every expression below follows the Python planner (which follows the reference) operation
// by operation, in float64 or float32 as there, so that with replayed draws both planners fill identical
// descriptors (tests/test_native_planner_gpu.py).
#include "common.cuh"

#include <vector>

#include <cmath>
#include <cstring>

namespace bfm {
namespace {

int failf(int code, const char *fmt, int a, int b) {
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}

// ---- Philox4x32-10, host side (same generator as the device fields, different streams) -----------------
struct Philox {
    uint32_t key[2];
    uint32_t ctr[4];
    uint32_t out[4];
    int have;
    static inline void mulhilo(uint32_t a, uint32_t b, uint32_t &hi, uint32_t &lo) {
        const uint64_t p = (uint64_t)a * b;
        hi = (uint32_t)(p >> 32);
        lo = (uint32_t)p;
    }
    void refill() {
        uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
        for (int r = 0; r < 10; ++r) {
            uint32_t hi0, lo0, hi1, lo1;
            mulhilo(0xD2511F53u, c0, hi0, lo0);
            mulhilo(0xCD9E8D57u, c2, hi1, lo1);
            const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
            c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
        have = 4;
        if (++ctr[0] == 0) ++ctr[1];
    }
    uint32_t u32() {
        if (!have) refill();
        return out[--have];
    }
};

inline uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// One stream of draws: native (Philox) or replayed from a flat array of doubles in consumption order.
struct Draws {
    Philox g;
    const double *replay;
    int64_t n_replay, pos;
    bool overrun;
    double spare;
    bool have_spare;

    void seed(uint64_t s, uint64_t sample) {
        const uint64_t k = splitmix64(s ^ splitmix64(sample));
        g.key[0] = (uint32_t)k; g.key[1] = (uint32_t)(k >> 32);
        g.ctr[0] = g.ctr[1] = 0; g.ctr[2] = 0x706c616eu; g.ctr[3] = 0;      // stream tag "plan"
        g.have = 0;
        have_spare = false;
    }
    double next_replay() {
        if (pos >= n_replay) { overrun = true; return 0.5; }
        return replay[pos++];
    }
    // uniform on [0,1) with 53 random bits (numpy random_sample)
    double rand() {
        if (replay) return next_replay();
        const uint64_t a = g.u32() >> 5, b = g.u32() >> 6;
        return (a * 67108864.0 + b) / 9007199254740992.0;
    }
    // float32 uniform on [0,1) with 24 random bits (torch.rand float32)
    float randf() {
        if (replay) return (float)next_replay();
        return (float)(g.u32() >> 8) * 5.9604644775390625e-8f;
    }
    // N(0,1), Box-Muller in float64
    double randn() {
        if (replay) return next_replay();
        if (have_spare) { have_spare = false; return spare; }
        const double u1 = 1.0 - rand(), u2 = rand();
        const double r = std::sqrt(-2.0 * std::log(u1)), t = 6.283185307179586 * u2;
        spare = r * std::sin(t);
        have_spare = true;
        return r * std::cos(t);
    }
    int randint(int n) {
        if (replay) return (int)next_replay();
        const int v = (int)(rand() * n);
        return v < n ? v : n - 1;
    }
};

// ---- bump allocator over the arena (host buffer and device twin share the layout) -----------------------
struct ArenaCursor {
    char *host;
    char *dev;
    int64_t cap, used;
    bool overflow;
    int64_t take(int64_t nbytes) {
        const int64_t off = (used + 15) / 16 * 16;
        if (off + nbytes > cap) { overflow = true; return 0; }
        used = off + nbytes;
        return off;
    }
};

inline double round_half_even(double v) { return std::nearbyint(v); }      // default rounding mode: to nearest even

inline void matmul3(const double a[9], const double b[9], double c[9]) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double acc = a[3 * i] * b[j];
            acc += a[3 * i + 1] * b[3 + j];
            acc += a[3 * i + 2] * b[6 + j];
            c[3 * i + j] = acc;
        }
}

// make_affine_matrix (Generator/utils.py:102-116): A = SHx SHy SHz Rx Ry Rz, row i scaled by s[i], float64
void affine_matrix(const double rot[3], const double sh[3], const double s[3], double A[9]) {
    const double c0 = std::cos(rot[0]), s0 = std::sin(rot[0]);
    const double c1 = std::cos(rot[1]), s1 = std::sin(rot[1]);
    const double c2 = std::cos(rot[2]), s2 = std::sin(rot[2]);
    const double SHx[9] = {1, 0, 0, sh[1], 1, 0, sh[2], 0, 1};
    const double SHy[9] = {1, sh[0], 0, 0, 1, 0, 0, sh[2], 1};
    const double SHz[9] = {1, 0, sh[0], 0, 1, sh[1], 0, 0, 1};
    const double Rx[9] = {1, 0, 0, 0, c0, -s0, 0, s0, c0};
    const double Ry[9] = {c1, 0, s1, 0, 1, 0, -s1, 0, c1};
    const double Rz[9] = {c2, -s2, 0, s2, c2, 0, 0, 0, 1};
    double t0[9], t1[9];
    matmul3(SHx, SHy, t0);
    matmul3(t0, SHz, t1);
    matmul3(t1, Rx, t0);
    matmul3(t0, Ry, t1);
    matmul3(t1, Rz, t0);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) A[3 * i + j] = t0[3 * i + j] * s[i];
}

struct ItemSetup {
    bool photo, flip;
    double spac, resolution[3], thickness[3];
};

int plan_item(const bfm_plan_cfg &cfg, const bfm_plan_item &it, const bfm_plan_out *outs, Draws &dr, uint64_t seed,
              uint64_t sample0, ArenaCursor &ar, bfm_gen_sample *descs, bfm_plan_info &info, bool native) {
    const int *size = cfg.size;
    // ---- read_input (datasets.py:563-588): first modality with u < prob whose volume exists, else synthetic
    int mode = 0;
    {
        const double u = dr.rand();
        if (u < it.input_prob[0] && it.real_vol[0]) mode = 1;
        else if (u < it.input_prob[1] && it.real_vol[1]) mode = 2;
        else if (u < it.input_prob[2] && it.real_vol[2]) mode = 3;
        else if (u < it.input_prob[3] && it.ct_vol) mode = 4;
    }
    info.input_mode = mode;
    // ---- get_setup_params (datasets.py:466-493)
    ItemSetup st;
    st.photo = cfg.low_res_only ? false : dr.rand() < cfg.photo_prob;
    (void)dr.rand();                                   // pathol_mode        (pathology is not planned here)
    (void)dr.rand();                                   // pathol_random_shape
    st.spac = st.photo ? 2.5 + 10 * dr.rand() : 0.0;
    st.flip = dr.randn() < cfg.flip_prob;
    if (st.photo) {
        st.resolution[0] = cfg.res[0]; st.resolution[1] = st.spac; st.resolution[2] = cfg.res[2];
        st.thickness[0] = cfg.res[0]; st.thickness[1] = 0.1; st.thickness[2] = cfg.res[2];
    } else {                                           // resolution_sampler (utils.py:34-57)
        double r = dr.rand();
        if (cfg.low_res_only) r = r * 0.5 + 0.5;
        for (int a = 0; a < 3; ++a) st.resolution[a] = st.thickness[a] = 1.0;
        if (r < 0.25) {
        } else if (r < 0.5) {
            const int idx = dr.randint(3);
            if (idx < 0 || idx > 2) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: replayed axis out of range");
            st.resolution[idx] = 2.5 + 6 * dr.rand();
            const double t = 4.0 + 2.0 * dr.rand();
            st.thickness[idx] = st.resolution[idx] < t ? st.resolution[idx] : t;
        } else if (r < 0.75) {
            const double base[3] = {1.3, 1.3, 4.8};
            for (int a = 0; a < 3; ++a) st.resolution[a] = st.thickness[a] = base[a] + 0.4 * dr.rand();
        } else {
            for (int a = 0; a < 3; ++a) st.resolution[a] = st.thickness[a] = 2.0 + 3.0 * dr.rand();
        }
    }
    // ---- random_affine_transform (datasets.py:187-201)
    double rot[3], sh[3], sc[3], A64[9];
    for (int a = 0; a < 3; ++a) rot[a] = (2 * cfg.max_rotation * dr.rand() - cfg.max_rotation) / 180.0 * M_PI;
    for (int a = 0; a < 3; ++a) sh[a] = 2 * cfg.max_shear * dr.rand() - cfg.max_shear;
    for (int a = 0; a < 3; ++a) sc[a] = 1 + (2 * cfg.max_scaling * dr.rand() - cfg.max_scaling);
    const double sfd = std::pow(sc[0] * sc[1] * sc[2], .33333333333);
    affine_matrix(rot, sh, sc, A64);
    // ---- random_nonlinear_transform (datasets.py:203-212): sizes and std; the field itself is drawn below
    int fs[3] = {0, 0, 0};
    float fs_std = 0.f;
    const float *fsmall_dev = nullptr;
    float *fsmall_host = nullptr;
    int64_t fsmall_n = 0;
    if (cfg.nonlinear_transform) {
        const double scale = cfg.nonlin_scale_min + dr.rand() * (cfg.nonlin_scale_max - cfg.nonlin_scale_min);
        for (int a = 0; a < 3; ++a) fs[a] = (int)round_half_even(scale * size[a]);
        if (st.photo) fs[1] = (int)round_half_even(size[1] / st.spac);
        fs_std = (float)(cfg.nonlin_std_max * dr.rand());
        for (int a = 0; a < 3; ++a)
            if (fs[a] < 1 || fs[a] > size[a] || !cfg.fwd[a][fs[a]].valid)
                return failf(BFM_E_UNSUPPORTED, "bfm_plan_batch: no zoom table for the %d -> %d deformation grid", fs[a],
                             size[a]);
        fsmall_n = (int64_t)fs[0] * fs[1] * fs[2] * 3;
        if (!native) {                                 // host-written: replayed values times float32(std)
            const int64_t off = ar.take(4 * fsmall_n);
            if (ar.overflow) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: arena overflow");
            fsmall_host = (float *)(ar.host + off);
            fsmall_dev = (const float *)(ar.dev + off);
            for (int64_t q = 0; q < fsmall_n; ++q) fsmall_host[q] = fs_std * dr.randf();
        }
    }
    info.photo_mode = st.photo; info.flip = st.flip; info.spac = st.spac;
    info.scaling_factor_distances = sfd;
    for (int a = 0; a < 3; ++a) {
        info.resolution[a] = st.resolution[a]; info.thickness[a] = st.thickness[a];
        info.c2[a] = (float)((it.src[a] - 1) / 2.0);
        info.fs[a] = fs[a];
    }
    for (int q = 0; q < 9; ++q) info.A[q] = (float)A64[q];

    // ---- samples of this item
    for (int k = 0; k < cfg.n_samples; ++k) {
        const bfm_plan_aug &ag = mode ? cfg.aug_real[k] : cfg.aug[k];
        bfm_gen_sample &s = descs[k];
        const bfm_plan_out &o = outs[k];
        std::memset(&s, 0, sizeof(s));
        // deformation
        bfm_deform &d = s.d;
        for (int a = 0; a < 3; ++a) {
            d.size[a] = size[a];
            d.src[a] = it.src[a];
            d.c2[a] = info.c2[a];
            d.ctr[a] = (float)((size[a] - 1) / 2.0);
        }
        for (int q = 0; q < 9; ++q) d.A[q] = info.A[q];
        d.photo = st.photo;
        if (cfg.nonlinear_transform) {
            for (int a = 0; a < 3; ++a) {
                const bfm_zoom_axis &z = cfg.fwd[a][fs[a]];
                d.fs[a] = fs[a];
                d.ftab.lo[a] = z.lo; d.ftab.hi[a] = z.hi; d.ftab.wl[a] = z.wl; d.ftab.wh[a] = z.wh;
                d.cand[a] = z.cand; d.ncand[a] = z.ncand;
            }
            d.fsmall = fsmall_dev;                     // native: patched after the host-written region is closed
        } else {
            for (int a = 0; a < 3; ++a) { d.cand[a] = cfg.ends[a]; d.ncand[a] = 2; }
        }
        if (mode) {
            // real-image input (augment_sample, datasets.py:306-336): gather straight from the volume; no contrast,
            // no GMM noise, no mixing draw
            s.real_input = mode == 4 ? 2 : 1;
            s.syn = const_cast<float *>(mode == 4 ? it.ct_vol : it.real_vol[mode - 1]);
        } else {
        s.labels = it.labels;
        s.label_is_u8 = it.label_is_u8;
        // ---- get_contrast (datasets.py:430-464): float32 like the torch tensors
        const int64_t ms_off = ar.take(2 * 256 * 4);
        if (ar.overflow) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: arena overflow");
        float *mu = (float *)(ar.host + ms_off), *sg = mu + 256;
        s.mu = (const float *)(ar.dev + ms_off);
        s.sigma = s.mu + 256;
        for (int q = 0; q < 256; ++q) mu[q] = dr.randf();
        for (int q = 0; q < 256; ++q) sg[q] = dr.randf();
        for (int q = 0; q < 256; ++q) {
            volatile float pm = mu[q] * 200.f, ps = sg[q] * 20.f;     // product and sum separately rounded
            mu[q] = pm + 25.f;
            sg[q] = ps + 5.f;
        }
        if (dr.rand() < cfg.ct_prob) {
            const float base[4] = {25.f, 90.f, 110.f, 150.f}, span[4] = {10.f, 20.f, 20.f, 50.f};
            float v[4];
            for (int g = 0; g < 4; ++g) {
                volatile float p = span[g] * dr.randf();
                v[g] = base[g] + p;
            }
            for (int q = 0; q < 256; ++q)
                if (cfg.ct_group[q] >= 0 && cfg.ct_group[q] < 4) mu[q] = v[cfg.ct_group[q]];
        }
        if (st.photo || dr.rand() < 0.5) mu[0] = 0.f;
        {   // partial-volume classes 100-149 / 150-199 / 200-249 blend (1,2) / (2,3) / (3,4) (datasets.py:452-462)
            float q2[5];
            for (int c = 0; c < 5; ++c) q2[c] = sg[c] * sg[c];
            float mu5[5];
            for (int c = 0; c < 5; ++c) mu5[c] = mu[c];
            for (int r = 0; r < 3; ++r)
                for (int t = 0; t < 50; ++t) {
                    volatile float vv = (float)t * 0.02f;
                    volatile float ww = 1.0f - vv;
                    volatile float a = mu5[1 + r] * ww, b = mu5[2 + r] * vv;
                    mu[100 + 50 * r + t] = a + b;
                    volatile float c = q2[1 + r] * ww, e = q2[2 + r] * vv;
                    volatile float sum = c + e;
                    sg[100 + 50 * r + t] = sqrtf(sum);
                }
            mu[250] = mu5[4];
            sg[250] = sg[4];
        }
        s.eps_gmm = it.eps_gmm[k];
        // ---- mixing draw (datasets.py:379): planned only for mix_synth_prob == 0
        if (dr.rand() < cfg.mix_synth_prob)
            return fail(BFM_E_UNSUPPORTED, "%s", "bfm_plan_batch: mixing with real modalities is not planned natively");
        }
        // ---- gamma (utils.py:568-572)
        s.gamma = (float)std::exp(ag.gamma_std * dr.randn());
        // ---- bias field (utils.py:574-585); none for CT inputs (utils.py:575-577)
        float bf_std = 0.f;
        if (mode != 4) {
        const double bscale = ag.bf_scale_min + dr.rand() * (ag.bf_scale_max - ag.bf_scale_min);
        int bs[3];
        for (int a = 0; a < 3; ++a) bs[a] = (int)round_half_even(bscale * size[a]);
        if (st.photo) bs[1] = (int)round_half_even(size[1] / st.spac);
        bf_std = (float)(ag.bf_std_min + (ag.bf_std_max - ag.bf_std_min) * dr.rand());
        for (int a = 0; a < 3; ++a) {
            if (bs[a] < 1 || bs[a] > size[a] || !cfg.fwd[a][bs[a]].valid)
                return failf(BFM_E_UNSUPPORTED, "bfm_plan_batch: no zoom table for the %d -> %d bias grid", bs[a], size[a]);
            const bfm_zoom_axis &z = cfg.fwd[a][bs[a]];
            s.bs[a] = bs[a];
            s.btab.lo[a] = z.lo; s.btab.hi[a] = z.hi; s.btab.wl[a] = z.wl; s.btab.wh[a] = z.wh;
        }
        if (!native) {
            const int64_t n = (int64_t)bs[0] * bs[1] * bs[2];
            const int64_t off = ar.take(4 * n);
            if (ar.overflow) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: arena overflow");
            float *bf = (float *)(ar.host + off);
            for (int64_t q = 0; q < n; ++q) bf[q] = dr.randf() * bf_std;
            s.bfsmall = (const float *)(ar.dev + off);
        }
        }
        s.gen_small = native ? ((k == 0 && cfg.nonlinear_transform ? 1 : 0) | (mode != 4 ? 2 : 0)) : 0;
        s.fs_std = fs_std;
        s.bf_std = bf_std;
        // ---- resample (utils.py:591-609)
        const double ru = dr.rand();
        double stds[3];
        int nsz[3];
        for (int a = 0; a < 3; ++a) {
            stds[a] = (0.85 + 0.3 * ru) * std::log(5.0) / M_PI * st.thickness[a] / cfg.res[a];
            if (st.thickness[a] <= cfg.res[a]) stds[a] = 0.0;
            nsz[a] = (int)(size[a] * cfg.res[a] / st.resolution[a]);
            if (nsz[a] < 1 || nsz[a] > size[a] || !cfg.inv[a][nsz[a]].valid)
                return failf(BFM_E_UNSUPPORTED, "bfm_plan_batch: no zoom table for the %d -> %d upsample", nsz[a], size[a]);
            s.new_size[a] = nsz[a];
            info.new_size[k][a] = nsz[a];
            const bfm_zoom_axis &z = cfg.inv[a][nsz[a]];
            s.utab.lo[a] = z.lo; s.utab.hi[a] = z.hi; s.utab.wl[a] = z.wl; s.utab.wh[a] = z.wh;
        }
        // banded passes in ascending factor order (stable), identity axes folded away
        int order[3] = {0, 1, 2};
        for (int i = 1; i < 3; ++i)
            for (int j = i; j > 0; --j) {
                const double fa = (double)nsz[order[j - 1]] / size[order[j - 1]], fb = (double)nsz[order[j]] / size[order[j]];
                if (fb < fa) { const int t = order[j]; order[j] = order[j - 1]; order[j - 1] = t; }
            }
        int nb = 0;
        for (int q = 0; q < 3; ++q) {
            const int a = order[q];
            if (nsz[a] == size[a] && stds[a] == 0) { s.zero_first[a] = 1; continue; }
            bfm_band &bd = s.band[nb++];
            const int half = stds[a] > 0 ? (int)std::ceil(3 * stds[a]) : 0;
            bd.T = 2 * half + 2;
            if (bd.T > 64) return fail(BFM_E_UNSUPPORTED, "%s", "bfm_plan_batch: blur kernel wider than 64 taps");
            bd.build = 1;
            bd.sigma = stds[a];
            bd.n_in = size[a]; bd.n_out = nsz[a]; bd.axis = a;
        }
        if (nb == 0) {
            bfm_band &bd = s.band[0];
            bd.start = cfg.ident_start; bd.w = cfg.ident_w;
            bd.T = 1; bd.n_in = size[2]; bd.n_out = size[2]; bd.axis = 2; bd.build = 0;
            nb = 1;
        }
        s.n_band = nb;
        // ---- noise (utils.py:633-635)
        s.noise_std = (float)(ag.noise_std_min + (ag.noise_std_max - ag.noise_std_min) * dr.rand());
        s.eps_noise = it.eps_noise[k];
        s.seed = native ? splitmix64(seed ^ splitmix64(0x5eedull + sample0 + k)) : 0;
        // ---- buffers
        s.flip = st.flip;
        s.zoom_order = cfg.bspline_zooming ? 3 : 0;          // draws nothing (datasets.py:337-340)
        if (!mode) { s.syn = o.syn; s.syn_pair_ok = (int)o.syn_pair_ok; }
        s.i_bf = o.i_bf; s.tmp[0] = o.tmp[0]; s.tmp[1] = o.tmp[1]; s.lowres = o.lowres;
        s.out = o.out; s.bflog_out = mode == 4 ? nullptr : o.bflog_out; s.residual = o.residual;
        if (k == 0) {
            s.n_aux = it.n_aux;
            for (int c = 0; c < it.n_aux; ++c) {
                s.aux_src[c] = it.aux_src[c]; s.aux_raw[c] = it.aux_raw[c]; s.aux_out[c] = it.aux_out[c];
            }
        }
    }
    return BFM_OK;
}

}  // namespace
}  // namespace bfm

using namespace bfm;

extern "C" int bfm_plan_batch(const bfm_plan_cfg *cfg, int n_items, const bfm_plan_item *items,
                              const bfm_plan_out *outs, uint64_t seed, uint64_t counter, void *arena_host,
                              void *arena_dev, int64_t arena_capacity, int64_t *arena_used, int64_t *upload_bytes,
                              bfm_gen_sample *descs_host, void **descs_dev, bfm_plan_info *info,
                              const double *replay, int64_t n_replay, int64_t *replay_used) {
    if (!cfg || !items || !outs || !arena_host || !arena_dev || !arena_used || !upload_bytes || !descs_host ||
        !descs_dev || !info || n_items <= 0)
        return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: null argument or empty batch");
    if (cfg->n_samples < 1 || cfg->n_samples > BFM_PLAN_MAX_SAMPLES)
        return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: n_samples out of range");
    for (int a = 0; a < 3; ++a)
        if (cfg->size[a] <= 0 || !cfg->fwd[a] || !cfg->inv[a] || !cfg->ends[a])
            return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: incomplete configuration");
    const bool native = replay == nullptr;
    const int ns = cfg->n_samples, total = n_items * ns;
    ArenaCursor ar{(char *)arena_host, (char *)arena_dev, arena_capacity, *arena_used, false};
    const int64_t start = (ar.used + 15) / 16 * 16;
    // host-written prefix: descriptor array, then per sample the mean/std tables (+ the small grids when replayed)
    const int64_t d_off = ar.take((int64_t)sizeof(bfm_gen_sample) * total);
    if (ar.overflow) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: arena overflow");
    Draws dr{};
    dr.replay = replay; dr.n_replay = n_replay; dr.pos = 0; dr.overrun = false;
    for (int n = 0; n < n_items; ++n) {
        if (native) dr.seed(seed, counter + n);
        for (int a = 0; a < 3; ++a)
            if (items[n].src[a] <= 0) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: non-positive source shape");
        if (!items[n].labels || items[n].n_aux < 0 || items[n].n_aux > BFM_MAX_AUX)
            return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: bad item");
        const int rc = plan_item(*cfg, items[n], outs + (int64_t)n * ns, dr, seed, (counter + n) * BFM_PLAN_MAX_SAMPLES,
                                 ar, descs_host + (int64_t)n * ns, info[n], native);
        if (rc) return rc;
    }
    if (dr.overrun) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: replay array exhausted");
    const int64_t host_end = ar.used;
    // device-only scratch: bounding boxes, band tables, maxima, target min/max, and (native) the small grids
    for (int q = 0; q < total; ++q) {
        bfm_gen_sample &s = descs_host[q];
        s.bbox = (int *)(ar.dev + ar.take(32));
        s.maxval = (float *)(ar.dev + ar.take(16));
        if (s.n_aux) s.aux_mm = (int *)(ar.dev + ar.take(8 * BFM_MAX_AUX));
        for (int p = 0; p < s.n_band; ++p) {
            bfm_band &bd = s.band[p];
            if (!bd.build) continue;
            bd.start = (const int *)(ar.dev + ar.take(4 * (int64_t)bd.n_out));
            bd.w = (const float *)(ar.dev + ar.take(4 * (int64_t)bd.n_out * bd.T));
        }
        if (native) {
            if (s.d.fs[0] > 0) {
                if (q % ns == 0)
                    s.d.fsmall = (const float *)(ar.dev + ar.take(4 * (int64_t)s.d.fs[0] * s.d.fs[1] * s.d.fs[2] * 3));
                else
                    s.d.fsmall = descs_host[q - q % ns].d.fsmall;      // one deformation per item
            }
            if (s.bs[0] > 0) s.bfsmall = (const float *)(ar.dev + ar.take(4 * (int64_t)s.bs[0] * s.bs[1] * s.bs[2]));
        }
        if (q % ns != 0) {                                             // samples of an item share the deformation:
            s.bbox = descs_host[q - q % ns].bbox;                      // one bounding box
        }
    }
    if (ar.overflow) return fail(BFM_E_INVALID, "%s", "bfm_plan_batch: arena overflow");
    std::memcpy(ar.host + d_off, descs_host, sizeof(bfm_gen_sample) * total);
    *descs_dev = ar.dev + d_off;
    *arena_used = ar.used;
    *upload_bytes = host_end - start;
    if (replay_used) *replay_used = dr.pos;
    (void)start;
    return BFM_OK;
}

// One call per batch for the common case (native draws, every target fused): lays the per-sample buffers out from a
// handful of base pointers, plans, ships the descriptors and launches the whole chain.  Python then only allocates
// the output tensors and makes this call (brainfm_b200/Generator/native.py::run_fast) -- the per-sample pointer
// arithmetic, three ctypes calls and ~20 kernel launches of bfm_gen_run happen here, without the interpreter lock.
extern "C" int bfm_plan_run(const bfm_plan_cfg *cfg, int n_items, bfm_plan_item *items, const bfm_step_bufs *bufs,
                            uint64_t seed, uint64_t counter, void *arena_host, void *arena_dev, int64_t arena_capacity,
                            int64_t arena_used_in, int64_t *arena_used_out, bfm_gen_sample *descs_host,
                            void **descs_dev, bfm_plan_info *info, void *stream) {
    if (!cfg || !items || !bufs || !arena_used_out || n_items <= 0 || n_items > 4096)
        return fail(BFM_E_INVALID, "%s", "bfm_plan_run: null argument or bad batch size");
    if (!bufs->out || !bufs->syn || !bufs->i_bf || !bufs->tmp || !bufs->lowres)
        return fail(BFM_E_INVALID, "%s", "bfm_plan_run: null buffer");
    const int ns = cfg->n_samples, total = n_items * ns;
    const int64_t N = (int64_t)cfg->size[0] * cfg->size[1] * cfg->size[2];
    const int64_t Np = (N + 3) & ~(int64_t)3;        // scratch slots keep the 16-byte alignment of their base
    std::vector<bfm_plan_out> outs((size_t)total);
    for (int q = 0; q < total; ++q) {
        bfm_plan_out &o = outs[q];
        o.out = bufs->out + q * N;
        o.bflog_out = bufs->bflog_out ? bufs->bflog_out + q * N : nullptr;
        o.residual = bufs->residual ? bufs->residual + q * N : nullptr;
        o.syn = bufs->syn + q * bufs->syn_stride;
        o.i_bf = bufs->i_bf + q * Np;
        o.tmp[0] = bufs->tmp + (2 * (int64_t)q) * Np;
        o.tmp[1] = bufs->tmp + (2 * (int64_t)q + 1) * Np;
        o.lowres = bufs->lowres + q * Np;
        o.syn_pair_ok = bufs->pair_ok;
    }
    int64_t k_aux = 0;
    for (int n = 0; n < n_items; ++n)
        for (int c = 0; c < items[n].n_aux && c < BFM_MAX_AUX; ++c) {
            if (!bufs->aux_out || !bufs->aux_raw) return fail(BFM_E_INVALID, "%s", "bfm_plan_run: null target buffer");
            items[n].aux_out[c] = bufs->aux_out + k_aux * N;
            items[n].aux_raw[c] = bufs->aux_raw + k_aux * Np;
            ++k_aux;
        }
    int64_t used = arena_used_in, upload = 0;
    const int64_t start = (arena_used_in + 15) / 16 * 16;
    int rc = bfm_plan_batch(cfg, n_items, items, outs.data(), seed, counter, arena_host, arena_dev, arena_capacity, &used,
                            &upload, descs_host, descs_dev, info, nullptr, 0, nullptr);
    if (rc) return rc;
    *arena_used_out = used;
    const int64_t nbytes = (upload + 15) / 16 * 16;
    rc = bfm_upload_pinned((char *)arena_dev + start, (const char *)arena_host + start, nbytes, stream);
    if (rc) return rc;
    return bfm_gen_run(descs_host, (const bfm_gen_sample *)*descs_dev, total, stream);
}

