"""bfm_plan_batch is HOST code: it can be exercised without a GPU (device addresses are just numbers to it).

  * replay mode against the oracle: affine matrix, centre, resolution / thickness, flip, photo mode and the
    low-res grid of the golden cases come out exactly as the oracle (hence the reference) computes them;
  * native mode: determinism, arena bounds, parameter ranges and branch frequencies of the in-library draws."""
import ctypes as C

import numpy as np
import pytest
import torch

from brainfm_b200 import _lib
from brainfm_b200.Generator import constants as K
from oracle import make_golden as mg
from tests._harness import oracle_case
from tests.test_chain_shapes_gpu import CASES as SHAPE_CASES

FAKE = 0x7f0000000000          # "device" addresses: never dereferenced by the planner


def make_cfg(size, gen, mix=0.0, aug_sets=None, real_sets=None):
    cfg = _lib.PlanCfg()
    cfg.size[:] = size
    cfg.res[:] = [1.0, 1.0, 1.0]
    cfg.low_res_only = int(bool(gen.low_res_only))
    cfg.nonlinear_transform = int(bool(gen.nonlinear_transform))
    for k in ('photo_prob', 'pathology_prob', 'random_shape_prob', 'flip_prob', 'max_rotation', 'max_shear',
              'max_scaling', 'nonlin_scale_min', 'nonlin_scale_max', 'nonlin_std_max', 'ct_prob'):
        setattr(cfg, k, float(getattr(gen, k)))
    cfg.mix_synth_prob = mix
    grp = np.full(256, -1, dtype=np.int8)
    C.memmove(cfg.ct_group, grp.ctypes.data, 256)
    aug_sets = aug_sets or [vars(gen)]
    cfg.n_samples = len(aug_sets)
    for k, vals in enumerate(aug_sets):
        for f, _ in _lib.PlanAug._fields_:
            setattr(cfg.aug[k], f, float(vals[f]))
            setattr(cfg.aug_real[k], f, float((real_sets or aug_sets)[k][f]))
    keep = []
    for ax in range(3):
        n = size[ax]
        fwd, inv = (_lib.ZoomAxis * (n + 1))(), (_lib.ZoomAxis * (n + 1))()
        for n_in in range(1, n + 1):
            for arr in (fwd, inv):
                z = arr[n_in]
                z.lo = z.hi = z.wl = z.wh = z.cand = FAKE
                z.ncand, z.valid = 4, 1
        keep += [fwd, inv]
        cfg.fwd[ax], cfg.inv[ax], cfg.ends[ax] = C.addressof(fwd), C.addressof(inv), FAKE
    cfg.ident_start = cfg.ident_w = FAKE
    return cfg, keep


def plan(cfg, n_items, src, seed=1, counter=0, replay=None, capacity=1 << 20, input_prob=None, real_vol=None,
         ct_vol=0):
    L = _lib.lib()
    ns = cfg.n_samples
    items = (_lib.PlanItem * n_items)()
    for it in items:
        it.labels, it.label_is_u8 = FAKE, 1
        it.src[:] = src
        if input_prob is not None:
            it.input_prob[:] = input_prob
            it.real_vol[:] = real_vol
            it.ct_vol = ct_vol
    outs = (_lib.PlanOut * (n_items * ns))()
    for o in outs:
        o.out = o.syn = o.i_bf = o.lowres = FAKE
        o.tmp[0] = o.tmp[1] = FAKE
    host = np.zeros(capacity, dtype=np.uint8)
    used, upload, consumed = C.c_int64(0), C.c_int64(0), C.c_int64(0)
    descs = (_lib.GenSample * (n_items * ns))()
    ddev = C.c_void_p(0)
    info = (_lib.PlanInfo * n_items)()
    rc = L.bfm_plan_batch(C.addressof(cfg), n_items, C.addressof(items), C.addressof(outs), seed, counter,
                          host.ctypes.data, FAKE, capacity, C.byref(used), C.byref(upload), C.addressof(descs),
                          C.byref(ddev), C.addressof(info), None if replay is None else replay.ctypes.data,
                          0 if replay is None else replay.size, C.byref(consumed))
    _lib.check(rc)
    return dict(descs=descs, info=info, host=host, used=used.value, upload=upload.value, consumed=consumed.value,
                descs_dev=ddev.value)


def flatten_log(log):
    vals = []
    for tag, v in log:
        if tag in ('gmm.eps', 'noise.eps'):
            continue
        vals.append(np.asarray(v.numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float64).reshape(-1))
    return np.ascontiguousarray(np.concatenate(vals))


# the odd and anisotropic grids of test_chain_shapes_gpu that the library plans (one sample per item, no mixing)
ODD = [k for k, v in SHAPE_CASES.items() if v[6] == "default" and "mix_synth_prob" not in v[4]]


@pytest.mark.parametrize("name", ["g64_s0", "g64_s1", "g64_s2", "g64_s3", "g64_s5_lowres", "g160_s0"] + ODD)
def test_replay_reproduces_the_oracle_setup(name):
    case = mg.CASES.get(name) or SHAPE_CASES[name]
    size, src, kind, seed, over, extra, option, stride = case
    item, orc = oracle_case(case)
    args = mg.cfg_for(size, over, option, ref=False)
    gen = dict(vars(args.generator))
    gen.update(vars(args.synth_image_generator))
    cfg, keep = make_cfg(list(mg.shape3(size)), args.generator, aug_sets=[gen])
    flat = flatten_log(orc.log)
    r = plan(cfg, 1, list(mg.shape3(src)), replay=flat)
    assert r['consumed'] == flat.size
    inf, s = r['info'][0], r['descs'][0]
    st = orc.setups
    assert bool(inf.photo_mode) == bool(st['photo_mode']) and bool(inf.flip) == bool(st['flip'])
    assert list(inf.resolution) == [float(v) for v in st['resolution']]
    assert list(inf.thickness) == [float(v) for v in st['thickness']]
    A = np.array(inf.A[:], dtype=np.float32).reshape(3, 3)
    assert np.array_equal(A, orc.deform['A'].numpy().astype(np.float32)), (A, orc.deform['A'])
    assert np.array_equal(np.array(inf.c2[:], dtype=np.float32), orc.deform['c2'].numpy().astype(np.float32))
    assert inf.scaling_factor_distances == float(orc.deform['scaling_factor_distances'])
    # the sample: input shape of the low-res grid is what the oracle's noise field has
    noise = [v for t, v in orc.log if t == 'noise.eps'][0]
    assert list(s.new_size) == list(noise.shape)
    small = [v for t, v in orc.log if t == 'nl.field'][0]
    assert list(s.d.fs) == list(small.shape[:3])
    # host-written small grid = float32(std) * draw, inside the uploaded prefix
    std = np.float32(args.generator.nonlin_std_max * [v for t, v in orc.log if t == 'nl.std'][0])
    off = s.d.fsmall - FAKE
    got = r['host'][off:off + 4 * small.numel()].view(np.float32)
    assert np.array_equal(got, (small.numpy().reshape(-1) * std).astype(np.float32))
    assert off + 4 * small.numel() <= r['upload'] and r['upload'] <= r['used']


def test_native_draws_are_deterministic_and_in_range():
    args = mg.cfg_for(160, {}, "default", ref=False)
    gen = dict(vars(args.generator))
    gen.update(vars(args.synth_image_generator))
    cfg, keep = make_cfg([160] * 3, args.generator, aug_sets=[gen])
    a = plan(cfg, 8, [160] * 3, seed=5, counter=16)
    b = plan(cfg, 8, [160] * 3, seed=5, counter=16)
    assert bytes(a['host'][:a['upload']]) == bytes(b['host'][:b['upload']])
    c = plan(cfg, 8, [160] * 3, seed=6, counter=16)
    assert bytes(a['host'][:a['upload']]) != bytes(c['host'][:c['upload']])
    # item n of a batch at counter c == item 0 of a batch at counter c+n (streams are keyed per item)
    d = plan(cfg, 1, [160] * 3, seed=5, counter=19)
    assert list(d['info'][0].A) == list(a['info'][3].A)
    g = args.generator
    n, photo, flip, cls = 0, 0, 0, np.zeros(4)
    for rep in range(250):
        r = plan(cfg, 8, [160] * 3, seed=9, counter=8 * rep)
        assert r['upload'] <= r['used'] <= 1 << 20
        for q in range(8):
            inf, s = r['info'][q], r['descs'][q]
            n += 1
            photo += inf.photo_mode
            flip += inf.flip
            res = np.array(inf.resolution[:])
            if not inf.photo_mode:
                k = 0 if (res == 1).all() else 1 if (res == 1).sum() == 2 else 2 if res[2] >= 4.8 and res[0] < 1.7 else 3
                cls[k] += 1
            A = np.array(inf.A[:]).reshape(3, 3)
            assert (1 - g.max_scaling) ** 3 * 0.7 < abs(np.linalg.det(A)) < (1 + g.max_scaling) ** 3 * 1.1
            assert all(round(g.nonlin_scale_min * 160) <= v <= round(g.nonlin_scale_max * 160) or inf.photo_mode
                       for v in s.d.fs)
            assert 0 <= s.fs_std <= g.nonlin_std_max and g.bf_std_min <= s.bf_std <= g.bf_std_max
            assert 5.0 <= s.noise_std <= 15.0 and 0.6 < s.gamma < 1.7
            assert all(1 <= v <= 160 for v in s.new_size) and 1 <= s.n_band <= 3
            off = s.mu - FAKE
            ms = r['host'][off:off + 2048].view(np.float32)
            assert ms[:100].max() <= 225 and ms[1:100].min() >= 25 and 5 <= ms[256:356].min() and ms[256:356].max() <= 25
            assert s.gen_small == 3
    assert abs(photo / n - g.photo_prob) < 0.03
    assert abs(flip / n - 0.6915) < 0.035
    assert np.all(np.abs(cls / cls.sum() - 0.25) < 0.04)


def test_brainid_item_shares_one_deformation():
    args = mg.cfg_for(64, {"generator.all_samples": 3, "generator.mild_samples": 1}, "brain_id", ref=False)
    sets = []
    for i in range(3):
        v = dict(vars(args.generator))
        v.update(vars(args.mild_generator if i < 1 else args.severe_generator))
        v.update(vars(args.synth_image_generator))
        sets.append(v)
    cfg, keep = make_cfg([64] * 3, args.generator, aug_sets=sets)
    r = plan(cfg, 2, [96] * 3, seed=3)
    d = r['descs']
    for item in range(2):
        a = d[3 * item]
        for k in (1, 2):
            b = d[3 * item + k]
            assert list(b.d.A) == list(a.d.A) and b.d.fsmall == a.d.fsmall and b.bbox == a.bbox
            assert b.gen_small == 2 and b.bfsmall != a.bfsmall and b.mu != a.mu
        assert a.gen_small == 3
    assert d[0].bbox != d[3].bbox
    assert d[0].bf_std <= args.mild_generator.bf_std_max + 1e-9


def test_unsupported_and_invalid_inputs_fail_loudly():
    args = mg.cfg_for(64, {}, "default", ref=False)
    gen = dict(vars(args.generator))
    gen.update(vars(args.synth_image_generator))
    cfg, keep = make_cfg([64] * 3, args.generator, mix=1.0, aug_sets=[gen])
    with pytest.raises(NotImplementedError):
        plan(cfg, 1, [64] * 3)
    cfg, keep = make_cfg([64] * 3, args.generator, aug_sets=[gen])
    with pytest.raises(ValueError):
        plan(cfg, 4, [64] * 3, capacity=4096)          # arena too small
    with pytest.raises(ValueError):
        plan(cfg, 1, [64] * 3, replay=np.zeros(5))     # replay array exhausted


def test_real_input_modes_are_drawn_like_read_input():
    """read_input (datasets.py:563-588): first of T1 / T2 / FLAIR with u < prob whose volume exists; real-input samples
    carry no contrast tables, gather from the modality's volume and use the real-image noise range."""
    args = mg.cfg_for(64, {}, "default", ref=False)
    gen = dict(vars(args.generator))
    syn = dict(gen); syn.update(vars(args.synth_image_generator))
    real = dict(gen); real.update(vars(args.real_image_generator))
    cfg, keep = make_cfg([64] * 3, args.generator, aug_sets=[syn], real_sets=[real])
    vols = [FAKE + 0x1000, 0, FAKE + 0x3000]                 # the subject has T1 and FLAIR, no T2
    counts = np.zeros(4)
    for rep in range(120):
        r = plan(cfg, 8, [64] * 3, seed=21, counter=8 * rep, input_prob=[0.25, 0.5, 0.75, 0.0], real_vol=vols)
        for q in range(8):
            inf, s = r['info'][q], r['descs'][q]
            counts[inf.input_mode] += 1
            if inf.input_mode:
                assert s.real_input == 1 and s.syn == vols[inf.input_mode - 1] and not s.mu and not s.labels
                assert 0.0 <= s.noise_std <= 0.02 + 1e-9
            else:
                assert s.real_input == 0 and s.syn == FAKE and s.mu and 5.0 <= s.noise_std <= 15.0
    frac = counts / counts.sum()
    assert counts[2] == 0                                    # no T2 volume: never drawn
    assert abs(frac[1] - 0.25) < 0.05 and abs(frac[3] - 0.5) < 0.06 and abs(frac[0] - 0.25) < 0.05
    # CT inputs: window flag, no bias grid, no bias_field_log output
    n_ct = 0
    for rep in range(20):
        r = plan(cfg, 8, [64] * 3, seed=3, counter=8 * rep, input_prob=[0, 0, 0, 0.9], real_vol=[0, 0, 0],
                 ct_vol=FAKE + 0x5000)
        for q in range(8):
            inf, s = r['info'][q], r['descs'][q]
            if inf.input_mode == 4:
                n_ct += 1
                assert s.real_input == 2 and s.syn == FAKE + 0x5000 and not s.bfsmall and not s.bflog_out
                assert list(s.bs) == [0, 0, 0] and s.gen_small in (0, 1)
            else:
                assert inf.input_mode == 0 and s.bfsmall
    assert 0.8 < n_ct / 160 < 0.98


@pytest.mark.parametrize("field", ["lowres", "tmp1", "i_bf", "syn", "out"])
def test_misaligned_buffers_are_refused_before_any_launch(field):
    """Every stage's argument check: the kernels take 128-bit accesses on the scratch (and on the outputs of a plane
    that is a multiple of 4) without testing the pointers, so a misaligned slot must come back as BFM_E_INVALID.  The
    descriptor is planned with (aligned) fake device addresses and then broken in exactly one field, so the check
    returns before anything is launched."""
    args = mg.cfg_for(64, {}, "default", ref=False)
    gen = dict(vars(args.generator))
    gen.update(vars(args.synth_image_generator))
    cfg, keep = make_cfg([64] * 3, args.generator, aug_sets=[gen])
    r = plan(cfg, 1, [96] * 3, seed=4)
    s = r['descs'][0]
    if field == "tmp1":                       # one float off: misaligned for 16-byte and for 8-byte slots
        s.tmp[1] = FAKE + 4
    else:
        setattr(s, field, FAKE + 4)
    L = _lib.lib()
    for stage in (L.bfm_gen_run, L.bfm_gen_plan, L.bfm_gen_bbox, L.bfm_gen_gmm, L.bfm_gen_warp, L.bfm_gen_resample,
                  L.bfm_gen_finish):
        assert stage(C.addressof(r['descs']), FAKE, 1, None) == _lib.BFM_E_INVALID
        assert "misaligned" in L.bfm_last_error().decode()


def test_layout_of_the_per_sample_buffers():
    """bfm_plan_layout, the one per-sample buffer layout of both batch paths (bfm_plan_run, NativePlanner.run): outputs
    advance by N floats per sample, the scratch by Npad = N rounded up to a multiple of 4 (two slots per sample for
    tmp), syn by syn_stride, and the fused targets by N / Npad per target in item order.  N is odd here (91 x 109 x 91)
    so that N and Npad differ."""
    L = _lib.lib()
    cfg = _lib.PlanCfg()
    cfg.size[:] = [91, 109, 91]
    cfg.n_samples = 2
    N = 91 * 109 * 91
    Np = N + 3
    assert N % 2 == 1 and Np % 4 == 0
    n_aux = [2, 0, 3]
    items = (_lib.PlanItem * 3)()
    for it, k in zip(items, n_aux):
        it.n_aux = k
    names = ("out", "bflog_out", "residual", "syn", "i_bf", "tmp", "lowres", "aux_out", "aux_raw")
    base = {f: FAKE + (k << 36) for k, f in enumerate(names)}
    stride = 2 * 902912                          # syn: float2 pairs of a padded source volume

    def layout(n_items=3, **over):
        bufs = _lib.StepBufs(**dict(base, **over))
        bufs.syn_stride, bufs.pair_ok = stride, 1
        outs = (_lib.PlanOut * (max(n_items, 1) * 2))()
        return L.bfm_plan_layout(C.addressof(cfg), n_items, C.addressof(items), C.addressof(bufs),
                                 C.addressof(outs)), outs

    rc, outs = layout()
    assert rc == _lib.BFM_OK
    for q in range(6):
        o = outs[q]
        assert (o.out, o.bflog_out, o.residual) == tuple(base[f] + 4 * q * N for f in ("out", "bflog_out", "residual"))
        assert o.syn == base["syn"] + 4 * q * stride and o.syn_pair_ok == 1
        assert o.i_bf == base["i_bf"] + 4 * q * Np and o.lowres == base["lowres"] + 4 * q * Np
        assert o.tmp[0] == base["tmp"] + 4 * (2 * q) * Np and o.tmp[1] == base["tmp"] + 4 * (2 * q + 1) * Np
    k = 0
    for it in items:
        for c in range(_lib.MAX_AUX):
            if c < it.n_aux:
                assert it.aux_out[c] == base["aux_out"] + 4 * k * N and it.aux_raw[c] == base["aux_raw"] + 4 * k * Np
                k += 1
            else:
                assert it.aux_out[c] is None and it.aux_raw[c] is None
    assert k == 5
    # no bias-field log / residual output requested: null in every sample
    rc, outs = layout(bflog_out=None, residual=None)
    assert rc == _lib.BFM_OK and all(o.bflog_out is None and o.residual is None for o in outs)
    # refusals
    for f in ("out", "syn", "i_bf", "tmp", "lowres"):
        assert layout(**{f: None})[0] == _lib.BFM_E_INVALID and "null buffer" in L.bfm_last_error().decode()
    for f in ("aux_out", "aux_raw"):
        assert layout(**{f: None})[0] == _lib.BFM_E_INVALID and "null target" in L.bfm_last_error().decode()
        assert layout(n_items=2, **{f: None})[0] == _lib.BFM_E_INVALID      # item 0 has targets
    items[0].n_aux = 0
    assert layout(n_items=2, aux_out=None, aux_raw=None)[0] == _lib.BFM_OK      # no target in the batch
    for n_items in (0, -1, 4097):
        assert layout(n_items=n_items)[0] == _lib.BFM_E_INVALID
    bufs, outs = _lib.StepBufs(**base), (_lib.PlanOut * 6)()
    for args in ((None, 3, C.addressof(items), C.addressof(bufs), C.addressof(outs)),
                 (C.addressof(cfg), 3, None, C.addressof(bufs), C.addressof(outs)),
                 (C.addressof(cfg), 3, C.addressof(items), None, C.addressof(outs)),
                 (C.addressof(cfg), 3, C.addressof(items), C.addressof(bufs), None)):
        assert L.bfm_plan_layout(*args) == _lib.BFM_E_INVALID
