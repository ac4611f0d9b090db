"""The cubic B-spline zoom back (`bspline_zooming`, datasets.py:337-340) on the fused chain: parity with the oracle
(same injected draws) through both planners, the finish stage alone against interpol.resize and the oracle's resize,
batching, and the routing that stays op-wise.  test_bspline_routing_covers_every_branch fails when the cases stop
reaching a branch of the new kernels (128-bit and scalar sides, flip, length-1 lines, the undegraded shortcut)."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from oracle import gen_oracle as go
from oracle import make_golden as mg
from tests._harness import ATOL, RTOL, compare, cuda_case, oracle_batch, oracle_case

pytestmark = pytest.mark.gpu

BS = {"generator.bspline_zooming": True}
ANISO, ANISO_SRC = (72, 61, 83), (101, 90, 97)
MNI2 = (91, 109, 91)
ORD_NEG_INF = -2139095041             # f2ord(-inf) (csrc/common.cuh): the initial value of a cubic sample's maximum


def _c(size, src, seed, over, extra=(), option="default", stride=2):
    return (size, src, "brain", seed, dict(BS, **over), list(extra), option, stride)


CASES = {
    "g64_bspline_s43": mg.CASES["g64_bspline_s43"],
    "g64_bspline_s41": mg.CASES["g64_bspline_s41"],                      # photo mode + flip
    "aniso_s0": _c(ANISO, ANISO_SRC, 0, {"task.T1": True}),
    "aniso_s2": _c(ANISO, ANISO_SRC, 2, {"task.T1": True}),
    "aniso_s3": _c(ANISO, ANISO_SRC, 3, {"task.T1": True}),      # undegraded, odd plane: no shortcut, cubic zoom
    "aniso_s5": _c(ANISO, ANISO_SRC, 5, {"task.T1": True}),
    "aniso_lowres_s0": _c(ANISO, ANISO_SRC, 0, {"generator.low_res_only": True}),
    "ident_s23": _c(64, 96, 23, {"task.super_resolution": True}),          # undegraded: k_gen_identity
    "clinical_s0": _c(64, 96, 0, {"task.super_resolution": True}),        # 64 x 64 x 22: identity x and y axes
    "realT1_s14": _c(64, 96, 14, {"modality_probs.HCP.T1": 1.0, "task.super_resolution": True}),
    "realCT_s16": _c(64, 96, 16, {"modality_probs.HCP.CT": 1.0, "task.CT": True}, ["CT"]),
    "brainid_s6": _c(64, 96, 6, {"generator.all_samples": 3, "generator.mild_samples": 1}, option="brain_id"),
}
NATIVE = ["g64_bspline_s43", "g64_bspline_s41", "aniso_s0", "aniso_lowres_s0", "ident_s23", "brainid_s6"]


# ---- routing: bfm_gen_finish's conditions (csrc/gen.cu), evaluated on the host copies of the descriptors ---------
def _identity(s):
    size = list(s.d.size)
    return (s.n_band == 1 and s.band[0].T == 1 and s.band[0].build == 0 and s.x_count == 0
            and list(s.new_size) == size and (size[1] * size[2]) % 4 == 0)


def finish_labels(s):
    if s.zoom_order != 3:
        return {"linear"}
    if _identity(s):
        return {"cubic_identity"}
    l0, l1, l2 = s.new_size
    out = {"cubic", "flip%d" % s.flip}
    out.add("prefilter_z_vec" if l2 % 4 == 0 else "prefilter_z_scalar")
    out.add("cubic_vec" if l2 % 4 == 0 else "cubic_scalar")
    if 1 in (l0, l1, l2):
        out.add("length1_line")
    if [l0, l1, l2] != list(s.d.size) and any(l == n for l, n in zip(s.new_size, s.d.size)):
        out.add("identity_axis")
    return out


REQUIRED = {"cubic", "flip0", "flip1", "prefilter_z_vec", "prefilter_z_scalar", "cubic_vec", "cubic_scalar",
            "cubic_identity", "identity_axis"}
SEEN = {}


def _note(key, ds):
    descs, _, B = ds._last_descs
    SEEN[key] = set().union(*[finish_labels(descs[b]) for b in range(B)])
    return descs, B


@functools.lru_cache(maxsize=None)
def _oracle(name):
    return oracle_case(CASES[name])


def _check(name, item, orc, got, ds, draws):
    assert draws.done(), "CUDA path consumed %d of %d draws" % (draws.pos, len(draws.log))
    assert ds.last_deform["_plan"].bbox_host() == orc.deform["lo"] + orc.deform["hi"]
    compare(mg.flatten(item), mg.flatten(got), name)


@pytest.mark.parametrize("planner", ["python", "native"])
@pytest.mark.parametrize("name", list(CASES))
def test_fused_cubic_zoom_matches_oracle(name, planner):
    if planner == "native" and name not in NATIVE:
        pytest.skip("covered by the python planner")
    item, orc = _oracle(name)
    got, ds, draws = cuda_case(CASES[name], orc.log, planner=planner)
    _check(name, item, orc, got, ds, draws)
    descs, B = _note((name, planner), ds)
    n_samples = 3 if CASES[name][6] == "brain_id" else 1
    assert B == n_samples and all(descs[b].zoom_order == 3 for b in range(B)), "the fused chain was not taken"
    if n_samples == 3:
        assert isinstance(got[4], list) and len(got[4]) == 3


# ---- the finish stage alone --------------------------------------------------------------------------------------
def _planned(name="aniso_s0"):
    item, orc = _oracle(name)
    _, ds, _ = cuda_case(CASES[name], orc.log, planner="python")
    return ds


def _finish_alone(ds, new_size, lowres, flip, size=None):
    """bfm_gen_finish on a copy of the planned descriptor with `lowres` (new_size) as its low-res volume (and, when
    given, `size` as the output grid)."""
    from brainfm_b200 import _lib
    descs, _, B = ds._last_descs
    s = _lib.GenSample()
    C.memmove(C.addressof(s), C.addressof(descs[0]), C.sizeof(s))
    if size is not None:
        s.d.size[:] = list(size)
    size = list(s.d.size)
    lo = lowres.cuda().contiguous()
    out = torch.full(size, float("nan"), device="cuda")
    mx = torch.tensor([ORD_NEG_INF], dtype=torch.int32, device="cuda")
    s.new_size[:] = list(new_size)
    s.lowres, s.out, s.maxval, s.flip = lo.data_ptr(), out.data_ptr(), mx.data_ptr(), int(flip)
    s.residual, s.n_aux = None, 0
    s.band[0].T = 2                          # never the undegraded class here
    assert finish_labels(s) & {"cubic"}
    dev = torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.lib().bfm_gen_finish(C.addressof(s), dev.data_ptr(), 1, st))
    torch.cuda.synchronize()
    return out.cpu(), mx.view(torch.float32)


def _ord2f(i):
    i = int(i)
    return np.array([i if i >= 0 else i ^ 0x7fffffff], dtype=np.int32).view(np.float32)[0]


@pytest.mark.parametrize("new_size,flip", [((1, 2, 3), 0), ((5, 3, 64), 1), ((2, 61, 5), 0), ((36, 20, 41), 1),
                                           ((3, 5, 1), 1)])
def test_finish_stage_alone_matches_interpol_resize(new_size, flip):
    from brainfm_b200 import interpol
    ds = _planned()
    size = list(ds.size)
    g = torch.Generator().manual_seed(sum(new_size))
    L = torch.rand(new_size, generator=g)
    L[torch.rand(new_size, generator=g) < 0.5] = 0.            # the zeros the noise clamp leaves: cubic overshoot < 0
    got, mx = _finish_alone(ds, new_size, L, flip)
    ref = interpol.resize(L.cuda()[None, None], shape=size, anchor='edge', interpolation=3, bound='dct2',
                          prefilter=True)[0, 0].cpu()
    orc = go.bspline_resize(L, size)
    for want, what in ((ref, "interpol.resize"), (orc, "oracle")):
        mref = torch.max(want)
        np.testing.assert_allclose(_ord2f(mx.view(torch.int32)[0]), mref.item(), rtol=RTOL, atol=ATOL, err_msg=what)
        w = want / mref
        w = torch.flip(w, [0]) if flip else w
        np.testing.assert_allclose(got.numpy(), w.numpy(), rtol=RTOL, atol=ATOL, err_msg=what)


# shared memory of k_gen_cubic_zoom: (min(ly, 32 * ly // s1 + 8) + 32) * lz floats + ~1 KB static.  Without the opt-in
# static + dynamic must fit 48 KB, so the sizes around that bound are pinned: just below 48 KB of dynamic memory (a
# 192^3 grid at ~1.1 mm: 48 416 bytes), above it, and a z line long enough that k_gen_prefilter_z's tile needs the
# opt-in too.
@pytest.mark.parametrize("size,new_size,smem", [((192, 192, 192), (40, 170, 178), 48416),
                                                ((192, 192, 256), (30, 180, 240), 67200),
                                                ((16, 64, 400), (7, 10, 390), 65520)])
def test_finish_stage_alone_with_large_shared_memory(size, new_size, smem):
    from brainfm_b200 import interpol
    ly, lz = new_size[1], new_size[2]
    assert (min(ly, 32 * ly // size[1] + 8) + 32) * lz * 4 == smem
    ds = _planned()
    g = torch.Generator().manual_seed(7)
    L = torch.rand(new_size, generator=g)
    L[torch.rand(new_size, generator=g) < 0.3] = 0.
    got, mx = _finish_alone(ds, new_size, L, 1, size=size)
    ref = interpol.resize(L.cuda()[None, None], shape=list(size), anchor='edge', interpolation=3, bound='dct2',
                          prefilter=True)[0, 0].cpu()
    mref = torch.max(ref)
    np.testing.assert_allclose(_ord2f(mx.view(torch.int32)[0]), mref.item(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got.numpy(), torch.flip(ref / mref, [0]).numpy(), rtol=RTOL, atol=ATOL)


def test_finish_stage_alone_with_negative_overshoot():
    """A volume whose cubic resize has negative voxels: the maximum (order-preserving encoding) and the normalised
    values still match."""
    ds = _planned()
    size = list(ds.size)
    L = torch.zeros((9, 8, 11))
    L[4, 3, 5] = 5.0
    L[2, 6, 2] = 1.0
    got, mx = _finish_alone(ds, L.shape, L, 0)
    orc = go.bspline_resize(L, size)
    assert (orc < 0).any() and (got < 0).any()
    np.testing.assert_allclose(_ord2f(mx.view(torch.int32)[0]), torch.max(orc).item(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got.numpy(), (orc / torch.max(orc)).numpy(), rtol=RTOL, atol=ATOL)
    # all-negative maximum is decoded too (a volume of negative values only)
    got2, mx2 = _finish_alone(ds, L.shape, -1.0 - L, 0)
    orc2 = go.bspline_resize(-1.0 - L, size)
    np.testing.assert_allclose(_ord2f(mx2.view(torch.int32)[0]), torch.max(orc2).item(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got2.numpy(), (orc2 / torch.max(orc2)).numpy(), rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("n_in,n_out", [(1, 64), (2, 61), (3, 83), (5, 72), (36, 72), (37, 61), (83, 83), (160, 160),
                                        (53, 160), (101, 64), (7, 3)])
def test_edge_anchored_coordinates_are_bit_exact(n_in, n_out):
    from brainfm_b200 import _lib
    out = torch.empty(n_out, dtype=torch.float32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.lib().bfm_gen_zoom_coords(n_in, n_out, out.data_ptr(), st))
    torch.cuda.synchronize()
    scale = n_in / n_out                       # gen_oracle.bspline_resize's expression
    want = (torch.arange(0., n_out, dtype=torch.float32) * scale + 0.5 * (scale - 1)).numpy()
    assert np.array_equal(out.cpu().numpy().view(np.int32), want.view(np.int32))


# ---- batching ----------------------------------------------------------------------------------------------------
BATCH = _c(MNI2, MNI2, 3, {"task.bias_field": False, "task.T1": True})
BATCH_SRCS = [MNI2, (96, 112, 100)]
BATCH_IDX = [0, 1, 1, 0]


def _flat(items):
    return [{k: v for k, v in mg.flatten(it).items() if isinstance(v, torch.Tensor)} for it in items]


def _identical(a, b, what):
    assert set(a) == set(b), what
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


def test_python_planner_batch_equals_single_items():
    items, orcs, log = oracle_batch(BATCH, BATCH_SRCS, BATCH_IDX)
    got, ds, draws = cuda_case(BATCH, log, planner="python", srcs=BATCH_SRCS, run=lambda d: d.generate_batch(BATCH_IDX))
    assert draws.done()
    descs, B = _note(("batch", "python"), ds)
    assert B == 4 and all(descs[b].zoom_order == 3 for b in range(B))
    for n, (it, g) in enumerate(zip(items, got)):
        compare(mg.flatten(it), mg.flatten(g), "batch item %d" % n)
    batch = _flat(got)
    for n, idx in enumerate(BATCH_IDX):
        alone, _, dr = cuda_case(BATCH, orcs[n].log, planner="python", srcs=BATCH_SRCS,
                                 run=lambda d, idx=idx: d.generate_batch([idx]))
        assert dr.done()
        _identical(batch[n], _flat(alone)[0], "python planner, item %d" % n)


@pytest.mark.parametrize("fast", [False, True])
def test_native_batch_items_equal_single_items(fast):
    _, ds, _ = cuda_case(BATCH, None, planner="native", srcs=BATCH_SRCS, run=lambda d: None)

    def gen(indices, counter):
        ds._native_planner(indices)
        ds._native.seed, ds._native.counter = 12345, counter
        items = ds.generate_batch_fast(indices) if fast else ds.generate_batch(indices)
        assert items is not None, "generate_batch_fast refused the batch"
        torch.cuda.synchronize()
        descs, _, B = ds._last_descs
        assert all(descs[b].zoom_order == 3 for b in range(B))
        return _flat(list(items))

    batch = gen(BATCH_IDX, 0)
    for n, idx in enumerate(BATCH_IDX):
        _identical(batch[n], gen([idx], n)[0], "native planner%s, item %d" % (" (fast)" if fast else "", n))


_DESC_FIELDS = ("zoom_order", "flip", "new_size", "noise_std", "gamma", "n_band", "zero_first", "real_input", "n_aux",
                "bs")


@pytest.mark.parametrize("name", ["g64_bspline_s41", "aniso_lowres_s0", "brainid_s6"])
def test_python_and_native_replay_plan_the_same_descriptors(name):
    item, orc = _oracle(name)
    got_p, ds_p, _ = cuda_case(CASES[name], orc.log, planner="python")
    dp, _, Bp = ds_p._last_descs
    fp = [{f: (list(v) if hasattr((v := getattr(dp[b], f)), "__len__") else v) for f in _DESC_FIELDS}
          for b in range(Bp)]
    bands_p = [[(dp[b].band[q].T, dp[b].band[q].n_in, dp[b].band[q].n_out, dp[b].band[q].axis, dp[b].band[q].sigma)
                for q in range(dp[b].n_band)] for b in range(Bp)]
    out_p = _flat([got_p])[0]
    got_n, ds_n, _ = cuda_case(CASES[name], orc.log, planner="native")
    dn, _, Bn = ds_n._last_descs
    assert Bn == Bp
    for b in range(Bn):
        fn = {f: (list(v) if hasattr((v := getattr(dn[b], f)), "__len__") else v) for f in _DESC_FIELDS}
        assert fn == fp[b], (name, b)
        assert [(dn[b].band[q].T, dn[b].band[q].n_in, dn[b].band[q].n_out, dn[b].band[q].axis, dn[b].band[q].sigma)
                for q in range(dn[b].n_band)] == bands_p[b]
    _identical(out_p, _flat([got_n])[0], name)


def test_device_pipeline_one_call_path_equals_the_general_path():
    """generate_batch_fast (bfm_plan_run, what DevicePipeline calls) against generate_batch with the same planner
    state, with bspline_zooming on."""
    from tests.test_pipeline_gpu import _dataset, _run
    ds, _ = _dataset()
    ds.synth_args.bspline_zooming = True
    for idx in ([0, 1, 2, 3], [3, 1]):
        ref = _run(ds, lambda: ds.generate_batch(idx))
        ref = [(a, b, c, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in d.items()},
                {k: v.clone() for k, v in e.items()}) for a, b, c, d, e in ref]
        descs, _, B = ds._last_descs
        assert all(descs[q].zoom_order == 3 for q in range(B))
        got = _run(ds, lambda: ds.generate_batch_fast(idx))
        assert got is not None and len(got) == len(idx)
        torch.cuda.synchronize()
        descs, _, B = ds._last_descs
        assert all(descs[q].zoom_order == 3 for q in range(B))
        for n, (r, g) in enumerate(zip(ref, got)):
            assert r[:3] == g[:3]
            for k in r[4]:
                assert torch.equal(r[4][k], g[4][k]), (n, k)
            assert torch.equal(r[3]['T1'], g[3]['T1'])
    from brainfm_b200.pipeline import DevicePipeline
    pipe = DevicePipeline(ds, depth=2)
    ref = _run(ds, lambda: ds.generate_batch_fast([0, 1, 2, 3]))
    ref_in = ref.input.clone()
    got = _run(ds, lambda: pipe.submit([0, 1, 2, 3]).wait())
    torch.cuda.synchronize()
    from brainfm_b200.Generator.native import LazyItems
    assert isinstance(got, LazyItems), "DevicePipeline did not take the one-call path (bfm_plan_run)"
    assert torch.equal(ref_in, got.input)


# ---- routing -----------------------------------------------------------------------------------------------------
def test_custom_steps_stay_op_wise_and_match_the_oracle():
    from brainfm_b200.Generator import constants as K
    name = "g64_bspline_s43"
    item, orc = _oracle(name)
    K.augmentation_funcs["noise_custom"] = K.augmentation_funcs["noise"]
    try:
        def run(ds):
            ds.augmentation_steps['synth'] = ["gamma", "bias_field", "resample", "noise_custom"]
            ds._last_descs = None
            return ds[0]
        got, ds, draws = cuda_case(name, orc.log, planner="python", run=run)
    finally:
        del K.augmentation_funcs["noise_custom"]
    assert ds._last_descs is None, "a custom step list must not take the fused chain"
    _check(name, item, orc, got, ds, draws)


def test_slab_mode_refuses_bspline_zooming():
    from brainfm_b200.Generator.slab import generate_slab
    for planner in ("python", "native"):
        _, ds, _ = cuda_case("g64_bspline_s43", None, planner=planner, run=lambda d: None)
        with pytest.raises(NotImplementedError):
            generate_slab(ds, 0, rank=0, world=1)


def test_bspline_routing_covers_every_branch():
    for name in CASES:
        if (name, "python") not in SEEN and (name, "native") not in SEEN:
            item, orc = _oracle(name)
            _, ds, _ = cuda_case(CASES[name], orc.log, planner="python")
            _note((name, "python"), ds)
    seen = set().union(*SEEN.values())
    assert REQUIRED <= seen, "branches no case reaches: %s" % sorted(REQUIRED - seen)
