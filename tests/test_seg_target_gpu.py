"""The segmentation target of the fused chain (bfm_gen_segmentation): one launch per batch writes the 56-channel one-hot
of every item.  Pinned against the reference fixtures, against the op-wise reader (read_and_deform_segmentation with
the item's own deformation) at odd and anisotropic grids, in mixed batches and for unusual label volumes, through the
one-call path (generate_batch_fast, DevicePipeline), and on the routing that keeps the op-wise reader."""
import os

import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from tests._harness import cuda_case, oracle_case

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SEG_FILE = "brainseg_with_extracerebral.nii"


class Calls:
    """Counts the calls of a library entry point (or of a Python function) while forwarding them."""

    def __init__(self, fn):
        self.fn, self.n = fn, 0

    def __call__(self, *a, **kw):
        self.n += 1
        return self.fn(*a, **kw)


@pytest.fixture
def stage_calls(monkeypatch):
    from brainfm_b200 import _lib
    L = _lib.lib()
    calls = {k: Calls(getattr(L, k)) for k in ("bfm_gen_segmentation", "bfm_label_warp_onehot")}
    for k, c in calls.items():
        monkeypatch.setattr(L, k, c)
    return calls


def _opwise(ds, seg_path, setups, deform):
    from brainfm_b200.Generator.utils import read_and_deform_segmentation
    return read_and_deform_segmentation(None, 'segmentation', seg_path, setups, deform, ds.device, cfg=ds.gen_args,
                                        onehotmatrix=ds.onehotmatrix, lut=ds.lut, vflip=ds.vflip)['segmentation']


def _seg_path(ds, k):
    return ds.names[0][k][:-len("T1w.nii")] + SEG_FILE


# ---- 1. the reference fixtures -----------------------------------------------------------------------------------
PARITY = ["g64_s0", "g64_s1", "g64_s2", "g64_s3", "g64_s5_lowres", "g160_s0", "g64_brainid_s6", "g64_realT1_s14",
          "g64_shift_s43"]


@pytest.mark.parametrize("planner", ["python", "native"])
@pytest.mark.parametrize("name", PARITY)
def test_segmentation_matches_reference_fixture(name, planner, stage_calls):
    if planner == "native" and name == "g64_shift_s43":
        pytest.skip("a random centre shift is planned in Python only")
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    _, orc = oracle_case(name)
    got, ds, draws = cuda_case(name, orc.log, planner=planner)
    assert draws.done()
    assert stage_calls["bfm_gen_segmentation"].n == 1 and stage_calls["bfm_label_warp_onehot"].n == 0
    seg = got[3]["segmentation"]
    assert seg.shape == (56, *ds.size)
    stride = int(gold["meta.stride"])
    out = {}
    mg.summarise("target.segmentation", seg, stride, out)
    keys = ["target.segmentation.argmax.sub", "target.segmentation.argmax.sum"]
    assert set(keys) <= set(out) and set(keys) <= set(gold.files), sorted(out)
    for k in keys:
        assert np.array_equal(out[k], gold[k]), k


# ---- 2. the batched stage against the op-wise reader ---------------------------------------------------------------
def _case(size, src, seed, over, extra=(), option="default"):
    return (size, src, "brain", seed, over, list(extra), option, 2)


SHAPES = {                                                   # (size, src): size[2] % 4 != 0 takes the scalar stores
    "aniso": ((72, 61, 83), (101, 90, 97)),
    "deep": ((40, 45, 270), (60, 64, 301)),
    "mni2": ((91, 109, 91), (91, 109, 91)),
    "vec": ((48, 56, 40), (60, 70, 52)),
}
VARIANTS = {                                                 # the flip is drawn as randn() < flip_prob (reference)
    "flip": {"generator.flip_prob": 10.0},
    "noflip": {"generator.flip_prob": -10.0},
    "photo": {"generator.photo_prob": 1.0, "generator.flip_prob": 0.5},
    "realT1": {"modality_probs.HCP.T1": 1.0},
}


def _items_against_opwise(ds, indices, seg_paths):
    """One generate_batch (python planner; every item's deformation is recorded as the item is finished), each
    segmentation against the op-wise reader with that item's deformation."""
    ctxs = []
    orig = ds._finish_item

    def finish(ctx, target, sample):
        ctxs.append((ctx["setups"], ctx["deform"], ctx["input_mode"]))
        return orig(ctx, target, sample)
    ds._finish_item = finish
    try:
        items = ds.generate_batch(list(indices))
    finally:
        ds._finish_item = orig
    modes = []
    for n, (it, (setups, deform, mode)) in enumerate(zip(items, ctxs)):
        ref = _opwise(ds, seg_paths[indices[n]], setups, deform)
        got = it[3]["segmentation"]
        assert got.shape == ref.shape
        assert torch.equal(got, ref), "item %d: one-hot differs in %d voxels" % (n, int((got != ref).sum()))
        assert torch.all(got.sum(0) == 1)
        modes.append((bool(setups["flip"]), bool(setups["photo_mode"]), mode))
    return modes


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("shape", list(SHAPES))
def test_batched_stage_equals_opwise_reader(shape, variant, stage_calls):
    size, src = SHAPES[shape]
    _, ds, _ = cuda_case(_case(size, src, 1, VARIANTS[variant]), None, planner="python", run=lambda d: None)
    np.random.seed(11)
    torch.manual_seed(11)
    modes = _items_against_opwise(ds, [0, 0, 0], [_seg_path(ds, 0)])
    assert stage_calls["bfm_gen_segmentation"].n == 1
    if variant == "flip":
        assert all(m[0] for m in modes)
    elif variant == "noflip":
        assert not any(m[0] for m in modes)
    elif variant == "photo":
        assert all(m[1] for m in modes)
    else:
        assert all(m[2] == "T1" for m in modes)


def test_native_general_path_equals_opwise_reader(stage_calls):
    """Native draws, one item per batch: ds.last_deform is the item's deformation (the default task set plans it)."""
    size, src = SHAPES["aniso"]
    _, ds, _ = cuda_case(_case(size, src, 1, {}), None, planner="native", run=lambda d: None)
    np.random.seed(5)
    for _ in range(4):
        it = ds.generate_batch([0])[0]
        ref = _opwise(ds, _seg_path(ds, 0), ds.last_setups, ds.last_deform)
        assert torch.equal(it[3]["segmentation"], ref)
    assert stage_calls["bfm_gen_segmentation"].n == 4 and stage_calls["bfm_label_warp_onehot"].n == 4


def test_mixed_batch_two_subjects_equals_opwise_reader(stage_calls):
    """Four items, two subjects of different source shapes, repeated indices: one launch, each item exact."""
    srcs = [(91, 109, 91), (96, 112, 100)]
    case = _case((91, 109, 91), srcs[0], 3, {})
    _, ds, _ = cuda_case(case, None, planner="python", srcs=srcs, run=lambda d: None)
    np.random.seed(2)
    _items_against_opwise(ds, [0, 1, 1, 0], [_seg_path(ds, 0), _seg_path(ds, 1)])
    assert stage_calls["bfm_gen_segmentation"].n == 1 and stage_calls["bfm_label_warp_onehot"].n == 4


def _odd_labels(shape, dtype):
    lab = mg.ti.seg_labels(shape).astype(np.float64)
    rng = np.random.RandomState(0)
    pick = rng.rand(*shape)
    lab[pick < 0.05] = 57                         # not in the label list
    lab[(pick >= 0.05) & (pick < 0.08)] = 99
    if dtype != np.uint8:
        lab[(pick >= 0.08) & (pick < 0.11)] = 10001   # >= len(lut)
        lab[(pick >= 0.11) & (pick < 0.14)] = 12345
        lab[(pick >= 0.14) & (pick < 0.17)] = -3      # negative
    return lab.astype(dtype)


@pytest.mark.parametrize("dtype", [np.int32, np.float32, np.uint8])
def test_label_volume_dtypes_and_out_of_list_labels(dtype, stage_calls):
    from brainfm_b200 import io as bio
    size, src = SHAPES["vec"]
    _, ds, _ = cuda_case(_case(size, src, 4, {}), None, planner="python", run=lambda d: None)
    path = _seg_path(ds, 0)
    bio.register_volume(path, _odd_labels(src, dtype))
    np.random.seed(8)
    _items_against_opwise(ds, [0, 0], [path])
    S = ds.cache.get(path, "i32")
    if dtype != np.uint8:
        assert bool((S < 0).any()) and bool((S >= 10000).any())
    cls = ds._seg_classes(path, src)
    assert cls.dtype == torch.uint8 and int(cls.max()) < 56


# ---- 3. one-call batches -------------------------------------------------------------------------------------------
def _native_ds(option="default", over=None, n=3, size=(48, 56, 40)):
    srcs = [tuple(v + d for v, d in zip(size, off)) for off in ((12, 14, 12), (8, 8, 8), (12, 14, 12))][:n]
    case = _case(size, srcs[0], 0, over or {}, option=option)
    _, ds, _ = cuda_case(case, None, planner="native", srcs=srcs, run=lambda d: None)
    return ds


def _run(ds, fn, seed=3):
    np.random.seed(seed)
    ds._native_planner([0])
    ds._native.seed, ds._native.counter = None, 0
    return fn()


def _snapshot(items):
    return [(a, b, c, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in d.items()},
             [{k: v.clone() for k, v in s.items()} for s in (e if isinstance(e, list) else [e])])
            for a, b, c, d, e in items]


def test_one_call_batches_equal_the_general_path(stage_calls):
    ds = _native_ds()
    assert {"bias_field", "segmentation"} <= set(ds.tasks) and "T1" not in ds.tasks
    for idx in ([0, 1, 2, 1], [2, 0]):
        ref = _snapshot(_run(ds, lambda: ds.generate_batch(idx)))
        got = _run(ds, lambda: ds.generate_batch_fast(idx))
        from brainfm_b200.Generator.native import LazyItems
        assert isinstance(got, LazyItems)
        torch.cuda.synchronize()
        assert tuple(got.targets["segmentation"].shape) == (len(idx), 56, *ds.size)
        for n, (r, g) in enumerate(zip(ref, _snapshot(got))):
            assert r[:3] == g[:3]
            assert list(r[3]) == list(g[3]), (list(r[3]), list(g[3]))
            for k, v in r[3].items():
                if torch.is_tensor(v):
                    assert torch.equal(v, g[3][k]), (n, k)
                else:
                    assert v == g[3][k], (n, k)
            assert len(r[4]) == len(g[4])
            for a, b in zip(r[4], g[4]):
                assert set(a) == set(b) and all(torch.equal(a[k], b[k]) for k in a)
            assert torch.equal(got.targets["segmentation"][n], g[3]["segmentation"])
            assert r[3]["bias_field"] == 0.
    assert stage_calls["bfm_label_warp_onehot"].n == 0


def test_device_pipeline_takes_the_one_call_path():
    from brainfm_b200.Generator.native import LazyItems
    from brainfm_b200.pipeline import DevicePipeline
    ds = _native_ds()
    ref = _run(ds, lambda: ds.generate_batch_fast([0, 1, 2, 0]))
    ref_seg = ref.targets["segmentation"].clone()
    pipe = DevicePipeline(ds, depth=2)
    got = _run(ds, lambda: pipe.submit([0, 1, 2, 0]).wait())
    torch.cuda.synchronize()
    assert isinstance(got, LazyItems), "DevicePipeline did not take the one-call path"
    assert torch.equal(ref_seg, got.targets["segmentation"])


def test_brainid_batch_has_one_segmentation_per_item(stage_calls):
    # >= 50 voxels per axis: the mild generator's bias grid (0.01-0.02 of the size) must round to >= 1 node
    ds = _native_ds(option="brain_id", over={"generator.all_samples": 3, "generator.mild_samples": 1}, size=(64, 64, 64))
    ref = _snapshot(_run(ds, lambda: ds.generate_batch([0, 1])))
    got = _run(ds, lambda: ds.generate_batch_fast([0, 1]))
    assert got is not None and got.input.shape[0] == 6
    assert tuple(got.targets["segmentation"].shape) == (2, 56, *ds.size)
    for n in range(2):
        assert len(got[n][4]) == 3
        assert torch.equal(got[n][3]["segmentation"], ref[n][3]["segmentation"])
    # the python planner gives every item its own segmentation too (one job per item, first descriptor)
    ds.planner = "python"
    np.random.seed(1)
    items = ds.generate_batch([0, 1])
    assert all(it[3]["segmentation"].shape == (56, *ds.size) for it in items)
    descs, _, B = ds._last_descs
    assert B == 6


# ---- 4. routing that keeps the op-wise reader ------------------------------------------------------------------------
def test_deform_one_hots_stays_opwise(stage_calls):
    ds = _native_ds(over={"generator.deform_one_hots": True})
    assert _run(ds, lambda: ds.generate_batch_fast([0, 1])) is None
    items = _run(ds, lambda: ds.generate_batch([0, 1]))
    assert stage_calls["bfm_gen_segmentation"].n == 0
    assert all(it[3]["segmentation"].shape == (56, *ds.size) for it in items)


def test_replaced_reader_stays_opwise(stage_calls, monkeypatch):
    from brainfm_b200.Generator import constants as K
    reader = Calls(K.processing_funcs["segmentation"])
    monkeypatch.setitem(K.processing_funcs, "segmentation", reader)
    ds = _native_ds()
    assert _run(ds, lambda: ds.generate_batch_fast([0, 1])) is None
    _run(ds, lambda: ds.generate_batch([0, 1]))
    ds.planner = "python"
    ds.generate_batch([2])
    assert reader.n == 3 and stage_calls["bfm_gen_segmentation"].n == 0


def test_segmentation_of_another_shape_stays_opwise(stage_calls):
    from brainfm_b200 import io as bio
    ds = _native_ds(n=2)
    path = _seg_path(ds, 1)
    src = (56, 64, 48)
    bio.register_volume(path, mg.ti.seg_labels((src[0] + 4, src[1], src[2])))   # same strides, 4 more x planes
    assert _run(ds, lambda: ds.generate_batch_fast([0, 1])) is None
    items = _run(ds, lambda: ds.generate_batch([0, 1]))
    # item 0 takes the stage, item 1 the op-wise reader
    assert stage_calls["bfm_gen_segmentation"].n == 1 and stage_calls["bfm_label_warp_onehot"].n == 1
    ref = _opwise(ds, path, ds.last_setups, ds.last_deform)
    assert torch.equal(items[1][3]["segmentation"], ref)


@pytest.mark.parametrize("task", ["distance", "registration"])
def test_distance_or_registration_keeps_the_general_path(task, stage_calls):
    srcs = [(60, 70, 52)]
    case = _case((48, 56, 40), srcs[0], 0, {"task." + task: True}, extra=[task])
    _, ds, _ = cuda_case(case, None, planner="native", srcs=srcs, run=lambda d: None)
    assert _run(ds, lambda: ds.generate_batch_fast([0])) is None
    it = _run(ds, lambda: ds.generate_batch([0]))[0]
    assert torch.is_tensor(it[3][task])
    ref = _opwise(ds, _seg_path(ds, 0), ds.last_setups, ds.last_deform)
    assert torch.equal(it[3]["segmentation"], ref)
    assert stage_calls["bfm_gen_segmentation"].n == 1


# ---- 5. the derived class map follows uploads ------------------------------------------------------------------------
def test_upload_of_the_segmentation_drops_the_class_map():
    ds = _native_ds(n=1)
    path = _seg_path(ds, 0)
    a = _run(ds, lambda: ds.generate_batch_fast([0, 0])).targets["segmentation"].clone()
    assert int(a[:, 1:].sum()) > 0
    zeros = torch.zeros(tuple(ds.cache.get(path, "i32").shape), dtype=torch.int32)
    ds.cache.upload(path, "i32", zeros)
    b = _run(ds, lambda: ds.generate_batch_fast([0, 0])).targets["segmentation"]
    torch.cuda.synchronize()
    assert bool((b[:, 0] == 1).all()) and int(b[:, 1:].sum()) == 0
