"""brainfm_b200.interpol.jitfields_compat: the `jitfields`-shaped front end that lets the REFERENCE's own
utils.interpol forward to libbfm (utils/interpol/backend.py:1, jitfields.py:28-95).

CPU part: the reference package (a checkout of the original project named by BFM_REFERENCE_ROOT, the variable
oracle/ref_shim.py reads; skipped without one) is imported with our module installed as `jitfields` and
`backend.jitfields = True`; our kernels cannot run without a GPU, so the six entry points of brainfm_b200.interpol.api are replaced by recorders that check the layout they receive and answer with the
reference's native implementation.  A call that goes reference API -> reference shim -> our front end -> (recorder)
-> back must then equal the reference's direct answer: that pins the argument marshalling in both directions.
Without a checkout, test_front_end_marshalling pins the front end's side of it: jitfields' keyword names and
channels-last layout in, this package's API calls and channels-first layout out, for every entry point.
GPU part: the front end against brainfm_b200.interpol.api itself (channels-last vs channels-first)."""
import importlib
import os
import sys
import tempfile

import numpy as np
import pytest
import torch

REF = os.path.join(os.environ.get("BFM_REFERENCE_ROOT", ""), "utils", "interpol")


@pytest.fixture(scope="module")
def ref_interpol():
    if not os.environ.get("BFM_REFERENCE_ROOT") or not os.path.isdir(REF):
        pytest.skip("no checkout of the original project (set BFM_REFERENCE_ROOT)")
    import brainfm_b200.interpol.jitfields_compat as jf
    tmp = tempfile.mkdtemp(prefix="ref_interpol_")
    os.symlink(REF, os.path.join(tmp, "interpol"))          # SURVEY appendix B-6: not via utils/ (shadows logging)
    saved = {k: sys.modules.get(k) for k in ("jitfields", "interpol")}
    sys.modules["jitfields"] = jf
    sys.path.insert(0, tmp)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mod = importlib.import_module("interpol")
    assert mod.jitfields.available and mod.jitfields.jitfields is jf
    yield mod
    sys.path.remove(tmp)
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v
    for k in [k for k in sys.modules if k == "interpol" or k.startswith("interpol.")]:
        sys.modules.pop(k, None)


def _record_into_reference(monkeypatch, ref, calls):
    """brainfm_b200.interpol.api.* -> recorders that run the reference's native code path (backend off)."""
    from brainfm_b200.interpol import api

    def native(name):
        fn = getattr(ref, name)

        def run(*a, **k):
            calls.append((name, [tuple(x.shape) if torch.is_tensor(x) else x for x in a], dict(k)))
            ref.backend.jitfields = False
            try:
                return fn(*a, **k)
            finally:
                ref.backend.jitfields = True
        return run
    for name in ("grid_pull", "grid_push", "grid_count", "grid_grad", "spline_coeff", "spline_coeff_nd", "resize",
                 "restrict"):
        monkeypatch.setattr(api, name, native(name))


@pytest.mark.parametrize("order,bound", [(1, "dct2"), (3, "zero"), (2, "dft")])
def test_reference_forwards_to_the_front_end(ref_interpol, monkeypatch, order, bound):
    ref = ref_interpol
    torch.manual_seed(order)
    B, C, shp, oshp = 2, 3, (7, 6, 5), (4, 5, 6)
    x = torch.rand(B, C, *shp)
    grid = torch.rand(B, *oshp, 3) * torch.tensor([s - 1.0 for s in shp])
    gin = torch.rand(B, *shp, 3) * torch.tensor([s - 1.0 for s in oshp])
    kw = dict(interpolation=order, bound=bound, extrapolate=True)
    ref.backend.jitfields = False
    want = dict(pull=ref.grid_pull(x, grid, **kw), push=ref.grid_push(x, gin, oshp, **kw),
                count=ref.grid_count(gin, oshp, **kw), grad=ref.grid_grad(x, grid, **kw),
                coeff=ref.spline_coeff_nd(x, interpolation=3, bound="dct2", dim=3),
                resize=ref.resize(x, shape=[9, 8, 7], anchor='e', interpolation=order, bound=bound, prefilter=False))
    calls = []
    _record_into_reference(monkeypatch, ref, calls)
    ref.backend.jitfields = True
    try:
        got = dict(pull=ref.grid_pull(x, grid, **kw), push=ref.grid_push(x, gin, oshp, **kw),
                   count=ref.grid_count(gin, oshp, **kw), grad=ref.grid_grad(x, grid, **kw),
                   coeff=ref.spline_coeff_nd(x, interpolation=3, bound="dct2", dim=3),
                   resize=ref.resize(x, shape=[9, 8, 7], anchor='e', interpolation=order, bound=bound, prefilter=False))
    finally:
        ref.backend.jitfields = False
    names = [c[0] for c in calls]
    assert names == ["grid_pull", "grid_push", "grid_count", "grid_grad", "spline_coeff_nd", "resize"], names
    # what libbfm's API received: channel-first tensors again, the reference's keyword meaning
    assert calls[0][1] == [(B, C, *shp), (B, *oshp, 3)] and calls[0][2]["interpolation"] == order
    assert calls[1][1][:2] == [(B, C, *shp), (B, *shp, 3)] and tuple(calls[1][1][2]) == oshp
    assert calls[3][1] == [(B, C, *shp), (B, *oshp, 3)] and calls[3][2]["bound"] == bound
    for k in want:
        assert got[k].shape == want[k].shape, k
        assert torch.equal(got[k], want[k]), k


def test_unbatched_and_channel_free_inputs(ref_interpol, monkeypatch):
    """The reference's shim inserts a channel axis for bare spatial inputs (jitfields.py:12-18)."""
    ref = ref_interpol
    x = torch.rand(6, 5, 4)
    grid = torch.rand(3, 3, 3, 3) * 3
    ref.backend.jitfields = False
    want = ref.grid_pull(x, grid, interpolation=1, bound='dct2', extrapolate=True)
    calls = []
    _record_into_reference(monkeypatch, ref, calls)
    ref.backend.jitfields = True
    try:
        got = ref.grid_pull(x, grid, interpolation=1, bound='dct2', extrapolate=True)
    finally:
        ref.backend.jitfields = False
    assert calls[0][1] == [(1, 6, 5, 4), (3, 3, 3, 3)]
    assert torch.equal(got, want)


def test_front_end_marshalling(monkeypatch):
    """Every entry point of the front end, without a GPU: the API functions are replaced by recorders that check the
    channel-first data they receive and answer with a known channel-first tensor, which must come back in jitfields'
    layout (channels last; pull / grad / push) or unchanged (count, spline_coeff*, resize, restrict)."""
    import brainfm_b200.interpol.jitfields_compat as jf
    from brainfm_b200.interpol import api
    torch.manual_seed(0)
    B, C, shp, oshp = 2, 3, (7, 6, 5), (4, 5, 6)
    xl = torch.rand(B, *shp, C)
    x = torch.movedim(xl, -1, 1)
    grid = torch.rand(B, *oshp, 3)
    gin = torch.rand(B, *shp, 3)
    calls = {}

    def answer(*shape):
        return torch.arange(float(np.prod(shape))).reshape(shape)

    def stub(name, out_shape, want_input, want_grid=None):
        def run(*a, **k):
            calls[name] = (a, k)
            if want_input is not None:
                assert torch.equal(a[0], want_input), name
            if want_grid is not None:
                assert a[1] is want_grid, name
            return answer(*out_shape)
        monkeypatch.setattr(api, name, run)

    stub("grid_pull", (B, C, *oshp), x, grid)
    stub("grid_grad", (B, C, *oshp, 3), x, grid)
    stub("grid_push", (B, C, *oshp), x, gin)
    stub("grid_count", (B, *oshp), None, None)
    stub("spline_coeff", (B, C, *shp), x)
    stub("spline_coeff_nd", (B, C, *shp), x)
    stub("resize", (B, C, 9, 8, 7), x)
    stub("restrict", (B, C, 3, 3, 2), x)
    kw = dict(bound="dft", extrapolate=False)
    full = dict(bound="dft", extrapolate=False, prefilter=True)

    got = jf.pull(xl, grid, order=3, prefilter=True, **kw)
    assert torch.equal(got, torch.movedim(answer(B, C, *oshp), 1, -1))
    assert calls["grid_pull"][1] == dict(interpolation=3, **full)
    out = torch.empty(B, *oshp, C)
    assert jf.pull(xl, grid, order=3, out=out, **kw) is out and torch.equal(out, got)

    got = jf.grad(xl, grid, order=1, prefilter=True, **kw)
    assert torch.equal(got, torch.movedim(answer(B, C, *oshp, 3), 1, -2))
    assert calls["grid_grad"][1] == dict(interpolation=1, **full)

    got = jf.push(xl, gin, oshp, order=2, prefilter=True, **kw)
    assert torch.equal(got, torch.movedim(answer(B, C, *oshp), 1, -1))
    assert calls["grid_push"][0][2] == oshp and calls["grid_push"][1] == dict(interpolation=2, **full)

    got = jf.count(gin, oshp, order=0, **kw)
    assert torch.equal(got, answer(B, *oshp))
    assert calls["grid_count"][0] == (gin, oshp) and calls["grid_count"][1] == dict(interpolation=0, **kw)

    for fn, inplace in ((jf.spline_coeff, False), (jf.spline_coeff_, True)):
        assert torch.equal(fn(x, 3, bound="dst2", dim=2), answer(B, C, *shp))
        assert calls["spline_coeff"][1] == dict(interpolation=3, bound="dst2", dim=2, inplace=inplace)
    for fn, inplace in ((jf.spline_coeff_nd, False), (jf.spline_coeff_nd_, True)):
        assert torch.equal(fn(x, 5, bound="dct1", ndim=3), answer(B, C, *shp))
        assert calls["spline_coeff_nd"][1] == dict(interpolation=5, bound="dct1", dim=3, inplace=inplace)

    assert torch.equal(jf.resize(x, shape=[9, 8, 7], ndim=3, anchor="c", order=1, bound="zero", prefilter=False),
                       answer(B, C, 9, 8, 7))
    assert calls["resize"][1] == dict(factor=None, shape=[9, 8, 7], anchor="c", interpolation=1, prefilter=False,
                                      bound="zero")
    assert torch.equal(jf.restrict(x, factor=2, ndim=3, anchor="e", order=2, bound="dct2", reduce_sum=True),
                       answer(B, C, 3, 3, 2))
    assert calls["restrict"][1] == dict(factor=2, shape=None, anchor="e", interpolation=2, reduce_sum=True,
                                        bound="dct2")


@pytest.mark.gpu
@pytest.mark.parametrize("order", [1, 3])
def test_front_end_equals_channel_first_api_on_gpu(order):
    import brainfm_b200.interpol as bi
    import brainfm_b200.interpol.jitfields_compat as jf
    torch.manual_seed(0)
    dev = "cuda"
    B, C, shp, oshp = 2, 3, (9, 8, 7), (5, 6, 4)
    x = torch.rand(B, C, *shp, device=dev)
    grid = torch.rand(B, *oshp, 3, device=dev) * torch.tensor([s - 1.0 for s in shp], device=dev)
    gin = torch.rand(B, *shp, 3, device=dev) * torch.tensor([s - 1.0 for s in oshp], device=dev)
    xl = torch.movedim(x, 1, -1).contiguous()
    kw = dict(bound='dct2', extrapolate=True)
    a = jf.pull(xl, grid, order=order, **kw)
    assert tuple(a.shape) == (B, *oshp, C)
    assert torch.equal(torch.movedim(a, -1, 1), bi.grid_pull(x, grid, interpolation=order, **kw))
    a = jf.push(xl, gin, oshp, order=order, **kw)
    assert tuple(a.shape) == (B, *oshp, C)
    np.testing.assert_allclose(torch.movedim(a, -1, 1).cpu().numpy(),
                               bi.grid_push(x, gin, oshp, interpolation=order, **kw).cpu().numpy(), rtol=1e-5, atol=1e-5)
    a = jf.grad(xl, grid, order=order, **kw)
    assert tuple(a.shape) == (B, *oshp, C, 3)
    assert torch.equal(torch.movedim(a, -2, 1), bi.grid_grad(x, grid, interpolation=order, **kw))
    np.testing.assert_allclose(jf.count(gin, oshp, order=order, **kw).cpu().numpy(),
                               bi.grid_count(gin, oshp, interpolation=order, **kw).cpu().numpy(), rtol=1e-5, atol=1e-5)
    assert torch.equal(jf.spline_coeff_nd(x, 3, bound='dct2', ndim=3), bi.spline_coeff_nd(x, 3, 'dct2', 3))
    out = torch.empty(B, *oshp, C, device=dev)
    assert jf.pull(xl, grid, order=order, out=out, **kw) is out
