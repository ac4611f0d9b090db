"""bfm_gen_segmentation without a GPU: the job struct's layout, the exported symbol, the argument checks (they run on the
host, before any launch), and the existing layout pins next to the new struct."""
import ctypes as C

import pytest

from brainfm_b200 import _lib


def test_job_struct_layout_and_symbol():
    assert C.sizeof(_lib.GenSeg) == 24
    assert [(f, getattr(_lib.GenSeg, f).offset) for f, _ in _lib.GenSeg._fields_] == [("sample", 0), ("cls", 8),
                                                                                         ("out", 16)]
    assert "bfm_gen_segmentation" in _lib.exported_symbols()
    assert C.sizeof(_lib.GenSample) == 976 and C.sizeof(_lib.PlanCfg) == 2288
    L = _lib.lib()
    assert L.bfm_abi_version() == _lib.ABI_VERSION == 8


def _call(descs, jobs, n_classes=56, vflip=None, n_desc=None):
    L = _lib.lib()
    vf = (C.c_int32 * 64)(*(vflip if vflip is not None else range(64)))
    rc = L.bfm_gen_segmentation(C.addressof(descs), 4096, len(descs) if n_desc is None else n_desc,
                                C.addressof(jobs), len(jobs), n_classes, C.addressof(vf), None)
    return rc, L.bfm_last_error().decode()


def _valid():
    descs = (_lib.GenSample * 2)()
    for s in descs:
        s.d.size[:] = [8, 8, 8]
        s.d.src[:] = [10, 10, 10]
        s.bbox = 1024
    jobs = (_lib.GenSeg * 2)()
    for q, j in enumerate(jobs):
        j.sample, j.cls, j.out = q, 2048, 1 << 20
    return descs, jobs


@pytest.mark.parametrize("what", ["null_out", "null_cls", "misaligned_out", "sample_range", "n_classes_0",
                                  "n_classes_65", "vflip_range", "no_bbox", "sizes_differ"])
def test_argument_checks_return_invalid(what):
    descs, jobs = _valid()
    kw = {}
    if what == "null_out":
        jobs[1].out = None
    elif what == "null_cls":
        jobs[0].cls = None
    elif what == "misaligned_out":
        jobs[1].out = (1 << 20) + 4
    elif what == "sample_range":
        jobs[1].sample = 2
    elif what == "n_classes_0":
        kw["n_classes"] = 0
    elif what == "n_classes_65":
        kw["n_classes"] = 65
    elif what == "vflip_range":
        kw["vflip"] = [56] + list(range(1, 64))
    elif what == "no_bbox":
        descs[1].bbox = None
    elif what == "sizes_differ":
        descs[1].d.size[2] = 12
    rc, msg = _call(descs, jobs, **kw)
    expect = _lib.BFM_E_UNSUPPORTED if what == "sizes_differ" else _lib.BFM_E_INVALID
    assert rc == expect, (what, rc, msg)
    assert msg.startswith("bfm_gen_segmentation")
