"""Host side of the cubic zoom back (`bspline_zooming`): the ABI fields sit in existing padding, the native planner
writes zoom_order into every descriptor without drawing anything, and every stage refuses an unknown zoom order
before it launches anything."""
import ctypes as C

import numpy as np
import pytest

from brainfm_b200 import _lib
from oracle import make_golden as mg
from tests._harness import oracle_case
from tests.test_native_planner_cpu import FAKE, flatten_log, make_cfg, plan


def test_abi_fields_sit_in_existing_padding():
    assert C.sizeof(_lib.GenSample) == 976 and C.sizeof(_lib.PlanCfg) == 2288
    assert _lib.GenSample.zoom_order.offset == 964
    assert _lib.PlanCfg.bspline_zooming.offset == 404
    assert _lib.GenSample.gmm_xr.offset == 968 and _lib.PlanCfg.aug.offset == 408


@pytest.mark.parametrize("name", ["g64_bspline_s43", "g64_bspline_s41"])
def test_native_replay_sets_zoom_order_and_draws_nothing(name):
    size, src, kind, seed, over, extra, option, stride = mg.CASES[name]
    item, orc = oracle_case(name)
    args = mg.cfg_for(size, over, option, ref=False)
    gen = dict(vars(args.generator))
    gen.update(vars(args.synth_image_generator))
    n = 1
    flat = flatten_log(orc.log)
    consumed = []
    for on in (0, 1):
        cfg, keep = make_cfg(list(mg.shape3(size)), args.generator, aug_sets=[gen] * n)
        cfg.bspline_zooming = on
        r = plan(cfg, 1, list(mg.shape3(src)), replay=flat)
        assert [r['descs'][q].zoom_order for q in range(n)] == [3 * on] * n
        consumed.append(r['consumed'])
    assert consumed[0] == consumed[1] == flat.size


@pytest.mark.parametrize("order", [1, 2, -1, 4])
def test_unknown_zoom_order_is_refused_before_any_launch(order):
    args = mg.cfg_for(64, {}, "default", ref=False)
    gen = dict(vars(args.generator))
    gen.update(vars(args.synth_image_generator))
    cfg, keep = make_cfg([64] * 3, args.generator, aug_sets=[gen])
    r = plan(cfg, 1, [96] * 3, seed=4)
    r['descs'][0].zoom_order = order
    L = _lib.lib()
    for stage in (L.bfm_gen_run, L.bfm_gen_plan, L.bfm_gen_bbox, L.bfm_gen_gmm, L.bfm_gen_warp, L.bfm_gen_resample,
                  L.bfm_gen_finish):
        assert stage(C.addressof(r['descs']), FAKE, 1, None) == _lib.BFM_E_INVALID
        assert "zoom_order" in L.bfm_last_error().decode()
