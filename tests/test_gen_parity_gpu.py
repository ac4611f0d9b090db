"""GPU parity of the fused generator chain against the oracle (same injected draws) and against the
reference-generated fixtures.  Tolerances are BASELINE.json's: integer / index outputs bit-exact, fp32
outputs within 1e-5 relative / 1e-4 absolute."""
import os

import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from tests._harness import ATOL, RTOL, cuda_case, oracle_case, to_np
from tests._harness import compare as _compare

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["g64_s0", "g64_s1", "g64_s2", "g64_s3", "g64_s5_lowres", "g64_full_s4", "g160_s0", "g64_pathol_s7",
         "g64_pathol_s12", "g64_left_s9", "g64_ident_s23", "g64_realT1_s14", "g64_realT2_s15", "g64_realCT_s16"]
# round 2: branches that were built but unpinned in round 1 -- SVF scaling-and-squaring ('surface' task), linearly warped
# one-hots, cubic B-spline zoom back, random centre shift, CT contrast groups, PDE-advected pathology shapes
CASES_R2 = ["g64_svf_s31", "g64_svf_s41", "g64_onehot_s43", "g64_onehot_s41", "g64_bspline_s43", "g64_bspline_s41",
            "g64_shift_s43", "g64_ct_s35", "g64_augpath_s47", "g64_augpath_s48"]


@pytest.mark.parametrize("name", CASES + CASES_R2)
def test_chain_matches_oracle(name):
    item, orc = oracle_case(name)
    got, ds, draws = cuda_case(name, orc.log)
    assert draws.done(), "CUDA path consumed %d of %d draws" % (draws.pos, len(draws.log))
    # integer side results: bounding box of the deformed grid
    assert ds.last_deform["_plan"].bbox_host() == orc.deform["lo"] + orc.deform["hi"]
    rep = _compare(mg.flatten(item), mg.flatten(got), name)
    # deformation / bias outputs are pure separately-rounded lerps: expect exact equality
    for k, v in rep.items():
        if "bias_field_log" in k:
            assert v == 0.0, (k, v)


def test_brainid_batch_matches_oracle():
    name = "g64_brainid_s6"
    item, orc = oracle_case(name)
    got, ds, draws = cuda_case(name, orc.log)
    assert draws.done()
    assert isinstance(got[4], list) and len(got[4]) == 3
    _compare(mg.flatten(item), mg.flatten(got), name)


@pytest.mark.parametrize("name", ["g64_s0", "g64_full_s4", "g160_s0", "g64_pathol_s7", "g64_left_s9", "g64_ident_s23", "g64_realT1_s14",
                                  "g64_realT2_s15", "g64_realCT_s16"] + CASES_R2)
def test_chain_matches_reference_fixture(name):
    """Directly against the fixture the unmodified reference produced (strided sub-sample + sums)."""
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    _, orc = oracle_case(name)
    got, ds, _ = cuda_case(name, orc.log)
    stride = int(gold["meta.stride"])
    assert list(gold["meta.bbox"]) == ds.last_deform["_plan"].bbox_host()
    for k, v in mg.flatten(got).items():
        if not isinstance(v, torch.Tensor):
            continue
        out = {}
        mg.summarise(k, v, stride, out)
        for kk, vv in out.items():
            if kk.endswith(".sub"):
                if gold[kk].dtype.kind == "f":
                    np.testing.assert_allclose(vv, gold[kk], rtol=RTOL, atol=ATOL, err_msg=kk)
                else:
                    assert np.array_equal(vv, gold[kk]), kk
            elif kk.endswith(".sum"):
                np.testing.assert_allclose(vv, gold[kk], rtol=1e-5, err_msg=kk)
    if "deform.F.sub" in gold.files:
        # 'surface' task: the integrated fields themselves (bfm_svf_step, datasets.py:214-223) against the REFERENCE's
        for key in ("F", "Fneg"):
            out = {}
            mg.summarise("deform." + key, ds.last_deform[key], stride, out)
            np.testing.assert_allclose(out["deform.%s.sub" % key], gold["deform.%s.sub" % key], rtol=RTOL, atol=ATOL)
            np.testing.assert_allclose(out["deform.%s.sum" % key], gold["deform.%s.sum" % key], rtol=1e-4, atol=1e-2)


@pytest.mark.parametrize("name", ["g64_svf_s31", "g64_svf_s41"])
def test_svf_integration_is_bit_exact(name):
    """Scaling and squaring (n_steps_svf_integration x `F += trilerp(F, id + F)`): separately rounded fp32 like the
    reference => F, Fneg and the coordinates of the deformed grid equal the oracle's bit for bit (the oracle's equal
    the reference's bit for bit: oracle/make_golden.py asserts it when the fixture is generated)."""
    _, orc = oracle_case(name)
    got, ds, _ = cuda_case(name, orc.log)
    for key in ("F", "Fneg"):
        a, b = to_np(ds.last_deform[key]), orc.deform[key].numpy()
        assert a.shape == b.shape
        assert np.array_equal(a, b), "%s: %d voxels differ, max %g" % (key, int((a != b).sum()), float(np.abs(a - b).max()))
    grid = ds.last_deform["grid"]
    for d in range(3):
        assert np.array_equal(to_np(grid[d]), orc.deform["rel"][d].numpy()), "coordinate plane %d" % d
    assert [int(v) for v in grid[3:]] == orc.deform["lo"] + orc.deform["hi"]


@pytest.mark.parametrize("name", ["g64_s0", "g64_s2", "g160_s0", "g64_s5_lowres"])
def test_pair_mode_is_identical_to_the_unpaired_gather(name, monkeypatch):
    """k_gen_warp_pk (float2 {synthetic, T1} gathers, packed f32x2 arithmetic) against k_gen_warp<1, 0>: same
    operations, bit-identical outputs."""
    _, orc = oracle_case(name)
    got_pk, ds, _ = cuda_case(name, orc.log)
    assert ds.pair_mode and ds._last_descs[0][0].syn_pair_ok == 1
    monkeypatch.setenv("BFM_PAIR_MODE", "0")
    got_np, ds2, _ = cuda_case(name, orc.log)
    assert not ds2.pair_mode and ds2._last_descs[0][0].syn_pair_ok == 0
    a, b = mg.flatten(got_pk), mg.flatten(got_np)
    for k, v in a.items():
        if isinstance(v, torch.Tensor):
            assert torch.equal(v, b[k]), k


def test_deform_grid_and_field_are_bit_exact():
    """deform_dict['grid'] (coordinates + bbox) against the oracle: separately rounded fp32 => exact."""
    name = "g64_s0"
    _, orc = oracle_case(name)
    got, ds, _ = cuda_case(name, orc.log)
    grid = ds.last_deform["grid"]
    for d in range(3):
        assert np.array_equal(to_np(grid[d]), orc.deform["rel"][d].numpy()), "coordinate plane %d" % d
    assert [int(v) for v in grid[3:]] == orc.deform["lo"] + orc.deform["hi"]


@pytest.mark.parametrize("n_in,n_out,sigma", [(160, 160, 0.0), (160, 25, 2.95), (160, 121, 0.51), (64, 13, 1.7),
                                             (160, 32, 5.0), (96, 96, 0.3), (160, 159, 0.0)])
def test_device_band_tables_match_host(n_in, n_out, sigma):
    """bfm_band_build (tables built on the GPU) against plan.band_host (numpy/torch, the op-level path)."""
    import ctypes as C
    from brainfm_b200 import _lib, plan
    start, w, T = plan.band_host(n_in, n_out, sigma)
    ds = torch.empty(n_out, dtype=torch.int32, device="cuda")
    dw = torch.empty((n_out, T), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib().bfm_band_build(n_in, n_out, float(sigma), T, ds.data_ptr(), dw.data_ptr(),
                                         C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert np.array_equal(to_np(ds), start)
    np.testing.assert_allclose(to_np(dw), w, rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(to_np(dw).sum(1), w.sum(1), rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("name", ["g64_s0", "g64_s5_lowres"])
def test_slab_mode_single_rank_matches_oracle(name):
    """Slab mode (x-slabs + plane exchange, Generator/slab.py) on one rank: same volume as the oracle."""
    from brainfm_b200.Generator.slab import generate_slab
    item, orc = oracle_case(name)
    ref = mg.flatten(item)
    got, ds, draws = cuda_case(name, orc.log, run=lambda ds: generate_slab(ds, 0, 0, 1))
    assert got["x_range"] == (0, int(ds.size[0]))
    np.testing.assert_allclose(to_np(got["input"]), to_np(ref["sample0.input"]), rtol=RTOL, atol=ATOL)
    if "bias_field_log" in got:
        assert np.array_equal(to_np(got["bias_field_log"]), to_np(ref["sample0.bias_field_log"]))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_slab_mode_two_ranks():
    """Two ranks over NCCL: assembled slabs == oracle within tolerance and == the single-rank slab run bit for bit."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for name in ("g64_s0", "g64_s5_lowres"):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", "29533",
                            os.path.join(root, "tests", "_slab_worker.py"), name],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("planner", ["python", "native"])
@pytest.mark.parametrize("world", [1, 3])
def test_slab_mode_without_injected_draws_does_not_depend_on_the_decomposition(world, planner):
    """The library's own noise (counter-based, keyed on absolute source / low-res voxels): a volume generated on W
    ranks equals the single-rank slab run bit for bit and the fused chain within tolerance.  The ranks share GPU 0
    (gloo stages the exchanged planes through the host), so this runs on a 1-GPU box."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, BFM_SLAB_ONE_GPU="1", BFM_SLAB_PLANNER=planner)
    worker = os.path.join(root, "tests", "_slab_noise_worker.py")
    cmd = [sys.executable, worker] if world == 1 else \
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
         "--master-addr", "127.0.0.1", "--master-port", "29541", worker]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=280, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.parametrize("planner", ["python", "native"])
def test_slab_mode_refuses_a_rank_without_planes(planner):
    """More ranks than planes: a rank that owns no plane raises instead of generating a slab.  Of 2 s0 + 1 ranks the
    middle one owns no plane whether the volume is flipped (slabs mirrored) or not."""
    from brainfm_b200.Generator.slab import generate_slab
    _, ds, _ = cuda_case("g64_s0", None, planner=planner, run=lambda d: None)
    s0 = int(ds.size[0])
    with pytest.raises(ValueError, match="owns no plane"):
        generate_slab(ds, 0, rank=s0, world=2 * s0 + 1)


@pytest.mark.parametrize("name", ["g64_s0", "g64_s2", "g160_s0"])
def test_full_bbox_scan_equals_candidate_result(name):
    """bfm_gen_bbox: with the candidate lists disabled (ncand = 0) the persistent full scan must give the same six
    integers as the candidate-voxel evaluation (and as the oracle)."""
    import ctypes as C
    from brainfm_b200 import _lib
    item, orc = oracle_case(name)
    got, ds, draws = cuda_case(name, orc.log, planner='python')
    descs, d_dev, B = ds._last_descs
    want = orc.deform["lo"] + orc.deform["hi"]
    assert ds.last_deform["_plan"].bbox_host() == want
    copy = (_lib.GenSample * B)()
    C.memmove(C.addressof(copy), C.addressof(descs), C.sizeof(copy))
    bb = torch.zeros(8 * B, dtype=torch.int32, device="cuda")
    for b in range(B):
        copy[b].d.ncand[:] = [0, 0, 0]
        copy[b].bbox = bb.data_ptr() + 32 * b
    host = np.frombuffer(copy, dtype=np.uint8).copy()
    dev = torch.from_numpy(host).cuda()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.lib().bfm_gen_bbox(C.addressof(copy), dev.data_ptr(), B, st))
    torch.cuda.synchronize()
    assert bb[:6].tolist() == want


@pytest.mark.parametrize("name,mode", [("g64_realT1_s14", "T1"), ("g64_realT2_s15", "T2"), ("g64_realCT_s16", "CT")])
def test_real_inputs_take_the_fused_chain(name, mode):
    """Real T1 / T2 / FLAIR inputs run through the fused chain (real_input descriptors, no GMM stage), not op by op."""
    item, orc = oracle_case(name)
    got, ds, draws = cuda_case(name, orc.log, planner='python')
    assert got[2] == mode == item[2]
    descs, _, B = ds._last_descs
    assert B == 1 and descs[0].real_input == (2 if mode == 'CT' else 1) and descs[0].labels is None
    _compare(mg.flatten(item), mg.flatten(got), name)
