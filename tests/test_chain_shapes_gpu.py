"""The fused chain at odd and anisotropic grids and in mixed batches, against the oracle (same injected draws).

The cubic fixtures of test_gen_parity_gpu have every extent a multiple of 32, so they only ever take one side of the
chain's vector / scalar pairs.  The cases here are chosen (by their draws) to take the other sides: flat GMM with
rows that straddle 4-groups, k_gen_warp<1, false> for a T1 target whose source z is not a multiple of 4, the scalar
normalisation of an odd output plane, the undegraded class through k_gen_band_z, band_z without the register
prefetch, the k loops of the warp and upsample kernels, partial row blocks, and batches that mix all of these with
per-sample scratch slots at odd offsets.  test_routing_covers_every_branch maps the descriptors of every launch to
the launchers' own routing conditions and fails when a case stops reaching the branch it is here for."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from tests._harness import compare, cuda_case, oracle_batch, oracle_case, to_np

pytestmark = pytest.mark.gpu

TS = {"task.T1": True, "task.segmentation": True}
ANISO, ANISO_SRC = (72, 61, 83), (101, 90, 97)
DEEP, DEEP_SRC = (40, 45, 270), (60, 64, 301)
MNI2 = (91, 109, 91)                              # the 2 mm MNI grid: N = 902 629 voxels, odd
BATCH_SRCS = [MNI2, (96, 112, 100)]               # subject 1: pairs refused (z % 4 = 3); subject 2: paired


def _c(size, src, seed, over, extra=(), option="default", stride=2):
    return (size, src, "brain", seed, over, list(extra), option, stride)


CASES = {
    "aniso_s0": _c(ANISO, ANISO_SRC, 0, TS),
    "aniso_s2": _c(ANISO, ANISO_SRC, 2, TS),
    "aniso_s3": _c(ANISO, ANISO_SRC, 3, TS),
    "aniso_s5": _c(ANISO, ANISO_SRC, 5, TS),
    "aniso_s6": _c(ANISO, ANISO_SRC, 6, TS),
    "aniso_lowres_s0": _c(ANISO, ANISO_SRC, 0, dict(TS, **{"generator.low_res_only": True})),
    "aniso_mix_s0": _c(ANISO, ANISO_SRC, 0, {"mix_synth_prob": 1.0, "task.T1": True, "task.T2": True}, ["T2"]),
    "deep_s0": _c(DEEP, DEEP_SRC, 0, TS),
    "deep_s3": _c(DEEP, DEEP_SRC, 3, TS),
    "deep_s4": _c(DEEP, DEEP_SRC, 4, TS),
    # an MNI 1 mm source (z = 182): pairs refused, flat GMM + k_gen_warp<1, false> into a 160^3 grid
    "mni1mm_s0": _c(160, (182, 218, 182), 0, {"task.T1": True}, stride=4),
    "mni1mm_s3": _c(160, (182, 218, 182), 3, {"task.T1": True}, stride=4),          # undegraded: k_gen_identity
    "brainid_s0": _c(MNI2, MNI2, 0, {"generator.all_samples": 3, "generator.mild_samples": 1}, option="brain_id"),
}
NATIVE = [k for k, v in CASES.items() if "mix_synth_prob" not in v[4]]      # the native planner does not mix
# a batch of 4 items from two subjects; tasks off but the T1 target, so that generate_batch_fast takes it too
BATCH = _c(MNI2, MNI2, 3, {"task.bias_field": False, "task.T1": True})
BATCH_IDX = [0, 1, 1, 0]

# ---- routing: the launchers' conditions (csrc/gen.cu), evaluated on the host copies of the descriptors -----------
K_PK_NODES, ZK_CAP, K_UR = 48, 96 * 1024, 32


def _use_pairs(s):
    return bool(s.syn_pair_ok and s.n_aux == 1 and not s.mix[0] and not s.real_input and s.d.src[2] % 4 == 0
                and not s.d.F_full and (not s.d.fsmall or s.d.fs[2] < K_PK_NODES)
                and (not s.bfsmall or s.bs[2] < K_PK_NODES))


def sample_labels(s, slot):
    """Branches of the fused chain that the sample in descriptor slot `slot` takes (bfm_gen_gmm ... bfm_gen_finish).
    'odd_slot_vec' marks a 128-bit tmp / lowres access in a slot that a stride of prod(size) floats misaligns."""
    size = list(s.d.size)
    N, plane = size[0] * size[1] * size[2], size[1] * size[2]
    out = set()
    if not s.real_input:
        out.add("gmm_flat" if s.d.src[2] % 4 else "gmm_planes")
    out.add("warp_pk" if _use_pairs(s) else "warp<%d,%s>" % (s.n_aux, "mix" if s.mix[0] else "false"))
    if size[2] > 256:
        out.add("warp_k_loop")
    vec_scratch = False
    ident = (s.n_band == 1 and s.band[0].T == 1 and s.band[0].build == 0 and list(s.new_size) == size)
    if ident and plane % 4 == 0:
        out.add("identity")
    else:
        if ident:
            out.add("undegraded_odd_plane")
        sh = list(size)
        for p in range(s.n_band):
            b = s.band[p]
            need_z = (b.n_out * ((b.T | 1) + 1) + 8 * (sh[2] + b.n_out + 4)) * 4
            if b.axis == 2 and need_z <= ZK_CAP:
                out.add("band_z")
                if sh[2] > 256:
                    out.add("band_z_no_prefetch")
            elif b.axis == 2 or sh[2] % 4:
                out.add("band<1>")
            else:
                out.add("band<4>")
                if p >= 1:
                    out.add("band<4>_on_tmp")
                    vec_scratch = True
                elif p < s.n_band - 1:
                    vec_scratch = True
            sh[b.axis] = b.n_out
    out.add("upsample")
    if s.new_size[2] % 4 == 0:
        out.add("upsample_vec")
        vec_scratch = True
    if size[2] > 160:
        out.add("upsample_k_loop")
    if size[1] % K_UR:
        out.add("partial_rows")
    out.add("normalize<4>" if plane % 4 == 0 else "normalize<1>")
    if vec_scratch and (slot * N) % 4:
        out.add("odd_slot_vec")
    return out


def launch_labels(descs, B):
    per = [sample_labels(descs[b], b) for b in range(B)]
    out = set().union(*per)
    if any("warp_pk" in p for p in per) and not all("warp_pk" in p for p in per):
        out.add("mixed_pairs")
    if {"gmm_flat", "gmm_planes"} <= out:
        out.add("mixed_gmm")
    return out


# every branch that only these shapes reach, and the common vector paths next to them
REQUIRED = {"gmm_flat", "gmm_planes", "warp<1,false>", "warp_pk", "warp<0,mix>", "normalize<1>", "normalize<4>",
            "undegraded_odd_plane", "identity", "band_z_no_prefetch", "band_z", "band<1>", "band<4>_on_tmp",
            "warp_k_loop", "upsample_k_loop", "upsample_vec", "partial_rows", "mixed_pairs", "mixed_gmm",
            "odd_slot_vec"}
SEEN = {}


def _note(key, ds):
    descs, _, B = ds._last_descs
    SEEN[key] = launch_labels(descs, B)


@functools.lru_cache(maxsize=None)
def _oracle(name):
    return oracle_case(CASES[name])


def _check_item(name, item, orc, got, ds, draws, coords):
    assert draws.done(), "CUDA path consumed %d of %d draws" % (draws.pos, len(draws.log))
    want = orc.deform["lo"] + orc.deform["hi"]
    rep = compare(mg.flatten(item), mg.flatten(got), name)
    for k, v in rep.items():
        if "bias_field_log" in k:
            assert v == 0.0, (name, k, v)
    if coords:
        assert ds.last_deform["_plan"].bbox_host() == want
        grid = ds.last_deform["grid"]
        for d in range(3):
            assert np.array_equal(to_np(grid[d]), orc.deform["rel"][d].numpy()), (name, "coordinate plane %d" % d)
        assert [int(v) for v in grid[3:]] == want


@pytest.mark.parametrize("planner", ["python", "native"])
@pytest.mark.parametrize("name", list(CASES))
def test_chain_matches_oracle_at_odd_shapes(name, planner):
    if planner == "native" and name not in NATIVE:
        pytest.skip("mixing with real modalities is planned in Python only")
    item, orc = _oracle(name)
    got, ds, draws = cuda_case(CASES[name], orc.log, planner=planner)
    _check_item(name, item, orc, got, ds, draws, coords=planner == "python")
    if CASES[name][6] == "brain_id":
        assert isinstance(got[4], list) and len(got[4]) == 3
    _note((name, planner), ds)


def _flat_items(items):
    return [{k: v for k, v in mg.flatten(it).items() if isinstance(v, torch.Tensor)} for it in items]


def _assert_identical(a, b, what):
    assert set(a) == set(b), what
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


def test_mixed_batch_matches_oracle_and_single_items():
    """Items of one launch that differ in source shape (pairs / no pairs, GMM planes / flat), band routing and low-res
    z, with scratch slots at odd offsets: each matches its oracle and equals the same item generated alone."""
    items, orcs, log = oracle_batch(BATCH, BATCH_SRCS, BATCH_IDX)
    got, ds, draws = cuda_case(BATCH, log, planner="python", srcs=BATCH_SRCS, run=lambda d: d.generate_batch(BATCH_IDX))
    assert draws.done()
    _note(("batch", "python"), ds)
    labels = SEEN[("batch", "python")]
    assert {"mixed_pairs", "mixed_gmm", "odd_slot_vec"} <= labels, sorted(labels)
    for n, (it, orc, g) in enumerate(zip(items, orcs, got)):
        _check_item("batch item %d" % n, it, orc, g, ds, draws, coords=False)
    batch = _flat_items(got)
    # the same item alone, B = 1: replay its own draws (item n of the batch is seeded by the draws before it)
    for n, idx in enumerate(BATCH_IDX):
        alone, _, dr = cuda_case(BATCH, orcs[n].log, planner="python", srcs=BATCH_SRCS,
                                 run=lambda d, idx=idx: d.generate_batch([idx]))
        assert dr.done()
        _assert_identical(batch[n], _flat_items(alone)[0], "python planner, item %d" % n)


@pytest.mark.parametrize("fast", [False, True])
def test_native_batch_items_equal_single_items(fast):
    """Native draws: item n of a batch at counter c is item 0 of a batch at counter c + n, bit for bit, through
    generate_batch and generate_batch_fast."""
    _, ds, _ = cuda_case(BATCH, None, planner="native", srcs=BATCH_SRCS, run=lambda d: None)

    def gen(indices, counter):
        ds._native_planner(indices)
        ds._native.seed, ds._native.counter = 12345, counter
        items = ds.generate_batch_fast(indices) if fast else ds.generate_batch(indices)
        assert items is not None, "generate_batch_fast refused the batch"
        torch.cuda.synchronize()
        descs, _, B = ds._last_descs
        return _flat_items(list(items)), launch_labels(descs, B)

    batch, labels = gen(BATCH_IDX, 0)
    assert {"mixed_pairs", "mixed_gmm"} <= labels, sorted(labels)
    for n, idx in enumerate(BATCH_IDX):
        alone, _ = gen([idx], n)
        _assert_identical(batch[n], alone[0], "native planner%s, item %d" % (" (fast)" if fast else "", n))


@pytest.mark.parametrize("name", ["aniso_s5", "deep_s0", "mni1mm_s0"])
def test_full_bbox_scan_equals_candidate_result_at_odd_shapes(name):
    """bfm_gen_bbox with the candidate lists disabled (ncand = 0): the persistent full scan gives the oracle's six
    integers at anisotropic grids too."""
    from brainfm_b200 import _lib
    item, orc = _oracle(name)
    got, ds, draws = cuda_case(CASES[name], orc.log, planner="python")
    descs, d_dev, B = ds._last_descs
    want = orc.deform["lo"] + orc.deform["hi"]
    assert ds.last_deform["_plan"].bbox_host() == want
    copy = (_lib.GenSample * B)()
    C.memmove(C.addressof(copy), C.addressof(descs), C.sizeof(copy))
    bb = torch.zeros(8 * B, dtype=torch.int32, device="cuda")
    for b in range(B):
        copy[b].d.ncand[:] = [0, 0, 0]
        copy[b].bbox = bb.data_ptr() + 32 * b
    dev = torch.from_numpy(np.frombuffer(copy, dtype=np.uint8).copy()).cuda()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.lib().bfm_gen_bbox(C.addressof(copy), dev.data_ptr(), B, st))
    torch.cuda.synchronize()
    assert bb[:6].tolist() == want


def test_routing_covers_every_branch():
    """The union of the branches every case above takes covers REQUIRED: a seed or configuration change that silently
    drops a path fails here.  Cases not run in this session are run now (python planner)."""
    for name in CASES:
        if (name, "python") not in SEEN and (name, "native") not in SEEN:
            item, orc = _oracle(name)
            _, ds, _ = cuda_case(CASES[name], orc.log, planner="python")
            _note((name, "python"), ds)
    if ("batch", "python") not in SEEN:
        _, _, log = oracle_batch(BATCH, BATCH_SRCS, BATCH_IDX)
        _, ds, _ = cuda_case(BATCH, log, planner="python", srcs=BATCH_SRCS, run=lambda d: d.generate_batch(BATCH_IDX))
        _note(("batch", "python"), ds)
    seen = set().union(*SEEN.values())
    assert REQUIRED <= seen, "branches no case reaches: %s" % sorted(REQUIRED - seen)
