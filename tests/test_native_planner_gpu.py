"""The native host planner (bfm_plan_batch, csrc/planner.cu) against the Python planner and the oracle.

Replay mode: the library consumes the oracle's recorded draws; the descriptors it fills must equal the Python
planner's field by field (bit-exact scalars, tables and small grids), and the generated sample must match the
oracle within BASELINE.json's tolerances.  Native mode: determinism under np.random.seed and sane outputs."""
import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from tests._harness import compare as _compare
from tests._harness import cuda_case, oracle_case, to_np

pytestmark = pytest.mark.gpu

CASES = ["g64_s0", "g64_s1", "g64_s2", "g64_s3", "g64_s5_lowres", "g160_s0", "g64_ident_s23", "g64_realT1_s14",
         "g64_realT2_s15", "g64_realCT_s16"]


def _read(ds, ptr, n, dtype):
    """n elements at device address ptr, which lies inside one of the dataset's arena slots."""
    for slot in range(len(ds.arena.slots)):
        base = ds.arena.slots[slot]["dev"].data_ptr()
        if base <= ptr < base + ds.arena.capacity:
            return ds.arena.view(ptr - base, n, dtype, slot=slot).cpu().numpy()
    raise AssertionError("pointer outside the arena")


def _scalars(s):
    d = s.d
    band = [(b.T, b.n_in, b.n_out, b.axis, b.build, b.sigma) for b in s.band[:s.n_band]]
    return dict(size=list(d.size), src=list(d.src), A=list(d.A), c2=list(d.c2), ctr=list(d.ctr), fs=list(d.fs),
                photo=d.photo, ncand=list(d.ncand), cand=list(d.cand), ftab=[list(d.ftab.lo), list(d.ftab.wh)],
                label_is_u8=s.label_is_u8, gamma=s.gamma, bs=list(s.bs), btab=[list(s.btab.lo), list(s.btab.wh)],
                flip=s.flip, band=band, n_band=s.n_band, zero_first=list(s.zero_first), noise_std=s.noise_std,
                new_size=list(s.new_size), utab=[list(s.utab.lo), list(s.utab.wh)], n_aux=s.n_aux,
                mixw=list(s.mixw), real_input=s.real_input)


@pytest.mark.parametrize("name", CASES + ["g64_brainid_s6"])
def test_replayed_native_plan_equals_python_plan(name):
    item, orc = oracle_case(name)
    _, ds_py, _ = cuda_case(name, orc.log, planner='python')
    py_descs, _, n_py = ds_py._last_descs
    py = []
    for q in range(n_py):
        s = py_descs[q]
        nf = s.d.fs[0] * s.d.fs[1] * s.d.fs[2] * 3
        py.append((_scalars(s), None if s.real_input else _read(ds_py, s.mu, 512, torch.float32),
                   _read(ds_py, s.d.fsmall, nf, torch.float32),
                   _read(ds_py, s.bfsmall, s.bs[0] * s.bs[1] * s.bs[2], torch.float32) if s.bfsmall else None))
    _, ds_c, draws = cuda_case(name, orc.log, planner='native')
    assert draws.done()
    c_descs, _, n_c = ds_c._last_descs
    assert n_c == n_py
    for q in range(n_c):
        s = c_descs[q]
        ref_sc, ref_ms, ref_f, ref_b = py[q]
        got_sc = _scalars(s)
        for k in ref_sc:
            assert got_sc[k] == ref_sc[k], (name, q, k, got_sc[k], ref_sc[k])
        nf = s.d.fs[0] * s.d.fs[1] * s.d.fs[2] * 3
        if not s.real_input:
            assert np.array_equal(_read(ds_c, s.mu, 512, torch.float32), ref_ms), (name, q, "mu/sigma tables")
        assert np.array_equal(_read(ds_c, s.d.fsmall, nf, torch.float32), ref_f), (name, q, "deformation grid")
        if ref_b is None:
            assert not s.bfsmall
        else:
            assert np.array_equal(_read(ds_c, s.bfsmall, s.bs[0] * s.bs[1] * s.bs[2], torch.float32), ref_b), (name, q)


@pytest.mark.parametrize("name", CASES)
def test_replayed_native_chain_matches_oracle(name):
    item, orc = oracle_case(name)
    got, ds, draws = cuda_case(name, orc.log, planner='native')
    assert draws.done()
    assert ds.last_deform["_plan"].bbox_host() == orc.deform["lo"] + orc.deform["hi"]
    rep = _compare(mg.flatten(item), mg.flatten(got), name)
    for k, v in rep.items():
        if "bias_field_log" in k:
            assert v == 0.0, (k, v)


def test_replayed_native_brainid_matches_oracle():
    name = "g64_brainid_s6"
    item, orc = oracle_case(name)
    got, ds, draws = cuda_case(name, orc.log, dataset_option=None, planner='native')
    assert draws.done()
    assert isinstance(got[4], list) and len(got[4]) == 3
    _compare(mg.flatten(item), mg.flatten(got), name)


def _native_dataset(batch=4, size=64):
    import bench
    from brainfm_b200 import io as bio
    bio.clear_registry()
    old = bench.SIZE
    bench.SIZE = size
    try:
        ds = bench.build_dataset(bench.make_inputs(batch), torch.device("cuda", 0))
    finally:
        bench.SIZE = old
    return ds


def test_native_mode_is_deterministic_and_sane():
    ds = _native_dataset()
    assert ds._native_planner([0, 1, 2, 3]) is not None, "bench configuration must be planned natively"
    outs = []
    for rep in range(2):
        np.random.seed(11)
        ds._native.seed, ds._native.counter = None, 0
        items = ds.generate_batch([0, 1, 2, 3])
        torch.cuda.synchronize()
        outs.append([to_np(it[4]['input']) for it in items])
        for it in items:
            x = it[4]['input']
            assert x.shape == (1, 64, 64, 64)
            assert torch.isfinite(x).all() and float(x.min()) >= 0 and abs(float(x.max()) - 1) < 1e-6
            t1 = it[3]['T1']
            assert torch.isfinite(t1).all() and float(t1.min()) >= 0 and float(t1.max()) <= 1 + 1e-6
            assert torch.isfinite(it[4]['bias_field_log']).all()
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
    # different items of one batch differ
    assert not np.array_equal(outs[0][0], outs[0][1])


def test_native_matches_python_planner_statistics():
    """Same distributions: photo / flip / resolution-class frequencies and parameter ranges over many plans."""
    ds = _native_dataset(batch=8)
    ds._native_planner(list(range(8)))
    np.random.seed(3)
    photo = flip = n = 0
    gam, nz, lowz = [], [], 0
    for rep in range(40):
        ds.generate_batch(list(range(8)))
        last = ds._native.last
        for q in range(8):
            inf, s = last['info'][q], last['descs'][q]
            photo += inf.photo_mode
            flip += inf.flip
            gam.append(s.gamma)
            nz.append(s.noise_std)
            lowz += int(list(s.new_size) != [64, 64, 64])
            n += 1
            A = np.array(inf.A[:]).reshape(3, 3)
            assert 0.5 < abs(np.linalg.det(A)) < 1.8
    torch.cuda.synchronize()
    assert abs(photo / n - 0.2) < 0.08                      # photo_prob 0.2
    assert abs(flip / n - 0.6915) < 0.09                    # P(N(0,1) < 0.5)
    assert 0.55 < lowz / n < 0.95                           # 1 - 0.8 * 0.25 = 0.8 of the samples are degraded
    assert 0.7 < min(gam) and max(gam) < 1.5 and abs(np.mean(np.log(gam))) < 0.03
    assert 5.0 <= min(nz) and max(nz) <= 15.0


def test_native_mode_draws_real_inputs():
    """modality_probs T1 = 0.5 (the reference's default table has real-image inputs for every dataset): the library
    planner draws the input mode per item; real and synthetic samples share one batched launch."""
    import bench
    from brainfm_b200 import io as bio
    from brainfm_b200.Generator import BaseGen
    bio.clear_registry()
    old = bench.SIZE
    bench.SIZE = 64
    try:
        import tempfile, os
        subs = bench.make_inputs(4)
        root = tempfile.mkdtemp(prefix="bfm_mix_")
        names = []
        for s, v in enumerate(subs):
            stem = os.path.join(root, "HCP.sub%02d." % s)
            bio.register_volume(stem + "T1w.nii", v["T1"])
            bio.register_volume(stem + "generation_labels.nii", v["Gen"])
            names.append(stem + "T1w.nii")
        with open(os.path.join(root, "train.txt"), "w") as f:
            f.write("\n".join(names) + "\n")
        cfg = bench.bench_cfg()
        cfg.split_root = root
        cfg.modality_probs.HCP.T1 = 0.5
        ds = BaseGen(cfg, "cuda", planner='native')
    finally:
        bench.SIZE = old
    np.random.seed(5)
    modes = []
    for rep in range(12):
        items = ds.generate_batch([0, 1, 2, 3])
        for it in items:
            modes.append(it[2])
            x = it[4]['input']
            assert torch.isfinite(x).all() and float(x.min()) >= 0 and abs(float(x.max()) - 1) < 1e-6
        descs = ds._native.last['descs']
        for q, it in enumerate(items):
            assert descs[q].real_input == (1 if it[2] == 'T1' else 0)
    assert set(modes) == {'synth', 'T1'}
    assert 0.25 < modes.count('T1') / len(modes) < 0.75


def test_native_planner_follows_changed_gen_args():
    """The cached bfm_plan_cfg is rebuilt when the caller changes generator parameters between batches."""
    ds = _native_dataset()
    np.random.seed(2)
    ds.generate_batch([0, 1, 2, 3])
    assert any(ds._native.last['descs'][q].gamma != 1.0 for q in range(4))
    ds.gen_args.generator.gamma_std = 0.0
    ds.gen_args.generator.flip_prob = -100.0          # randn() < -100 never holds
    ds.generate_batch([0, 1, 2, 3])
    torch.cuda.synchronize()
    for q in range(4):
        assert ds._native.last['descs'][q].gamma == 1.0 and ds._native.last['descs'][q].flip == 0
