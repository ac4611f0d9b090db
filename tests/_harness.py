"""Shared helpers of the GPU parity tests: run the oracle on a named case, then feed its recorded draws to
the CUDA generator."""
import os
import tempfile

import numpy as np
import torch

from oracle import gen_oracle as go
from oracle import make_golden as mg

RTOL, ATOL = 1e-5, 1e-4


def _case(case):
    """A key of make_golden.CASES or a case tuple of the same layout (sizes: int = cube, or 3-tuple)."""
    return mg.CASES[case] if isinstance(case, str) else tuple(case)


def oracle_case(name):
    (item, orc) = mg.run_oracle(name)
    return item, orc


def oracle_batch(case, srcs, indices):
    """One oracle per item of a batch, drawn after ONE seed_all in item order (what generate_batch does): item n
    uses subject indices[n], whose source shape is srcs[indices[n]].  Returns the items, the oracles and the
    concatenated draw log."""
    size, src, kind, seed, over, extra, option, stride = _case(case)
    args = mg.cfg_for(size, over, option, ref=False)
    orcs = [go.GeneratorOracle(args, mg.build_volumes(srcs[i], kind, extra), case_name="HCP.sub%02d" % (i + 1),
                               brain_id=(option == "brain_id")) for i in indices]
    go.seed_all(seed)
    items = [o.sample() for o in orcs]
    return items, orcs, [e for o in orcs for e in o.log]


def cuda_case(name, log, dataset_option=None, run=None, planner='auto', srcs=None):
    """The CUDA generator with the draws of `log` replayed (None: the generator's own draws).  srcs: source shapes of the registered subjects
    HCP.sub01, HCP.sub02, ... (default: the case's one source); `run(ds)` replaces ds[0]."""
    from brainfm_b200 import io as bio
    from brainfm_b200.draws import ReplayDraws
    from brainfm_b200.Generator import dataset_options
    size, src, kind, seed, over, extra, option, stride = _case(name)
    root = tempfile.mkdtemp(prefix="bfm_case_")
    bio.clear_registry()
    t1s = []
    for k, shape in enumerate(srcs or [src]):
        vols = mg.build_volumes(shape, kind, extra)
        stem = os.path.join(root, "HCP.sub%02d." % (k + 1))
        bio.register_volume(stem + "T1w.nii", vols["T1"])
        bio.register_volume(stem + "generation_labels.nii", vols["Gen"])
        bio.register_volume(stem + "brainseg_with_extracerebral.nii", vols["segmentation"])
        if "T2" in vols:
            bio.register_volume(stem + "T2w.nii", vols["T2"])
        if "CT" in vols:
            bio.register_volume(stem + "CT.nii", vols["CT"])
        if "distance" in vols:
            for key, v in zip(["lp_dist_map", "lw_dist_map", "rp_dist_map", "rw_dist_map"], vols["distance"]):
                bio.register_volume(stem + key + ".nii", v)
        if "registration" in vols:
            for key, v in zip(["mni_reg.x", "mni_reg.y", "mni_reg.z"], vols["registration"]):
                bio.register_volume(stem + key + ".nii", v)
        t1s.append(stem + "T1w.nii")
    with open(os.path.join(root, "train.txt"), "w") as f:
        f.write("".join(t + "\n" for t in t1s))
    args = mg.cfg_for(size, over, option, ref=False)
    args.split_root = root
    draws = ReplayDraws(log) if log is not None else None
    ds = dataset_options[dataset_option or option](args, "cuda", draws=draws, planner=planner)
    item = ds[0] if run is None else run(ds)
    torch.cuda.synchronize()
    return item, ds, draws


def to_np(v):
    return v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)


def compare(ref, got, name):
    """Flattened items (make_golden.flatten): scalars and one-hot segmentations bit-exact, every other volume within
    RTOL / ATOL.  Returns the largest absolute difference per key."""
    assert set(ref) == set(got), (name, sorted(set(ref) ^ set(got)))
    report = {}
    for k, a in ref.items():
        b = got[k]
        if not isinstance(a, torch.Tensor):
            assert float(a) == float(b), (name, k)
            continue
        a, b = to_np(a), to_np(b)
        assert a.shape == b.shape, (name, k, a.shape, b.shape)
        if "segmentation" in k and np.all((a == 0) | (a == 1)):
            assert np.array_equal(a, b), "%s %s: one-hot differs in %d voxels" % (name, k, int((a != b).sum()))
        else:
            np.testing.assert_allclose(b, a, rtol=RTOL, atol=ATOL, err_msg="%s %s" % (name, k))
        report[k] = float(np.abs(a.astype(np.float64) - b).max())
    return report
