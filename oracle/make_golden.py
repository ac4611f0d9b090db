"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, through oracle/ref_shim.py) in the build container, and checks the oracle
restatement (oracle/gen_oracle.py) against it on the spot.

    python -m oracle.make_golden            # from the repo root, build container only

Fixtures hold strided sub-samples of every output volume plus full-volume float64 sums, maxima and
the integer side results (bounding box, low-res size), and the library versions that produced them.
"""
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shim as rs                      # noqa: E402
from oracle import gen_oracle as go                    # noqa: E402
from tests import _inputs as ti                        # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def sub(a, stride):
    a = np.asarray(a)
    sl = tuple(slice(None, None, stride) if n > 8 else slice(None) for n in a.shape)
    return np.ascontiguousarray(a[sl])


def summarise(name, t, stride, out):
    a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    if a.ndim == 4 and a.shape[0] == 56 and np.all((a == 0) | (a == 1)) and np.all(a.sum(0) == 1):
        a = a.argmax(0).astype(np.uint8)           # hard one-hot -> label index (lossless)
        name = name + ".argmax"
    elif a.ndim == 4 and a.shape[0] == 56:         # deform_one_hots: linearly warped (soft) one-hots
        stride = 2 * stride
    out[name + ".sub"] = sub(a, stride)
    out[name + ".sum"] = np.float64(a.astype(np.float64).sum())
    out[name + ".max"] = np.float64(a.max())
    out[name + ".shape"] = np.array(a.shape)


CASES = {
    # name: (size, source shape, label kind, seed, cfg overrides, extra volumes, dataset_option, stride)
    "g64_s0": (64, 96, "block", 0, {}, [], "default", 2),
    "g64_s1": (64, 96, "block", 1, {}, [], "default", 2),
    "g64_s2": (64, 96, "brain", 2, {}, [], "default", 2),
    "g64_s3": (64, 96, "brain", 3, {}, [], "default", 2),
    "g64_s5_lowres": (64, 96, "brain", 5, {"generator.low_res_only": True}, [], "default", 2),
    "g64_full_s4": (64, 96, "brain", 4, {"mix_synth_prob": 1.0, "task.T1": True, "task.T2": True, "task.CT": True,
                                         "task.segmentation": True, "task.distance": True,
                                         "task.registration": True, "task.super_resolution": True},
                    ["T2", "CT", "distance", "registration"], "default", 2),
    "g64_brainid_s6": (64, 96, "brain", 6, {"generator.all_samples": 3, "generator.mild_samples": 1}, [],
                       "brain_id", 2),
    "g160_s0": (160, 192, "brain", 0, {}, [], "default", 4),
    # undegraded resolution class (identity band + identity zoom), no flip, with the super-resolution residual
    "g64_ident_s23": (64, 96, "brain", 23, {"task.super_resolution": True}, [], "default", 2),
    # real-image inputs (read_input draws the modality): T1 with the default tasks, T2 with every image target
    "g64_realT1_s14": (64, 96, "brain", 14, {"modality_probs.HCP.T1": 1.0, "task.super_resolution": True}, [],
                       "default", 2),
    "g64_realT2_s15": (64, 96, "brain", 15, {"modality_probs.HCP.T2": 1.0, "task.T1": True, "task.T2": True},
                       ["T2"], "default", 2),
    "g64_realCT_s16": (64, 96, "brain", 16, {"modality_probs.HCP.CT": 1.0, "task.CT": True}, ["CT"], "default", 2),
    # left hemisphere only: photo mode forced, no flip, source masked by (left label) & (MNI x < 0), left label list
    "g64_left_s9": (64, 96, "brain", 9, {"generator.left_hemis_only": True, "task.segmentation": True,
                                         "task.distance": True, "task.registration": True},
                    ["distance", "mni"], "default", 2),
    # pathology: random Perlin shape encoded into the synthetic image.  The reference's branch only runs when the
    # crop covers the whole output shape (datasets.py:391-398 index the deformed image with crop-shaped masks),
    # hence source shape == output shape here.
    "g64_pathol_s7": (64, 64, "brain", 7, {"task.pathology": True, "generator.pathology_prob": 1.0,
                                           "generator.random_shape_prob": 1.0}, [], "default", 2),
    "g64_pathol_s12": (64, 64, "brain", 12, {"task.pathology": True, "generator.pathology_prob": 1.0,
                                             "generator.random_shape_prob": 1.0}, [], "default", 2),
    # ---- round 2: branches that were built but unpinned (VERDICT r1 weak 1-2)
    # 'surface' task: SVF scaling-and-squaring of the nonlinear field (datasets.py:214-223), F / Fneg full-resolution,
    # full bbox scan, k_gen_warp FIELD == 2
    "g64_svf_s31": (64, 96, "brain", 31, {"task.surface": True}, [], "default", 2),
    "g64_svf_s41": (64, 96, "brain", 41, {"task.surface": True}, [], "default", 2),          # photo mode + flip
    # one-hot segmentation warped linearly (utils.py:404-416)
    "g64_onehot_s43": (64, 96, "brain", 43, {"task.segmentation": True, "generator.deform_one_hots": True}, [],
                       "default", 2),
    "g64_onehot_s41": (64, 96, "brain", 41, {"task.segmentation": True, "generator.deform_one_hots": True}, [],
                       "default", 2),                                                          # photo mode + flip
    # cubic B-spline zoom back to the grid (datasets.py:337-340, interpol.resize)
    "g64_bspline_s43": (64, 96, "brain", 43, {"generator.bspline_zooming": True}, [], "default", 2),
    "g64_bspline_s41": (64, 96, "brain", 41, {"generator.bspline_zooming": True}, [], "default", 2),
    # random centre shift (datasets.py:195-200)
    "g64_shift_s43": (64, 96, "brain", 43, {"generator.random_shift": True}, [], "default", 2),
    # CT-like contrast groups (datasets.py:349, get_contrast)
    "g64_ct_s35": (64, 96, "brain", 35, {"generator.ct_prob": 1.0}, [], "default", 2),
    # pathology shape advected by the ShapeID PDE inside the chain (utils.py:514-522)
    "g64_augpath_s47": (64, 64, "brain", 47, {"task.pathology": True, "generator.pathology_prob": 1.0,
                                              "generator.random_shape_prob": 1.0,
                                              "generator.augment_pathology": True}, [], "default", 2),
    "g64_augpath_s48": (64, 64, "brain", 48, {"task.pathology": True, "generator.pathology_prob": 1.0,
                                              "generator.random_shape_prob": 1.0,
                                              "generator.augment_pathology": True}, [], "default", 2),
}


def shape3(n):
    """An int means a cube; a 3-tuple is taken as (x, y, z)."""
    return tuple(int(v) for v in n) if isinstance(n, (tuple, list)) else (int(n),) * 3


def build_volumes(src, kind, extra):
    shp = shape3(src)
    lab = ti.block_labels(shp) if kind == "block" else ti.brain_like_labels(shp)
    vols = {"Gen": lab, "T1": ti.smooth_image(shp, 0.0), "segmentation": ti.seg_labels(shp)}
    if "T2" in extra:
        vols["T2"] = ti.smooth_image(shp, 1.0)
    if "CT" in extra:
        vols["CT"] = ti.smooth_image(shp, 2.0) * 8 - 500
    if "distance" in extra:
        vols["distance"] = [ti.smooth_image(shp, 0.3 * i) for i in range(4)]
    if "registration" in extra:
        vols["registration"] = [ti.smooth_image(shp, 0.7 * i) * 50 for i in range(3)]
    if "mni" in extra:           # signed MNI-like coordinates: x < 0 on one side of a wavy mid-sagittal surface
        ax = [np.arange(n, dtype=np.float32) - (n - 1) / 2 for n in shp]
        base = [ax[0][:, None, None], ax[1][None, :, None], ax[2][None, None, :]]
        wob = [ti.smooth_image(shp, 0.7 * i) for i in range(3)]
        vols["registration"] = [(base[i] + 3 * (wob[i] - wob[i].mean()) / wob[i].std()).astype(np.float32)
                                for i in range(3)]
    return vols


def cfg_for(size, over, option, ref):
    if ref:
        args = rs.load_generator_cfg()
        base = ti.default_cfg(shape3(size))
        for k, v in vars(base.task).items():
            setattr(args.task, k, v)
        args.generator.size = list(shape3(size))
        args.mix_synth_prob = 0.0
        args.dataset_names = ["HCP"]
        args.modality_probs.HCP = ti.ns(T1=0., T2=0., FLAIR=0., CT=0., synth=1.)
    else:
        args = ti.default_cfg(shape3(size))
    args.dataset_option = option
    for k, v in over.items():
        node = args
        parts = k.split(".")
        for p in parts[:-1]:
            node = getattr(node, p)
        setattr(node, parts[-1], v)
    return args


def run_reference(name):
    size, src, kind, seed, over, extra, option, stride = CASES[name]
    rs.install()
    import Generator
    vols = build_volumes(src, kind, extra)
    files = {"T1w": vols["T1"], "generation_labels": vols["Gen"], "brainseg_with_extracerebral": vols["segmentation"]}
    if "T2" in vols:
        files["T2w"] = vols["T2"]
    if "CT" in vols:
        files["CT"] = vols["CT"]
    if "distance" in vols:
        for k, v in zip(["lp_dist_map", "lw_dist_map", "rp_dist_map", "rw_dist_map"], vols["distance"]):
            files[k] = v
    if "registration" in vols:
        for k, v in zip(["mni_reg.x", "mni_reg.y", "mni_reg.z"], vols["registration"]):
            files[k] = v
    root, t1 = rs.make_subject(files)
    # get_info() gates T2 / CT on os.path.isfile (datasets.py:547-560): create empty marker files
    for suffix in ("T2w", "CT"):
        if suffix in files:
            open(os.path.join(root, "HCP.sub01.%s.nii" % suffix), "w").close()
    args = cfg_for(size, over, option, ref=True)
    args.split_root = root
    ds = Generator.build_datasets(args, "cpu")["all"]
    # keep the reference's deformation dict (F / Fneg of the 'surface' task are not part of the item)
    inner = ds.generate_deformation

    def keep(*a, **k):
        ds.last_deform = inner(*a, **k)
        return ds.last_deform
    ds.generate_deformation = keep
    go.seed_all(seed)
    return ds[0], ds


def run_oracle(name):
    """name: a key of CASES or a case tuple of the same layout."""
    size, src, kind, seed, over, extra, option, stride = CASES[name] if isinstance(name, str) else name
    vols = build_volumes(src, kind, extra)
    args = cfg_for(size, over, option, ref=False)
    orc = go.GeneratorOracle(args, vols, brain_id=(option == "brain_id"))
    go.seed_all(seed)
    return orc.sample(), orc


def flatten(item):
    _, dsname, mode, target, sample = item
    out = {}
    for k, v in target.items():
        if isinstance(v, torch.Tensor):
            out["target." + k] = v
        elif k != "name":
            out["target." + k] = np.float64(v)
    samples = sample if isinstance(sample, list) else [sample]
    for i, s in enumerate(samples):
        for k, v in s.items():
            out["sample%d.%s" % (i, k)] = v
    return out


def compare(ref, orc, name):
    worst = 0.0
    assert set(ref) == set(orc), (name, sorted(set(ref) ^ set(orc)))
    for k in ref:
        a, b = ref[k], orc[k]
        if isinstance(a, torch.Tensor):
            a, b = a.numpy(), b.numpy()
            assert a.shape == b.shape, (name, k, a.shape, b.shape)
            if not np.array_equal(a, b):
                d = float(np.abs(a.astype(np.float64) - b).max())
                worst = max(worst, d)
                print("   %-28s max|diff| %.3e (n_diff=%d)" % (k, d, int((a != b).sum())))
        else:
            assert float(a) == float(b), (name, k, a, b)
    return worst


def main(argv):
    names = argv or list(CASES)
    os.makedirs(GOLD, exist_ok=True)
    for name in names:
        stride = CASES[name][-1]
        item, ds = run_reference(name)
        ref = flatten(item)
        (oitem, orc) = run_oracle(name)
        worst = compare(ref, flatten(oitem), name)
        out = {}
        for k, v in ref.items():
            if isinstance(v, torch.Tensor):
                summarise(k, v, stride, out)
            else:
                out[k] = v
        out["meta.bbox"] = np.array(orc.deform["lo"] + orc.deform["hi"])
        rd = getattr(ds, "last_deform", None)
        if rd is not None and rd.get("Fneg") is not None:       # integrated fields: reference values, oracle checked
            for key in ("F", "Fneg"):
                a, b = rd[key].numpy(), orc.deform[key].numpy()
                assert np.array_equal(a, b), (name, key, float(np.abs(a - b).max()))
                summarise("deform." + key, rd[key], stride, out)
            g = [int(v) for v in rd["grid"][3:]]
            assert g == [g[0], g[1], g[2], g[3], g[4], g[5]] and \
                [g[0], g[1], g[2]] == list(orc.deform["lo"]) and [g[3], g[4], g[5]] == list(orc.deform["hi"]), (g, orc.deform["lo"])
        out["meta.factors"] = np.asarray(orc.aux["factors"])
        out["meta.flip"] = np.array(bool(orc.setups["flip"]))
        out["meta.photo"] = np.array(bool(orc.setups["photo_mode"]))
        out["meta.stride"] = np.array(stride)
        out["meta.versions"] = np.array("torch %s numpy %s" % (torch.__version__, np.__version__))
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
        print("%-16s oracle-vs-reference worst |diff| = %.3e   keys=%d  flip=%s photo=%s factors=%s" % (
            name, worst, len(ref), orc.setups["flip"], orc.setups["photo_mode"], np.round(orc.aux["factors"], 3)))


if __name__ == "__main__":
    main(sys.argv[1:])
