"""brainfm_b200.io readers (nib.load replacement, Generator/utils.py:296-305): NIfTI-1 and MGH / MGZ files written here
byte by byte from the formats' specifications, the reference's shipped files/gca.mgz when a checkout of the original
project is named by BFM_REFERENCE_ROOT, and the committed benchmark label map derived from it."""
import gzip
import os
import struct

import numpy as np
import pytest

from brainfm_b200 import io as bio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GCA = os.path.join(os.environ.get("BFM_REFERENCE_ROOT", ""), "files", "gca.mgz")


def _nifti_bytes(data, endian="<", slope=0.0, inter=0.0, sform=None, pixdim=(1.0, 1.0, 1.0)):
    code = {np.dtype("u1"): 2, np.dtype("i2"): 4, np.dtype("i4"): 8, np.dtype("f4"): 16, np.dtype("f8"): 64,
            np.dtype("i1"): 256, np.dtype("u2"): 512}[data.dtype]
    hdr = bytearray(352)
    struct.pack_into(endian + "i", hdr, 0, 348)
    dim = [data.ndim] + list(data.shape) + [1] * (7 - data.ndim)
    struct.pack_into(endian + "8h", hdr, 40, *dim)
    struct.pack_into(endian + "h", hdr, 70, code)
    struct.pack_into(endian + "h", hdr, 72, 8 * data.dtype.itemsize)
    struct.pack_into(endian + "8f", hdr, 76, 1.0, *pixdim, 0, 0, 0, 0)
    struct.pack_into(endian + "f", hdr, 108, 352.0)
    struct.pack_into(endian + "2f", hdr, 112, slope, inter)
    if sform is not None:
        struct.pack_into(endian + "h", hdr, 254, 1)
        struct.pack_into(endian + "12f", hdr, 280, *np.asarray(sform, dtype=np.float32)[:3].reshape(-1))
    hdr[344:348] = b"n+1\0"
    return bytes(hdr) + data.astype(data.dtype.newbyteorder(endian)).tobytes(order="F")


def _mgh_bytes(data):
    typ = {np.dtype("u1"): 0, np.dtype("i4"): 1, np.dtype("f4"): 3, np.dtype("i2"): 4}[data.dtype]
    w, h, d = data.shape[:3]
    nf = data.shape[3] if data.ndim == 4 else 1
    hdr = bytearray(284)
    struct.pack_into(">7i", hdr, 0, 1, w, h, d, nf, typ, 0)
    return bytes(hdr) + data.astype(data.dtype.newbyteorder(">")).tobytes(order="F")


@pytest.mark.parametrize("dtype", ["u1", "i2", "i4", "f4", "f8", "u2"])
@pytest.mark.parametrize("endian", ["<", ">"])
def test_nifti_reader(tmp_path, dtype, endian):
    rng = np.random.RandomState(3)
    a = (rng.rand(5, 7, 6) * 100).astype(dtype)
    aff = np.array([[0.0, -1.5, 0, 10], [2.0, 0, 0, -3], [0, 0, 1.25, 7], [0, 0, 0, 1]])
    p = str(tmp_path / "v.nii")
    open(p, "wb").write(_nifti_bytes(a, endian, sform=aff))
    v = bio.load(p)
    assert np.array_equal(np.asarray(v.get_fdata()), a.astype(np.float64))
    np.testing.assert_allclose(v.affine, aff, rtol=1e-6)


def test_nifti_gz_scaling_and_pixdim(tmp_path):
    a = np.arange(4 * 3 * 2, dtype=np.int16).reshape(4, 3, 2)
    p = str(tmp_path / "s.nii.gz")
    with gzip.open(p, "wb") as f:
        f.write(_nifti_bytes(a, slope=2.0, inter=1.0, pixdim=(0.5, 2.0, 3.0)))
    v = bio.load(p)
    assert np.array_equal(np.asarray(v.get_fdata()), a * 2.0 + 1.0)
    assert np.allclose(np.diag(v.affine), [0.5, 2.0, 3.0, 1.0])
    # the reference's retry: the path without '.gz' resolves to the gzipped file (Generator/utils.py:299-302)
    assert np.array_equal(np.asarray(bio.load(p[:-3]).get_fdata()), a * 2.0 + 1.0)
    with pytest.raises(FileNotFoundError):
        bio.load(str(tmp_path / "missing.nii"))


@pytest.mark.parametrize("dtype", ["u1", "i4", "f4", "i2"])
def test_mgh_reader(tmp_path, dtype):
    rng = np.random.RandomState(5)
    a = (rng.rand(6, 4, 5) * 200).astype(dtype)
    p = str(tmp_path / "v.mgh")
    open(p, "wb").write(_mgh_bytes(a))
    assert np.array_equal(np.asarray(bio.load(p).get_fdata()), a.astype(np.float64))
    pz = str(tmp_path / "v.mgz")
    with gzip.open(pz, "wb") as f:
        f.write(_mgh_bytes(a))
    assert np.array_equal(np.asarray(bio.load(pz).get_fdata()), a.astype(np.float64))
    frames = (rng.rand(3, 4, 5, 2) * 50).astype(dtype)
    open(p, "wb").write(_mgh_bytes(frames))
    assert np.array_equal(np.asarray(bio.load(p).get_fdata()), frames.astype(np.float64))


def test_registry_takes_precedence(tmp_path):
    a = np.ones((2, 2, 2), dtype=np.float32)
    bio.register_volume("/nowhere/x.nii", a)
    try:
        assert bio.exists("/nowhere/x.nii") and np.array_equal(np.asarray(bio.load("/nowhere/x.nii").get_fdata()), a)
    finally:
        bio.clear_registry()
    assert not bio.exists("/nowhere/x.nii")


def test_benchmark_label_map_fixture():
    """The committed bench label map: 160^3 uint8, the documented checksum, values < 256 as the 256-entry LUT needs."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "atlas_gca_L160_u8.npz"))
    L = z["L160"]
    assert L.shape == (160, 160, 160) and L.dtype == np.uint8
    assert int(L.astype(np.int64).sum()) == int(z["checksum"][0])
    assert 0.5 < (L > 0).mean() < 0.6 and L.max() == 233


@pytest.mark.skipif(not os.environ.get("BFM_REFERENCE_ROOT") or not os.path.exists(GCA),
                    reason="no checkout of the original project (set BFM_REFERENCE_ROOT)")
def test_reference_atlas_and_the_fixture_derived_from_it():
    """files/gca.mgz, the only real volume the reference ships (SURVEY.md 2.1 row 20): 256^3, integer valued 0..233,
    non-zero bounding box 152 x 176 x 184; the committed fixture is the documented crop of it."""
    a = np.asarray(bio.load(GCA).get_fdata())
    assert a.shape == (256, 256, 256) and a.min() == 0 and a.max() == 233 and np.all(a == np.round(a))
    nz = np.nonzero(a)
    assert [int(x.max()) + 1 - int(x.min()) for x in nz] == [152, 176, 184]
    z = np.load(os.path.join(ROOT, "tests", "golden", "atlas_gca_L160_u8.npz"))
    o = [int(v) for v in z["origin"]]
    assert np.array_equal(z["L160"], a[o[0]:o[0] + 160, o[1]:o[1] + 160, o[2]:o[2] + 160].astype(np.uint8))
