"""Per-voxel primitives, target readers and augmentation operators of the generator -- same names,
arguments and error behaviour as the reference's Generator/utils.py, computed by libbfm (sm_100a CUDA).

All tensors must live on a CUDA device: there is no CPU implementation in this package."""
import ctypes as C

import numpy as np
import torch

from .. import _lib, io as bio
from ..draws import HostDraws
from ..plan import (band_host, device_tables, gaussian_taps_host, make_deform, zoom_newsize, zoom_tables_host)

_DRAWS = HostDraws()


def _stream():
    # raw handle of torch's current stream on the current device (torch.cuda.current_stream() builds a Stream object
    # and costs ~15 us per call, which adds up on the per-batch host path)
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


def scratch_stride(N):
    """Floats per sample slot of the fused chain's scratch (i_bf, tmp, lowres, aux_raw): N rounded up to a multiple of
    4, so that every slot keeps the 16-byte alignment the 128-bit kernel paths need (include/bfm.h)."""
    return (int(N) + 3) // 4 * 4


def syn_stride(src):
    """Floats per sample slot of the fused chain's `syn` scratch for a label map of shape `src`: float2 {synthetic,
    target} pairs (bfm_gen_sample.syn_pair_ok) over the source volume with the volume cache's padding
    (DeviceVolumeCache._pad), the volume rounded up to a multiple of 4 floats."""
    s0, s1, s2 = (int(v) for v in src[:3])
    return 2 * ((s0 * s1 * s2 + s1 * s2 + s2 + 1 + 3) // 4 * 4)


def _need_cuda(t, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.BfmError("%s must be a CUDA tensor: brainfm_b200 has no CPU path" % what)


def pack_to_device(arrays, device):
    """Concatenate small host arrays into one device byte buffer (one H2D copy); returns (buffer, addresses)."""
    offs, total = [], 0
    for a in arrays:
        total = (total + 15) // 16 * 16
        offs.append(total)
        total += a.nbytes
    host = np.zeros(max(total, 16), dtype=np.uint8)
    for a, o in zip(arrays, offs):
        host[o:o + a.nbytes] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    dev = torch.from_numpy(host).to(device)
    base = dev.data_ptr()
    return dev, [base + o for o in offs]


class _MiniArena:
    """plan.Arena-compatible packer for a single plan that owns its tables: device addresses are known up
    front (fixed-capacity device buffer), the host image is uploaded once by finalize()."""

    def __init__(self, device, capacity=1 << 20):
        self.host = np.zeros(capacity, dtype=np.uint8)
        self.dev = torch.empty(capacity, dtype=torch.uint8, device=device)
        self.base = self.dev.data_ptr()
        self.used = 0

    def put(self, arr):
        a = np.ascontiguousarray(arr)
        off = (self.used + 15) // 16 * 16
        if off + a.nbytes > self.host.size:
            raise MemoryError("deformation plan tables exceed the mini arena")
        self.host[off:off + a.nbytes] = a.view(np.uint8).reshape(-1)
        self.used = off + a.nbytes
        return self.base + off

    def finalize(self):
        n = max(self.used, 16)
        self.dev[:n].copy_(torch.from_numpy(self.host[:n]))


# ------------------------------------------------------------------------------------------------
# resolution sampling / small helpers (host)
# ------------------------------------------------------------------------------------------------
def resolution_sampler(low_res_only=False, draws=None):
    """Acquisition resolution and slice thickness (Generator/utils.py:34-57)."""
    rng = draws or _DRAWS
    r = rng.rand("res.class")
    if low_res_only:
        r = r * 0.5 + 0.5
    resolution = np.array([1.0, 1.0, 1.0])
    thickness = np.array([1.0, 1.0, 1.0])
    if r < 0.25:
        pass
    elif r < 0.5:
        idx = rng.randint("res.axis", 3)
        resolution[idx] = 2.5 + 6 * rng.rand("res.u")
        thickness[idx] = np.min([resolution[idx], 4.0 + 2.0 * rng.rand("res.u2")])
    elif r < 0.75:
        resolution = np.array([1.3, 1.3, 4.8]) + 0.4 * rng.rand3("res.u3")
        thickness = resolution.copy()
    else:
        resolution = 2.0 + 3.0 * rng.rand3("res.u3")
        thickness = resolution.copy()
    return resolution, thickness


_AFF = np.zeros((6, 3, 3))                     # SHx SHy SHz Rx Ry Rz templates (unit diagonal filled below)
for _q in range(6):
    _AFF[_q] = np.eye(3)


def make_affine_matrix(rot, sh, s):
    """A = SHx SHy SHz Rx Ry Rz with row i scaled by s[i], float64 (Generator/utils.py:102-116).  Same numpy
    operations as the reference (np.cos/np.sin on the 3-vectors, five BLAS `@` products in the same order, the
    row scaling); only the six factor matrices are written into a preallocated buffer instead of being built
    from nested lists."""
    cr, sr = np.cos(rot).tolist(), np.sin(rot).tolist()
    sh = sh.tolist() if isinstance(sh, np.ndarray) else list(sh)
    m = _AFF
    m[0, 1, 0] = sh[1]; m[0, 2, 0] = sh[2]                                       # SHx
    m[1, 0, 1] = sh[0]; m[1, 2, 1] = sh[2]                                       # SHy
    m[2, 0, 2] = sh[0]; m[2, 1, 2] = sh[1]                                       # SHz
    m[3, 1, 1] = cr[0]; m[3, 1, 2] = -sr[0]; m[3, 2, 1] = sr[0]; m[3, 2, 2] = cr[0]     # Rx
    m[4, 0, 0] = cr[1]; m[4, 0, 2] = sr[1]; m[4, 2, 0] = -sr[1]; m[4, 2, 2] = cr[1]     # Ry
    m[5, 0, 0] = cr[2]; m[5, 0, 1] = -sr[2]; m[5, 1, 0] = sr[2]; m[5, 1, 1] = cr[2]     # Rz
    A = m[0] @ m[1] @ m[2] @ m[3] @ m[4] @ m[5]
    return A * np.asarray(s)[:, None]          # row r scaled by s[r]


def binarize(p, thres):
    """Threshold at thres * max (Generator/utils.py:65-72)."""
    t = thres * p.max()
    return (p >= t).to(p.dtype)


def make_gaussian_kernel(sigma, device):
    """Normalised Gaussian taps on [-ceil(3 sigma), ceil(3 sigma)] (Generator/utils.py:74-81)."""
    taps, _ = gaussian_taps_host(sigma)
    return torch.from_numpy(taps).to(device)


def gaussian_blur_3d(input, stds, device=None):
    """Separable zero-padded Gaussian blur, axes with std == 0 skipped (Generator/utils.py:83-94)."""
    _need_cuda(input, "input")
    x = input.contiguous().float()
    nx, ny, nz = x.shape
    L = _lib.lib()
    for ax in range(3):
        if stds[ax] > 0:
            taps, half = gaussian_taps_host(stds[ax])
            t = torch.from_numpy(taps).to(x.device)
            y = torch.empty_like(x)
            _lib.check(L.bfm_blur_axis(x.data_ptr(), y.data_ptr(), nx, ny, nz, ax, t.data_ptr(), half, _stream()))
            x = y
    return torch.squeeze(x)


# ------------------------------------------------------------------------------------------------
# samplers
# ------------------------------------------------------------------------------------------------
def fast_3D_interp_torch(X, II, JJ, KK, mode='linear', default_value_linear=0.0):
    """Trilinear / nearest sampling of X at voxel coordinates (Generator/utils.py:119-196)."""
    if II is None:
        return X
    if mode not in ('linear', 'nearest'):
        raise Exception('mode must be linear or nearest')
    _need_cuda(X, "X")
    L = _lib.lib()
    X4 = X if X.dim() == 4 else X[..., None]
    nx, ny, nz, Cn = X4.shape
    I = II.contiguous().float()
    J = JJ.contiguous().float()
    K = KK.contiguous().float()
    n = I.numel()
    if mode == 'nearest':
        Xc = X4.contiguous()
        out = torch.empty((*II.shape, Cn), dtype=X.dtype, device=X.device)
        _lib.check(L.bfm_nearest_pull(Xc.data_ptr(), Xc.element_size(), nx, ny, nz, Cn, I.data_ptr(), J.data_ptr(),
                                      K.data_ptr(), n, out.data_ptr(), _stream()))
    else:
        Xc = X4.contiguous().float()
        out = torch.empty((*II.shape, Cn), dtype=torch.float32, device=X.device)
        dptr, dval = None, 0.0
        if isinstance(default_value_linear, torch.Tensor):
            dflt = default_value_linear.to(device=X.device, dtype=torch.float32).reshape(1)
            dptr = dflt.data_ptr()
        else:
            dval = float(default_value_linear)
        _lib.check(L.bfm_trilerp_pull(Xc.data_ptr(), nx, ny, nz, Cn, I.data_ptr(), J.data_ptr(), K.data_ptr(), n,
                                      dval, dptr, out.data_ptr(), _stream()))
    return out[..., 0] if Cn == 1 else out


def myzoom_torch(X, factor, aff=None):
    """Separable linear zoom with edge clamp (Generator/utils.py:200-257)."""
    _need_cuda(X, "X")
    L = _lib.lib()
    X4 = (X if X.dim() == 4 else X[..., None]).contiguous().float()
    a, b, c, Cn = X4.shape
    factor = np.asarray(factor, dtype=np.float64) * np.ones(3)
    new = zoom_newsize((a, b, c), factor)
    tabs = [zoom_tables_host((a, b, c)[d], factor[d], int(new[d])) for d in range(3)]
    flat = [t for tab in tabs for t in tab]
    keep, addr = pack_to_device(flat, X.device)
    out = torch.empty((int(new[0]), int(new[1]), int(new[2]), Cn), dtype=torch.float32, device=X.device)
    args = [X4.data_ptr(), a, b, c, Cn]
    for d in range(3):
        args += [addr[4 * d], addr[4 * d + 1], addr[4 * d + 2], addr[4 * d + 3], int(new[d])]
    _lib.check(L.bfm_zoom_linear(*args, out.data_ptr(), _stream()))
    Y = out[..., 0] if Cn == 1 else out
    if aff is not None:
        aff_new = aff.copy()
        aff_new[:-1] = aff_new[:-1] / factor
        aff_new[:-1, -1] = aff_new[:-1, -1] - aff[:-1, :-1] @ (0.5 - 0.5 / (factor * np.ones(3)))
        return Y, aff_new
    return Y


# ------------------------------------------------------------------------------------------------
# deformation plan (what deform_dict carries besides the reference's keys)
# ------------------------------------------------------------------------------------------------
class DeformPlan:
    """Device-side description of one random deformation: affine + small nonlinear grid + zoom tables +
    the bounding box of the deformed grid in the source volume.  Owns its device buffers."""

    def __init__(self, size, src, A, c2, fsmall_host, photo, device, F_full=None, arena=None, lazy=False,
                 fsmall_dev=None):
        self.size = [int(v) for v in size]
        self.src = [int(v) for v in src[:3]]
        self.device = torch.device(device)
        self.A_host = np.asarray(A, dtype=np.float32)
        self.c2_host = np.asarray(c2, dtype=np.float32)
        self.photo = bool(photo)
        self.F_full = F_full
        fptr = F_full.data_ptr() if F_full is not None else None
        if fsmall_host is not None:
            fsmall_host = np.ascontiguousarray(fsmall_host, dtype=np.float32)
        tables = device_tables(self.device)
        self._arena, self._bbox = None, None
        if arena is not None:
            # the small grid lives in the caller's arena slot: valid until that slot is recycled
            self.struct = make_deform(tables, arena, self.size, self.src, self.A_host, self.c2_host, fsmall_host,
                                      photo, fptr, fsmall_dev=fsmall_dev)
            self.bbox_ptr, self._bbox_off = arena.reserve(32)
            self._arena, self._slot = arena, arena.cur
        else:
            ar = _MiniArena(self.device)
            self.struct = make_deform(tables, ar, self.size, self.src, self.A_host, self.c2_host, fsmall_host,
                                      photo, fptr)
            ar.finalize()
            self._keep = ar.dev
            self._bbox = torch.empty(8, dtype=torch.int32, device=self.device)
            self.bbox_ptr = self._bbox.data_ptr()
        self._bbox_host = None
        self.have_bbox = False
        if not lazy:
            if arena is not None:
                arena.commit()
            self.compute_bbox()

    @property
    def bbox(self):
        """Device tensor view of the 6 bounding-box ints (+2 of scratch)."""
        if self._bbox is None:
            self._bbox = self._arena.view(self._bbox_off, 8, torch.int32, slot=self._slot)
        return self._bbox

    def compute_bbox(self):
        if not self.have_bbox:
            _lib.check(_lib.lib().bfm_deform_grid(C.byref(self.struct), self.bbox_ptr, None, _stream()))
            self.have_bbox = True

    def bbox_host(self):
        """[x1,y1,z1,x2,y2,z2] -- one 24-byte D2H, only when somebody asks (datasets.py:296-301)."""
        if self._bbox_host is None:
            self._bbox_host = [int(v) for v in self.bbox[:6].tolist()]
        return self._bbox_host

    def coords(self):
        """bbox-relative xx2, yy2, zz2 as the reference's deform_grid returns them."""
        out = torch.empty((3, *self.size), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().bfm_deform_grid(C.byref(self.struct), self.bbox_ptr, out.data_ptr(), _stream()))
        return out[0], out[1], out[2]


class DeformDict(dict):
    """deform_dict with the reference's keys; 'grid' and 'F' are materialised on first access."""

    def __missing__(self, key):
        plan = dict.__getitem__(self, '_plan')
        if key in ('A', 'c2'):
            self[key] = torch.from_numpy(np.array(plan.A_host if key == 'A' else plan.c2_host)).to(plan.device)
            return self[key]
        if key == 'F':
            # full-resolution nonlinear field (datasets.py:209-212), only when somebody asks for it
            small = dict.get(self, '_Fsmall')
            if small is None:
                self['F'] = None
                return None
            F = myzoom_torch(small.to(plan.device), np.array(plan.size) / np.array(small.shape[:3]))
            if dict.get(self, '_photo'):
                F[:, :, :, 1] = 0
            self['F'] = F
            return F
        if key == 'grid':
            xx2, yy2, zz2 = plan.coords()
            x1, y1, z1, x2, y2, z2 = plan.bbox_host()
            self['grid'] = [xx2, yy2, zz2, x1, y1, z1, x2, y2, z2]
            return self['grid']
        raise KeyError(key)


def _plan_of(deform_dict):
    if '_plan' not in deform_dict:
        raise _lib.BfmError("deform_dict was not produced by brainfm_b200 (no '_plan' entry)")
    return dict.__getitem__(deform_dict, '_plan')


def _cache(device):
    """The device's one volume cache (shared with BaseGen: an uploaded / refreshed volume is seen by every reader)."""
    return bio.shared_cache(device)


# ------------------------------------------------------------------------------------------------
# target readers (processing_funcs)
# ------------------------------------------------------------------------------------------------
def read_image(file_name):
    img = bio.load(file_name)
    aff = img.affine
    res = np.sqrt(np.sum(abs(aff[:-1, :-1]), axis=0))
    return img, aff, res


def read_and_deform(file_name, dtype, deform_dict, device, mask, default_value_linear_mode=None,
                    deform_mode='linear', mean=0., scale=1., minmax_out=None):
    """Crop-read + trilinear warp of one volume (Generator/utils.py:296-321), fused into one gather kernel
    over the device-resident volume (no host crop, no H2D per sample)."""
    if default_value_linear_mode is not None and default_value_linear_mode != 'max':
        raise ValueError('Not support default_value_linear_mode:', default_value_linear_mode)
    if deform_mode != 'linear':
        raise NotImplementedError("read_and_deform supports deform_mode='linear' only")
    plan = _plan_of(deform_dict)
    img = bio.load(file_name)
    res = np.sqrt(np.sum(abs(img.affine[:-1, :-1]), axis=0))
    vol = _cache(plan.device).get(file_name, 'f32')
    if list(vol.shape[:3]) != plan.src:
        raise ValueError("volume shape %s does not match the deformation's source shape %s" % (tuple(vol.shape), plan.src))
    if mask is not None:
        # left hemisphere only (utils.py:307-311): I -= mean; I /= scale; I[mask == 0] = 0 on a (padded) copy of the
        # volume -- `mask` is the full-volume mask of BaseGen.get_left_hemis_mask
        if tuple(mask.shape) != tuple(vol.shape):
            raise ValueError("mask shape %s does not match the volume %s" % (tuple(mask.shape), tuple(vol.shape)))
        pad = int(vol.shape[1]) * int(vol.shape[2]) + int(vol.shape[2]) + 1
        buf = torch.zeros(vol.numel() + pad, dtype=torch.float32, device=plan.device)
        view = buf[:vol.numel()].view(vol.shape)
        torch.sub(vol, float(mean), out=view)
        view.div_(float(scale))
        view[mask == 0] = 0
        vol, mean, scale = view, 0., 1.
    out = torch.empty(plan.size, dtype=torch.float32, device=plan.device)
    scratch = torch.empty(1, dtype=torch.float32, device=plan.device)
    _lib.check(_lib.lib().bfm_warp_volume(C.byref(plan.struct), plan.bbox_ptr, vol.data_ptr(), float(mean),
                                          float(scale), 1 if default_value_linear_mode == 'max' else 0,
                                          scratch.data_ptr(), out.data_ptr(),
                                          None if minmax_out is None else minmax_out.data_ptr(), _stream()))
    return out, res


def _normalise_flip(x, flip, minmax=True, post=1.0, mm=None):
    L = _lib.lib()
    out = torch.empty_like(x)
    nx = x.shape[0]
    plane = x.numel() // nx
    if minmax:
        if mm is None:
            mm = torch.empty(2, dtype=torch.float32, device=x.device)
            _lib.check(L.bfm_minmax(x.data_ptr(), x.numel(), mm.data_ptr(), _stream()))
        _lib.check(L.bfm_shift_scale_flip(x.data_ptr(), out.data_ptr(), nx, plane, mm.data_ptr(), mm.data_ptr() + 4,
                                          1.0, 1 if flip else 0, _stream()))
    else:
        _lib.check(L.bfm_shift_scale_flip(x.data_ptr(), out.data_ptr(), nx, plane, None, None, float(post),
                                          1 if flip else 0, _stream()))
    return out


def read_and_deform_image(exist_keys, task_name, file_name, setups, deform_dict, device, mask=None, **kwargs):
    """Warp, min-max normalise, flip (Generator/utils.py:324-343)."""
    mm = torch.empty(2, dtype=torch.float32, device=_plan_of(deform_dict).device)
    Idef, _ = read_and_deform(file_name, torch.float, deform_dict, device, mask, minmax_out=mm)
    Idef = _normalise_flip(Idef, setups['flip'], mm=mm)
    update_dict = {task_name: Idef[None]}
    dm = file_name[:-4] + '.defacingmask.nii'
    if bio.exists(dm):
        Idef_DM, _ = read_and_deform(dm, torch.float, deform_dict, device, mask)
        Idef_DM = torch.clamp(Idef_DM, min=0.)
        Idef_DM /= torch.max(Idef_DM)
        update_dict.update({task_name + '_DM': Idef_DM[None]})    # reference leaves the mask unflipped (utils.py:336-338)
    return update_dict


def read_and_deform_CT(exist_keys, task_name, file_name, setups, deform_dict, device, mask=None, **kwargs):
    """CT target: /1000, flip, no normalisation (Generator/utils.py:345-364)."""
    Idef, _ = read_and_deform(file_name, torch.float, deform_dict, device, mask, scale=1000)
    if setups['flip']:
        Idef = _normalise_flip(Idef, True, minmax=False)
    update_dict = {'CT': Idef[None]}
    dm = file_name[:-4] + '.defacingmask.nii'
    if bio.exists(dm):                                     # defacing mask (Generator/utils.py:353-359)
        Idef_DM, _ = read_and_deform(dm, torch.float, deform_dict, device, mask)
        Idef_DM = torch.clamp(Idef_DM, min=0.)
        Idef_DM /= torch.max(Idef_DM)
        update_dict.update({task_name + '_DM': Idef_DM[None]})    # the reference leaves the mask unflipped (:357-359)
    return update_dict


def read_and_deform_distance(exist_keys, task_name, file_names, setups, deform_dict, device, mask=None, cfg=None,
                             **kwargs):
    """Four surface-distance maps, default = crop max, L/R swap on flip, / scaling, clamp
    (Generator/utils.py:366-392)."""
    if mask is not None:                                   # left hemisphere only: two maps (utils.py:373-374)
        file_names = file_names[:2]
    maps = [read_and_deform(f, torch.float, deform_dict, device, mask, default_value_linear_mode='max', mean=128.,
                            scale=20)[0] for f in file_names]
    if mask is not None:
        Idef = torch.stack(maps, dim=0)
    else:
        lp, lw, rp, rw = maps
        if setups['flip']:
            lp, rp = _normalise_flip(rp, True, minmax=False), _normalise_flip(lp, True, minmax=False)
            lw, rw = _normalise_flip(rw, True, minmax=False), _normalise_flip(lw, True, minmax=False)
        Idef = torch.stack([lp, lw, rp, rw], dim=0)
    Idef /= deform_dict['scaling_factor_distances']
    Idef = torch.clamp(Idef, min=-cfg.max_surf_distance, max=cfg.max_surf_distance)
    return {'distance': Idef}


def read_and_deform_registration(exist_keys, task_name, file_names, setups, deform_dict, device, mask=None, **kwargs):
    """MNI coordinate maps /10000, x sign flipped on flip (Generator/utils.py:458-471)."""
    reg = [read_and_deform(f, torch.float, deform_dict, device, mask, scale=10000)[0] for f in file_names]
    if setups['flip']:
        reg = [_normalise_flip(reg[0], True, minmax=False, post=-1.0), _normalise_flip(reg[1], True, minmax=False),
               _normalise_flip(reg[2], True, minmax=False)]
    return {'registration': torch.stack(reg, dim=0)}


def read_and_deform_surface(exist_keys, task_name, file_name, setups, deform_dict, device, mask=None, size=None,
                            **kwargs):
    """White / pial surface vertices carried through the INVERSE deformation (Generator/utils.py:479-533):
    V <- (V - c2) Ainv^T, V += trilerp(Fneg, V + c2), V += c2; on flip the x coordinate is mirrored and left / right
    swap.  `deform_dict['Fneg']` is the integrated negative field ('surface' task, datasets.py:214-223).  The
    faces are returned untouched.  Ainv is formed on the host like the reference's CPU `torch.inverse`."""
    Fneg, A, c2 = deform_dict['Fneg'], deform_dict['A'], deform_dict['c2']
    if Fneg is None:
        raise ValueError("read_and_deform_surface needs deform_dict['Fneg'] (enable the 'surface' task)")
    if size is None:
        size = list(Fneg.shape[:3])
    mat = bio.load_surface(file_name.split('.nii')[0] + '.mat')
    dev = Fneg.device
    Ainv = torch.inverse(A.detach().float().cpu()).to(dev)
    c2 = c2.to(dev).float()
    out = {}
    for v, f in (('Vlw', 'Flw'), ('Vrw', 'Frw'), ('Vlp', 'Flp'), ('Vrp', 'Frp')):
        V = torch.tensor(np.asarray(mat[v]), dtype=torch.float, device=dev)
        V = V - c2[None, :]
        V = V @ torch.transpose(Ainv, 0, 1)
        V = V + fast_3D_interp_torch(Fneg, V[:, 0] + c2[0], V[:, 1] + c2[1], V[:, 2] + c2[2])
        V = V + c2[None, :]
        out[v] = V
        out[f] = torch.tensor(np.asarray(mat[f]), dtype=torch.int, device=dev)
    if setups['flip']:
        for v in ('Vlw', 'Vrw', 'Vlp', 'Vrp'):
            out[v][:, 0] = size[0] - 1 - out[v][:, 0]
        for a, b in (('Vlw', 'Vrw'), ('Vlp', 'Vrp'), ('Flw', 'Frw'), ('Flp', 'Frp')):
            out[a], out[b] = out[b], out[a]
    return {k: out[k] for k in ('Vlw', 'Flw', 'Vrw', 'Frw', 'Vlp', 'Flp', 'Vrp', 'Frp')}


def read_and_deform_bias_field(exist_keys, task_name, file_name, setups, deform_dict, device, mask=None, **kwargs):
    """Real bias-field target (Generator/utils.py:473-477; the reference swaps `mask` and `device`, which is
    harmless there only because mask is None)."""
    Idef, _ = read_and_deform(file_name, torch.float, deform_dict, device, mask)
    if setups['flip']:
        Idef = _normalise_flip(Idef, True, minmax=False)
    return {'bias_field': Idef[None]}


def read_and_deform_segmentation(exist_keys, task_name, file_name, setups, deform_dict, device, mask=None, cfg=None,
                                 onehotmatrix=None, lut=None, vflip=None, **kwargs):
    """Nearest-neighbour label warp -> LUT -> one-hot -> flip + L/R channel swap -> channels first
    (Generator/utils.py:394-424), one integer kernel, bit-exact."""
    plan = _plan_of(deform_dict)
    S = _cache(plan.device).get(file_name, 'i32')
    if mask is not None:                                   # S[mask == 0] = 0 (utils.py:400-401)
        S = torch.where(mask != 0, S, torch.zeros((), dtype=S.dtype, device=S.device)).contiguous()
    n_classes = int(onehotmatrix.shape[0])
    if cfg is not None and cfg.generator.deform_one_hots:
        onehot = onehotmatrix[lut[S.long()]]
        xx2, yy2, zz2 = deform_dict['grid'][:3]
        x1, y1, z1, x2, y2, z2 = deform_dict['grid'][3:]
        Sdef_OneHot = fast_3D_interp_torch(onehot[x1:x2, y1:y2, z1:z2].contiguous(), xx2, yy2, zz2)
        if setups['flip']:
            Sdef_OneHot = torch.flip(Sdef_OneHot, [0])[:, :, :, torch.as_tensor(vflip, device=S.device)]
        return {'segmentation': Sdef_OneHot.permute([3, 0, 1, 2])}
    lut32 = lut.to(device=plan.device, dtype=torch.int32)
    vf = torch.as_tensor(np.asarray(vflip), dtype=torch.int32, device=plan.device)
    out = torch.empty((n_classes, *plan.size), dtype=torch.float32, device=plan.device)
    _lib.check(_lib.lib().bfm_label_warp_onehot(C.byref(plan.struct), plan.bbox_ptr, S.data_ptr(),
                                                lut32.data_ptr(), int(lut32.numel()), n_classes, vf.data_ptr(),
                                                1 if setups['flip'] else 0, out.data_ptr(), None, _stream()))
    return {'segmentation': out}


def read_and_deform_pathology(exist_keys, task_name, file_name, setups, deform_dict, device, mask=None, augment=False,
                              pde_func=None, t=None, shape_gen_args=None, thres=0., **kwargs):
    """Pathology probability target (Generator/utils.py:428-455).  Only the `file_name is None` branch is on
    the default configuration's path; the random-shape / PDE branch lives in brainfm_b200.ShapeID."""
    plan = _plan_of(deform_dict)
    if file_name is None:
        z = torch.zeros(plan.size, device=plan.device)[None]
        return {'pathology': z, 'pathology_prob': z.clone()}
    from ..ShapeID.perlin3d import generate_shape_3d
    if file_name == 'random_shape':
        draws = kwargs.get('draws') or _DRAWS
        # np.random.uniform(a, b) == a + (b - a) * random_sample()
        percentile = shape_gen_args.mask_percentile_min + (shape_gen_args.mask_percentile_max -
                                                           shape_gen_args.mask_percentile_min) * draws.rand("pathol.percentile")
        _, Pdef = generate_shape_3d(tuple(plan.size), shape_gen_args.perlin_res, percentile, plan.device,
                                    draws=draws)
    else:
        Pdef, _ = read_and_deform(file_name, torch.float, deform_dict, device, None)
    if augment:
        Pdef = augment_pathology(Pdef, pde_func, t, shape_gen_args, device, draws=kwargs.get('draws'))
    P = binarize(Pdef, thres)
    if P.mean() <= shape_gen_args.pathol_tol:
        z = torch.zeros(plan.size, device=plan.device)[None]
        return {'pathology': z, 'pathology_prob': z.clone()}
    return {'pathology': P[None], 'pathology_prob': Pdef[None]}


def augment_pathology(Pprob, pde_func, t, shape_gen_args, device, draws=None):
    """Advect a pathology probability map with a random divergence-free velocity field
    (Generator/utils.py:542-560)."""
    from ..ShapeID.DiffEqs.adjoint import odeint_adjoint as odeint
    from ..ShapeID.perlin3d import generate_velocity_3d
    Pprob = torch.squeeze(Pprob)
    nt = (draws or _DRAWS).randint("pathol.nt", shape_gen_args.max_nt) + 1
    if nt <= 1:
        return Pprob
    pde_func.V_dict = generate_velocity_3d(Pprob.shape, shape_gen_args.perlin_res, shape_gen_args.V_multiplier, device)
    return odeint(pde_func, Pprob[None], t[:nt], shape_gen_args.dt, method=shape_gen_args.integ_method)[-1, 0]


# ------------------------------------------------------------------------------------------------
# augmentation operators (augmentation_funcs) -- the op-by-op path; BaseGen fuses the stock sequence
# ------------------------------------------------------------------------------------------------
def add_gamma_transform(I, aux_dict, cfg, device=None, draws=None, **kwargs):
    """300 * (I/300) ** exp(gamma_std * n) (Generator/utils.py:568-572)."""
    _need_cuda(I, "I")
    rng = draws or _DRAWS
    gamma = float(np.float32(np.exp(cfg.gamma_std * rng.randn1("gamma.n"))))
    return 300.0 * (I / 300.0) ** gamma, aux_dict


def add_bias_field(I, aux_dict, cfg, input_mode, setups, size, device=None, draws=None, **kwargs):
    """Multiplicative smooth bias field exp(zoom(small random grid)) (Generator/utils.py:574-589)."""
    _need_cuda(I, "I")
    if input_mode == 'CT':
        aux_dict.update({'high_res': I})
        return I, aux_dict
    rng = draws or _DRAWS
    bf_scale = cfg.bf_scale_min + rng.rand1("bf.scale") * (cfg.bf_scale_max - cfg.bf_scale_min)
    size_BF_small = np.round(bf_scale * np.array(size)).astype(int).tolist()
    if setups['photo_mode']:
        size_BF_small[1] = np.round(size[1] / setups['spac']).astype(int)
    std = torch.tensor(cfg.bf_std_min + (cfg.bf_std_max - cfg.bf_std_min) * rng.rand1("bf.std"), dtype=torch.float)
    BFsmall = (std * rng.torch_randn("bf.field", size_BF_small)).to(I.device)
    BFlog = myzoom_torch(BFsmall, np.array(size) / size_BF_small)
    I_bf = I * torch.exp(BFlog)
    aux_dict.update({'BFlog': BFlog, 'high_res': I_bf})
    return I_bf, aux_dict


def resample_resolution(I, aux_dict, setups, res, size, device=None, draws=None, **kwargs):
    """Slice-thickness blur + trilinear downsample to the acquisition grid (Generator/utils.py:591-609),
    evaluated as one banded linear map per axis."""
    _need_cuda(I, "I")
    rng = draws or _DRAWS
    stds = (0.85 + 0.3 * rng.rand("rs.u")) * np.log(5) / np.pi * setups['thickness'] / res
    stds[setups['thickness'] <= res] = 0.0
    new_size = (np.array(size) * res / setups['resolution']).astype(int)
    factors = np.array(new_size) / np.array(size)
    L = _lib.lib()
    x = I.contiguous().float()
    shape = list(x.shape)
    for ax in range(3):
        start, w, T = band_host(int(size[ax]), int(new_size[ax]), float(stds[ax]))
        keep, (p_start, p_w) = pack_to_device([start, w], x.device)
        out_shape = list(shape)
        out_shape[ax] = int(new_size[ax])
        y = torch.empty(out_shape, dtype=torch.float32, device=x.device)
        shp = (C.c_int * 3)(*shape)
        _lib.check(L.bfm_band_axis(x.data_ptr(), y.data_ptr(), shp, ax, int(new_size[ax]), p_start, p_w, T, -1.0,
                                   None, 0, _stream()))
        x, shape = y, out_shape
    aux_dict.update({'factors': factors})
    return x, aux_dict


def add_noise(I, aux_dict, cfg, device=None, draws=None, **kwargs):
    """max(0, I + sigma * N(0,1)) (Generator/utils.py:633-638)."""
    _need_cuda(I, "I")
    rng = draws or _DRAWS
    noise_std = float(np.float32(cfg.noise_std_min + (cfg.noise_std_max - cfg.noise_std_min) * rng.rand1("noise.u")[0]))
    eps = rng.field_randn("noise.eps", tuple(I.shape))
    eps = torch.randn(I.shape, dtype=torch.float, device=I.device) if eps is None else eps.to(I.device)
    I_noisy = I + noise_std * eps
    I_noisy[I_noisy < 0] = 0
    return I_noisy, aux_dict
