"""One large volume across several GPUs: x-slabs of the output grid with plane (halo) exchange.

The reference has no spatial decomposition (SURVEY.md 2.1, 8e); its generator simply cannot hold the
intermediates of a 512^3 sample next to a training job.  Here the OUTPUT grid is cut into x-slabs, one per
rank; every rank holds the (integer) source label map and draws the same random numbers (same seeds), so the
deformation, the contrast tables and the GMM image are identical everywhere without any traffic (the GMM noise
is counter-based, keyed on the absolute source voxel).  Only two stages have a stencil along x and therefore
an exchange step, both point-to-point between neighbouring ranks (parallel.exchange_planes -> NCCL send/recv):

  1. the slice-profile blur + downsample along x needs ceil(3*sigma)+1 planes of the warped image from each
     neighbour (<= 17 planes of 512^2 floats = 17.8 MB per side);
  2. the zoom back to the training grid needs the 1-2 low-res planes next to the slab.

The global maximum of I / max(I) is one scalar all-reduce.  Either planner fills the fused chain's bfm_gen_sample
descriptor (the library planner in bfm_plan_batch; the Python planner, which replays injected draws and plans BrainID
items, in BaseGen._build_descs), and one body runs it: the fused chain's band order and tables, its noise and its zoom
tables, so the volume equals what generate_batch produces for the same draws within the float tolerance.  Both
volume-sized noise fields are counter-based (GMM noise keyed on the absolute source voxel, acquisition noise on the
absolute low-res voxel, bfm_add_noise_at), so a volume generated on W ranks is bit-identical to the same volume
generated in slab mode on one rank -- with injected draws or without (tests/test_gen_parity_gpu.py,
tests/_slab_worker.py).
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from .. import _lib, parallel as par
from ..plan import resample_coords_host, zoom_tables_host
from .utils import _stream, scratch_stride

_HOST_TABS = {}


def _band_ranges_host(n_in, n_out):
    """floor of the low-res sample positions along one axis (the band's first tap is floor - ceil(3 sigma)); cached."""
    key = ('band', int(n_in), int(n_out))
    hit = _HOST_TABS.get(key)
    if hit is None:
        lo = np.floor(resample_coords_host(n_in, n_out)[0]).astype(np.int64)
        hit = _HOST_TABS[key] = (lo, np.clip(lo, 0, n_in - 1))
    return hit


def _zoom_ranges_host(n_in, n_out):
    """lo / hi source planes of the zoom back along one axis (host copy of the device table); cached."""
    key = ('zoom', int(n_in), int(n_out))
    hit = _HOST_TABS.get(key)
    if hit is None:
        t = zoom_tables_host(n_in, 1 / (n_in / n_out), n_out)
        hit = _HOST_TABS[key] = (t[0].astype(np.int64), t[1].astype(np.int64))
    return hit


def _all_reduce_max(t, world, group):
    """Element-wise maximum over the ranks of a float or int32 tensor."""
    if world > 1:
        if dist.get_backend(group) == "gloo":              # ranks sharing one GPU (tests): reduce on the host
            h = t.cpu()
            dist.all_reduce(h, op=dist.ReduceOp.MAX, group=group)
            return h.to(t.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return t


def _owned(s0, world, flip):
    """[begin, end) of the planes of the (unflipped) grid each rank computes; with a flip the slabs are mirrored so
    that the planes a rank computes are the ones it owns in the flipped output."""
    return [list(par.slab_bounds(s0, (world - 1 - r) if flip else r, world)) for r in range(world)]


def _plan_native(native, idx, patch):
    """Library planner: ONE bfm_plan_batch call plans the volume (a few microseconds, against ~1 ms for the Python
    planner); bfm_gen_plan draws the small grids and builds the band tables on the device."""
    plan = native.run([idx], patch=patch, plan_only=True)
    descs = plan['descs']
    bfl = plan['bfl'][0] if plan['bfl'] is not None else None
    keys = plan['ents'][0]['aux']
    return descs, plan['d_dev'], plan['arena'], bfl, keys, None, bool(descs[0].flip)


def _plan_python(ds, idx, patch):
    """Python planner (replayed draws; BrainID items, of which the first sample is sliced): the host draws of one item
    and its descriptor from BaseGen._build_descs.  No real-image target rides on the gather (n_aux = 0)."""
    arena = ds.arena.begin()
    ctx = ds._prologue_host(idx, arena)
    if not ds._fast_ok(ctx['input_mode']):
        raise NotImplementedError("slab mode covers synthetic inputs with the stock augmentation chain")
    setups, target = ctx['setups'], {}
    for a in ds._gen_arg_sets()[0]:
        ds.update_gen_args(a)
    p = ds._plan_synth(setups, target)
    if p['mix'] is not None:
        raise NotImplementedError("slab mode does not mix real modalities into the synthetic image")
    job = ds._job(setups, ctx['deform'], target, p)
    descs, results = ds._build_descs([job], arena)
    patch(descs)
    d_dev = arena.put_struct_array(descs)
    arena.commit()
    ds._last_descs = (descs, d_dev, 1)
    job['plan'].have_bbox = True                 # the body's bfm_gen_bbox computes it before anything reads it
    ds.last_setups, ds.last_deform = setups, ctx['deform']
    return descs, d_dev, arena, results[0].get('bias_field_log'), [], p['eps_noise'], bool(setups['flip'])


def _slab(ds, rank, world, group, descs, d_dev, arena, bfl, keys, eps, flip):
    """This rank's slab of the one planned sample `descs[0]`.  The bbox / GMM / warp stages evaluate only the owned
    planes; the banded passes run in the descriptor's order (ascending factor, identity axes folded away into the
    `zero_first` masks) with its tables.  The x pass and the zoom back address the exchanged plane buffers through a
    base pointer biased by the first plane they hold, so the whole-volume tables are used as they are (no per-slab
    copies of tables).  eps: injected acquisition-noise draws of the whole low-res volume, or None."""
    L = _lib.lib()
    s = descs[0]
    if s.real_input or s.mix[0]:
        raise NotImplementedError("slab mode covers synthetic inputs without mixing")
    s0, s1, s2 = [int(v) for v in ds.size]
    owned = _owned(s0, world, flip)
    c0, c1 = owned[rank]
    h, st, dev = C.addressof(descs), _stream(), ds.device
    for fn in (L.bfm_gen_plan, L.bfm_gen_bbox, L.bfm_gen_gmm, L.bfm_gen_warp):
        _lib.check(fn(h, d_dev, 1, st))
    N = s0 * s1 * s2
    cur = ds._ws['i_bf'][:N].view(s0, s1, s2)[c0:c1]
    dims = [s0, s1, s2]
    new = [int(v) for v in s.new_size[:]]
    identity = s.n_band == 1 and s.band[0].T == 1 and s.band[0].build == 0
    low_owned = [list(o) for o in owned]
    if identity:
        cur = cur.clone()                      # the noise is added in place; i_bf is persistent scratch
    else:
        for q in range(s.n_band):
            b = s.band[q]
            a, T, n_out = int(b.axis), int(b.T), int(b.n_out)
            first = 0                          # first output row of the pass (the x pass computes this rank's rows)
            src, shape = cur.data_ptr(), [cur.shape[0], dims[1], dims[2]]
            if a == 0:
                # ---- x pass: ceil(3 sigma) + 1 planes from each neighbour
                lo, centre = _band_ranges_host(s0, n_out)
                start = lo - (T - 2) // 2
                low_owned, needed = [], []
                for r in range(world):
                    b_, e_ = owned[r]
                    o = np.nonzero((centre >= b_) & (centre < e_))[0]
                    low_owned.append([int(o[0]), int(o[-1]) + 1] if o.size else [0, 0])
                    ob, oe = low_owned[-1]
                    if oe > ob:
                        needed.append([int(max(0, start[ob:oe].min())), int(min(s0, start[ob:oe].max() + T))])
                    else:
                        needed.append([owned[r][0], owned[r][0]])
                ext = par.exchange_planes(cur, owned, needed, rank, world, group)
                first, oe = low_owned[rank]
                n_out = oe - first
                src, shape = ext.data_ptr() - needed[rank][0] * 4 * dims[1] * dims[2], [s0, dims[1], dims[2]]
            oshape = list(shape)
            oshape[a] = n_out
            y = torch.empty(oshape, dtype=torch.float32, device=dev)
            if y.numel():
                _lib.check(L.bfm_band_axis(src, y.data_ptr(), (C.c_int * 3)(*shape), a, n_out, b.start + 4 * first,
                                           b.w + 4 * first * T, T, -1.0, None, 0, st))
            cur = y
            dims[a] = int(b.n_out)
    ob, oe = low_owned[rank]
    low = cur
    # ---- strict `> 0` masks of the identity axes, then the noise: injected draws are sliced and added like the fused
    # chain does (k_gen_band / k_gen_identity: separately rounded, clamped at 0); otherwise the chain's counter-based
    # stream 1 keyed on the ABSOLUTE low-res voxel (the assembled volume does not depend on the number of ranks)
    if low.numel():
        if s.zero_first[0] and ob == 0:
            low[0].zero_()
        if s.zero_first[1]:
            low[:, 0].zero_()
        if s.zero_first[2]:
            low[:, :, 0].zero_()
        if eps is not None:
            low = torch.clamp(low + float(s.noise_std) * eps[ob:oe].to(dev), min=0)
        else:
            _lib.check(L.bfm_add_noise_at(low.data_ptr(), low.numel(), float(s.noise_std), int(s.seed), 1,
                                          ob * dims[1] * dims[2], st))
    if identity:
        out = low
    else:
        # ---- back to the training grid: low-res planes lo[c0] .. hi[c1-1] (1-2 from the neighbours)
        zlo, zhi = _zoom_ranges_host(new[0], s0)
        need_low = [[int(zlo[o[0]]), int(zhi[o[1] - 1]) + 1] if o[1] > o[0] else [0, 0] for o in owned]
        lext = par.exchange_planes(low, low_owned, need_low, rank, world, group)
        nb = need_low[rank][0]
        out = torch.empty((c1 - c0, s1, s2), dtype=torch.float32, device=dev)
        u = s.utab
        args = [lext.data_ptr() - nb * 4 * new[1] * new[2], new[0], new[1], new[2], 1,
                u.lo[0] + 4 * c0, u.hi[0] + 4 * c0, u.wl[0] + 4 * c0, u.wh[0] + 4 * c0, c1 - c0,
                u.lo[1], u.hi[1], u.wl[1], u.wh[1], s1, u.lo[2], u.hi[2], u.wl[2], u.wh[2], s2]
        _lib.check(L.bfm_zoom_linear(*args, out.data_ptr(), st))
    # ---- I / max(I) with the global maximum (datasets.py:342-343), then the flip
    mx = _all_reduce_max(out.max().reshape(1), world, group)
    fin = torch.empty_like(out)
    _lib.check(L.bfm_shift_scale_flip(out.data_ptr(), fin.data_ptr(), c1 - c0, s1 * s2, None, mx.data_ptr(), 1.0,
                                      1 if flip else 0, st))
    x0, x1 = (s0 - c1, s0 - c0) if flip else (c0, c1)
    sample = {'input': fin[None], 'x_range': (x0, x1)}
    if bfl is not None and s.bflog_out:
        sample['bias_field_log'] = bfl[:, x0:x1]
    # ---- real-image targets that ride on the gather (read_and_deform_image, Generator/utils.py:324-343): the warp
    # wrote this rank's planes of the raw warped volume and reduced ITS min / max; `Idef -= min; Idef /= max` needs the
    # volume's: one all-reduce of 2 * n_aux order-preserving ints (MAX of {-min, max}), then the normalise + flip pass
    n_aux = int(s.n_aux)
    if n_aux:
        base = arena.slots[arena.cur]["dev"].data_ptr()
        mm = arena.view(s.aux_mm - base, 2 * n_aux, torch.int32).clone()
        mm[0::2] = -mm[0::2]
        mm = _all_reduce_max(mm, world, group)
        mm[0::2] = -mm[0::2]
        mmf = torch.where(mm >= 0, mm, mm ^ 0x7fffffff).view(torch.float32)         # ord2f (csrc/common.cuh)
        for a in range(n_aux):
            raw = ds._ws['aux_raw'][a * scratch_stride(N):][:N].view(s0, s1, s2)[c0:c1]
            tgt = torch.empty((c1 - c0, s1, s2), dtype=torch.float32, device=dev)
            _lib.check(L.bfm_shift_scale_flip(raw.data_ptr(), tgt.data_ptr(), c1 - c0, s1 * s2,
                                              mmf[2 * a:2 * a + 1].data_ptr(), mmf[2 * a + 1:2 * a + 2].data_ptr(), 1.0,
                                              1 if flip else 0, st))
            sample[keys[a]] = tgt[None]
    arena.mark_done()
    return sample


def generate_slab(ds, idx, rank=None, world=None, group=None):
    """This rank's x-slab of sample `idx` of dataset `ds` (BaseGen): {'input': (1, nx, s1, s2),
    'bias_field_log': (1, nx, s1, s2) or absent, 'T1' / 'T2' / 'FLAIR': (1, nx, s1, s2) for the real-image targets that
    ride on the fused gather (library planner), 'x_range': (x0, x1)} with x0:x1 the owned planes of the final
    (flipped) output volume.  Every rank must call this with the same generator seeds.  Raises ValueError when this
    rank owns no plane (more ranks than planes)."""
    if rank is None:
        rank = dist.get_rank(group) if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size(group) if dist.is_initialized() else 1
    if getattr(ds.synth_args, 'bspline_zooming', False):
        # the cubic zoom's dct2 prefilter is a recursion along the whole x axis: no fixed halo covers it
        raise NotImplementedError("slab mode does not cover bspline_zooming")
    s0 = int(ds.size[0])
    # the GMM stage only synthesises the source planes this slab gathers from (bfm_gen_bbox reduces the range)
    xr = torch.empty(2, dtype=torch.int32, device=ds.device) if world > 1 else None

    def patch(descs):
        # the owned planes depend on the planned flip: set before the descriptor travels to the device
        c0, c1 = _owned(s0, world, descs[0].flip)[rank]
        if c1 <= c0:
            raise ValueError("slab mode: rank %d owns no plane (%d planes over %d ranks)" % (rank, s0, world))
        descs[0].x_begin, descs[0].x_count = c0, c1 - c0
        if xr is not None:
            descs[0].gmm_xr = xr.data_ptr()

    ds.cache.begin_batch()
    native = ds._native_planner([idx]) if not getattr(ds.rng, 'replay', False) else None
    if native is not None and native.n_samples == 1:
        plan = _plan_native(native, idx, patch)
    else:
        plan = _plan_python(ds, idx, patch)
    return _slab(ds, rank, world, group, *plan)
