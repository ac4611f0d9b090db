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

The global maximum of I / max(I) is one scalar all-reduce.  Per voxel the arithmetic is that of the op-level
path (resample_resolution -> add_noise -> myzoom_torch) and both volume-sized noise fields are counter-based (GMM
noise keyed on the absolute source voxel, acquisition noise on the absolute low-res voxel, bfm_add_noise_at), so a
volume generated on W ranks is bit-identical to the same volume generated in slab mode on one rank -- with injected
draws or without (tests/test_gen_parity_gpu.py, tests/_slab_worker.py).
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from .. import _lib, parallel as par
from ..plan import band_host, resample_coords_host, zoom_tables_host
from .utils import _stream, scratch_stride


def _band_axis(x, axis, n_out, start, w, T, arena):
    # tables through the pinned plan arena (asynchronous upload): a pageable host->device copy would wait for all
    # queued GPU work every time and serialise host and device
    p_start = arena.put(np.ascontiguousarray(start, dtype=np.int32))
    p_w = arena.put(np.ascontiguousarray(w, dtype=np.float32))
    arena.commit()
    shape = list(x.shape)
    out_shape = list(shape)
    out_shape[axis] = int(n_out)
    y = torch.empty(out_shape, dtype=torch.float32, device=x.device)
    if y.numel() and x.numel():
        _lib.check(_lib.lib().bfm_band_axis(x.data_ptr(), y.data_ptr(), (C.c_int * 3)(*shape), axis, int(n_out),
                                            p_start, p_w, int(T), -1.0, None, 0, _stream()))
    return y


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


def _mx_all_reduce(mx, world, group):
    if world > 1:
        if dist.get_backend(group) == "gloo":              # ranks sharing one GPU (tests): reduce on the host
            h_mx = mx.cpu()
            dist.all_reduce(h_mx, op=dist.ReduceOp.MAX, group=group)
            mx = h_mx.to(mx.device)
        else:
            dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    return mx


def _generate_slab_native(ds, native, idx, rank, world, group):
    """Slab mode on the library planner: ONE bfm_plan_batch call plans the volume (a few microseconds, against ~1 ms
    for the Python planner), the band tables are built on the device by bfm_gen_plan, the zoom tables come from the
    device-resident cache, and the banded passes run in the fused chain's order (ascending factor, identity axes
    skipped) with the fused chain's tables -- so the assembled volume equals what generate_batch produces for the same
    planner state, up to the order-independent parts.  The x pass and the zoom back address the exchanged plane
    buffers through a base pointer biased by the first plane they hold, so the whole-volume tables are used as they
    are (no per-slab copies of tables)."""
    L = _lib.lib()
    s0, s1, s2 = [int(v) for v in ds.size]
    state = {}

    def patch(descs, info):
        flip = bool(descs[0].flip)
        # planes of the (unflipped) grid this rank computes; with a flip the slabs are mirrored so that the planes
        # a rank computes are the ones it owns in the flipped output
        owned = [list(par.slab_bounds(s0, (world - 1 - r) if flip else r, world)) for r in range(world)]
        c0, c1 = owned[rank]
        if c1 <= c0:
            raise ValueError("slab mode: rank %d owns no plane (%d planes over %d ranks)" % (rank, s0, world))
        descs[0].x_begin, descs[0].x_count = c0, c1 - c0
        # the GMM stage only synthesises the source planes this slab gathers from (bfm_gen_bbox reduces the range)
        xr = None
        if world > 1:
            xr = torch.empty(2, dtype=torch.int32, device=ds.device)
            descs[0].gmm_xr = xr.data_ptr()
        state.update(flip=flip, owned=owned, xr=xr)

    plan = native.run([idx], patch=patch, plan_only=True)
    descs, d_dev = plan['descs'], plan['d_dev']
    s = descs[0]
    if s.real_input or s.mix[0]:
        raise NotImplementedError("slab mode covers synthetic inputs without mixing")
    flip, owned = state['flip'], state['owned']
    c0, c1 = owned[rank]
    h, st = C.addressof(descs), _stream()
    for fn in (L.bfm_gen_plan, L.bfm_gen_bbox, L.bfm_gen_gmm, L.bfm_gen_warp):
        _lib.check(fn(h, d_dev, 1, st))
    N = s0 * s1 * s2
    dev = plan['out'].device
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
                ob, oe = low_owned[rank]
                y = torch.empty((max(oe - ob, 0), dims[1], dims[2]), dtype=torch.float32, device=dev)
                if y.numel():
                    plane_bytes = 4 * dims[1] * dims[2]
                    _lib.check(L.bfm_band_axis(ext.data_ptr() - needed[rank][0] * plane_bytes, y.data_ptr(),
                                               (C.c_int * 3)(s0, dims[1], dims[2]), 0, oe - ob, b.start + 4 * ob,
                                               b.w + 4 * ob * T, T, -1.0, None, 0, st))
            else:
                shape = [cur.shape[0], dims[1], dims[2]]
                oshape = list(shape)
                oshape[a] = n_out
                y = torch.empty(oshape, dtype=torch.float32, device=dev)
                if y.numel():
                    _lib.check(L.bfm_band_axis(cur.data_ptr(), y.data_ptr(), (C.c_int * 3)(*shape), a, n_out, b.start,
                                               b.w, T, -1.0, None, 0, st))
            cur = y
            dims[a] = n_out
    ob, oe = low_owned[rank]
    low = cur
    # ---- strict `> 0` masks of the identity axes, then the noise (counter-based stream 1 keyed on the ABSOLUTE low-res
    # voxel: the assembled volume does not depend on the number of ranks)
    if low.numel():
        if s.zero_first[0] and ob == 0:
            low[0].zero_()
        if s.zero_first[1]:
            low[:, 0].zero_()
        if s.zero_first[2]:
            low[:, :, 0].zero_()
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
    mx = _mx_all_reduce(out.max().reshape(1), world, group)
    fin = torch.empty_like(out)
    _lib.check(L.bfm_shift_scale_flip(out.data_ptr(), fin.data_ptr(), c1 - c0, s1 * s2, None, mx.data_ptr(), 1.0,
                                      1 if flip else 0, st))
    x0, x1 = (s0 - c1, s0 - c0) if flip else (c0, c1)
    sample = {'input': fin[None], 'x_range': (x0, x1)}
    if plan['bfl'] is not None and s.bflog_out:
        sample['bias_field_log'] = plan['bfl'][0][:, x0:x1]
    # ---- real-image targets that ride on the gather (read_and_deform_image, Generator/utils.py:324-343): the warp
    # wrote this rank's planes of the raw warped volume and reduced ITS min / max; `Idef -= min; Idef /= max` needs the
    # volume's: one all-reduce of 2 * n_aux order-preserving ints (MAX of {-min, max}), then the normalise + flip pass
    n_aux = int(s.n_aux)
    if n_aux:
        arena = plan['arena']
        base = arena.slots[arena.cur]["dev"].data_ptr()
        mm = arena.view(s.aux_mm - base, 2 * n_aux, torch.int32).clone()
        mm[0::2] = -mm[0::2]
        if world > 1:
            if dist.get_backend(group) == "gloo":
                h_mm = mm.cpu()
                dist.all_reduce(h_mm, op=dist.ReduceOp.MAX, group=group)
                mm = h_mm.to(dev)
            else:
                dist.all_reduce(mm, op=dist.ReduceOp.MAX, group=group)
        mm[0::2] = -mm[0::2]
        mmf = torch.where(mm >= 0, mm, mm ^ 0x7fffffff).view(torch.float32)         # ord2f (csrc/common.cuh)
        keys = [k for k, _ in plan['metas'][0][5]]
        for a in range(n_aux):
            raw = ds._ws['aux_raw'][a * scratch_stride(N):][:N].view(s0, s1, s2)[c0:c1]
            tgt = torch.empty((c1 - c0, s1, s2), dtype=torch.float32, device=dev)
            _lib.check(L.bfm_shift_scale_flip(raw.data_ptr(), tgt.data_ptr(), c1 - c0, s1 * s2,
                                              mmf[2 * a:2 * a + 1].data_ptr(), mmf[2 * a + 1:2 * a + 2].data_ptr(), 1.0,
                                              1 if flip else 0, st))
            sample[keys[a]] = tgt[None]
    plan['arena'].mark_done()
    return sample


def generate_slab(ds, idx, rank=None, world=None, group=None):
    """This rank's x-slab of sample `idx` of dataset `ds` (BaseGen): {'input': (1, nx, s1, s2),
    'bias_field_log': (1, nx, s1, s2) or absent, 'T1' / 'T2' / 'FLAIR': (1, nx, s1, s2) for the real-image targets that
    ride on the fused gather (library planner), 'x_range': (x0, x1)} with x0:x1 the owned planes of the final
    (flipped) output volume.  Every rank must call this with the same generator seeds."""
    if rank is None:
        rank = dist.get_rank(group) if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size(group) if dist.is_initialized() else 1
    if getattr(ds.synth_args, 'bspline_zooming', False):
        # the cubic zoom's dct2 prefilter is a recursion along the whole x axis: no fixed halo covers it
        raise NotImplementedError("slab mode does not cover bspline_zooming")
    ds.cache.begin_batch()
    native = ds._native_planner([idx]) if not getattr(ds.rng, 'replay', False) else None
    if native is not None and native.n_samples == 1:
        return _generate_slab_native(ds, native, idx, rank, world, group)
    L = _lib.lib()
    size = [int(v) for v in ds.size]
    s0, s1, s2 = size
    arena = ds.arena.begin()
    ctx = ds._prologue_host(idx, arena)
    if not ds._fast_ok(ctx['input_mode']):
        raise NotImplementedError("slab mode covers synthetic inputs with the stock augmentation chain")
    setups = ctx['setups']
    target = {}
    for a in ds._gen_arg_sets()[0]:
        ds.update_gen_args(a)
    p = ds._plan_synth(setups, target)
    if p['mix'] is not None:
        raise NotImplementedError("slab mode does not mix real modalities into the synthetic image")
    job = ds._job(setups, ctx['deform'], target, p)
    descs, results = ds._build_descs([job], arena)
    flip = bool(setups['flip'])
    # planes of the (unflipped) grid this rank computes; with a flip the slabs are mirrored so that the planes
    # a rank computes are the ones it owns in the flipped output
    owned = [list(par.slab_bounds(s0, (world - 1 - r) if flip else r, world)) for r in range(world)]
    c0, c1 = owned[rank]
    descs[0].x_begin, descs[0].x_count = c0, c1 - c0
    if world > 1:
        xr = torch.empty(2, dtype=torch.int32, device=ds.device)      # source planes this slab gathers from (GMM range)
        descs[0].gmm_xr = xr.data_ptr()
    d_dev = arena.put_struct_array(descs)
    arena.commit()
    ds._last_descs = (descs, d_dev, 1)
    h, st = C.addressof(descs), _stream()
    _lib.check(L.bfm_gen_bbox(h, d_dev, 1, st))
    job['plan'].have_bbox = True
    _lib.check(L.bfm_gen_gmm(h, d_dev, 1, st))
    _lib.check(L.bfm_gen_warp(h, d_dev, 1, st))
    N = s0 * s1 * s2
    i_bf = ds._ws['i_bf'][:N].view(s0, s1, s2)[c0:c1]

    # ---- resolution degradation: x first (needs neighbours' planes), then y and z on the slab
    new = [int(v) for v in p['new_size']]
    stds = [float(v) for v in p['stds']]
    start, w, T = band_host(s0, new[0], stds[0])
    centre = np.clip(np.floor(resample_coords_host(s0, new[0])[0]).astype(np.int64), 0, s0 - 1)
    low_owned = []
    for r in range(world):
        b, e = owned[r]
        o = np.nonzero((centre >= b) & (centre < e))[0]
        low_owned.append([int(o[0]), int(o[-1]) + 1] if o.size else [0, 0])
    needed = []
    for r in range(world):
        ob, oe = low_owned[r]
        if oe > ob:
            needed.append([int(max(0, start[ob:oe].min())), int(min(s0, start[ob:oe].max() + T))])
        else:
            needed.append([owned[r][0], owned[r][0]])
    ext = par.exchange_planes(i_bf, owned, needed, rank, world, group)
    ob, oe = low_owned[rank]
    x = _band_axis(ext, 0, oe - ob, start[ob:oe] - needed[rank][0], w[ob:oe], T, arena)
    for ax in (1, 2):
        st_a, w_a, T_a = band_host(size[ax], new[ax], stds[ax])
        x = _band_axis(x, ax, new[ax], st_a, w_a, T_a, arena)
    # ---- noise (add_noise, utils.py:633-638): injected draws are sliced; otherwise the chain's counter-based stream 1,
    # keyed on the ABSOLUTE low-res voxel -- the assembled volume does not depend on the number of ranks, and equals
    # what the fused chain (generate_batch) draws for the same seed
    if p['eps_noise'] is not None:
        eps = p['eps_noise'][ob:oe].to(x.device)
        low = torch.clamp(x + float(p['noise_std']) * eps, min=0)
    else:
        low = x.contiguous()
        _lib.check(L.bfm_add_noise_at(low.data_ptr(), low.numel(), float(p['noise_std']), int(p['seed']), 1,
                                      ob * new[1] * new[2], _stream()))

    # ---- back to the training grid: low-res planes lo[c0] .. hi[c1-1] (1-2 from the neighbours)
    up = 1 / (np.array(new) / np.array(size))
    tabs = [zoom_tables_host(new[a], up[a], size[a]) for a in range(3)]
    need_low = []
    for r in range(world):
        b, e = owned[r]
        need_low.append([int(tabs[0][0][b:e].min()), int(tabs[0][1][b:e].max()) + 1] if e > b else [0, 0])
    lext = par.exchange_planes(low, low_owned, need_low, rank, world, group)
    nb = need_low[rank][0]
    t0 = (tabs[0][0][c0:c1] - nb, tabs[0][1][c0:c1] - nb, tabs[0][2][c0:c1], tabs[0][3][c0:c1])
    flat = [np.ascontiguousarray(t) for t in t0] + [t for tab in tabs[1:] for t in tab]
    addr = [arena.put(np.ascontiguousarray(t)) for t in flat]
    arena.commit()
    out = torch.empty((c1 - c0, s1, s2), dtype=torch.float32, device=low.device)
    if out.numel():
        args = [lext.data_ptr(), lext.shape[0], new[1], new[2], 1]
        for d, n_out in enumerate((c1 - c0, s1, s2)):
            args += [addr[4 * d], addr[4 * d + 1], addr[4 * d + 2], addr[4 * d + 3], int(n_out)]
        _lib.check(L.bfm_zoom_linear(*args, out.data_ptr(), _stream()))
    # ---- I / max(I) with the global maximum (datasets.py:342-343), then the flip
    mx = _mx_all_reduce(out.max().reshape(1) if out.numel() else torch.zeros(1, device=low.device), world, group)
    # one pass: I / max and the flip of the slab's planes (bfm_shift_scale_flip: true division like the reference)
    if out.numel():
        fin = torch.empty_like(out)
        _lib.check(L.bfm_shift_scale_flip(out.data_ptr(), fin.data_ptr(), c1 - c0, s1 * s2, None, mx.data_ptr(), 1.0,
                                          1 if flip else 0, _stream()))
        out = fin
    sample = {}
    if flip:
        x0, x1 = s0 - c1, s0 - c0
    else:
        x0, x1 = c0, c1
    sample['input'] = out[None]
    if 'bias_field_log' in results[0]:
        sample['bias_field_log'] = results[0]['bias_field_log'][:, x0:x1]
    sample['x_range'] = (x0, x1)
    arena.mark_done()
    ds.last_setups, ds.last_deform = setups, ctx['deform']
    return sample
