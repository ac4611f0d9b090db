"""Batched planning through the native host planner (libbfm `bfm_plan_batch`, csrc/planner.cu).

`BaseGen.generate_batch` plans every item in Python (draws from the numpy/torch global generators in the
reference's order, ~250 us per sample).  When nothing in the configuration needs Python per sample -- synthetic or
real T1 / T2 / FLAIR / CT inputs (drawn per item like read_input), stock augmentation chain, no mixing with real
modalities, no pathology / surface task, no random shift -- the whole batch is planned by ONE call into
the library instead: the same arithmetic in C, draws from an in-library Philox stream keyed on (seed, item counter)
(the seed itself is one draw of numpy's global generator, so `np.random.seed` still makes a run reproducible), small
random grids drawn on the device.
With a `ReplayDraws` source the planner runs in replay mode and consumes the recorded draws (parity tests).
"""
import ctypes as C
from collections import defaultdict

import numpy as np
import torch

from .. import _lib
from ..draws import HostDraws
from . import constants as K
from .utils import DeformDict, DeformPlan, _stream, scratch_stride


def _ptr(t):
    return 0 if t is None else t.data_ptr()


class NativePlanner:
    def __init__(self, ds):
        self.ds = ds
        self.device = ds.device
        self.size = [int(v) for v in ds.size]
        self.N = int(np.prod(self.size))
        self.n_samples = len(ds._gen_arg_sets())
        self.counter = 0
        self.seed = None
        self._keep = []
        self.cfg = self._build_cfg()
        self._fp = self.fingerprint()
        self.last = None
        self._prep = {}
        self._prep_version = -1
        self._items = {}
        self._item_version = -1
        self._other_targets = None

    _KEYS = ('photo_prob', 'pathology_prob', 'random_shape_prob', 'flip_prob', 'max_rotation', 'max_shear',
             'max_scaling', 'nonlin_scale_min', 'nonlin_scale_max', 'nonlin_std_max', 'ct_prob', 'low_res_only',
             'nonlinear_transform')

    def fingerprint(self):
        """The parameter values the cached bfm_plan_cfg was built from; `refresh()` rebuilds it when the caller has
        changed gen_args since (curricula, update_gen_args with new values)."""
        ds = self.ds
        a = ds.synth_args
        fp = [getattr(a, k) for k in self._KEYS] + [getattr(a, 'bspline_zooming', False), ds.gen_args.mix_synth_prob,
                                                    tuple(ds.size)]
        for mode in ('synth', 'T1'):
            for overrides in ds._gen_arg_sets(mode):
                for o in overrides:
                    fp.append(tuple(sorted(vars(o).items())))
        base = vars(ds.gen_args.generator)
        fp += [base[f] for f in ('gamma_std', 'bf_scale_min', 'bf_scale_max', 'bf_std_min', 'bf_std_max')]
        return fp

    def refresh(self):
        fp = self.fingerprint()
        if fp != self._fp:
            self.cfg = self._build_cfg()
            self._fp = fp

    # ---- eligibility ------------------------------------------------------------------------------
    @staticmethod
    def config_ok(ds):
        a = ds.synth_args
        if a.left_hemis_only or a.random_shift:
            return False
        if ds.gen_args.mix_synth_prob > 0 or 'surface' in ds.tasks or 'pathology' in ds.tasks:
            return False
        if not ds._stock_chain('synth'):
            return False
        if len(ds._gen_arg_sets()) > _lib.PLAN_MAX_SAMPLES:
            return False
        return True

    def item_ok(self, input_prob, modalities):
        """Inputs the library plans: synthetic, and real T1 / T2 / FLAIR / CT volumes of the label map's shape."""
        ds = self.ds
        if any(input_prob.get(m, 0) > 0 and m in modalities for m in ('T1', 'T2', 'FLAIR', 'CT')):
            if not ds._stock_chain('real'):
                return False
            shape = list(ds.cache.get(modalities['Gen'], 'gen').shape[:3])
            for m in ('T1', 'T2', 'FLAIR', 'CT'):
                if input_prob.get(m, 0) > 0 and m in modalities and \
                        list(ds.cache.get(modalities[m], 'f32').shape[:3]) != shape:
                    return False
        return True

    # ---- configuration (built once) ------------------------------------------------------------------
    def _build_cfg(self):
        ds, size = self.ds, self.size
        a = ds.synth_args
        cfg = _lib.PlanCfg()
        cfg.size[:] = size
        cfg.res[:] = [float(v) for v in ds.res_training_data]
        cfg.low_res_only = int(bool(a.low_res_only))
        cfg.bspline_zooming = int(bool(getattr(a, 'bspline_zooming', False)))
        cfg.nonlinear_transform = int(bool(a.nonlinear_transform))
        for k in ('photo_prob', 'pathology_prob', 'random_shape_prob', 'flip_prob', 'max_rotation', 'max_shear',
                  'max_scaling', 'nonlin_scale_min', 'nonlin_scale_max', 'nonlin_std_max', 'ct_prob'):
            setattr(cfg, k, float(getattr(a, k)))
        cfg.mix_synth_prob = float(ds.gen_args.mix_synth_prob)
        grp = np.full(256, -1, dtype=np.int8)
        from .datasets import ct_brightness_group
        for g, name in enumerate(('darker', 'dark', 'bright', 'brighter')):
            for l in ct_brightness_group[name]:
                grp[l] = g
        C.memmove(cfg.ct_group, grp.ctypes.data, 256)
        # per-sample parameter ranges: generator values with the overrides of each sample applied in order
        base = dict(vars(ds.gen_args.generator))           # snapshot: update_gen_args mutates the shared namespace
        for mode, dst in (('synth', cfg.aug), ('T1', cfg.aug_real)):
            sets = ds._gen_arg_sets(mode)
            cfg.n_samples = len(sets)
            vals = dict(base)
            for k, overrides in enumerate(sets):
                for o in overrides:                         # overrides accumulate from sample to sample, like
                    vals.update(vars(o))                    # update_gen_args on the shared namespace (datasets.py:634-636)
                for f, _ in _lib.PlanAug._fields_:
                    setattr(dst[k], f, float(vals[f]))
        # zoom-table directories
        tables = ds.tables
        tables.prebuild(size)
        ends, dirs = [], []
        for ax in range(3):
            n_out = size[ax]
            fwd = (_lib.ZoomAxis * (n_out + 1))()
            inv = (_lib.ZoomAxis * (n_out + 1))()
            for n_in in range(1, n_out + 1):
                for arr, factor in ((fwd, n_out / n_in), (inv, 1 / (n_in / n_out))):
                    z = arr[n_in]
                    z.lo, z.hi, z.wl, z.wh = tables.zoom(n_in, factor, n_out)
                    z.valid = int(int(np.round(n_in * factor)) == n_out)
                fwd[n_in].cand, fwd[n_in].ncand = tables.cand(n_in, n_out / n_in, n_out)
            dirs.append((fwd, inv))
            cfg.fwd[ax] = C.addressof(fwd)
            cfg.inv[ax] = C.addressof(inv)
            cfg.ends[ax] = tables.ends(n_out)[0]
        ident = torch.cat([torch.arange(size[2], dtype=torch.int32, device=self.device).view(torch.float32),
                           torch.ones(size[2], dtype=torch.float32, device=self.device)])
        cfg.ident_start = ident.data_ptr()
        cfg.ident_w = ident.data_ptr() + 4 * size[2]
        self._keep += [dirs, ident]
        return cfg

    # ---- per-batch preparation, cached ------------------------------------------------------------------
    def _prepare(self, indices, use_cache=True):
        """PlanItem array + per-item metadata of a batch of dataset indices.  Everything in here depends only on the
        indices and on WHICH tensors the device cache holds, so it is built once per index tuple and reused until the
        cache's membership changes (`DeviceVolumeCache.version`: a new volume, an eviction, a clear); uploads and
        refreshes overwrite cached volumes in place and keep it valid.  On a hit the volumes are only touched (LRU
        order + eviction epoch).  Saves ~0.15 ms of ctypes stores and dictionary look-ups per batch of 8."""
        ds = self.ds
        key = tuple(int(i) for i in indices)
        cache = ds.cache
        if self._prep_version != cache.version:
            self._prep.clear()               # entries hold references to cached tensors: drop them with the old set
            self._prep_version = cache.version
        ent = self._prep.get(key)
        if use_cache and ent is not None and ent['version'] == cache.version:
            cache.touch(ent['keys'])
            return ent
        B = len(key)
        items = (_lib.PlanItem * B)()
        metas, keys = [], []
        n_aux_total, src_pad = 0, 0
        for n, idx in enumerate(key):
            dataset_name, input_prob, t1_path, age = ds.idx_to_path(idx)
            mods = ds.get_info(t1_path)
            lab = cache.get(mods['Gen'], 'gen')
            keys.append((mods['Gen'], 'gen'))
            it = items[n]
            it.labels = lab.data_ptr()
            it.label_is_u8 = 1 if lab.dtype == torch.uint8 else 0
            src = [int(v) for v in lab.shape[:3]]
            it.src[:] = src
            for q, m in enumerate(('T1', 'T2', 'FLAIR', 'CT')):
                it.input_prob[q] = float(input_prob.get(m, 0))
            for q, m in enumerate(('T1', 'T2', 'FLAIR')):
                if m in mods and input_prob.get(m, 0) > 0:
                    it.real_vol[q] = cache.get(mods[m], 'f32').data_ptr()
                    keys.append((mods[m], 'f32'))
            if 'CT' in mods and input_prob.get('CT', 0) > 0:
                it.ct_vol = cache.get(mods['CT'], 'f32').data_ptr()
                keys.append((mods['CT'], 'f32'))
            aux = ds._fused_aux_volumes(mods, src)
            it.n_aux = len(aux)
            for c, (k_, vol) in enumerate(aux):
                it.aux_src[c] = vol.data_ptr()
                keys.append((mods[k_], 'f32'))
            n_aux_total += len(aux)
            src_pad = max(src_pad, src[0] * src[1] * src[2] + src[1] * src[2] + src[2] + 1)
            metas.append((idx, dataset_name, t1_path, age, dict(mods), aux, src))
        ent = dict(items=items, metas=metas, n_aux_total=n_aux_total, src_pad=src_pad, keys=keys,
                   version=cache.version, ok=None)
        if use_cache:
            if len(self._prep) > 256 or self._prep_version != cache.version:      # volumes were loaded while preparing
                self._prep.clear()
                self._prep_version = cache.version
            self._prep[key] = ent
        return ent

    def batch_ok(self, indices):
        """item_ok for every index of the batch (cached with the batch's preparation)."""
        ds = self.ds
        ent = self._prepare(indices)
        if ent['ok'] is None:
            ent['ok'] = all(self.item_ok(ds.idx_to_path(m[0])[1], m[4]) for m in ent['metas'])
        return ent['ok']

    # ---- one batch, lean path ------------------------------------------------------------------------------
    def fast_ok(self):
        """run_fast covers native draws with every requested target riding on the fused gather (no op-wise target
        readers, no replay, no stage timers)."""
        ds = self.ds
        if getattr(ds.rng, 'replay', False):
            return False
        other = self._other_targets
        if other is None:
            other = self._other_targets = any(t in K.processing_funcs and t not in ('T1', 'T2', 'FLAIR')
                                              for t in ds.tasks)
        return not other

    def _item_entry(self, idx):
        """Per-INDEX cached PlanItem bytes + metadata (valid while the device cache holds the same tensors)."""
        ds, cache = self.ds, self.ds.cache
        if self._item_version != cache.version:
            self._items.clear()
            self._item_version = cache.version
        ent = self._items.get(idx)
        if ent is not None:
            return ent
        prep = self._prepare([idx], use_cache=False)
        meta = prep['metas'][0]
        ent = dict(raw=bytes(prep['items']), meta=meta, keys=prep['keys'], n_aux=len(meta[5]),
                   src_pad=prep['src_pad'], ok=self.item_ok(ds.idx_to_path(idx)[1], meta[4]),
                   needs_plan=len(meta[5]) < sum(1 for k in ('T1', 'T2', 'FLAIR') if k in meta[4]),
                   case_name=_case_name(meta[2]))
        if self._item_version != cache.version:              # volumes were loaded while preparing
            self._items.clear()
            self._item_version = cache.version
        self._items[idx] = ent
        return ent

    def run_fast(self, indices):
        """generate_batch for the common case in ONE library call (bfm_plan_run: buffer lay-out, planning, descriptor
        upload, every stage launch) and a few dozen microseconds of Python: per-index cached PlanItems are copied into
        the batch array, the output tensors are allocated, and the per-item result tuples are built only when somebody
        indexes the returned sequence (`LazyItems`; `.input` / `.bias_field_log` / `.targets` are the collated batch
        tensors a trainer consumes).  Returns None when the batch needs the general path (`run`)."""
        ds, L = self.ds, _lib.lib()
        tr = getattr(ds, '_trace', None)           # development aid: host time stamps of the last call
        if tr is not None:
            import time as _t
            tr.clear()
            tr.append(('start', _t.perf_counter()))
        B = len(indices)
        ns = self.n_samples
        total = B * ns
        ents = []
        for idx in indices:
            e = self._item_entry(int(idx))
            if not e['ok'] or e['needs_plan']:
                return None
            ents.append(e)
        if self.seed is None:
            self.seed = int(np.random.randint(0, 2 ** 62))
        ds.hemis_mask = None
        size, N, dev = self.size, self.N, self.device
        items = (_lib.PlanItem * B)()
        isz = C.sizeof(_lib.PlanItem)
        base = C.addressof(items)
        touch = ds.cache.touch
        n_aux_total, src_pad = 0, 0
        for n, e in enumerate(ents):
            C.memmove(base + n * isz, e['raw'], isz)
            touch(e['keys'])
            n_aux_total += e['n_aux']
            if e['src_pad'] > src_pad:
                src_pad = e['src_pad']
        src_pad = (src_pad + 3) // 4 * 4 * 2                 # float2 {synthetic, target} pairs (syn_pair_ok)
        if tr is not None:
            tr.append(('items', _t.perf_counter()))
        want_bflog = ds._want_bflog('synth')
        want_res = 'super_resolution' in ds.tasks
        # Outputs come from the CALLER's stream pool when a pipeline set one (DevicePipeline): the caching allocator keeps
        # one pool of free blocks per stream, and with the outputs in the lanes' pools a lane was measured to run out of
        # free 131 MB blocks and cudaMalloc three new ones (1.3-200 ms) while a dozen sat free in the other pools.  Safe:
        # every submit() orders the lane after the caller's stream, so a block the consumer freed is only rewritten
        # after the consumer's work on it (see pipeline._DeviceTicket.wait).
        als = getattr(ds, '_alloc_stream', None)
        if als is not None:
            lane_stream = torch.cuda.current_stream(dev)
            torch.cuda.set_stream(als)
        out = torch.empty((total, 1, *size), dtype=torch.float32, device=dev)
        bfl = torch.empty((total, 1, *size), dtype=torch.float32, device=dev) if want_bflog else None
        res = torch.empty((total, 1, *size), dtype=torch.float32, device=dev) if want_res else None
        aux_all = torch.empty((n_aux_total, 1, *size), dtype=torch.float32, device=dev) if n_aux_total else None
        if als is not None:
            torch.cuda.set_stream(lane_stream)
        if tr is not None:
            tr.append(('outputs', _t.perf_counter()))
        syn_ws = ds._workspace('syn', total * src_pad, zero=True)
        if ds._ws.get('syn_stride') != src_pad:
            if 'syn_stride' in ds._ws:
                syn_ws.zero_()
            ds._ws['syn_stride'] = src_pad
        bufs = _lib.StepBufs()
        bufs.out = out.data_ptr()
        bufs.bflog_out = bfl.data_ptr() if bfl is not None else None
        bufs.residual = res.data_ptr() if res is not None else None
        bufs.syn = syn_ws.data_ptr()
        bufs.syn_stride = src_pad
        Np = scratch_stride(N)
        bufs.i_bf = ds._workspace('i_bf', total * Np).data_ptr()
        bufs.tmp = ds._workspace('tmp', total * 2 * Np).data_ptr()
        bufs.lowres = ds._workspace('lowres', total * Np).data_ptr()
        if n_aux_total:
            bufs.aux_out = aux_all.data_ptr()
            bufs.aux_raw = ds._workspace('aux_raw', n_aux_total * Np).data_ptr()
        bufs.pair_ok = 1 if ds.pair_mode else 0
        if tr is not None:
            tr.append(('workspaces', _t.perf_counter()))
        arena = ds.arena.begin()
        if tr is not None:
            tr.append(('arena', _t.perf_counter()))
        slot = arena.slots[arena.cur]
        descs = (_lib.GenSample * total)()
        descs_dev = C.c_void_p(0)
        info = (_lib.PlanInfo * B)()
        used = C.c_int64(0)
        _lib.check(L.bfm_plan_run(C.addressof(self.cfg), B, base, C.addressof(bufs), self.seed, self.counter,
                                  slot["host"].data_ptr(), slot["dev"].data_ptr(), arena.capacity, arena.used,
                                  C.byref(used), C.addressof(descs), C.byref(descs_dev), C.addressof(info), _stream()))
        if tr is not None:
            tr.append(('plan_run', _t.perf_counter()))
        self.counter += B
        arena.used = arena.committed = used.value
        arena.mark_done()
        self.last = dict(descs=descs, descs_dev=descs_dev.value, info=info, total=total,
                         keep=(out, bfl, res, aux_all, items), arena_slot=arena.cur)
        if tr is not None:
            tr.append(('done', _t.perf_counter()))
        ds._last_descs = (descs, descs_dev.value, total)
        ds._last_out = out
        return LazyItems(ds, ents, info, ns, out, bfl, res, aux_all)

    # ---- one batch ---------------------------------------------------------------------------------------
    def run(self, indices, timers=None, patch=None, plan_only=False):
        """Plan the batch in the library and run the fused chain.
        patch(descs, info): optional hook called after planning and BEFORE the descriptors travel to the device (slab
        mode sets x_begin / x_count there, which depend on the planned flip).  plan_only: stop after the upload and
        return the plan (descs, device address, info, output tensors) without launching any stage."""
        ds, L = self.ds, _lib.lib()
        size, N, ns = self.size, self.N, self.n_samples
        B = len(indices)
        total = B * ns
        dev = self.device
        rng = ds.rng
        replay = getattr(rng, 'replay', False)
        if self.seed is None and not replay:
            self.seed = int(np.random.randint(0, 2 ** 62))
        ds.hemis_mask = None
        want_bflog = ds._want_bflog('synth')
        want_res = 'super_resolution' in ds.tasks
        # ---- items: volumes from the device cache (prepared once per index tuple, see _prepare)
        prep = self._prepare(indices, use_cache=not replay)     # replayed draws park eps pointers in the items
        items, metas, n_aux_total, src_pad = prep['items'], prep['metas'], prep['n_aux_total'], prep['src_pad']
        src_pad = (src_pad + 3) // 4 * 4
        # ---- outputs (fresh) and persistent scratch
        out = torch.empty((total, 1, *size), dtype=torch.float32, device=dev)
        bfl = torch.empty((total, 1, *size), dtype=torch.float32, device=dev) if want_bflog else None
        res = torch.empty((total, 1, *size), dtype=torch.float32, device=dev) if want_res else None
        aux_all = torch.empty((n_aux_total, 1, *size), dtype=torch.float32, device=dev) if n_aux_total else None
        # syn holds float2 {synthetic, T1} pairs for samples with one fused target (bfm_gen_sample.syn_pair_ok)
        src_pad *= 2
        syn_ws = ds._workspace('syn', total * src_pad, zero=True)
        if ds._ws.get('syn_stride') != src_pad:
            if 'syn_stride' in ds._ws:
                syn_ws.zero_()
            ds._ws['syn_stride'] = src_pad
        Np = scratch_stride(N)
        p_ibf = ds._workspace('i_bf', total * Np).data_ptr()
        p_tmp = ds._workspace('tmp', total * 2 * Np).data_ptr()
        p_low = ds._workspace('lowres', total * Np).data_ptr()
        p_raw = ds._workspace('aux_raw', n_aux_total * Np).data_ptr() if n_aux_total else 0
        outs = (_lib.PlanOut * total)()
        o_np = np.frombuffer(outs, dtype=np.uint64).reshape(total, 9)
        q = np.arange(total, dtype=np.uint64)
        step, pstep = np.uint64(4 * N), np.uint64(4 * Np)
        o_np[:, 0] = np.uint64(out.data_ptr()) + q * step
        o_np[:, 1] = (np.uint64(bfl.data_ptr()) + q * step) if want_bflog else 0
        o_np[:, 2] = (np.uint64(res.data_ptr()) + q * step) if want_res else 0
        o_np[:, 3] = np.uint64(syn_ws.data_ptr()) + q * np.uint64(4 * src_pad)
        o_np[:, 4] = np.uint64(p_ibf) + q * pstep
        o_np[:, 5] = np.uint64(p_tmp) + (2 * q) * pstep
        o_np[:, 6] = np.uint64(p_tmp) + (2 * q + 1) * pstep
        o_np[:, 7] = np.uint64(p_low) + q * pstep
        o_np[:, 8] = 1 if ds.pair_mode else 0
        k_aux = 0
        for n in range(B):
            it = items[n]
            for c in range(it.n_aux):
                it.aux_out[c] = aux_all.data_ptr() + 4 * N * k_aux
                it.aux_raw[c] = p_raw + 4 * Np * k_aux
                k_aux += 1
        # ---- draws to replay (parity tests): scalars and small arrays flattened in log order
        keep = []
        flat, n_flat = None, 0
        if replay:
            vals, k_eps = [], defaultdict(int)
            while not rng.done():
                tag, v = rng.log[rng.pos]
                rng.pos += 1
                if tag in ('gmm.eps', 'noise.eps'):
                    t = v.to(dev).float().contiguous()
                    keep.append(t)
                    arr = items[0].eps_gmm if tag == 'gmm.eps' else items[0].eps_noise
                    arr[k_eps[tag]] = t.data_ptr()
                    k_eps[tag] += 1
                else:
                    vals.append(np.asarray(v.numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float64).reshape(-1))
            flat = np.ascontiguousarray(np.concatenate(vals))
            n_flat = flat.size
            if B != 1:
                raise ValueError("replayed draws drive one item at a time")
        # ---- plan
        arena = ds.arena.begin()
        slot = arena.slots[arena.cur]
        start = (arena.used + 15) // 16 * 16
        used, upload = C.c_int64(arena.used), C.c_int64(0)
        descs = (_lib.GenSample * total)()
        descs_dev = C.c_void_p(0)
        info = (_lib.PlanInfo * B)()
        consumed = C.c_int64(0)
        _lib.check(L.bfm_plan_batch(C.addressof(self.cfg), B, C.addressof(items), C.addressof(outs),
                                    self.seed or 0, self.counter, slot["host"].data_ptr(), slot["dev"].data_ptr(),
                                    arena.capacity, C.byref(used), C.byref(upload), C.addressof(descs),
                                    C.byref(descs_dev), C.addressof(info),
                                    flat.ctypes.data if replay else None, n_flat, C.byref(consumed)))
        if replay and consumed.value != n_flat:
            raise AssertionError("native planner consumed %d of %d replayed draws" % (consumed.value, n_flat))
        self.counter += B
        arena.used = used.value
        st = _stream()
        if patch is not None:
            patch(descs, info)
            C.memmove(slot["host"].data_ptr() + (descs_dev.value - slot["dev"].data_ptr()), C.addressof(descs),
                      C.sizeof(descs))
        nbytes = (upload.value + 15) // 16 * 16
        _lib.check(L.bfm_upload_pinned(slot["dev"].data_ptr() + start, slot["host"].data_ptr() + start, nbytes, st))
        arena.committed = arena.used
        if plan_only:
            self.last = dict(descs=descs, descs_dev=descs_dev.value, info=info, total=total,
                             keep=(out, bfl, res, aux_all, keep), arena_slot=arena.cur)
            ds._last_descs = (descs, descs_dev.value, total)
            return dict(descs=descs, d_dev=descs_dev.value, info=info, out=out, bfl=bfl, res=res, aux=aux_all,
                        arena=arena, metas=metas)
        # ---- per-item context (targets that do not ride on the fused gather need a DeformPlan)
        h, d_dev = C.addressof(descs), descs_dev.value
        other_targets = self._other_targets
        if other_targets is None:
            other_targets = self._other_targets = any(t in K.processing_funcs and t not in ('T1', 'T2', 'FLAIR')
                                                      for t in ds.tasks)
        need_plans = other_targets or any(len(m[5]) < sum(1 for k in ('T1', 'T2', 'FLAIR') if k in m[4]) for m in metas)

        def setups_of(inf):
            return {'resolution': np.array(inf.resolution[:]), 'thickness': np.array(inf.thickness[:]),
                    'photo_mode': bool(inf.photo_mode), 'pathol_mode': False, 'pathol_random_shape': False,
                    'spac': inf.spac if inf.photo_mode else None, 'flip': bool(inf.flip), 'hemis': 'both'}

        ctxs = []
        for n, (idx, dataset_name, t1_path, age, mods, aux, src) in enumerate(metas):
            inf = info[n]
            # the set-up dictionary is only read by the op-wise target readers (and kept as ds.last_setups)
            setups = setups_of(inf) if (need_plans or n == B - 1) else None
            ctxs.append(dict(idx=idx, dataset_name=dataset_name, case_name=_case_name(t1_path),
                             input_mode=_INPUT_MODES[inf.input_mode],
                             age=age, setups=setups, modalities=mods, aux=aux, src=src, n=n))

        def stage(name, fn):
            if timers is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            _lib.check(fn(h, d_dev, total, st))
            if timers is not None:
                e1.record()
                timers.setdefault(name, []).append((e0, e1))

        if timers is None and not need_plans:
            _lib.check(L.bfm_gen_run(h, d_dev, total, st))
        else:
            stage('plan', L.bfm_gen_plan)
            stage('bbox', L.bfm_gen_bbox)
        aux_views = aux_all.unbind(0) if aux_all is not None else ()
        k_aux = 0
        targets = []
        for ctx in ctxs:
            n = ctx['n']
            target = defaultdict(ds._default_target)
            target['name'] = ctx['case_name']
            fused = {}
            for key, _ in ctx['aux']:
                fused[key] = aux_views[k_aux]
                k_aux += 1
            deform = self._deform_dict(ctx, descs[n * ns], info[n], arena) if need_plans else None
            ctx['deform'] = deform
            ds.modalities = ctx['modalities']
            for key in ('T1', 'T2', 'FLAIR'):
                if key in fused:
                    target[key] = fused[key]
                elif key in ctx['modalities']:
                    target.update(ds.read_and_deform_target(ctx['idx'], target.keys(), key, ctx['input_mode'],
                                                            ctx['setups'], deform))
                else:
                    target[key] = 0.
            if other_targets:
                for task_name in ds.tasks:
                    if task_name in K.processing_funcs.keys() and task_name not in ('T1', 'T2', 'FLAIR'):
                        target.update(ds.read_and_deform_target(ctx['idx'], target.keys(), task_name,
                                                                ctx['input_mode'], ctx['setups'], deform))
            target['pathology'] = 0.
            target['pathology_prob'] = 0.
            targets.append(target)
        if timers is not None or need_plans:
            stage('gmm', L.bfm_gen_gmm)
            stage('warp', L.bfm_gen_warp)
            stage('resample', L.bfm_gen_resample)
            stage('finish', L.bfm_gen_finish)
        arena.mark_done()
        # ---- results
        out_v = out.unbind(0)
        bfl_v = bfl.unbind(0) if bfl is not None else None
        res_v = res.unbind(0) if res is not None else None
        results = []
        for q_ in range(total):
            s = {}
            if res_v is not None:
                s['high_res_residual'] = res_v[q_]
            s['input'] = out_v[q_]
            if bfl_v is not None and info[q_ // ns].input_mode != 4:      # no bias field on CT inputs
                s['bias_field_log'] = bfl_v[q_]
            results.append(s)
        tuples = []
        for ctx, target in zip(ctxs, targets):
            n = ctx['n']
            sample = results[n * ns:(n + 1) * ns] if ds._list_samples else results[n * ns]
            if ctx['age'] is not None:
                target['age'] = ctx['age']
            tuples.append((ds.datasets_num, ctx['dataset_name'], ctx['input_mode'], target, sample))
        if ctxs:
            ds.last_setups, ds.last_deform = ctxs[-1]['setups'], ctxs[-1]['deform']
        self.last = dict(descs=descs, descs_dev=d_dev, info=info, total=total, keep=(out, bfl, res, aux_all, keep),
                         arena_slot=arena.cur)
        ds._last_descs = (descs, d_dev, total)
        ds._last_out = out
        return tuples

    def _deform_dict(self, ctx, desc, inf, arena):
        """A DeformDict around the planned deformation, for targets computed by the op-wise entry points."""
        ds = self.ds
        plan = DeformPlan.__new__(DeformPlan)
        plan.size = list(self.size)
        plan.src = list(ctx['src'])
        plan.device = self.device
        plan.A_host = np.array(inf.A[:], dtype=np.float32).reshape(3, 3)
        plan.c2_host = np.array(inf.c2[:], dtype=np.float32)
        plan.photo = bool(inf.photo_mode)
        plan.F_full = None
        plan.struct = _lib.Deform.from_buffer_copy(desc.d)
        plan.bbox_ptr = desc.bbox
        plan._bbox = None
        plan._arena, plan._slot = arena, arena.cur
        plan._bbox_off = desc.bbox - arena.slots[arena.cur]["dev"].data_ptr()
        plan._bbox_host = None
        plan.have_bbox = True
        fs = list(inf.fs[:])
        small = None
        if fs[0] > 0:
            off = desc.d.fsmall - arena.slots[arena.cur]["dev"].data_ptr()
            small = arena.view(off, fs[0] * fs[1] * fs[2] * 3, torch.float32).view(*fs, 3)
        return DeformDict({'scaling_factor_distances': inf.scaling_factor_distances, 'Fneg': None, '_plan': plan,
                           '_Fsmall': small, '_photo': bool(inf.photo_mode)})

    # ---- what the last batch looked like (bench.py) ---------------------------------------------------------
    def last_shapes(self):
        """[(bbox ints, new_size)] of every sample of the last batch (one small D2H per sample)."""
        torch.cuda.synchronize()
        last = self.last
        arena = self.ds.arena
        base = arena.slots[last['arena_slot']]["dev"].data_ptr()
        rows = []
        ns = self.n_samples
        for q in range(last['total']):
            d = last['descs'][q]
            bb = arena.view(d.bbox - base, 8, torch.int32, slot=last['arena_slot'])[:6].tolist()
            rows.append((bb, list(last['info'][q // ns].new_size[q % ns])))
        return rows


_INPUT_MODES = ('synth', 'T1', 'T2', 'FLAIR', 'CT')


def _case_name(t1_path):
    import os
    return os.path.basename(t1_path).split('.T1w.nii')[0]


class LazyItems:
    """What `run_fast` returns: the batch as collated device tensors (`input`: (B * n_samples, 1, *size), `bias_field_log`,
    `high_res_residual`, `targets[key]`: (B, 1, *size)) and, on demand, the reference-shaped per-item tuples
    `(datasets_num, dataset_name, input_mode, target, sample)` -- a sequence: len(), indexing and iteration build
    them exactly as `NativePlanner.run` does."""

    def __init__(self, ds, ents, info, ns, out, bfl, res, aux_all):
        self._ds, self._ents, self._info, self._ns = ds, ents, info, ns
        self.input, self.bias_field_log, self.high_res_residual = out, bfl, res
        self._aux = aux_all
        self._built = None

    @property
    def targets(self):
        """{key: (n_items_with_that_target, 1, *size)} of the fused real-image targets, in item order."""
        out, k = {}, 0
        for e in self._ents:
            for key, _ in e['meta'][5]:
                out.setdefault(key, []).append(self._aux[k])
                k += 1
        return {key: torch.stack(v) for key, v in out.items()}

    def _build(self):
        if self._built is not None:
            return self._built
        ds, ns, info = self._ds, self._ns, self._info
        out_v = self.input.unbind(0)
        bfl_v = self.bias_field_log.unbind(0) if self.bias_field_log is not None else None
        res_v = self.high_res_residual.unbind(0) if self.high_res_residual is not None else None
        aux_v = self._aux.unbind(0) if self._aux is not None else ()
        tuples, k_aux = [], 0
        for n, e in enumerate(self._ents):
            idx, dataset_name, t1_path, age, mods, aux, src = e['meta']
            inf = info[n]
            target = defaultdict(ds._default_target)
            target['name'] = e['case_name']
            fused = {}
            for key, _ in aux:
                fused[key] = aux_v[k_aux]
                k_aux += 1
            for key in ('T1', 'T2', 'FLAIR'):
                target[key] = fused[key] if key in fused else 0.
            target['pathology'] = 0.
            target['pathology_prob'] = 0.
            if age is not None:
                target['age'] = age
            results = []
            for q in range(n * ns, (n + 1) * ns):
                smp = {}
                if res_v is not None:
                    smp['high_res_residual'] = res_v[q]
                smp['input'] = out_v[q]
                if bfl_v is not None and inf.input_mode != 4:          # no bias field on CT inputs
                    smp['bias_field_log'] = bfl_v[q]
                results.append(smp)
            sample = results if ds._list_samples else results[0]
            tuples.append((ds.datasets_num, dataset_name, _INPUT_MODES[inf.input_mode], target, sample))
        self._built = tuples
        return tuples

    def __len__(self):
        return len(self._ents)

    def __getitem__(self, n):
        return self._build()[n]

    def __iter__(self):
        return iter(self._build())
