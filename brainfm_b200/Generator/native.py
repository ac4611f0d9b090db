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
import os
import time
from collections import defaultdict

import numpy as np
import torch

from .. import _lib
from . import constants as K
from .utils import DeformDict, DeformPlan, _stream, syn_stride


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
        self._ents = {}                  # dataset index -> _entry
        self._version = -1               # cache.version the entries were built under

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

    # ---- per-index preparation, cached ---------------------------------------------------------------------
    def _entry(self, idx):
        """PlanItem bytes + metadata of one dataset index.  Everything in here depends only on the index and on WHICH
        tensors the device cache holds, so it is built once per index and reused until the cache's membership changes
        (`DeviceVolumeCache.version`: a new volume, an eviction, a clear); uploads and refreshes overwrite cached
        volumes in place and keep it valid.  On a hit the volumes are touched (LRU order + eviction epoch), so that
        looking up the batch's other entries cannot evict them.  What depends on the task list is decided per batch."""
        ds, cache = self.ds, self.ds.cache
        if self._version != cache.version:
            self._ents.clear()               # entries point at cached tensors: drop them with the old set
            self._version = cache.version
        ent = self._ents.get(idx)
        if ent is not None:
            cache.touch(ent['keys'])
            return ent
        dataset_name, input_prob, t1_path, age = ds.idx_to_path(idx)
        mods = dict(ds.get_info(t1_path))
        lab = cache.get(mods['Gen'], 'gen')
        keys = [(mods['Gen'], 'gen')]
        it = _lib.PlanItem()
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
        for c, (k, vol) in enumerate(aux):
            it.aux_src[c] = vol.data_ptr()
            keys.append((mods[k], 'f32'))
        ent = dict(raw=bytes(it), keys=keys, idx=idx, dataset_name=dataset_name, case_name=_case_name(t1_path),
                   age=age, mods=mods, src=src, aux=[k for k, _ in aux], syn_stride=syn_stride(src),
                   item_ok=self.item_ok(input_prob, mods),
                   # every real-image target the subject has rides on the gather (else: op-wise readers, run)
                   all_fused=len(aux) == sum(1 for k in ('T1', 'T2', 'FLAIR') if k in mods))
        if self._version != cache.version:              # volumes were loaded while preparing
            self._ents.clear()
            self._version = cache.version
        self._ents[idx] = ent
        return ent

    def batch_ok(self, indices):
        """item_ok for every index of the batch."""
        return all(self._entry(int(i))['item_ok'] for i in indices)

    @staticmethod
    def _items(ents):
        """A fresh PlanItem array of the batch (the layout writes the target pointers into it, replay the injected
        draws), its number of fused real-image targets and its syn stride."""
        items = (_lib.PlanItem * len(ents))()
        isz, base = C.sizeof(_lib.PlanItem), C.addressof(items)
        n_aux, stride = 0, 0
        for n, e in enumerate(ents):
            C.memmove(base + n * isz, e['raw'], isz)
            n_aux += len(e['aux'])
            if e['syn_stride'] > stride:
                stride = e['syn_stride']
        return items, n_aux, stride

    def _seg_maps(self, ents):
        """Per item: the class map of the batched segmentation stage (bfm_gen_segmentation), or None (no segmentation
        target, or the op-wise reader).  Looked up per batch: the cache drops a map when its volume is uploaded."""
        ds = self.ds
        if not ds._seg_stage_ok():
            return [None] * len(ents)
        return [ds._seg_classes(e['mods']['segmentation'], e['src']) for e in ents]

    def _outputs(self, total, n_aux, n_seg):
        """(out, bias_field_log, high_res_residual, fused targets, segmentation) tensors of a batch.  They come from
        the CALLER's stream pool when a pipeline set one (DevicePipeline): the caching allocator keeps one pool of free
        blocks per stream, and with the outputs in the lanes' pools a lane was measured to run out of free 131 MB blocks
        and cudaMalloc three new ones (1.3-200 ms) while a dozen sat free in the other pools.  Safe: every submit()
        orders the lane after the caller's stream, so a block the consumer freed is only rewritten after the consumer's
        work on it (see pipeline._DeviceTicket.wait)."""
        ds, size, dev = self.ds, self.size, self.device
        als = getattr(ds, '_alloc_stream', None)
        if als is not None:
            lane_stream = torch.cuda.current_stream(dev)
            torch.cuda.set_stream(als)
        shape = (total, 1, *size)
        out = torch.empty(shape, dtype=torch.float32, device=dev)
        bfl = torch.empty(shape, dtype=torch.float32, device=dev) if ds._want_bflog('synth') else None
        res = torch.empty(shape, dtype=torch.float32, device=dev) if 'super_resolution' in ds.tasks else None
        aux = torch.empty((n_aux, 1, *size), dtype=torch.float32, device=dev) if n_aux else None
        seg = torch.empty((n_seg, int(ds.onehotmatrix.shape[0]), *size), dtype=torch.float32, device=dev) \
            if n_seg else None
        if als is not None:
            torch.cuda.set_stream(lane_stream)
        return out, bfl, res, aux, seg

    def _bufs(self, outputs, n_aux, stride):
        """bfm_step_bufs of a batch: base addresses of its outputs and of the persistent scratch (BaseGen._scratch)."""
        out, bfl, res, aux, _ = outputs
        bufs = _lib.StepBufs()
        bufs.out, bufs.bflog_out, bufs.residual, bufs.aux_out = _ptr(out), _ptr(bfl), _ptr(res), _ptr(aux)
        bufs.syn, bufs.i_bf, bufs.tmp, bufs.lowres, bufs.aux_raw = self.ds._scratch(out.shape[0], n_aux, stride)
        bufs.syn_stride = stride
        bufs.pair_ok = 1 if self.ds.pair_mode else 0
        return bufs

    def _keep_last(self, descs, d_dev, info, arena, outputs, *keep):
        """The last batch's plan (tests, bench.py's `last_shapes`) and what its kernels still read or write."""
        total = len(descs)
        self.last = dict(descs=descs, descs_dev=d_dev, info=info, total=total, keep=(outputs,) + keep,
                         arena_slot=arena.cur)
        self.ds._last_descs = (descs, d_dev, total)
        self.ds._last_out = outputs[0]

    # ---- one batch, lean path ------------------------------------------------------------------------------
    def fast_ok(self):
        """run_fast covers native draws with every requested target riding on the fused gather or coming from the
        batched segmentation stage (no op-wise target readers, no replay, no stage timers).  `bias_field` and `CT`
        targets are the 0. placeholder of a subject without that file (checked per item by run_fast)."""
        ds = self.ds
        if getattr(ds.rng, 'replay', False):
            return False
        for t in ds.tasks:
            if t not in K.processing_funcs or t in ('T1', 'T2', 'FLAIR', 'CT', 'bias_field'):
                continue
            if t == 'segmentation' and ds._seg_stage_ok():
                continue
            return False
        return True

    def run_fast(self, indices):
        """generate_batch for the common case in ONE library call (bfm_plan_run: buffer lay-out, planning, descriptor
        upload, every stage launch) and a few dozen microseconds of Python: per-index cached PlanItems are copied into
        the batch array, the output tensors are allocated, and the per-item result tuples are built only when somebody
        indexes the returned sequence (`LazyItems`; `.input` / `.bias_field_log` / `.targets` are the collated batch
        tensors a trainer consumes).  Returns None when the batch needs the general path (`run`)."""
        ds, L = self.ds, _lib.lib()
        tr = getattr(ds, '_trace', None)           # development aid: host time stamps of the last call
        if tr is not None:
            tr.clear()
            tr.append(('start', time.perf_counter()))
        absent = [t for t in ('CT', 'bias_field') if t in ds.tasks]      # only as the 0. of a file the item lacks
        ents = []
        for i in indices:
            e = self._entry(int(i))
            if not (e['item_ok'] and e['all_fused']) or absent and not e['mods'].keys().isdisjoint(absent):
                return None
            ents.append(e)
        B, ns = len(ents), self.n_samples
        total = B * ns
        cls = self._seg_maps(ents)
        jobs = [(n * ns, c) for n, c in enumerate(cls) if c is not None]
        if 'segmentation' in ds.tasks and len(jobs) < B:
            return None
        if self.seed is None:
            self.seed = int(np.random.randint(0, 2 ** 62))
        ds.hemis_mask = None
        items, n_aux, stride = self._items(ents)
        if tr is not None:
            tr.append(('items', time.perf_counter()))
        outputs = self._outputs(total, n_aux, len(jobs))
        if tr is not None:
            tr.append(('outputs', time.perf_counter()))
        bufs = self._bufs(outputs, n_aux, stride)
        if tr is not None:
            tr.append(('workspaces', time.perf_counter()))
        arena = ds.arena.begin()
        if tr is not None:
            tr.append(('arena', time.perf_counter()))
        slot = arena.slots[arena.cur]
        descs = (_lib.GenSample * total)()
        descs_dev = C.c_void_p(0)
        info = (_lib.PlanInfo * B)()
        used = C.c_int64(0)
        _lib.check(L.bfm_plan_run(C.addressof(self.cfg), B, C.addressof(items), C.addressof(bufs), self.seed,
                                  self.counter, slot["host"].data_ptr(), slot["dev"].data_ptr(), arena.capacity,
                                  arena.used, C.byref(used), C.addressof(descs), C.byref(descs_dev), C.addressof(info),
                                  _stream()))
        if tr is not None:
            tr.append(('plan_run', time.perf_counter()))
        self.counter += B
        arena.used = arena.committed = used.value
        if jobs:                               # reads the descriptors and boxes of this arena slot: before mark_done
            ds._segmentation_stage(descs, descs_dev.value, total, jobs, out=outputs[4])
        arena.mark_done()
        self._keep_last(descs, descs_dev.value, info, arena, outputs, items, cls)
        if tr is not None:
            tr.append(('done', time.perf_counter()))
        return LazyItems(ds, ents, info, ns, outputs, cls)

    # ---- one batch ---------------------------------------------------------------------------------------
    def run(self, indices, timers=None, patch=None, plan_only=False):
        """Plan the batch in the library and run the fused chain.
        patch(descs): optional hook called after planning and BEFORE the descriptors travel to the device (slab
        mode sets x_begin / x_count there, which depend on the planned flip).  plan_only: stop after the upload and
        return the plan (descs, device address, info, output tensors) without launching any stage."""
        ds, L = self.ds, _lib.lib()
        ns, B = self.n_samples, len(indices)
        total = B * ns
        dev = self.device
        rng = ds.rng
        replay = getattr(rng, 'replay', False)
        if self.seed is None and not replay:
            self.seed = int(np.random.randint(0, 2 ** 62))
        ds.hemis_mask = None
        ents = [self._entry(int(i)) for i in indices]
        items, n_aux, stride = self._items(ents)
        cls = [None] * B if plan_only else self._seg_maps(ents)
        jobs = [(n * ns, c) for n, c in enumerate(cls) if c is not None]
        outputs = self._outputs(total, n_aux, len(jobs))
        bufs = self._bufs(outputs, n_aux, stride)
        outs = (_lib.PlanOut * total)()
        _lib.check(L.bfm_plan_layout(C.addressof(self.cfg), B, C.addressof(items), C.addressof(bufs),
                                     C.addressof(outs)))
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
            patch(descs)
            C.memmove(slot["host"].data_ptr() + (descs_dev.value - slot["dev"].data_ptr()), C.addressof(descs),
                      C.sizeof(descs))
        nbytes = (upload.value + 15) // 16 * 16
        _lib.check(L.bfm_upload_pinned(slot["dev"].data_ptr() + start, slot["host"].data_ptr() + start, nbytes, st))
        arena.committed = arena.used
        h, d_dev = C.addressof(descs), descs_dev.value
        if plan_only:
            self._keep_last(descs, d_dev, info, arena, outputs, keep)
            out, bfl, res, aux, _ = outputs
            return dict(descs=descs, d_dev=d_dev, info=info, out=out, bfl=bfl, res=res, aux=aux, arena=arena,
                        ents=ents)
        # ---- per-item context (targets that do not ride on the fused gather need a DeformPlan)
        need_plans = any(t in K.processing_funcs and t not in ('T1', 'T2', 'FLAIR', 'segmentation') for t in ds.tasks) \
            or ('segmentation' in ds.tasks and any(c is None for c in cls)) or not all(e['all_fused'] for e in ents)
        # the set-up dictionary is only read by the op-wise target readers (and kept as ds.last_setups)
        setups = [_setups(info[n]) if (need_plans or n == B - 1) else None for n in range(B)]
        deforms = [self._deform_dict(e['src'], descs[n * ns], info[n], arena) if need_plans else None
                   for n, e in enumerate(ents)]

        def read(n, key, target):
            ds.modalities = ents[n]['mods']
            return ds.read_and_deform_target(ents[n]['idx'], target.keys(), key, _INPUT_MODES[info[n].input_mode],
                                             setups[n], deforms[n])

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
        if jobs:
            ds._segmentation_stage(descs, d_dev, total, jobs, out=outputs[4], timers=timers)
        tuples = list(LazyItems(ds, ents, info, ns, outputs, cls, read))      # op-wise readers: after the bbox stage
        if timers is not None or need_plans:
            stage('gmm', L.bfm_gen_gmm)
            stage('warp', L.bfm_gen_warp)
            stage('resample', L.bfm_gen_resample)
            stage('finish', L.bfm_gen_finish)
        arena.mark_done()
        ds.last_setups, ds.last_deform = setups[-1], deforms[-1]
        self._keep_last(descs, d_dev, info, arena, outputs, cls, keep)
        return tuples

    def _deform_dict(self, src, desc, inf, arena):
        """A DeformDict around the planned deformation, for targets computed by the op-wise entry points."""
        plan = DeformPlan.__new__(DeformPlan)
        plan.size = list(self.size)
        plan.src = list(src)
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


def _setups(inf):
    """The set-up dictionary of a planned item (what get_setup_params returns)."""
    return {'resolution': np.array(inf.resolution[:]), 'thickness': np.array(inf.thickness[:]),
            'photo_mode': bool(inf.photo_mode), 'pathol_mode': False, 'pathol_random_shape': False,
            'spac': inf.spac if inf.photo_mode else None, 'flip': bool(inf.flip), 'hemis': 'both'}


def _case_name(t1_path):
    return os.path.basename(t1_path).split('.T1w.nii')[0]


def _absent(n, key, target):
    return {key: 0.}                  # read_and_deform_target of a file the subject does not have


class LazyItems:
    """The batch as collated device tensors (`input`: (B * n_samples, 1, *size), `bias_field_log`, `high_res_residual`,
    `targets[key]`: (B, 1, *size)) and, on demand, the reference-shaped per-item tuples
    `(datasets_num, dataset_name, input_mode, target, sample)` -- a sequence: len(), indexing and iteration build
    them.  `run_fast` returns it; `run` lists it, with `read(n, key, target)` computing the op-wise targets of item n
    (by default every target that neither rides on the fused gather nor comes from the segmentation stage is the 0. of
    a file the subject does not have)."""

    def __init__(self, ds, ents, info, ns, outputs, seg_maps, read=_absent):
        self._ds, self._ents, self._info, self._ns, self._read = ds, ents, info, ns, read
        self.input, self.bias_field_log, self.high_res_residual, self._aux, self._seg = outputs
        self._seg_maps = seg_maps
        self._built = None

    @property
    def targets(self):
        """{key: (n_items_with_that_target, 1, *size)} of the fused real-image targets, in item order, and
        'segmentation': the (B, n_classes, *size) one-hots when the task is on."""
        out, k = {}, 0
        for e in self._ents:
            for key in e['aux']:
                out.setdefault(key, []).append(self._aux[k])
                k += 1
        out = {key: torch.stack(v) for key, v in out.items()}
        if self._seg is not None:
            out['segmentation'] = self._seg
        return out

    def _build(self):
        if self._built is not None:
            return self._built
        ds, ns, info, read = self._ds, self._ns, self._info, self._read
        out_v = self.input.unbind(0)
        bfl_v = self.bias_field_log.unbind(0) if self.bias_field_log is not None else None
        res_v = self.high_res_residual.unbind(0) if self.high_res_residual is not None else None
        aux_v = iter(self._aux.unbind(0) if self._aux is not None else ())
        seg_v = iter(self._seg.unbind(0) if self._seg is not None else ())
        tuples = []
        for n, e in enumerate(self._ents):
            inf = info[n]
            target = defaultdict(ds._default_target)
            target['name'] = e['case_name']
            fused = {key: next(aux_v) for key in e['aux']}
            for key in ('T1', 'T2', 'FLAIR'):
                if key in fused:
                    target[key] = fused[key]
                elif key in e['mods']:
                    target.update(read(n, key, target))
                else:
                    target[key] = 0.
            for key in ds.tasks:
                if key == 'segmentation' and self._seg_maps[n] is not None:
                    target[key] = next(seg_v)
                elif key in K.processing_funcs and key not in ('T1', 'T2', 'FLAIR'):
                    target.update(read(n, key, target))
            target['pathology'] = 0.
            target['pathology_prob'] = 0.
            if e['age'] is not None:
                target['age'] = e['age']
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
            tuples.append((ds.datasets_num, e['dataset_name'], _INPUT_MODES[inf.input_mode], target, sample))
        self._built = tuples
        return tuples

    def __len__(self):
        return len(self._ents)

    def __getitem__(self, n):
        return self._build()[n]

    def __iter__(self):
        return iter(self._build())
