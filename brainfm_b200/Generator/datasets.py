"""BaseGen / BrainIDGen: the on-the-fly synthetic-data generator (mirror of Generator/datasets.py:25-757)
computed by libbfm's sm_100a kernels.

Same constructor, `__len__`, `__getitem__` 5-tuple, `names/mild_samples/all_samples` attributes, operator
registries and random-draw order as the reference.  Differences that are deliberate:
  * volumes are decoded once into a device-resident cache and cropped by indexing inside the gather kernels
    (no per-sample host crop + H2D);
  * the stock augmentation sequence ['gamma','bias_field','resample','noise'] runs as the fused batched chain
    (bfm_gen_*); any other sequence, or a re-registered operator, runs op by op through augmentation_funcs;
  * the two volume-sized N(0,1) fields are generated in-kernel (Philox) unless draws are injected.
"""
import ctypes as C
import glob
import os
from collections import defaultdict

import numpy as np
import torch
from torch.utils.data import Dataset

from .. import _lib, io as bio
from ..draws import HostDraws
from ..plan import Arena, band_host, device_tables, set_zoom_tab, zoom_newsize
from . import constants as K
from .utils import (DeformDict, DeformPlan, _stream, fast_3D_interp_torch, make_affine_matrix, myzoom_torch,
                    read_and_deform_image, resolution_sampler, scratch_stride)

ct_brightness_group = {
    'darker': [4, 5, 14, 15, 24, 31, 72],
    'dark': [2, 7, 16, 77, 30],
    'bright': [3, 8, 17, 18, 28, 10, 11, 12, 13, 26],
    'brighter': [],
}

_STOCK_STEPS = ['gamma', 'bias_field', 'resample', 'noise']

# partial-volume blend weights of get_contrast (datasets.py:452): 0.02 * torch.arange(50) in float32
_PV_V = np.arange(50).astype(np.float32) * np.float32(0.02)
_PV_W = np.float32(1) - _PV_V
_GMM_SCALE = np.array([[200], [20]], dtype=np.float32)     # mus = 25 + 200*u, sigmas = 5 + 20*u (datasets.py:432-433)
_GMM_SHIFT = np.array([[25], [5]], dtype=np.float32)


class BaseGen(Dataset):
    """BaseGen dataset (Generator/datasets.py:25-681)."""

    def __init__(self, gen_args, device='cuda', draws=None, planner='auto'):
        """planner: 'python' -- every item is planned in Python with draws from the numpy/torch global generators
        in the reference's order; 'native' -- batches are planned by the library (bfm_plan_batch, Generator/native.py;
        raises if the configuration needs the Python planner); 'auto' -- native whenever the configuration allows it
        and the draw source is the default one."""
        if not torch.cuda.is_available():
            raise _lib.BfmError("brainfm_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        _lib.lib()
        if planner not in ('auto', 'python', 'native'):
            raise ValueError("planner must be 'auto', 'python' or 'native'")
        self.planner = planner
        self._native = None
        self.gen_args = gen_args
        self.split = gen_args.split
        self.synth_args = self.gen_args.generator
        self.shape_gen_args = gen_args.pathology_shape_generator
        self.real_image_args = gen_args.real_image_generator
        self.synth_image_args = gen_args.synth_image_generator
        self.augmentation_steps = vars(gen_args.augmentation_steps)
        self.input_prob = vars(gen_args.modality_probs)
        self.device = torch.device('cuda' if device in ('cpu', None) else device)
        if self.device.type != 'cuda':
            raise _lib.BfmError("device must be a CUDA device")
        self.rng = draws or HostDraws()
        self.cache = bio.shared_cache(self.device)     # one cache per device, shared with the op-wise target readers
        self.arena = Arena(self.device)
        self.tables = device_tables(self.device)
        self._ws = {}                  # persistent device scratch of the fused chain (see _workspace)
        # float2 {synthetic, T1} pairs in `syn` + k_gen_warp_pk for samples with one fused target (bfm.h: syn_pair_ok)
        self.pair_mode = os.environ.get('BFM_PAIR_MODE', '1') != '0'
        self._info = {}                # t1 path -> modality table
        self._inputs = {}              # volume path -> (img, aff, res)
        self._c2 = {}                  # source shape -> centre (float32)
        self._hemis_key = ()           # (segmentation path, registration path) of the current left-hemisphere mask
        self.hemis_mask = None
        self.write_bflog = None        # None: follow the task list; True/False: force
        self.prepare_tasks()
        self.prepare_paths()
        self.prepare_grid()
        self.prepare_one_hot()
        self.tables.prebuild(self.size)

    def __len__(self):
        return sum([len(self.names[i]) for i in range(len(self.names))])

    # ---- bookkeeping (datasets.py:52-184) --------------------------------------------------------
    def idx_to_path(self, idx):
        cnt = 0
        for i, l in enumerate(self.datasets_len):
            if cnt <= idx < cnt + l:
                name = self.names[i][idx - cnt]
                age = self.ages[i][os.path.basename(name).split('.T1w')[0]] if len(self.ages) > 0 else None
                return self.datasets[i], vars(self.input_prob[self.datasets[i]]), name, age
            cnt += l
        raise IndexError(idx)

    def prepare_paths(self):
        if len(self.gen_args.dataset_names) < 1:
            datasets = []
            for g in glob.glob(os.path.join(self.gen_args.data_root, '*' + 'T1w.nii')):
                d = os.path.basename(g)
                d = d[:d.find('.')]
                if d not in datasets:
                    datasets.append(d)
        else:
            datasets = self.gen_args.dataset_names
        names = []
        if 'age' in self.tasks:
            self.split = self.split + '_age'
        if self.gen_args.split_root is not None:
            with open(os.path.join(self.gen_args.split_root, self.split + '.txt'), 'r') as f:
                split_names = [s.strip() for s in f.readlines()]
            for d in datasets:
                names.append([n for n in split_names if os.path.basename(n).startswith(d)])
        ages = []
        if 'age' in self.tasks:
            with open(os.path.join(self.gen_args.split_root, 'participants_age.txt'), 'r') as f:
                rows = [line.strip().split(' ') for line in f.readlines()]
            for d in datasets:
                ages.append({n: float(a) for n, a in rows if n.startswith(d)})
        self.ages = ages
        self.names = names
        self.datasets = datasets
        self.datasets_num = len(datasets)
        self.datasets_len = [len(n) for n in names]
        self.pathology_type = None

    def prepare_tasks(self):
        self.tasks = [key for (key, value) in vars(self.gen_args.task).items() if value]
        if 'bias_field' in self.tasks and 'segmentation' not in self.tasks:
            self.tasks += ['segmentation']
        self.t, self.adv_pde = None, None
        if 'pathology' in self.tasks and self.synth_args.augment_pathology and self.synth_args.random_shape_prob < 1.:
            from ..ShapeID.DiffEqs.pde import AdvDiffPDE
            self.t = torch.from_numpy(np.arange(self.shape_gen_args.max_nt) * self.shape_gen_args.dt).to(self.device)
            self.adv_pde = AdvDiffPDE(data_spacing=[1., 1., 1.], perf_pattern='adv', V_type='vector_div_free',
                                      V_dict={}, BC=self.shape_gen_args.bc, dt=self.shape_gen_args.dt,
                                      device=self.device)

    def prepare_grid(self):
        self.size = list(self.synth_args.size)
        self.res_training_data = np.array([1.0, 1.0, 1.0])
        self.c = torch.tensor((np.array(self.size) - 1) / 2, dtype=torch.float)

    def prepare_one_hot(self):
        if self.synth_args.left_hemis_only:
            label_list = K.label_list_segmentation_brainseg_left
        else:
            label_list = K.label_list_segmentation_brainseg_with_extracerebral
        n_labels = len(label_list)
        lut = torch.zeros(10000, dtype=torch.long)
        for l in range(n_labels):
            lut[label_list[l]] = l
        self.lut = lut.to(self.device)
        self.onehotmatrix = torch.eye(n_labels, dtype=torch.float, device=self.device)
        nn_ = K.n_neutral_labels_brainseg_with_extracerebral
        nlat = int((n_labels - nn_) / 2.0)
        self.vflip = np.concatenate([np.array(range(nn_)), np.array(range(nn_ + nlat, n_labels)),
                                     np.array(range(nn_, nn_ + nlat))])

    def get_info(self, t1):
        hit = self._info.get(t1)
        if hit is not None:
            self.modalities = dict(hit)
            return self.modalities
        stem = t1[:-7]
        self.modalities = {'T1': t1, 'Gen': stem + 'generation_labels.nii',
                           'segmentation': stem + self.gen_args.segment_prefix + '.nii',
                           'distance': [stem + 'lp_dist_map.nii', stem + 'lw_dist_map.nii', stem + 'rp_dist_map.nii',
                                        stem + 'rw_dist_map.nii'],
                           'registration': [stem + 'mni_reg.x.nii', stem + 'mni_reg.y.nii', stem + 'mni_reg.z.nii']}
        for key, suffix in (('T1_DM', 'T1w.defacingmask.nii'), ('T2', 'T2w.nii'), ('T2_DM', 'T2w.defacingmask.nii'),
                            ('FLAIR', 'FLAIR.nii'), ('FLAIR_DM', 'FLAIR.defacingmask.nii'), ('CT', 'CT.nii'),
                            ('CT_DM', 'CT.defacingmask.nii')):
            if bio.exists(stem + suffix):
                self.modalities[key] = stem + suffix
        self._info[t1] = dict(self.modalities)
        return self.modalities

    # ---- random setup (datasets.py:466-493, 563-590) ---------------------------------------------
    def read_input(self, idx):
        dataset_name, input_prob, t1_path, age = self.idx_to_path(idx)
        case_name = os.path.basename(t1_path).split('.T1w.nii')[0]
        self.modalities = self.get_info(t1_path)
        prob = self.rng.rand("input.mode")
        input_mode = 'synth'
        for m in ('T1', 'T2', 'FLAIR', 'CT'):
            if prob < input_prob[m] and m in self.modalities:
                input_mode = m
                break
        path = self.modalities['Gen' if input_mode == 'synth' else input_mode]
        hit = self._inputs.get(path)
        if hit is None:
            img = bio.load(path)
            aff = img.affine
            hit = (img, aff, np.sqrt(np.sum(abs(aff[:-1, :-1]), axis=0)))
            self._inputs[path] = hit
        img, aff, res = hit
        return dataset_name, case_name, input_mode, img, aff, res, age

    def get_setup_params(self):
        a, rng = self.synth_args, self.rng
        hemis = 'left' if a.left_hemis_only else 'both'
        if a.low_res_only:
            photo_mode = False
        elif a.left_hemis_only:
            photo_mode = True
        else:
            photo_mode = rng.rand("setup.photo") < a.photo_prob
        pathol_mode = rng.rand("setup.pathol") < a.pathology_prob
        pathol_random_shape = rng.rand("setup.rshape") < a.random_shape_prob
        spac = 2.5 + 10 * rng.rand("setup.spac") if photo_mode else None
        flip = rng.randn("setup.flip") < a.flip_prob if not a.left_hemis_only else False
        if photo_mode:
            resolution = np.array([self.res_training_data[0], spac, self.res_training_data[2]])
            thickness = np.array([self.res_training_data[0], 0.1, self.res_training_data[2]])
        else:
            resolution, thickness = resolution_sampler(a.low_res_only, draws=rng)
        return {'resolution': resolution, 'thickness': thickness, 'photo_mode': photo_mode, 'pathol_mode': pathol_mode,
                'pathol_random_shape': pathol_random_shape, 'spac': spac, 'flip': flip, 'hemis': hemis}

    # ---- deformation (datasets.py:187-303) --------------------------------------------------------
    def random_affine_transform(self, shp):
        """A (3,3) and c2 (3,) as float32 numpy arrays (the reference's float32 tensors, datasets.py:187-201).
        The per-component float64 arithmetic is evaluated on python floats (same IEEE operations in the same
        order as the reference's numpy expressions on 3-vectors)."""
        a, rng = self.synth_args, self.rng
        mr, ms, mc = a.max_rotation, a.max_shear, a.max_scaling
        rotations = np.array([(2 * mr * u - mr) / 180.0 * np.pi for u in rng.rand3("aff.rot").tolist()])
        shears = [(2 * ms * u - ms) for u in rng.rand3("aff.shear").tolist()]
        scalings = [1 + (2 * mc * u - mc) for u in rng.rand3("aff.scale").tolist()]
        scaling_factor_distances = (scalings[0] * scalings[1] * scalings[2]) ** .33333333333
        A = make_affine_matrix(rotations, shears, scalings).astype(np.float32)
        key = tuple(int(v) for v in shp[0:3])
        c2 = self._c2.get(key)
        if c2 is None:
            c2 = self._c2[key] = ((np.array(key) - 1) / 2).astype(np.float32)
        if a.random_shift:
            max_shift = torch.tensor(np.array(shp[0:3]) - self.size, dtype=torch.float) / 2
            max_shift[max_shift < 0] = 0
            c2 = (torch.from_numpy(c2) + (2 * (max_shift * rng.torch_rand("aff.shift", 3, dtype=torch.float64))
                                          - max_shift)).to(torch.float32).numpy()
        return scaling_factor_distances, A, c2

    def random_nonlinear_transform(self, photo_mode, spac, arena=None):
        """Returns the SMALL random grid (host float32, [sx,sy,sz,3]) and, with an arena, its device address:
        the draw is written straight into the pinned plan arena.  The full-resolution field F is never
        materialised unless somebody reads deform_dict['F'] or the SVF integration is requested."""
        a, rng = self.synth_args, self.rng
        nonlin_scale = a.nonlin_scale_min + float(rng.rand1("nl.scale")[0]) * (a.nonlin_scale_max - a.nonlin_scale_min)
        size_F_small = [int(round(nonlin_scale * n)) for n in self.size]     # np.round: half to even, like round()
        if photo_mode:
            size_F_small[1] = int(round(self.size[1] / spac))
        nonlin_std = a.nonlin_std_max * rng.rand("nl.std")
        shape = [*size_F_small, 3]
        if arena is None:
            return nonlin_std * rng.torch_randn("nl.field", shape), None
        dev, view = arena.alloc_tensor(shape)
        rng.torch_randn("nl.field", shape, out=view)
        view.mul_(float(nonlin_std))
        return view, dev

    def _full_field(self, Fsmall, photo_mode):
        F = myzoom_torch(Fsmall.to(self.device), np.array(self.size) / np.array(Fsmall.shape[:3]))
        if photo_mode:
            F[:, :, :, 1] = 0
        return F

    def _integrate_svf(self, F):
        n = self.synth_args.n_steps_svf_integration
        L = _lib.lib()
        F = F.contiguous()
        if F.dtype == torch.float32 and F.is_cuda:
            # one library call; the field stays in 16-byte records between the steps (bfm_svf_integrate)
            out = torch.empty_like(F)
            scratch = torch.empty(2 * 4 * int(np.prod(self.size)), dtype=torch.float32, device=F.device)
            _lib.check(L.bfm_svf_integrate(F.data_ptr(), out.data_ptr(), *[int(v) for v in self.size], int(n),
                                           float(1.0 / (2.0 ** n)), scratch.data_ptr(), _stream()))
            return out
        cur = (F * (1.0 / (2.0 ** n))).contiguous()
        nxt = torch.empty_like(cur)
        for _ in range(n):
            _lib.check(L.bfm_svf_step(cur.data_ptr(), nxt.data_ptr(), *self.size, _stream()))
            cur, nxt = nxt, cur
        return cur

    def generate_deformation(self, setups, shp, arena=None, lazy=False):
        scaling_factor_distances, A, c2 = self.random_affine_transform(shp)
        Fsmall, F, Fneg, fdev = None, None, None, None
        if self.synth_args.nonlinear_transform:
            Fsmall, fdev = self.random_nonlinear_transform(setups['photo_mode'], setups['spac'], arena)
            if 'surface' in self.tasks:
                full = self._full_field(Fsmall, setups['photo_mode'])
                F, Fneg = self._integrate_svf(full), self._integrate_svf(-full)
        plan = DeformPlan(self.size, shp, A, c2,
                          None if (Fsmall is None or F is not None) else Fsmall.numpy(), setups['photo_mode'],
                          self.device, F_full=F, arena=arena, lazy=lazy, fsmall_dev=fdev)
        # 'A', 'c2' and 'F' (device tensors in the reference) are materialised on first access
        d = DeformDict({'scaling_factor_distances': scaling_factor_distances, 'Fneg': Fneg, '_plan': plan,
                        '_Fsmall': None if Fsmall is None else Fsmall.clone(), '_photo': setups['photo_mode']})
        if F is not None or Fsmall is None:
            d['F'] = F
        return d

    def deform_grid(self, shp, A, c2, F):
        """Reference-shaped entry point (datasets.py:264-303): F is a full-resolution field or None."""
        plan = DeformPlan(self.size, shp, A.detach().cpu().numpy(), c2.detach().cpu().float().numpy(), None, False,
                          self.device, F_full=None if F is None else F.contiguous().float())
        xx2, yy2, zz2 = plan.coords()
        return (xx2, yy2, zz2, *plan.bbox_host())

    def get_left_hemis_mask(self, grid):
        """Left-hemisphere mask (datasets.py:251-262): (lut[seg] > 0) & (MNI x < 0).  The reference evaluates it on
        the bounding-box crop of every sample; here it is a FULL-volume uint8 device tensor computed once per
        subject (the kernels index the full source volume, and the crop of the full mask is the crop's mask)."""
        if not self.synth_args.left_hemis_only:
            self.hemis_mask = None
            return
        key = (self.modalities['segmentation'], self.modalities['registration'][0])

        def build():
            S = self.cache.get(key[0], 'i32')
            X = self.cache.get(key[1], 'f32')
            return ((self.lut[S.long()] > 0) & (X < 0)).to(torch.uint8)
        self.hemis_mask = self.cache.derived('left_hemis_mask', key, build)     # dropped when a dependency is uploaded
        self._hemis_key = key

    # ---- targets (datasets.py:593-631) -------------------------------------------------------------
    def read_and_deform_target(self, idx, exist_keys, task_name, input_mode, setups, deform_dict, linear_weights=None):
        if task_name == 'pathology':
            p_prob_path, augment, thres = None, False, 0.1
            if self.pathology_type is None and setups['pathol_mode']:
                if setups['pathol_random_shape']:
                    p_prob_path, augment, thres = 'random_shape', False, self.shape_gen_args.pathol_thres
                else:
                    p_prob_path = self.rng.choice("pathol.path", K.pathology_prob_paths)
                    augment, thres = self.synth_args.augment_pathology, self.shape_gen_args.pathol_thres
            return K.processing_funcs[task_name](exist_keys, task_name, p_prob_path, setups, deform_dict, self.device,
                                                 mask=self.hemis_mask, augment=augment, pde_func=self.adv_pde,
                                                 t=self.t, shape_gen_args=self.shape_gen_args, thres=thres,
                                                 draws=self.rng)
        if task_name in self.modalities:
            return K.processing_funcs[task_name](exist_keys, task_name, self.modalities[task_name], setups,
                                                 deform_dict, self.device, mask=self.hemis_mask, cfg=self.gen_args,
                                                 onehotmatrix=self.onehotmatrix, lut=self.lut, vflip=self.vflip)
        return {task_name: 0.}

    def update_gen_args(self, new_args):
        for key, value in vars(new_args).items():
            vars(self.gen_args.generator)[key] = value

    # ---- contrast (datasets.py:430-464) ------------------------------------------------------------
    def get_contrast(self, photo_mode, out=None):
        """256-entry mean / std tables incl. partial-volume blends (datasets.py:430-464).  The random draws are
        torch's; the blends are evaluated in numpy float32 with the reference's operation order (every product
        and sum separately rounded): the means reproduce the torch float32 results bit for bit; the blended
        stds can differ in the last bit because torch's CPU sqrt (MKL vsSqrt) is not correctly rounded
        while numpy's is.  `out`: optional (2, 256) float32 CPU tensor (a view of the plan arena) that receives
        the two tables in place."""
        rng = self.rng
        if out is None:
            out = torch.empty((2, 256), dtype=torch.float32)
        mus, sigmas = out[0], out[1]
        rng.torch_rand("gmm.mu", 256, out=mus)
        rng.torch_rand("gmm.sigma", 256, out=sigmas)
        ms = out.numpy()
        # 25 + 200*u, 5 + 20*u in float32: product then sum, separately rounded, as torch evaluates them
        np.multiply(ms, _GMM_SCALE, out=ms)
        np.add(ms, _GMM_SHIFT, out=ms)
        m, sg = ms[0], ms[1]
        if rng.rand("gmm.ct") < self.synth_args.ct_prob:
            for name, (base, span) in (('darker', (25, 10)), ('dark', (90, 20)), ('bright', (110, 20)),
                                       ('brighter', (150, 50))):
                v = base + span * rng.torch_rand("gmm.ct." + name, 1)[0]
                for l in ct_brightness_group[name]:
                    mus[l] = v
        if photo_mode or rng.rand1("gmm.bg") < 0.5:
            m[0] = 0
        # labels 100-149 / 150-199 / 200-249 blend classes (1,2) / (2,3) / (3,4): three rows at once
        m[100:250].reshape(3, 50)[:] = m[1:4, None] * _PV_W + m[2:5, None] * _PV_V
        m[250] = m[4]
        q = sg[:5] * sg[:5]
        sg[100:250].reshape(3, 50)[:] = np.sqrt(q[1:4, None] * _PV_W + q[2:5, None] * _PV_V)
        sg[250] = sg[4]
        return mus, sigmas

    # ---- host-side plan of one synthetic sample (all scalar draws, reference order) ----------------
    def _stock_chain(self, input_mode):
        steps = self.augmentation_steps['synth'] if input_mode == 'synth' else self.augmentation_steps['real']
        return list(steps) == _STOCK_STEPS and all(K.augmentation_funcs.get(k) is K._STOCK_AUGMENTATION[k]
                                                   for k in _STOCK_STEPS)

    def _plan_synth(self, setups, target, arena=None, real=False):
        """Draws of generate_sample + the stock augmentation chain, in the reference's order
        (datasets.py:357-428, utils.py:568-638).  With an arena the array-shaped draws (mean/std tables, bias
        grid) are written straight into the pinned plan arena and `p` carries their device addresses."""
        cfg, rng, size = self.gen_args.generator, self.rng, self.size
        p = {'real': real}
        if real:
            # real-image input (augment_sample, datasets.py:306-336): no contrast, no GMM noise, no mixing draw
            p['mu'] = p['sigma'] = p['eps_gmm'] = p['mix'] = None
        else:
            if arena is not None:
                p['musigma_dev'], ms = arena.alloc_tensor((2, 256))
                p['mu'], p['sigma'] = self.get_contrast(setups['photo_mode'], out=ms)
            else:
                p['mu'], p['sigma'] = self.get_contrast(setups['photo_mode'])
            p['eps_gmm'] = rng.field_randn("gmm.eps")
            p['mix'] = None
            if rng.rand("mix.u") < self.gen_args.mix_synth_prob:
                v = rng.torch_rand("mix.v", 4)
                v[2] = 0 if 'T2' not in self.modalities else v[2]
                v[3] = 0 if 'FLAIR' not in self.modalities else v[3]
                v /= torch.sum(v)
                p['mix'] = v
        # gamma
        p['gamma'] = np.float32(np.exp(cfg.gamma_std * rng.randn1("gamma.n")))
        # bias field (none for CT inputs, utils.py:575-577)
        if real == 'CT':
            p['bfsmall'], p['bf_shape'] = None, None
            return self._plan_tail(p, setups, cfg, rng, size)
        bf_scale = cfg.bf_scale_min + float(rng.rand1("bf.scale")[0]) * (cfg.bf_scale_max - cfg.bf_scale_min)
        small = [int(round(bf_scale * n)) for n in size]                    # np.round: half to even, like round()
        if setups['photo_mode']:
            small[1] = int(round(size[1] / setups['spac']))
        std = float(np.float32(cfg.bf_std_min + (cfg.bf_std_max - cfg.bf_std_min) * float(rng.rand1("bf.std")[0])))
        if arena is not None:
            p['bfsmall_dev'], bf = arena.alloc_tensor(small)
            rng.torch_randn("bf.field", small, out=bf)
        else:
            bf = rng.torch_randn("bf.field", small)
        p['bfsmall'] = bf.mul_(std).numpy()                                  # float32(std) * randn, in float32
        p['bf_shape'] = small
        return self._plan_tail(p, setups, cfg, rng, size)

    def _plan_tail(self, p, setups, cfg, rng, size):
        # resample
        res = self.res_training_data
        stds = (0.85 + 0.3 * rng.rand("rs.u")) * np.log(5) / np.pi * setups['thickness'] / res
        stds[setups['thickness'] <= res] = 0.0
        p['stds'] = stds
        p['new_size'] = (np.array(size) * res / setups['resolution']).astype(int)
        p['factors'] = np.array(p['new_size']) / np.array(size)
        # noise
        u = rng.rand1("noise.u")
        p['noise_std'] = np.float32((cfg.noise_std_min + (cfg.noise_std_max - cfg.noise_std_min) * u)[0])
        p['eps_noise'] = rng.field_randn("noise.eps")
        p['seed'] = rng.seed64()
        return p

    # ---- fused batched launch ----------------------------------------------------------------------
    def _workspace(self, name, numel, dtype=torch.float32, zero=False):
        """Persistent device scratch of the fused chain, grown on demand.  Reuse across batches is safe because
        all work is ordered on one stream; nothing in here is ever returned to the caller."""
        t = self._ws.get(name)
        if t is None or t.numel() < numel:
            t = (torch.zeros if zero else torch.empty)(int(numel), dtype=dtype, device=self.device)
            self._ws[name] = t
        return t

    def _build_descs(self, jobs, arena):
        """Fill one bfm_gen_sample per job.  Per sample only the small random grids and the two 256-entry
        tables travel through the arena; zoom tables come from the device-resident cache, the banded
        blur-o-downsample tables are built on the GPU (bfm_gen_plan), scratch volumes are persistent.
        jobs: dicts(plan=DeformPlan, flip, labels, p=<_plan_synth>, want_bflog, want_residual, aux=[(key, vol)])."""
        B = len(jobs)
        dev, size, tables = self.device, tuple(self.size), self.tables
        N = int(np.prod(size))
        descs = (_lib.GenSample * B)()
        out = torch.empty((B, 1, *size), dtype=torch.float32, device=dev)
        n_bfl = sum(1 for j in jobs if j['want_bflog'])
        n_res = sum(1 for j in jobs if j['want_residual'])
        n_aux = sum(len(j.get('aux') or ()) for j in jobs)
        bfl_all = torch.empty((n_bfl, 1, *size), dtype=torch.float32, device=dev) if n_bfl else None
        res_all = torch.empty((n_res, 1, *size), dtype=torch.float32, device=dev) if n_res else None
        aux_all = torch.empty((n_aux, 1, *size), dtype=torch.float32, device=dev) if n_aux else None
        # persistent scratch: syn is zero-initialised once and afterwards only ever holds finite values
        src_pad = max(int(np.prod(j['plan'].src)) + j['plan'].src[1] * j['plan'].src[2] + j['plan'].src[2] + 1
                      for j in jobs)
        src_pad = 2 * ((src_pad + 3) // 4 * 4)         # room for float2 {synthetic, T1} pairs (syn_pair_ok)
        syn_ws = self._workspace('syn', B * src_pad, zero=True)
        if self._ws.get('syn_stride') != src_pad:      # slots moved: stale data no longer lines up, start clean
            if 'syn_stride' in self._ws:
                syn_ws.zero_()
            self._ws['syn_stride'] = src_pad
        Np = scratch_stride(N)
        i_bf_ws = self._workspace('i_bf', B * Np)
        tmp_ws = self._workspace('tmp', B * 2 * Np)
        low_ws = self._workspace('lowres', B * Np)
        raw_ws = self._workspace('aux_raw', n_aux * Np) if n_aux else None
        p_syn, p_ibf, p_tmp, p_low = syn_ws.data_ptr(), i_bf_ws.data_ptr(), tmp_ws.data_ptr(), low_ws.data_ptr()
        keep = [out, bfl_all, res_all, aux_all]
        results = []
        k_bfl = k_res = k_aux = 0
        for b, job in enumerate(jobs):
            s, p, plan = descs[b], job['p'], job['plan']
            s.d = plan.struct
            if p.get('real'):
                # the warp gathers straight from the cached (finite, padded) real volume; nothing is synthesised
                s.real_input = 2 if p['real'] == 'CT' else 1
                s.syn = job['real_vol'].data_ptr()
            else:
                lab = job['labels']
                s.labels = lab.data_ptr()
                s.label_is_u8 = 1 if lab.dtype == torch.uint8 else 0
                if 'musigma_dev' in p:
                    s.mu, s.sigma = p['musigma_dev'], p['musigma_dev'] + 1024
                else:
                    s.mu = arena.put(p['mu'].numpy())
                    s.sigma = arena.put(p['sigma'].numpy())
                if p['eps_gmm'] is not None:
                    e = p['eps_gmm'].to(dev).contiguous()
                    keep.append(e)
                    s.eps_gmm = e.data_ptr()
                s.syn = p_syn + 4 * b * src_pad
                s.syn_pair_ok = 1 if self.pair_mode else 0
            s.seed = int(p['seed'])
            s.bbox = plan.bbox_ptr
            if p['mix'] is not None:
                for q in range(4):
                    s.mixw[q] = float(p['mix'][q])
            s.gamma = float(p['gamma'])
            bfs = p['bfsmall']
            if bfs is not None:
                s.bfsmall = p['bfsmall_dev'] if 'bfsmall_dev' in p else arena.put(bfs)
                s.bs[:] = bfs.shape
                s.btab = tables.zoom_tab(bfs.shape, size)
            s.i_bf = p_ibf + 4 * b * Np
            sample = {}
            if job['want_bflog']:
                s.bflog_out = bfl_all[k_bfl].data_ptr()
                sample['bias_field_log'] = bfl_all[k_bfl]
                k_bfl += 1
            s.flip = 1 if job['flip'] else 0
            s.zoom_order = 3 if self.synth_args.bspline_zooming else 0
            # resolution degradation: banded passes in ascending factor order, identity axes folded away
            new = [int(v) for v in p['new_size']]
            order = sorted(range(3), key=lambda a: new[a] / size[a])
            nb = 0
            for a in order:
                sigma = float(p['stds'][a])
                if new[a] == size[a] and sigma == 0:
                    s.zero_first[a] = 1
                    continue
                bd = s.band[nb]
                half = int(np.ceil(3 * sigma)) if sigma > 0 else 0
                T = 2 * half + 2
                if T <= 64:
                    # tables built on the device by bfm_gen_plan into arena scratch
                    bd.start, _ = arena.reserve(4 * new[a])
                    bd.w, _ = arena.reserve(4 * new[a] * T)
                    bd.T, bd.build, bd.sigma = T, 1, sigma
                else:
                    start, w, T = band_host(size[a], new[a], sigma)
                    bd.start, bd.w, bd.T, bd.build = arena.put(start), arena.put(w), T, 0
                bd.n_in, bd.n_out, bd.axis = size[a], new[a], a
                nb += 1
            if nb == 0:
                bd = s.band[0]
                bd.start = arena.put(np.arange(size[2], dtype=np.int32))
                bd.w = arena.put(np.ones(size[2], dtype=np.float32))
                bd.T, bd.n_in, bd.n_out, bd.axis, bd.build = 1, size[2], size[2], 2, 0
                nb = 1
            s.n_band = nb
            s.noise_std = float(p['noise_std'])
            if p['eps_noise'] is not None:
                e = p['eps_noise'].to(dev).contiguous()
                keep.append(e)
                s.eps_noise = e.data_ptr()
            s.tmp[0] = p_tmp + 4 * (2 * b) * Np
            s.tmp[1] = p_tmp + 4 * (2 * b + 1) * Np
            s.lowres = p_low + 4 * b * Np
            s.new_size[:] = new
            s.utab = tables.zoom_tab(new, size, inverse=True)
            s.maxval, _ = arena.reserve(16)
            s.out = out[b].data_ptr()
            if job['want_residual']:
                s.residual = res_all[k_res].data_ptr()
                sample['high_res_residual'] = res_all[k_res]
                k_res += 1
            # real-image targets warped by the same gather (read_and_deform_image)
            aux = job.get('aux') or ()
            s.n_aux = len(aux)
            job['aux_out'] = {}
            if aux:
                s.aux_mm, _ = arena.reserve(8 * _lib.MAX_AUX)
            for c, (key, vol) in enumerate(aux):
                s.aux_src[c] = vol.data_ptr()
                s.aux_raw[c] = raw_ws.data_ptr() + 4 * k_aux * Np
                s.aux_out[c] = aux_all[k_aux].data_ptr()
                job['aux_out'][key] = aux_all[k_aux]
                k_aux += 1
            sample['input'] = out[b]
            job['_new_size'] = new
            # key order of the reference's sample dict (datasets.py:345-352)
            results.append({k: sample[k] for k in ('high_res_residual', 'input', 'bias_field_log') if k in sample})
        self._keep = keep
        self._last_out = out
        return descs, results

    def _run_chain(self, jobs, arena, targets_fn=None, timers=None):
        """Planned jobs -> device.  Stage order: plan + bbox (batched) -> targets_fn() (per-sample target
        kernels, which need the bbox and may feed the mixing step) -> gmm -> warp -> resample -> finish (all
        batched)."""
        L = _lib.lib()
        B = len(jobs)
        descs, results = self._build_descs(jobs, arena)
        d_dev = arena.put_struct_array(descs)
        arena.commit()
        h = C.addressof(descs)
        st = _stream()

        def stage(name, fn, dptr):
            if timers is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            _lib.check(fn(h, dptr, B, st))
            if timers is not None:
                e1.record()
                timers.setdefault(name, []).append((e0, e1))

        stage('plan', L.bfm_gen_plan, d_dev)
        stage('bbox', L.bfm_gen_bbox, d_dev)
        for job in jobs:
            job['plan'].have_bbox = True
        if targets_fn is not None:
            if timers is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            targets_fn()
            if timers is not None:
                e1.record()
                timers.setdefault('targets', []).append((e0, e1))
            patched = False
            for b, job in enumerate(jobs):
                if job['p']['mix'] is None:
                    continue
                tg = job['target']
                mt = [tg['T1'][0].contiguous(),
                      tg['T2'][0].contiguous() if 'T2' in job['modalities'] else None,
                      tg['FLAIR'][0].contiguous() if 'FLAIR' in job['modalities'] else None]
                for q, t in enumerate(mt):
                    if t is not None:
                        self._keep.append(t)
                        descs[b].mix[q] = t.data_ptr()
                patched = True
            if patched:
                d_dev = arena.put_struct_array(descs)
                arena.commit()
        stage('gmm', L.bfm_gen_gmm, d_dev)
        stage('warp', L.bfm_gen_warp, d_dev)
        stage('resample', L.bfm_gen_resample, d_dev)
        stage('finish', L.bfm_gen_finish, d_dev)
        arena.mark_done()
        self._last_descs = (descs, d_dev, B)
        return results

    def _labels(self):
        lab = self.cache.get(self.modalities['Gen'], 'gen')
        if self.hemis_mask is None:
            return lab
        mask = self.hemis_mask                                # G[hemis_mask == 0] = 0 (datasets.py:367-368)
        return self.cache.derived('gen_masked', (self.modalities['Gen'],) + tuple(self._hemis_key),
                                  lambda: torch.where(mask != 0, lab, torch.zeros((), dtype=lab.dtype,
                                                                                  device=lab.device)).contiguous())

    def _want_bflog(self, input_mode):
        if input_mode == 'CT':                          # no bias field on CT (utils.py:575-577, datasets.py:351)
            return False
        if self.write_bflog is not None:
            return bool(self.write_bflog)
        return 'bias_field' in self.tasks and input_mode != 'CT'

    def _job(self, setups, deform_dict, target, p, input_mode='synth'):
        real = input_mode != 'synth'
        return dict(plan=deform_dict['_plan'], flip=setups['flip'], labels=None if real else self._labels(), p=p,
                    real_vol=self.cache.get(self.modalities[input_mode], 'f32') if real else None,
                    target=target, modalities=dict(self.modalities), want_bflog=self._want_bflog(input_mode),
                    want_residual='super_resolution' in self.tasks)

    # ---- reference-shaped sample generation ---------------------------------------------------------
    def generate_sample(self, name, G, setups, deform_dict, res, target):
        """GMM synthesis + augmentation of one sample (datasets.py:357-428)."""
        P = target['pathology'] if 'pathology' in target else None
        has_pathol = isinstance(P, torch.Tensor) and bool(P.sum() > 0)       # host sync, datasets.py:390
        if has_pathol or not self._stock_chain('synth'):
            return self._generate_sample_opwise(setups, deform_dict, res, target, has_pathol)
        deform_dict['_plan'].compute_bbox()
        p = self._plan_synth(setups, target)
        arena = self.arena.begin()
        sample = self._run_chain([self._job(setups, deform_dict, target, p)], arena, targets_fn=lambda: None)[0]
        target['pathology'] = 0.
        target['pathology_prob'] = 0.
        return target['pathology'], target['pathology_prob'], sample

    def _generate_sample_opwise(self, setups, deform_dict, res, target, has_pathol=False):
        """Op-by-op path through the registries (custom or reordered augmentation steps, pathology encoding)."""
        rng = self.rng
        L, st = _lib.lib(), _stream()
        mus, sigmas = self.get_contrast(setups['photo_mode'])
        xx2, yy2, zz2, x1, y1, z1, x2, y2, z2 = deform_dict['grid']
        # GMM image over the bbox crop (datasets.py:364-372): one kernel reading the cached label volume in place
        lab = self._labels()
        src = (C.c_int * 3)(*[int(v) for v in lab.shape[:3]])
        box = (C.c_int * 6)(int(x1), int(y1), int(z1), int(x2), int(y2), int(z2))
        crop = (int(x2 - x1), int(y2 - y1), int(z2 - z1))
        lab_u8 = 1 if lab.dtype == torch.uint8 else 0
        if not lab_u8 and lab.dtype != torch.float32:
            lab = lab.float()
        eps = rng.field_randn("gmm.eps")
        eps = None if eps is None else eps.to(self.device, torch.float32).contiguous()
        tab = torch.stack([mus.float(), sigmas.float()]).to(self.device)          # (2, 256), one upload
        SYN = torch.empty(crop, dtype=torch.float32, device=self.device)
        _lib.check(L.bfm_gmm_crop(lab.data_ptr(), lab_u8, src, box, tab[0].data_ptr(), tab[1].data_ptr(),
                                  0 if eps is None else eps.data_ptr(), int(rng.seed64()) if eps is None else 0,
                                  SYN.data_ptr(), st))
        SYN = fast_3D_interp_torch(SYN.contiguous(), xx2, yy2, zz2)
        if rng.rand("mix.u") < self.gen_args.mix_synth_prob:
            v = rng.torch_rand("mix.v", 4)
            v[2] = 0 if 'T2' not in self.modalities else v[2]
            v[3] = 0 if 'FLAIR' not in self.modalities else v[3]
            v /= torch.sum(v)
            SYN = v[0] * SYN + v[1] * target['T1'][0]
            if 'T2' in self.modalities:
                SYN += v[2] * target['T2'][0]
            if 'FLAIR' in self.modalities:
                SYN += v[3] * target['FLAIR'][0]
        if has_pathol:
            # datasets.py:390-406, quirks included: the masks have the crop's shape, so this branch (like the
            # reference's) only works when the crop covers the whole output shape; SYN_cerebral is warped twice
            if tuple(SYN.shape) != crop:
                raise RuntimeError("pathology encoding needs the bbox crop to cover the output shape "
                                   "(the reference's masks have the crop's shape, datasets.py:391-400)")
            SYN = SYN.contiguous()
            SYN_cerebral = torch.empty_like(SYN)
            sums = torch.empty(4, dtype=torch.float64, device=self.device)
            _lib.check(L.bfm_pathol_cerebral(SYN.data_ptr(), lab.data_ptr(), lab_u8, src, box, SYN_cerebral.data_ptr(),
                                             sums.data_ptr(), st))
            SYN_cerebral = fast_3D_interp_torch(SYN_cerebral, xx2, yy2, zz2).contiguous()
            for key in ('pathology', 'pathology_prob'):
                t = target[key]
                if not t.is_contiguous():
                    t = target[key] = t.contiguous()
                if t.numel() != SYN_cerebral.numel() or t.dtype not in (torch.float32, torch.float64):
                    t[SYN_cerebral[None] == 0] = 0                      # unusual shapes / dtypes: tensor expression
                else:
                    _lib.check(L.bfm_zero_where_zero(t.data_ptr(), int(t.dtype == torch.float64),
                                                     SYN_cerebral.data_ptr(), t.numel(), st))
            wm_sum, wm_n, gm_sum, gm_n = sums.tolist()                  # host sync (the reference's bool(gm > wm))
            wm_mean = wm_sum / wm_n if wm_n else float('nan')
            gm_mean = gm_sum / gm_n if gm_n else float('nan')
            pathol_direction = self.get_pathology_direction('synth', bool(gm_mean > wm_mean))
        else:
            pathol_direction = None
            target['pathology'] = 0.
            target['pathology_prob'] = 0.
        SYN[SYN < 0.] = 0.
        return target['pathology'], target['pathology_prob'], self.augment_sample(
            None, SYN, setups, deform_dict, res, target, pathol_direction=pathol_direction)

    def augment_sample(self, name, I_def, setups, deform_dict, res, target, pathol_direction=None, input_mode='synth'):
        """Augmentation of an already deformed image through the operator registry (datasets.py:306-354)."""
        sample = {}
        if not isinstance(I_def, torch.Tensor):
            raise NotImplementedError("real-image inputs go through read_and_deform; pass a deformed tensor")
        if input_mode == 'CT':
            I_def = torch.clamp(I_def, min=0., max=80.)
        P = target['pathology'] if 'pathology' in target else None
        if isinstance(P, torch.Tensor) and bool(P.sum() > 0):            # datasets.py:321-326
            I_def = self.encode_pathology(I_def, P, target['pathology_prob'], pathol_direction)
            I_def[I_def < 0.] = 0.
        else:
            target['pathology'] = 0.
            target['pathology_prob'] = 0.
        aux_dict = {}
        steps = self.augmentation_steps['synth'] if input_mode == 'synth' else self.augmentation_steps['real']
        for func_name in steps:
            I_def, aux_dict = K.augmentation_funcs[func_name](I=I_def, aux_dict=aux_dict, cfg=self.gen_args.generator,
                                                             input_mode=input_mode, setups=setups, size=self.size,
                                                             res=res, device=self.device, draws=self.rng)
        if self.synth_args.bspline_zooming:
            from .. import interpol
            I_def = interpol.resize(I_def, shape=self.size, anchor='edge', interpolation=3, bound='dct2',
                                    prefilter=True)
        else:
            I_def = myzoom_torch(I_def, 1 / aux_dict['factors'])
        maxi = torch.max(I_def)
        I_final = I_def / maxi
        flip = setups['flip']
        if 'super_resolution' in self.tasks:
            SRresidual = aux_dict['high_res'] / maxi - I_final
            sample.update({'high_res_residual': torch.flip(SRresidual, [0])[None] if flip else SRresidual[None]})
        sample.update({'input': torch.flip(I_final, [0])[None] if flip else I_final[None]})
        if 'bias_field' in self.tasks and input_mode != 'CT':
            sample.update({'bias_field_log': torch.flip(aux_dict['BFlog'], [0])[None] if flip else aux_dict['BFlog'][None]})
        return sample

    def encode_pathology(self, I, P, Pprob, pathol_direction=None):
        """Paint a lesion into the image: I += Pprob * N(mu_p, sigma_p), mu_p = +-(3/4 + u/4) * mean(I | P),
        sigma_p = u'/4 * mean(I | P) (datasets.py:496-518; same tensor expressions, hence the same dtype
        promotions: P / Pprob are float64 for random shapes, the image stays float32)."""
        rng = self.rng
        if pathol_direction is None:       # True: T2/FLAIR-resembled, False: T1-resembled
            pathol_direction = rng.choice("pathol.dir", [True, False])
        P, Pprob = torch.squeeze(P), torch.squeeze(Pprob)
        fast = (I.dtype == torch.float32 and P.dtype == Pprob.dtype and P.dtype in (torch.float32, torch.float64)
                and P.shape == I.shape and Pprob.shape == I.shape)
        if fast:
            L, st = _lib.lib(), _stream()
            I = I if I.is_contiguous() else I.contiguous()
            P, Pprob = P.contiguous(), Pprob.contiguous()
            dbl = int(P.dtype == torch.float64)
            sums = torch.empty(2, dtype=torch.float64, device=self.device)
            _lib.check(L.bfm_masked_mean(I.data_ptr(), P.data_ptr(), dbl, I.numel(), sums.data_ptr(), st))
            I_mu = (sums[0] / sums[1]).to(P.dtype if dbl else torch.float32)           # 0-dim, like the reference's
        else:
            I_mu = (I * P).sum() / P.sum()
        pth_mus = 3 * I_mu / 4 + I_mu / 4 * rng.torch_rand("pathol.mus", 10000).to(self.device)
        pth_mus = pth_mus if pathol_direction else -pth_mus
        pth_sigmas = I_mu / 4 * rng.torch_rand("pathol.sigmas", 10000).to(self.device)
        eps = rng.field_randn("pathol.eps", tuple(P.shape))
        if fast and pth_mus.dtype == torch.float32:
            eps = None if eps is None else eps.to(self.device, torch.float32).contiguous()
            pth_mus, pth_sigmas = pth_mus.contiguous(), pth_sigmas.contiguous()
            _lib.check(L.bfm_encode_pathology(I.data_ptr(), P.data_ptr(), Pprob.data_ptr(), dbl, pth_mus.data_ptr(),
                                              pth_sigmas.data_ptr(), pth_mus.numel(),
                                              0 if eps is None else eps.data_ptr(),
                                              int(rng.seed64()) if eps is None else 0, I.numel(), st))
            return I
        p_mask = torch.round(P).long()
        eps = torch.randn(p_mask.shape, dtype=torch.float, device=self.device) if eps is None else eps.to(self.device)
        I += Pprob * (pth_mus[p_mask] + pth_sigmas[p_mask] * eps)
        I[I < 0] = 0
        return I

    def get_pathology_direction(self, input_mode, pathol_direction=None):
        if pathol_direction is not None:
            return pathol_direction
        if input_mode in ['T1', 'CT']:
            return False
        if input_mode in ['T2', 'FLAIR']:
            return True
        return self.rng.choice("pathol.dir", [True, False])

    # ---- __getitem__ (datasets.py:638-681) ----------------------------------------------------------
    def _prologue_host(self, idx, arena):
        """Host-only part of an item: input mode, setup and deformation draws (reference order)."""
        if torch.is_tensor(idx):
            idx = idx.tolist()
        dataset_name, case_name, input_mode, img, aff, res, age = self.read_input(idx)
        setups = self.get_setup_params()
        deform_dict = self.generate_deformation(setups, img.shape, arena=arena, lazy=True)
        self.get_left_hemis_mask(None)
        return dict(idx=idx, dataset_name=dataset_name, case_name=case_name, input_mode=input_mode, img=img, res=res,
                    age=age, setups=setups, deform=deform_dict, modalities=dict(self.modalities),
                    hemis_mask=self.hemis_mask)

    def _targets(self, ctx, default):
        """Per-sample target kernels (needs the bounding box on the device)."""
        self.modalities = ctx['modalities']
        self.hemis_mask = ctx.get('hemis_mask')
        idx, input_mode, setups, deform_dict = ctx['idx'], ctx['input_mode'], ctx['setups'], ctx['deform']
        target = ctx.get('target')
        if target is None:
            target = defaultdict(default)
        target['name'] = ctx['case_name']
        fused = ctx.get('fused_job')
        for key in ('T1', 'T2', 'FLAIR'):
            if fused is not None and key in fused['aux_out']:
                target[key] = fused['aux_out'][key]          # written by the fused chain (warp + finish stages)
            else:
                target.update(self.read_and_deform_target(idx, target.keys(), key, input_mode, setups, deform_dict))
        for task_name in self.tasks:
            if task_name in K.processing_funcs.keys() and task_name not in ['T1', 'T2', 'FLAIR']:
                target.update(self.read_and_deform_target(idx, target.keys(), task_name, input_mode, setups,
                                                          deform_dict))
        return target

    def _fused_image_targets(self, ctx, jobs):
        """Real-image targets (T1/T2/FLAIR, read_and_deform_image) that can ride on the synthetic image's gather:
        stock reader, no defacing mask, no hemisphere mask, same volume shape, and no job of this item mixes real
        modalities into the synthetic image (mixing needs the normalised targets BEFORE the warp)."""
        if self.hemis_mask is not None or any(j['p']['mix'] is not None for j in jobs):
            return []
        return self._fused_aux_volumes(ctx['modalities'], ctx['deform']['_plan'].src)

    def _fused_aux_volumes(self, mods, src):
        out = []
        for key in ('T1', 'T2', 'FLAIR'):
            if key not in mods or (key + '_DM') in mods or K.processing_funcs.get(key) is not read_and_deform_image:
                continue
            vol = self.cache.get(mods[key], 'f32')
            if list(vol.shape[:3]) == list(src):
                out.append((key, vol))
        return out[:_lib.MAX_AUX]

    def _native_planner(self, indices):
        """The NativePlanner to use for this batch, or None (Python planner)."""
        if self.planner == 'python':
            return None
        from .native import NativePlanner
        ok = NativePlanner.config_ok(self) and (self.planner == 'native' or type(self.rng) is HostDraws)
        if ok:
            if self._native is None:
                self._native = NativePlanner(self)
            else:
                self._native.refresh()
            ok = self._native.batch_ok(indices)
        if not ok and self.planner == 'native':
            raise NotImplementedError("this configuration needs the Python planner (planner='python' or 'auto')")
        return self._native if ok else None

    def _real_input(self, input_mode, setups, deform_dict, res, target):
        from .utils import read_and_deform
        I, _ = read_and_deform(self.modalities[input_mode], torch.float, deform_dict, self.device, self.hemis_mask)
        return self.augment_sample(None, I, setups, deform_dict, res, target,
                                   pathol_direction=self.get_pathology_direction(input_mode), input_mode=input_mode)

    def _finish_item(self, ctx, target, sample):
        setups = ctx['setups']
        if setups['flip'] and isinstance(target['pathology'], torch.Tensor):
            target['pathology'] = torch.flip(target['pathology'], [1])
            target['pathology_prob'] = torch.flip(target['pathology_prob'], [1])
        if ctx['age'] is not None:
            target['age'] = ctx['age']
        self.last_setups, self.last_deform = setups, ctx['deform']
        return self.datasets_num, ctx['dataset_name'], ctx['input_mode'], target, sample

    def _fast_ok(self, input_mode, src_shape=None):
        """Fused chain: synthetic inputs, and real T1 / T2 / FLAIR / CT inputs whose volume has the shape of the
        deformation's source grid, with the stock augmentation chain."""
        if 'pathology' in self.tasks:
            return False
        if input_mode == 'synth':
            return self._stock_chain('synth')
        if input_mode not in ('T1', 'T2', 'FLAIR', 'CT') or self.hemis_mask is not None or \
                not self._stock_chain(input_mode):
            return False
        vol = self.cache.get(self.modalities[input_mode], 'f32')
        return src_shape is None or list(vol.shape[:3]) == [int(v) for v in src_shape[:3]]

    def _gen_arg_sets(self, input_mode='synth'):
        """Parameter overrides applied before each sample of an item (datasets.py:664-669, 728-745)."""
        return [[self.synth_image_args if input_mode == 'synth' else self.real_image_args]]

    _default_target = staticmethod(lambda: None)
    _list_samples = False

    def generate_batch(self, indices, timers=None):
        """Several items in one go: all host draws first (reference order, item by item), then ONE batched launch
        per stage of the fused chain.  Returns a list of __getitem__ tuples."""
        self.cache.begin_batch()          # volumes looked up from here on stay alive until the launches are enqueued
        native = self._native_planner(indices)
        if native is not None:
            return native.run(indices, timers=timers)
        arena = self.arena.begin()
        ctxs, jobs, spans, slow = [], [], [], {}
        for n, idx in enumerate(indices):
            ctx = self._prologue_host(idx, arena)
            ctxs.append(ctx)
            mode = ctx['input_mode']
            if not self._fast_ok(mode, ctx['img'].shape):
                slow[n] = True
                spans.append((0, 0))
                continue
            ctx['target'] = defaultdict(self._default_target)
            first = len(jobs)
            for arg_sets in self._gen_arg_sets(mode):
                for a in arg_sets:
                    self.update_gen_args(a)
                jobs.append(self._job(ctx['setups'], ctx['deform'], ctx['target'],
                                      self._plan_synth(ctx['setups'], ctx['target'], arena,
                                                       real=mode if mode != 'synth' else False),
                                      mode))
            spans.append((first, len(jobs)))
            aux = self._fused_image_targets(ctx, jobs[first:])
            if aux:
                jobs[first]['aux'] = aux
                ctx['fused_job'] = jobs[first]

        def run_targets():
            for n, ctx in enumerate(ctxs):
                if n not in slow:
                    self._targets(ctx, self._default_target)

        self._last_jobs = jobs
        results = self._run_chain(jobs, arena, targets_fn=run_targets, timers=timers) if jobs else []
        items = []
        for n, ctx in enumerate(ctxs):
            if n in slow:
                items.append(self._slow_item(ctx))
                continue
            target = ctx['target']
            target['pathology'] = 0.
            target['pathology_prob'] = 0.
            a, b = spans[n]
            sample = results[a:b] if self._list_samples else results[a]
            items.append(self._finish_item(ctx, target, sample))
        return items

    def generate_batch_fast(self, indices):
        """generate_batch through `NativePlanner.run_fast` (one library call per batch, lazily built result tuples), or
        None when the configuration / batch needs the general path."""
        if self.planner == 'python':
            return None
        self.cache.begin_batch()
        from .native import NativePlanner
        if not (NativePlanner.config_ok(self) and (self.planner == 'native' or type(self.rng) is HostDraws)):
            return None
        if self._native is None:
            self._native = NativePlanner(self)
        else:
            self._native.refresh()
        if not self._native.fast_ok():
            return None
        return self._native.run_fast(indices)

    def _slow_item(self, ctx):
        """Op-by-op path: real-image inputs, custom augmentation sequences, pathology."""
        self.arena.commit()
        ctx['deform']['_plan'].compute_bbox()
        target = self._targets(ctx, self._default_target)
        setups, deform_dict, res, input_mode = ctx['setups'], ctx['deform'], ctx['res'], ctx['input_mode']
        samples = []
        for arg_sets in self._gen_arg_sets():
            for a in arg_sets[:-1]:
                self.update_gen_args(a)
            if input_mode == 'synth':
                self.update_gen_args(self.synth_image_args)
                target['pathology'], target['pathology_prob'], sample = \
                    self.generate_sample(ctx['case_name'], ctx['img'], setups, deform_dict, res, target)
            else:
                self.update_gen_args(self.real_image_args)
                sample = self._real_input(input_mode, setups, deform_dict, res, target)
            samples.append(sample)
        return self._finish_item(ctx, target, samples if self._list_samples else samples[0])

    def __getitem__(self, idx):
        return self.generate_batch([idx])[0]


class BrainIDGen(BaseGen):
    """Intra-subject augmentation: one deformation, `all_samples` contrasts; the first `mild_samples` use
    mild_generator parameters, the rest severe_generator (Generator/datasets.py:687-757).  All samples of one
    item run as ONE batched launch of the fused chain."""

    _default_target = staticmethod(lambda: 1.)
    _list_samples = True

    def __init__(self, gen_args, device='cuda', draws=None, planner='auto'):
        self.all_samples = gen_args.generator.all_samples        # _gen_arg_sets may be asked early
        self.mild_samples = gen_args.generator.mild_samples
        self.mild_generator_args = gen_args.mild_generator
        self.severe_generator_args = gen_args.severe_generator
        super(BrainIDGen, self).__init__(gen_args, device, draws, planner)
        self.all_samples = gen_args.generator.all_samples
        self.mild_samples = gen_args.generator.mild_samples
        self.mild_generator_args = gen_args.mild_generator
        self.severe_generator_args = gen_args.severe_generator

    def _gen_arg_sets(self, input_mode='synth'):
        last = self.synth_image_args if input_mode == 'synth' else self.real_image_args
        return [[self.mild_generator_args if i < self.mild_samples else self.severe_generator_args, last]
                for i in range(self.all_samples)]
