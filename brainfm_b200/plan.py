"""Host-side planning for the CUDA kernels: the per-axis index/weight tables the reference builds with
float32 `torch.arange` (myzoom_torch, Generator/utils.py:205-236), the banded blur-o-downsample maps of
resample_resolution (utils.py:74-94, 591-609), and a pinned-host/device arena that ships all of a batch's
small arrays to the GPU in one asynchronous copy."""
import ctypes as C

import time

import numpy as np
import torch

from . import _lib

_ALIGN = 16


_ZOOM_CACHE = {}
_CAND_CACHE = {}


def zoom_tables_host(n_in, factor, n_out):
    """lo, hi (int32), wl, wh (float32) of one axis of myzoom_torch -- computed with the reference's own
    float32 torch expressions (SURVEY.md 3.3 item 5: float32 arange is not float64-then-cast).  Memoised: the
    tables only depend on (n_in, factor, n_out) and a generator sees a few hundred distinct keys."""
    key = (int(n_in), float(factor), int(n_out))
    hit = _ZOOM_CACHE.get(key)
    if hit is None:
        hit = _zoom_tables_host(*key)
        _ZOOM_CACHE[key] = hit
    return hit


def _zoom_tables_host(n_in, factor, n_out):
    factor = float(factor)
    delta = (1.0 - factor) / (2.0 * factor)
    v = torch.arange(delta, delta + n_out / factor, 1 / factor, dtype=torch.float32)[:n_out]
    v = v.clamp(min=0, max=n_in - 1)
    lo = torch.floor(v).int()
    hi = (lo + 1).clamp(max=n_in - 1)
    wh = v - lo
    wl = 1 - wh
    return (lo.numpy().astype(np.int32), hi.numpy().astype(np.int32), wl.numpy().astype(np.float32),
            wh.numpy().astype(np.float32))


def zoom_candidates_host(n_in, factor, n_out):
    key = (int(n_in), float(factor), int(n_out))
    hit = _CAND_CACHE.get(key)
    if hit is None:
        hit = _zoom_candidates_host(*key)
        _CAND_CACHE[key] = hit
    return hit


def _zoom_candidates_host(n_in, factor, n_out):
    """Output indices next to a kink of the piecewise-linear zoom weights along one axis: the ends, every
    change of the lower source node, and the transitions into / out of the edge clamp.  Between two
    consecutive candidates the interpolation weight is (up to rounding) affine in the index, so a field
    zoomed this way is multilinear between candidates and attains its extrema on them."""
    factor = float(factor)
    delta = (1.0 - factor) / (2.0 * factor)
    v = torch.arange(delta, delta + n_out / factor, 1 / factor, dtype=torch.float32)[:n_out].numpy()
    seg = np.floor(np.clip(v, 0, n_in - 1)).astype(np.int64) * 4 + (v < 0) * 1 + (v > n_in - 1) * 2
    k = np.nonzero(seg[1:] != seg[:-1])[0] + 1
    cand = np.unique(np.concatenate([[0, n_out - 1], k, k - 1]))
    return cand.astype(np.int32)


def zoom_newsize(shape, factor):
    return np.round(np.asarray(shape) * np.asarray(factor, dtype=np.float64)).astype(int)


def gaussian_taps_host(sigma):
    """make_gaussian_kernel (utils.py:74-81), same float32 torch expressions."""
    sl = int(np.ceil(3 * sigma))
    ts = torch.linspace(-sl, sl, 2 * sl + 1, dtype=torch.float32)
    g = torch.exp((-(ts / sigma) ** 2 / 2))
    return (g / g.sum()).numpy(), sl


def resample_coords_host(n_in, n_out):
    """Low-res sample positions along one axis: float64 np.arange then float32 (utils.py:595-605)."""
    f = n_out / n_in
    delta = (1.0 - f) / (2.0 * f)
    return np.arange(delta, delta + n_out / f, 1 / f)[:n_out].astype(np.float32), f


def band_host(n_in, n_out, sigma):
    """Banded matrix of (zero-padded Gaussian correlation) followed by (masked 2-tap linear sampling)
    along one axis.  Returns start[n_out] int32, w[n_out, T] float32, T."""
    v, _ = resample_coords_host(n_in, n_out)
    ok = (v > 0) & (v <= np.float32(n_in - 1))
    fx = np.floor(v)
    lo = fx.astype(np.int64)
    hi = np.minimum(lo + 1, n_in - 1)
    wh = (v - fx).astype(np.float32)
    wl = (np.float32(1) - wh).astype(np.float32)
    if sigma > 0:
        g, half = gaussian_taps_host(sigma)
        g = g.astype(np.float64)
    else:
        g, half = np.ones(1, dtype=np.float64), 0
    L = 2 * half + 1
    T = L + 1
    W = np.zeros((n_out, T), dtype=np.float64)
    W[:, :L] += wl.astype(np.float64)[:, None] * g[None, :]
    shift = (hi - lo).astype(bool)
    W[shift, 1:] += wh.astype(np.float64)[shift, None] * g[None, :]
    W[~shift, :L] += wh.astype(np.float64)[~shift, None] * g[None, :]
    W[~ok] = 0
    start = (lo - half).astype(np.int32)
    return start, W.astype(np.float32), T


class Arena:
    """A ring of pinned-host / device byte buffers.  All small per-batch arrays (tables, LUTs, small random
    grids, the descriptor array) are packed into the host side and shipped with ONE async copy."""

    def __init__(self, device, capacity=8 << 20, slots=3):
        self.device = torch.device(device)
        self.capacity = capacity
        self.slots = []
        for _ in range(slots):
            host = torch.empty(capacity, dtype=torch.uint8).pin_memory()
            dev = torch.empty(capacity, dtype=torch.uint8, device=self.device)
            self.slots.append(dict(host=host, dev=dev, np=host.numpy(), event=None))
        self.cur = -1
        self.used = 0
        self.committed = 0
        self.wait_s = 0.0                # host time spent waiting for a free slot (= for the GPU), cumulative

    def begin(self):
        self.cur = (self.cur + 1) % len(self.slots)
        s = self.slots[self.cur]
        if s["event"] is not None:
            if not s["event"].query():                   # the GPU is behind: the host waits here (and only here)
                t0 = time.perf_counter()
                s["event"].synchronize()
                self.wait_s += time.perf_counter() - t0
        self.used = 0
        self.committed = 0
        self.base = s["dev"].data_ptr()
        return self

    def put(self, arr):
        """Copy a numpy array into the host buffer; returns its DEVICE address."""
        a = np.ascontiguousarray(arr)
        n = a.nbytes
        off = (self.used + _ALIGN - 1) // _ALIGN * _ALIGN
        if off + n > self.capacity:
            raise MemoryError("plan arena overflow (%d + %d > %d)" % (off, n, self.capacity))
        self.slots[self.cur]["np"][off:off + n] = a.view(np.uint8).reshape(-1)
        self.used = off + n
        return self.base + off

    def reserve(self, nbytes):
        """Uninitialised device scratch inside the arena (bbox ints, max scalars); returns (address, offset)."""
        off = (self.used + _ALIGN - 1) // _ALIGN * _ALIGN
        if off + nbytes > self.capacity:
            raise MemoryError("plan arena overflow")
        self.used = off + nbytes
        return self.base + off, off

    def alloc_tensor(self, shape, dtype=torch.float32):
        """Uninitialised array INSIDE the pinned host buffer: (device address, CPU tensor view).  Draws written
        into the view (torch.rand(..., out=view)) reach the device with the slot's single copy."""
        n = 1
        for v in shape:
            n *= int(v)
        item = 4 if dtype in (torch.float32, torch.int32) else torch.empty((), dtype=dtype).element_size()
        off = (self.used + _ALIGN - 1) // _ALIGN * _ALIGN
        if off + n * item > self.capacity:
            raise MemoryError("plan arena overflow")
        self.used = off + n * item
        view = self.slots[self.cur]["host"][off:off + n * item].view(dtype).view(*shape)
        return self.base + off, view

    def put_struct_array(self, arr):
        n = C.sizeof(arr)
        off = (self.used + _ALIGN - 1) // _ALIGN * _ALIGN
        if off + n > self.capacity:
            raise MemoryError("plan arena overflow")
        C.memmove(self.slots[self.cur]["host"].data_ptr() + off, C.addressof(arr), n)
        self.used = off + n
        return self.base + off

    def commit(self, stream=None):
        """Ship everything put() since the last commit: one asynchronous copy on the current stream, done by a
        kernel that reads the pinned host buffer (bfm_upload_pinned) -- a cudaMemcpyAsync would queue behind
        whatever bulk uploads are sitting in the copy engine's FIFO (HostPipeline)."""
        s = self.slots[self.cur]
        if self.used > self.committed:
            a = self.committed // _ALIGN * _ALIGN
            b = min((self.used + _ALIGN - 1) // _ALIGN * _ALIGN, self.capacity)
            st = C.c_void_p(torch._C._cuda_getCurrentRawStream(self.device.index if self.device.index is not None
                                                               else torch._C._cuda_getDevice()))
            _lib.check(_lib.lib().bfm_upload_pinned(s["dev"].data_ptr() + a, s["host"].data_ptr() + a, b - a, st))
            self.committed = self.used

    def mark_done(self):
        ev = torch.cuda.Event()
        ev.record()
        self.slots[self.cur]["event"] = ev

    def view(self, off, count, dtype, slot=None):
        """Device tensor view of arena bytes [off, off+count*itemsize) of a slot (default: the current one)."""
        item = torch.empty((), dtype=dtype).element_size()
        return self.slots[self.cur if slot is None else slot]["dev"][off:off + count * item].view(dtype)


class DeviceTables:
    """Device-resident cache of the per-axis myzoom_torch tables and of the bounding-box candidate lists.  Both
    depend only on (n_in, factor, n_out); a generator sees a few hundred distinct keys, so after warm-up no
    table is rebuilt or copied again (a miss costs one small synchronous upload)."""

    def __init__(self, device):
        self.device = torch.device(device)
        self._zoom = {}
        self._cand = {}
        self._keep = []

    def _upload(self, arrays):
        offs, total = [], 0
        for a in arrays:
            total = (total + _ALIGN - 1) // _ALIGN * _ALIGN
            offs.append(total)
            total += a.nbytes
        host = np.zeros(max(total, _ALIGN), dtype=np.uint8)
        for a, o in zip(arrays, offs):
            host[o:o + a.nbytes] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        dev = torch.from_numpy(host).to(self.device)
        self._keep.append(dev)
        base = dev.data_ptr()
        return [base + o for o in offs]

    def prebuild(self, size):
        """Build and upload, in one copy, the tables of every zoom the generator can ask for on a grid of this
        size: n_in -> n_out for n_in = 1..n_out with the factor n_out/n_in (small random grids) and with
        1/(n_in/n_out) (low-res grid back to the training grid), plus the candidate lists.  A table miss later on
        still works but costs a synchronous upload in the middle of the stream."""
        todo_z, todo_c = [], []
        for n_out in sorted(set(int(v) for v in size)):
            for n_in in range(1, n_out + 1):
                for factor in (n_out / n_in, 1 / (n_in / n_out)):
                    key = (n_in, float(factor), n_out)
                    if key not in self._zoom and key not in [k for k, _ in todo_z]:
                        todo_z.append((key, zoom_tables_host(*key)))
                key = (n_in, float(n_out / n_in), n_out)
                if key not in self._cand:
                    todo_c.append((key, zoom_candidates_host(*key)))
        if not todo_z and not todo_c:
            return
        arrays = [a for _, tabs in todo_z for a in tabs] + [c for _, c in todo_c]
        addrs = self._upload(arrays)
        for n, (key, _) in enumerate(todo_z):
            self._zoom[key] = tuple(addrs[4 * n:4 * n + 4])
        base = 4 * len(todo_z)
        for n, (key, c) in enumerate(todo_c):
            self._cand[key] = (addrs[base + n], int(c.size))

    def zoom(self, n_in, factor, n_out):
        """Device addresses (lo, hi, wl, wh) of one axis."""
        key = (int(n_in), float(factor), int(n_out))
        hit = self._zoom.get(key)
        if hit is None:
            hit = tuple(self._upload(zoom_tables_host(*key)))
            self._zoom[key] = hit
        return hit

    def cand(self, n_in, factor, n_out):
        """(device address, count) of the candidate list of one axis."""
        key = (int(n_in), float(factor), int(n_out))
        hit = self._cand.get(key)
        if hit is None:
            c = zoom_candidates_host(*key)
            hit = (self._upload([c])[0], int(c.size))
            self._cand[key] = hit
        return hit

    def zoom_tab(self, n_in, n_out, inverse=False):
        """A filled _lib.ZoomTab for the three axes of a zoom from shape n_in to shape n_out (cached; assign it
        to a descriptor field with `desc.tab = ...`, a struct copy).  The factor is what the caller of
        myzoom_torch passes: n_out/n_in (deformation and bias grids, datasets.py:210, utils.py:585), or with
        inverse=True 1/(n_in/n_out) (back to the training grid, datasets.py:340)."""
        key = (tuple(n_in), tuple(n_out), inverse)
        hit = self._zoom.get(key)
        if hit is None:
            a, b = np.array(key[0]), np.array(key[1])
            factor = 1 / (a / b) if inverse else b / a
            assert tuple(zoom_newsize(key[0], factor)) == key[1], (key, factor)
            hit = _lib.ZoomTab()
            set_zoom_tab(hit, self, key[0], factor, key[1])
            self._zoom[key] = hit
        return hit

    def deform_template(self, size, fs):
        """A _lib.Deform with everything that only depends on (output size, small-grid shape) filled in: zoom
        tables, candidate lists, centre.  fs=None: no nonlinear field."""
        key = ("deform", tuple(size), None if fs is None else tuple(fs))
        hit = self._zoom.get(key)
        if hit is None:
            hit = _lib.Deform()
            for a in range(3):
                hit.size[a] = int(size[a])
                hit.ctr[a] = float(np.float32((size[a] - 1) / 2))
            if fs is None:
                for a in range(3):
                    hit.cand[a], hit.ncand[a] = self.ends(size[a])
            else:
                factor = np.array(size) / np.array(fs)
                assert tuple(zoom_newsize(fs, factor)) == tuple(size), (fs, size)
                hit.ftab = self.zoom_tab(fs, size)
                for a in range(3):
                    hit.fs[a] = int(fs[a])
                    hit.cand[a], hit.ncand[a] = self.cand(fs[a], factor[a], int(size[a]))
            self._zoom[key] = hit
        return hit

    def ends(self, n_out):
        """Candidate list {0, n_out-1} of an axis without a nonlinear field."""
        key = ("ends", int(n_out))
        hit = self._cand.get(key)
        if hit is None:
            hit = (self._upload([np.array([0, n_out - 1], dtype=np.int32)])[0], 2)
            self._cand[key] = hit
        return hit


_TABLES = {}


def device_tables(device):
    key = str(torch.device(device))
    if key not in _TABLES:
        _TABLES[key] = DeviceTables(device)
    return _TABLES[key]


def set_zoom_tab(tab, tables, n_in, factors, n_out):
    """Point a _lib.ZoomTab at the cached device tables of the three axes."""
    for ax in range(3):
        lo, hi, wl, wh = tables.zoom(n_in[ax], factors[ax], n_out[ax])
        tab.lo[ax], tab.hi[ax], tab.wl[ax], tab.wh[ax] = lo, hi, wl, wh


def make_deform(tables, arena, size, src, A, c2, fsmall_host, photo, F_full_ptr=None, fsmall_dev=None):
    """A filled _lib.Deform: the cached template of (size, small-grid shape) plus this sample's affine, source
    shape and small random grid (the only array that goes through the arena; fsmall_dev: it is already there)."""
    fs = None if fsmall_host is None else tuple(fsmall_host.shape[:3])
    d = _lib.Deform.from_buffer_copy(tables.deform_template(size, fs))
    d.src[:] = [int(v) for v in src[:3]]
    d.A[:] = np.asarray(A, dtype=np.float32).reshape(-1).tolist()
    d.c2[:] = np.asarray(c2, dtype=np.float32).tolist()
    d.photo = int(bool(photo))
    if F_full_ptr is not None:
        d.F_full = F_full_ptr
        d.ncand[:] = [0, 0, 0]
    if fsmall_host is not None:
        d.fsmall = fsmall_dev if fsmall_dev is not None else arena.put(fsmall_host)
    return d
