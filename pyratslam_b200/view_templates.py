"""View templates on the B200: the reference's class surface over the CUDA sweep kernel.

``ViewTemplates`` / ``ViewTemplate`` keep the names, arguments and decisions of
``ratslam/view_templates.py`` -- ``ViewTemplates.match(input, pc_x, pc_y, pc_th)``
returns the best stored template or creates one (strict ``>`` threshold test,
first minimum wins) -- while the library lives in HBM as one ``[capacity, 32,
32]`` tensor and every match is a single streaming sweep
(``csrc/view_templates.cu``) instead of a Python loop over templates.

``ShardedViewTemplates`` splits a very large library by contiguous template
ranges over the ranks of a ``torch.distributed`` group; the only exchange is one
8-byte MIN all-reduce of the packed ``(score << 32 | index)`` key per query.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native as nat
from .sharding import decide, reduce_packed_key, unpack_key

_KEY_NONE = (1 << 64) - 1


def flat_cell_index(locations, shape):
    """Template locations ``[n, 3]`` -> the C-order flat pose cell ``x*Y*Th + y*Th + th`` each one injects into, or -1
    where ``PoseCellEnsemble.inject`` raises ``IndexError``: coordinates are truncated the way ``int()`` does, a
    coordinate in ``[-n, 0)`` wraps like a numpy index, anything else (out of range, not finite) is -1."""
    loc = np.asarray(locations, dtype=np.float64).reshape(-1, 3)
    dims = np.asarray(shape, dtype=np.int64).reshape(1, 3)
    ok = np.isfinite(loc).all(axis=1)
    v = np.trunc(np.where(np.isfinite(loc), loc, 0.0))
    ok &= ((v >= -dims) & (v < dims)).all(axis=1)
    c = np.where(ok[:, None], v, 0.0).astype(np.int64)
    c = np.where(c < 0, c + dims, c)
    X, Y, Th = (int(s) for s in shape)
    return np.where(ok, c[:, 0] * (Y * Th) + c[:, 1] * Th + c[:, 2], -1).astype(np.int64)


class ViewTemplate:
    """One stored view, tied to the pose cell that was most active when it was created
    (``view_templates.py:4-37``)."""

    max_offset = 8

    def __init__(self, pc_x, pc_y, pc_th, index, template=None, _owner=None):
        self.pc_x, self.pc_y, self.pc_th = pc_x, pc_y, pc_th
        self.index = index
        self._template = template
        self._owner = _owner
        self.max_offset = 8

    @property
    def template(self):
        if self._template is None and self._owner is not None:
            self._template = self._owner._fetch_template(self.index)
        return self._template

    def match(self, new_template):
        """Score of ``new_template`` against this one (``view_templates.py:16-28``), computed on the device."""
        nat.require_cuda()
        a = np.ascontiguousarray(self.template)
        b = np.ascontiguousarray(new_template)
        if a.ndim != 2 or a.shape != b.shape:
            raise ValueError("operands could not be broadcast together with shapes %r %r" % (a.shape, b.shape))
        R, C = a.shape
        dev = torch.device("cuda", torch.cuda.current_device())
        key = torch.empty(1, dtype=torch.int64, device=dev)
        if a.dtype == np.uint8 and b.dtype == np.uint8:
            ta, tb = torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)
            nat.check(nat.lib().prs_vt_sweep_any_u8(ta.data_ptr(), 1, tb.data_ptr(), R, C, self.max_offset, 0,
                                                    key.data_ptr(), None, nat.stream_ptr()), "prs_vt_sweep_any_u8")
            return np.uint64(int(key.item()) >> 32)
        ta = torch.from_numpy(a.astype(np.float32)).to(dev)
        tb = torch.from_numpy(b.astype(np.float32)).to(dev)
        nat.check(nat.lib().prs_vt_sweep_any_f32(ta.data_ptr(), 1, tb.data_ptr(), R, C, self.max_offset, 0,
                                                 key.data_ptr(), None, nat.stream_ptr()), "prs_vt_sweep_any_f32")
        return np.array([int(key.item()) >> 32], dtype=np.uint32).view(np.float32)[0]

    def location(self):
        return (self.pc_x, self.pc_y, self.pc_th)

    def get_index(self):
        return self.index


class _TemplateList:
    """``ViewTemplates.templates``: behaves like the reference's Python list of ``ViewTemplate`` objects,
    but the objects are made on demand so that a 10^6-entry library is not 10^6 Python objects."""

    def __init__(self, owner):
        self._o = owner
        self._cache = {}

    def __len__(self):
        return self._o._n

    def __getitem__(self, i):
        n = self._o._n
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(n))]
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError("list index out of range")
        t = self._cache.get(i)
        if t is None:
            x, y, th = self._o._loc[i]
            t = ViewTemplate(self._o._loc_cast(x), self._o._loc_cast(y), self._o._loc_cast(th), i, None, self._o)
            self._cache[i] = t
        return t

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class ViewTemplates:
    """Drop-in for ``ratslam/view_templates.py:ViewTemplates`` with a device-resident library."""

    def __init__(self, x_range, y_range, x_step, y_step, im_x, im_y, match_threshold, mode="ref", capacity=1024,
                 device=None):
        nat.require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.x_range, self.y_range = tuple(x_range), tuple(y_range)
        self.x_step, self.y_step = int(x_step), int(y_step)
        self.im_x, self.im_y = int(im_x), int(im_y)
        # view_templates.py:44 with Python-2 integer division
        self.shape = ((x_range[1] - x_range[0]) // x_step, (y_range[1] - y_range[0]) // y_step)
        self.match_threshold = match_threshold
        self.mode = {"ref": nat.VT_MODE_REF, "circular": nat.VT_MODE_CIRCULAR}[mode]
        # rows are selected by y_range (base / im_x is the row index), columns by x_range
        cnt = lambda lo, hi, st: (hi - lo - 1) - (hi - lo - 1) // st  # noqa: E731
        self._n_rows = cnt(y_range[0], y_range[1], y_step)
        self._n_cols = cnt(x_range[0], x_range[1], x_step)
        if self._n_rows * self._n_cols != self.shape[0] * self.shape[1]:
            raise ValueError("cannot reshape array of size %d into shape %r"
                             % (self._n_rows * self._n_cols, self.shape))
        # 32x32 (the reference configuration) takes the tuned kernels; any other shape the general one
        # (a non-square image takes the mask path: the reference builds its mask with row = base / im_x but reshapes it
        # to (im_x, im_y), view_templates.py:48-57, and only the mask itself reproduces that)
        self._fast = tuple(self.shape) == (32, 32) and self._n_rows == 32 and self._n_cols == 32 and self.im_x == self.im_y
        if not self._fast and mode != "ref":
            raise NotImplementedError("circular mode is implemented for 32x32 templates")
        self._mask = None
        self._mask_dev = None
        self._n = 0
        self._dtype = None           # torch dtype of the library, fixed by the first frame
        self._lib = None             # [capacity, 32, 32]
        self._capacity = int(capacity)
        self._loc = np.zeros((self._capacity, 3), dtype=np.float64)
        self._loc_is_int = True
        # the device-side twin of _loc for the frame plans' injection node: int64 [capacity] flat pose cells
        # (flat_cell_index of a grid of shape _cell_shape), rows [0, _cell_n) in step with _loc
        self._cell_dev = None
        self._cell_shape = None
        self._cell_n = 0
        self.templates = _TemplateList(self)
        self._key =torch.empty(1, dtype=torch.int64, device=self.device)
        self._key_pin = torch.empty(1, dtype=torch.int64).pin_memory()
        self._frame_dev = torch.empty((self.im_x, self.im_y), dtype=torch.uint8, device=self.device)
        self._tpl_u8 = torch.empty(tuple(self.shape), dtype=torch.uint8, device=self.device)
        self._frame_pin = torch.empty((self.im_x, self.im_y), dtype=torch.uint8).pin_memory()
        self._scratch = torch.empty(4096, dtype=torch.uint8, device=self.device)
        self.last_score = None       # best score of the most recent match() (None when the library was empty)

    # ------------------------------------------------------------------ reference attributes
    @property
    def mask(self):
        """The boolean sub-sampling mask of view_templates.py:48-57 (built lazily; the device path does not need it)."""
        if self._mask is None:
            base = np.arange(self.im_x * self.im_y)
            row, col = base // self.im_x, base % self.im_x
            m = ((row > self.y_range[0]) & (row < self.y_range[1]) & (col > self.x_range[0]) & (col < self.x_range[1])
                 & ((row - self.y_range[0]) % self.y_step != 0) & ((col - self.x_range[0]) % self.x_step != 0))
            self._mask = m.reshape((self.im_x, self.im_y))
        return self._mask

    def __len__(self):
        return self._n

    def _loc_cast(self, v):
        return int(v) if self._loc_is_int else float(v)

    def _fetch_template(self, i):
        if self._dtype == torch.uint8 and self._fast:
            out = torch.empty((32, 32), dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.device):
                nat.check(nat.lib().prs_vt_unpack_u8(self._lib.data_ptr(), int(i), out.data_ptr(), nat.stream_ptr()),
                          "prs_vt_unpack_u8")
            return out.cpu().numpy()
        return self._lib[i].cpu().numpy()

    # ------------------------------------------------------------------ library management
    # uint8 libraries are stored bit-sliced ("packed", 1088 B per template, see csrc/view_templates.cu);
    # float32 libraries are plain [capacity, 32, 32].
    def _alloc(self, torch_dtype, capacity):
        if torch_dtype == torch.uint8 and self._fast:
            nbytes = int(nat.lib().prs_vt_packed_bytes(int(capacity)))
            return torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        return torch.empty((capacity,) + tuple(self.shape), dtype=torch_dtype, device=self.device)

    def _ensure_lib(self, torch_dtype):
        if self._lib is None:
            self._dtype = torch_dtype
            self._lib = self._alloc(torch_dtype, self._capacity)
        elif self._dtype != torch_dtype:
            raise TypeError("library holds %s templates, got a %s frame" % (self._dtype, torch_dtype))

    def _grow(self, need):
        if need <= self._capacity:
            return
        cap = max(need, self._capacity * 2)
        new = self._alloc(self._dtype, cap)
        if self._dtype == torch.uint8 and self._fast:
            new[: self._lib.numel()].copy_(self._lib)      # whole 32-template groups, position independent
        else:
            new[: self._n].copy_(self._lib[: self._n])
        self._lib = new
        loc = np.zeros((cap, 3), dtype=np.float64)
        loc[: self._n] = self._loc[: self._n]
        self._loc = loc
        if self._cell_dev is not None:
            cells = torch.full((cap,), -1, dtype=torch.int64, device=self.device)
            cells[: self._cell_dev.numel()].copy_(self._cell_dev)
            self._cell_dev = cells
        self._capacity = cap

    def _cell_table(self, shape):
        """The device location table for a pose-cell grid of ``shape`` (created on first use, all rows -1)."""
        shape = tuple(int(s) for s in shape)
        if self._cell_dev is None or self._cell_shape != shape or self._cell_dev.numel() < self._capacity:
            self._cell_dev = torch.full((self._capacity,), -1, dtype=torch.int64, device=self.device)
            self._cell_shape, self._cell_n = shape, 0
        return self._cell_dev

    def _cell_sync(self, stream):
        """Copy the rows of templates appended outside the frame plans (``match`` / ``create`` / ``load_library``) into
        the device table, on ``stream``."""
        if self._cell_dev is None or self._cell_n >= self._n:
            self._cell_n = min(self._cell_n, self._n)
            return
        rows = torch.from_numpy(flat_cell_index(self._loc[self._cell_n: self._n], self._cell_shape))
        with torch.cuda.stream(stream):
            self._cell_dev[self._cell_n: self._n].copy_(rows)
        self._cell_n = self._n

    def _store(self, tpl_dev, first, count):
        """Write ``count`` row-major templates into slots ``first..``."""
        if self._dtype == torch.uint8 and self._fast:
            nat.check(nat.lib().prs_vt_pack_u8(tpl_dev.data_ptr(), int(count), self._lib.data_ptr(), int(first),
                                               nat.stream_ptr()), "prs_vt_pack_u8")
        else:
            self._lib[first: first + count].copy_(tpl_dev.reshape((count,) + tuple(self.shape)))

    def load_library(self, templates, locations=None):
        """Bulk-load ``templates[n, 32, 32]`` (uint8 or float32; numpy or torch) as templates 0..n-1."""
        t = templates if isinstance(templates, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(templates))
        if t.dtype not in (torch.uint8, torch.float32):
            raise TypeError("templates must be uint8 or float32")
        if tuple(t.shape[1:]) != tuple(self.shape):
            raise ValueError("library templates are %r, this matcher uses %r" % (tuple(t.shape[1:]), tuple(self.shape)))
        n = t.shape[0]
        self._dtype = t.dtype
        self._capacity = max(n, 32)
        with torch.cuda.device(self.device):
            src = t.to(self.device).contiguous()
            if t.dtype == torch.uint8 and self._fast:
                self._lib = self._alloc(torch.uint8, self._capacity)
                self._store(src, 0, n)
            else:
                self._lib = src
                self._capacity = n
        self._n = n
        self._loc = np.zeros((self._capacity, 3), dtype=np.float64)
        if locations is not None:
            self._loc[:n] = np.asarray(locations, np.float64)
        self._cell_dev, self._cell_n = None, 0
        self.templates = _TemplateList(self)

    def _append(self, tpl_dev, pc_x, pc_y, pc_th):
        self._grow(self._n + 1)
        self._store(tpl_dev, self._n, 1)
        self._loc[self._n] = (pc_x, pc_y, pc_th)
        if not all(float(v).is_integer() for v in (pc_x, pc_y, pc_th)):
            self._loc_is_int = False
        self._n += 1
        return self.templates[self._n - 1]

    # ------------------------------------------------------------------ matching
    def _subsample(self, input):
        """Frame -> device template ``[32, 32]`` in the library dtype (view_templates.py:64)."""
        if isinstance(input, torch.Tensor):
            fr = input
        else:
            fr = np.asarray(input)
        is_u8 = (fr.dtype == torch.uint8) if isinstance(fr, torch.Tensor) else (fr.dtype == np.uint8)
        if tuple(fr.shape) != (self.im_x, self.im_y):
            # The reference's numpy accepted a frame smaller than the mask as long as every selected pixel was inside it
            # (ros_scenario.py publishes 128x128 frames against the 256x256 mask): the fast uint8 path takes such frames
            # with their own row stride; anything else is the IndexError numpy raises.
            covers = (fr.ndim == 2 and self._fast and is_u8 and fr.shape[0] >= self.y_range[1]
                      and fr.shape[1] >= self.x_range[1])
            if not covers:
                raise IndexError("boolean index did not match indexed array: frame %r, mask %r"
                                 % (tuple(fr.shape), (self.im_x, self.im_y)))
            t = fr if isinstance(fr, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(fr))
            t = t.to(self.device).contiguous()
            nat.check(nat.lib().prs_vt_extract_u8(
                t.data_ptr(), int(t.shape[0]), int(t.shape[1]), self.y_range[0], self.y_range[1], self.y_step,
                self.x_range[0], self.x_range[1], self.x_step, self._tpl_u8.data_ptr(), self._n_rows, self._n_cols,
                nat.stream_ptr()), "prs_vt_extract_u8")
            return self._tpl_u8, torch.uint8
        if not self._fast:
            if self._mask_dev is None:
                self._mask_dev = torch.from_numpy(self.mask).to(self.device)
            t = fr if isinstance(fr, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(fr))
            t = t.to(self.device)
            if not is_u8:
                t = t.to(torch.float32)
            return t[self._mask_dev].reshape(tuple(self.shape)).contiguous(), (torch.uint8 if is_u8 else torch.float32)
        if is_u8:
            if isinstance(fr, torch.Tensor):
                self._frame_dev.copy_(fr, non_blocking=True)
            else:
                self._frame_pin.numpy()[...] = fr
                self._frame_dev.copy_(self._frame_pin, non_blocking=True)
            nat.check(nat.lib().prs_vt_extract_u8(
                self._frame_dev.data_ptr(), self.im_x, self.im_y, self.y_range[0], self.y_range[1], self.y_step,
                self.x_range[0], self.x_range[1], self.x_step, self._tpl_u8.data_ptr(), self._n_rows, self._n_cols,
                nat.stream_ptr()), "prs_vt_extract_u8")
            return self._tpl_u8, torch.uint8
        # float frames: ordinary SAD in float32
        t = fr if isinstance(fr, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(fr))
        t = t.to(self.device, torch.float32)
        r0, c0 = self.y_range[0] + 1, self.x_range[0] + 1
        if self.x_step != 2 or self.y_step != 2:
            m = torch.from_numpy(self.mask).to(self.device)
            return t[m].reshape(32, 32).contiguous(), torch.float32
        return t[r0: self.y_range[1]: 2, c0: self.x_range[1]: 2].contiguous(), torch.float32

    def _sweep(self, tpl, torch_dtype, key_dev, scores_ptr=None):
        lib_ptr = self._lib.data_ptr() if self._n else None
        if not self._fast:
            fn = nat.lib().prs_vt_sweep_any_u8 if torch_dtype == torch.uint8 else nat.lib().prs_vt_sweep_any_f32
            nat.check(fn(lib_ptr, self._n, tpl.data_ptr(), int(self.shape[0]), int(self.shape[1]), ViewTemplate.max_offset,
                         0, key_dev.data_ptr(), scores_ptr, nat.stream_ptr()), "prs_vt_sweep_any")
        elif torch_dtype == torch.uint8:
            nat.check(nat.lib().prs_vt_sweep_packed_u8(lib_ptr, self._n, tpl.data_ptr(), self.mode, 0,
                                                       key_dev.data_ptr(), scores_ptr, self._scratch.data_ptr(),
                                                       nat.stream_ptr()), "prs_vt_sweep_packed_u8")
        else:
            nat.check(nat.lib().prs_vt_sweep_f32(lib_ptr, self._n, tpl.data_ptr(), self.mode, 0, key_dev.data_ptr(),
                                                 scores_ptr, nat.stream_ptr()), "prs_vt_sweep_f32")

    def _decode(self, key, torch_dtype):
        """``(score, index)`` from the packed key, or ``(None, -1)`` when nothing was compared."""
        key &= _KEY_NONE
        if key == _KEY_NONE:
            return None, -1
        hi, idx = key >> 32, key & 0xFFFFFFFF
        if torch_dtype == torch.uint8:
            return int(hi), int(idx)
        return float(np.array([hi], dtype=np.uint32).view(np.float32)[0]), int(idx)

    def scores(self, input):
        """Per-template scores of a frame against the whole library (numpy array); for inspection and tests."""
        with torch.cuda.device(self.device):
            tpl, td = self._subsample(input)
            self._ensure_lib(td)
            out = torch.empty(self._n, dtype=torch.int32 if td == torch.uint8 else torch.float32, device=self.device)
            self._sweep(tpl, td, self._key, out.data_ptr())
            res = out.cpu().numpy()
            return res.view(np.uint32).astype(np.int64) if td == torch.uint8 else res

    def match(self, input, pc_x, pc_y, pc_th):
        """Best stored template for this frame, or a newly created one (``view_templates.py:63-75``)."""
        with torch.cuda.device(self.device):
            tpl, td = self._subsample(input)
            self._ensure_lib(td)
            self._sweep(tpl, td, self._key)
            self._key_pin.copy_(self._key, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            score, idx = self._decode(int(self._key_pin[0]), td)
            self.last_score = score
            if score is None or score > self.match_threshold:
                return self._append(tpl, pc_x, pc_y, pc_th)
            return self.templates[idx]

    # north_star spelling: force creation of a template from a frame
    def create(self, input, pc_x, pc_y, pc_th):
        with torch.cuda.device(self.device):
            tpl, td = self._subsample(input)
            self._ensure_lib(td)
            t = self._append(tpl, pc_x, pc_y, pc_th)
            torch.cuda.current_stream().synchronize()   # the pinned staging frame may be rewritten by the next call
            return t


class ShardedViewTemplates:
    """A template library split by contiguous index ranges over the ranks of a process group.

    Rank r holds templates ``[base_r, base_r + n_r)``.  A query sweeps the local shard and the ranks' packed keys
    are MIN-reduced, which yields the global minimum score and, among equal scores, the lowest global index --
    ``numpy.argmin`` semantics (``view_templates.py:73``).  New templates are appended to the last rank's shard so
    global indices stay contiguous.

    ``exchange`` selects how the keys meet: ``"fused"`` -- one small kernel per query that writes this rank's key
    into every peer's CUDA-IPC-mapped buffer over NVLink, waits for the peers' keys, reduces them and (for
    ``match``) takes the create-or-match decision and appends on the device, the 32-byte result landing in pinned
    host memory (``csrc/sharded.cu``) -- or ``"nccl"``: a MIN all-reduce of the int64 key through
    ``torch.distributed``.  ``"auto"`` uses the fused exchange and falls back to NCCL, with a warning, when the
    peers' buffers cannot be mapped.  ``self.exchange`` names what is in use.
    """

    def __init__(self, local_templates, base_index, match_threshold, mode="ref", group=None, device=None,
                 exchange="auto", capacity=None):
        import torch.distributed as dist
        nat.require_cuda()
        self._dist = dist
        self.group = group
        self._distributed = dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank(group) if self._distributed else 0
        self.world = dist.get_world_size(group) if self._distributed else 1
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        t = local_templates if isinstance(local_templates, torch.Tensor) else torch.from_numpy(
            np.ascontiguousarray(local_templates))
        if t.dtype not in (torch.uint8, torch.float32):
            raise TypeError("templates must be uint8 or float32")
        self._n = int(t.shape[0])
        self._dtype = t.dtype
        self._owner = self.rank == self.world - 1          # created templates go to the last rank's shard
        self._cap = max(self._n + (64 if self._owner else 0), 32) if capacity is None else max(int(capacity), self._n, 32)
        self._scratch = torch.empty(4096, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            self._lib = self._alloc(self._cap)
            src = t.to(self.device).contiguous()
            if self._n:
                if self._dtype == torch.uint8:
                    nat.check(nat.lib().prs_vt_pack_u8(src.data_ptr(), self._n, self._lib.data_ptr(), 0,
                                                       nat.stream_ptr()), "prs_vt_pack_u8")
                else:
                    self._lib[: self._n].copy_(src)
            torch.cuda.current_stream().synchronize()
        del src
        self.base_index = int(base_index)
        self.match_threshold = match_threshold
        self.mode = {"ref": nat.VT_MODE_REF, "circular": nat.VT_MODE_CIRCULAR}[mode]
        self._key = torch.empty(1, dtype=torch.int64, device=self.device)
        self._keys_pin = torch.zeros(64, dtype=torch.int64).pin_memory()
        self._res_pin = torch.zeros(ctypes.sizeof(nat.ShardResult), dtype=torch.uint8).pin_memory()
        self._res = nat.ShardResult.from_address(self._res_pin.data_ptr())
        if self._distributed:
            counts = torch.tensor([self._n], dtype=torch.int64, device=self.device)
            allc = [torch.zeros_like(counts) for _ in range(self.world)]
            dist.all_gather(allc, counts, group=group)
            self.n_total = int(sum(int(c.item()) for c in allc))
        else:
            self.n_total = self._n
        self._xchg = None
        self.exchange = "nccl"
        if exchange not in ("auto", "fused", "nccl"):
            raise ValueError("exchange must be 'auto', 'fused' or 'nccl'")
        if exchange != "nccl":
            self._connect(strict=exchange == "fused")

    # ------------------------------------------------------------------ set-up
    def _alloc(self, capacity):
        if self._dtype == torch.uint8:
            nbytes = int(nat.lib().prs_vt_packed_bytes(int(capacity)))
            return torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        return torch.empty((capacity, 32, 32), dtype=torch.float32, device=self.device)

    def _connect(self, strict):
        """Create this rank's exchange buffer and map the peers' (CUDA IPC handles all-gathered through the group)."""
        dist = self._dist
        L = nat.lib()
        with torch.cuda.device(self.device):
            h = ctypes.c_void_p()
            nat.check(L.prs_xchg_create(self.world, self.rank, ctypes.byref(h)), "prs_xchg_create")
            ok = 1
            if self.world > 1:
                mine = torch.zeros(nat.XCHG_HANDLE_BYTES, dtype=torch.uint8)
                nat.check(L.prs_xchg_export(h, mine.data_ptr()), "prs_xchg_export")
                on_gpu = dist.get_backend(self.group) == "nccl"
                mine = mine.to(self.device) if on_gpu else mine
                allh = [torch.zeros_like(mine) for _ in range(self.world)]
                dist.all_gather(allh, mine, group=self.group)
                handles = torch.stack([a.cpu() for a in allh]).contiguous()
                rc = L.prs_xchg_connect(h, handles.data_ptr())
                msg = L.prs_last_error().decode(errors="replace") if rc != 0 else ""
                flag = torch.tensor([1 if rc == 0 else 0], dtype=torch.int64, device=self.device if on_gpu else "cpu")
                dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)   # all ranks take the same path
                ok = int(flag.item())
                if not ok:
                    L.prs_xchg_destroy(h)
                    if strict:
                        raise nat.NativeError("fused exchange unavailable: %s" % (msg or "a peer could not map the buffers"))
                    import warnings
                    warnings.warn("ShardedViewTemplates: CUDA IPC mapping failed (%s); using the NCCL all-reduce" % msg)
                    return
            self._xchg = h
            self.exchange = "fused"

    def set_exchange(self, name):
        """Switch between the fused device-side exchange and the NCCL all-reduce (every rank must do the same)."""
        if name == "nccl":
            if self._xchg is not None:
                self._xchg_off, self._xchg = self._xchg, None
            self.exchange = "nccl"
        elif name == "fused":
            if self._xchg is None:
                if getattr(self, "_xchg_off", None) is None:
                    raise nat.NativeError("the fused exchange was never connected")
                self._xchg, self._xchg_off = self._xchg_off, None
            self.exchange = "fused"
        else:
            raise ValueError("exchange must be 'fused' or 'nccl'")

    def close(self):
        if self._xchg is None and getattr(self, "_xchg_off", None) is not None:
            self._xchg, self._xchg_off = self._xchg_off, None
        if self._xchg is not None:
            with torch.cuda.device(self.device):
                nat.lib().prs_xchg_destroy(self._xchg)
            self._xchg = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return self.n_total

    def _grow(self, need):
        if need <= self._cap:
            return
        cap = max(need, self._cap * 2)
        new = self._alloc(cap)
        if self._dtype == torch.uint8:
            new[: self._lib.numel()].copy_(self._lib)        # whole 32-template groups, position independent
        else:
            new[: self._n].copy_(self._lib[: self._n])
        self._lib, self._cap = new, cap

    def _store_local(self, query_dev):
        """Append the query to this rank's shard: ONE slot is written (``prs_vt_pack_u8(first=n)``)."""
        self._grow(self._n + 1)
        if self._dtype == torch.uint8:
            nat.check(nat.lib().prs_vt_pack_u8(query_dev.data_ptr(), 1, self._lib.data_ptr(), self._n, nat.stream_ptr()),
                      "prs_vt_pack_u8")
        else:
            self._lib[self._n].copy_(query_dev.reshape(32, 32))
        self._n += 1

    # ------------------------------------------------------------------ matching
    def local_sweep(self, query_dev, key=None):
        """Launch the local sweep; the packed key is left in ``key`` (a one-element int64 device tensor, default
        ``self._key``) on the device."""
        key = self._key if key is None else key
        lib_ptr = self._lib.data_ptr() if self._n else None
        if self._dtype == torch.uint8:
            nat.check(nat.lib().prs_vt_sweep_packed_u8(lib_ptr, self._n, query_dev.data_ptr(), self.mode,
                                                       self.base_index, key.data_ptr(), None,
                                                       self._scratch.data_ptr(), nat.stream_ptr()),
                      "prs_vt_sweep_packed_u8")
        else:
            nat.check(nat.lib().prs_vt_sweep_f32(lib_ptr, self._n, query_dev.data_ptr(), self.mode, self.base_index,
                                                 key.data_ptr(), None, nat.stream_ptr()), "prs_vt_sweep_f32")
        return key

    def _check_status(self):
        if self._res.status != 0:
            raise nat.NativeError("sharded exchange %d timed out waiting for a peer rank" % self._res.seq)

    def match_keys(self, queries_dev):
        """``match_key`` for a batch of queries ``[Q, 32, 32]``: Q local sweeps, ONE exchange of the Q packed keys
        and one read-back -- the exchange and the synchronisation are paid once per batch, not once per query.
        Returns a list of ``(score, index)``, identical on every rank."""
        Q = int(queries_dev.shape[0])
        keys = torch.empty(Q, dtype=torch.int64, device=self.device)
        is_float = self._dtype != torch.uint8
        with torch.cuda.device(self.device):
            for i in range(Q):
                self.local_sweep(queries_dev[i], keys[i:i + 1])
            if self._xchg is None:
                host = reduce_packed_key(keys, self.group).cpu().numpy()
                return [unpack_key(int(k), is_float=is_float) for k in host]
            out = []
            for q0 in range(0, Q, 64):                          # the exchange kernel carries up to 64 keys
                nq = min(64, Q - q0)
                nat.check(nat.lib().prs_vt_shard_exchange(self._xchg, keys[q0:].data_ptr(), nq, self._keys_pin.data_ptr(),
                                                          self._res_pin.data_ptr(), nat.stream_ptr()),
                          "prs_vt_shard_exchange")
                nat.check(nat.lib().prs_xchg_wait(self._xchg, self._res_pin.data_ptr(), 30.0), "prs_xchg_wait")
                self._check_status()
                out += [unpack_key(int(k), is_float=is_float) for k in self._keys_pin[:nq].tolist()]
        return out

    def match_key(self, query_dev):
        """Global ``(score, index)`` of the best match over all shards; identical on every rank."""
        is_float = self._dtype != torch.uint8
        with torch.cuda.device(self.device):
            if self._xchg is None:
                k = int(reduce_packed_key(self.local_sweep(query_dev), self.group).item())
                return unpack_key(k, is_float=is_float)
            return unpack_key(self._query(query_dev, 0).key, is_float=is_float)

    def _query(self, query_dev, decide):
        """Sweep + exchange (+ decision) + wait for the pinned record, one library call (``prs_vt_shard_query``)."""
        nat.check(nat.lib().prs_vt_shard_query(
            self._xchg, nat.PRS_U8 if self._dtype == torch.uint8 else nat.PRS_F32, self._lib.data_ptr(), self._n,
            query_dev.data_ptr(), self.mode, self.base_index, self._key.data_ptr(), self._scratch.data_ptr(), decide,
            float(self.match_threshold), self.n_total, 1 if self._owner else 0, self._res_pin.data_ptr(),
            nat.stream_ptr()), "prs_vt_shard_query")
        self._check_status()
        return self._res

    def match(self, query_dev):
        """``(index, created)`` with the reference's create-or-match rule applied identically on every rank."""
        if self._xchg is None:
            score, idx = self.match_key(query_dev)
            index, created = decide(score, idx, self.n_total, self.match_threshold)
            if created:
                if self._owner:
                    with torch.cuda.device(self.device):
                        self._store_local(query_dev)
                self.n_total += 1
            return index, created
        with torch.cuda.device(self.device):
            if self._owner:
                self._grow(self._n + 1)                        # room for the template the kernel may append
            self._query(query_dev, 1)
            created = bool(self._res.created)
            if created:
                if self._owner:
                    self._n += 1
                self.n_total += 1
            return int(self._res.template_index), created
