"""Pose-cell network on the B200: the reference's class surface over the CUDA library.

``PoseCellNetwork`` keeps the names, arguments and return values of
``ratslam/posecell_network.py:22-353`` -- ``update`` / ``inject`` /
``path_integration`` / ``get_pc_max``, the ``posecells`` / ``max_pc`` /
``kernel_3d`` attributes -- while the state lives on the device and every step is
a launch of the kernels in ``csrc/`` through the C ABI
(``include/pyratslam_b200.h``).  The reference's ``Convolution`` operator
(``ratslam/convolution.py``) has no counterpart here: it is replaced outright.

``PoseCellEnsemble`` is the batched form (BASELINE config 4): B independent
networks of one shape, each with its own global inhibition and odometry stream.
"""
from __future__ import annotations

import ctypes
import math

import numpy as np
import torch

from . import _native as nat
from . import kernels as K


def _as_np_dtype(dtype):
    if dtype in (None, "float32", np.float32, torch.float32):
        return np.float32
    if dtype in ("float64", np.float64, torch.float64, float):
        return np.float64
    raise TypeError("Data type specified is not currently supported: %r" % (dtype,))  # convolution.py:25


_PATHS = {0: "generic", 1: "resident", 2: "tiled", 3: "cluster", 4: "pair"}



_HOST_TABLES = None


def _host_tables():
    """The filter tables of ``PoseCellNetwork.__init__`` (posecell_network.py:24-59), computed once per process."""
    global _HOST_TABLES
    if _HOST_TABLES is None:
        fd = K.build_diff_gaussian_set_2d()
        _HOST_TABLES = {
            "kernel_3d": K.diff_gaussian(order=3),
            "filter_dict_2d": fd,
            "separable": K.separable_dog_factors(),
            "f2d": np.ascontiguousarray(np.stack([fd[(0, 0)], fd[(-1, -1)]])),
            "f1d": np.ascontiguousarray(K.theta_filter_table(nat.OG_RANGE)),
        }
    return _HOST_TABLES


def _raw_stream(dev_index):
    """The current CUDA stream of ``dev_index`` as an integer handle (torch's C accessor: no Stream object)."""
    try:
        return torch._C._cuda_getCurrentRawStream(dev_index)
    except AttributeError:  # pragma: no cover - older torch
        return torch.cuda.current_stream(dev_index).cuda_stream

class PoseCellEnsemble:
    """B independent pose-cell networks of one shape, resident on one GPU."""

    def __init__(self, shape, n_networks=1, global_inhibition=K.PC_GLOBAL_INHIB, dtype=np.float32, device=None,
                 active_set=0):
        nat.require_cuda()
        if len(shape) != 3:
            raise ValueError("shape must be (X, Y, Th)")
        self.shape = tuple(int(s) for s in shape)
        self.n_networks = int(n_networks)
        self.np_dtype = _as_np_dtype(dtype)
        self.torch_dtype = torch.float32 if self.np_dtype == np.float32 else torch.float64
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        X, Y, Th = self.shape
        B = self.n_networks

        # host tables, float64, as the reference computes them (they depend on the module constants only: computed
        # once per process, every network gets its own copies of what it exposes as attributes)
        tables = _host_tables()
        self.kernel_3d = tables["kernel_3d"].copy()
        self.pc_vtrans_scale = K.PC_CELL_X_SIZE
        self.pc_vrot_scale = 2.0 * math.pi / Th
        self.filter_dict_2d = {k: v.copy() for k, v in tables["filter_dict_2d"].items()}
        self.filter_dict_2d_precision = 10
        ge, gi, aE, aI = tables["separable"]
        f2d, f1d = tables["f2d"], tables["f1d"]
        mid = Th // 2
        ang = (np.arange(Th) - mid) * self.pc_vrot_scale
        self._cos = np.ascontiguousarray(np.cos(ang))
        self._sin = np.ascontiguousarray(np.sin(ang))
        dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
        ge = np.ascontiguousarray(ge)
        gi = np.ascontiguousarray(gi)
        cfg = nat.PcConfig(X, Y, Th, B, nat.PRS_F32 if self.np_dtype == np.float32 else nat.PRS_F64,
                           self.pc_vtrans_scale, self.pc_vrot_scale, dp(ge), dp(gi), aE, aI, dp(f2d), dp(f1d),
                           dp(self._cos), dp(self._sin))
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_create(ctypes.byref(cfg), ctypes.byref(self._h)), "prs_pc_create")
        dev, td = self.device, self.torch_dtype
        self._state = torch.zeros((B, Th, X, Y), dtype=td, device=dev)       # theta-major, see the header
        self._gi = torch.empty(B, dtype=td, device=dev)
        self.global_inhibition = global_inhibition
        self._odom = torch.zeros((B, 2), dtype=torch.float64, device=dev)
        self._argmax = torch.zeros(B, dtype=torch.int64, device=dev)
        self._total = torch.zeros(B, dtype=td, device=dev)
        self._err = torch.zeros(B, dtype=torch.int32, device=dev)
        self._odom_pin = torch.zeros((B, 2), dtype=torch.float64).pin_memory()
        self._res_pin = torch.zeros((B, 4), dtype=torch.int32).pin_memory()   # (x, y, th, err) per network
        self._res_np = self._res_pin.numpy()
        self._odom_np = self._odom_pin.numpy()
        # fixed addresses and the bound entry point of the single-call update (PoseCellNetwork.update)
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self._state_ptr = self._state.data_ptr()
        self._gi_ptr = self._gi.data_ptr()
        self._odom_pin_ptr = self._odom_pin.data_ptr()
        self._res_pin_ptr = self._res_pin.data_ptr()
        self._update_host = nat.lib().prs_pc_update_host
        self.max_pc = np.zeros((B, 3), dtype=np.int64)
        # bumped by every call that changes the device state; users that cache something derived from the state on
        # the device (the frame plans of ros_simulate cache the arg-max) compare it with the value they last saw
        self._state_gen = 0
        if active_set:
            self.set_option("active_set", active_set)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                nat.lib().prs_pc_destroy(h)
            except Exception:
                pass
            self._h = None

    # ------------------------------------------------------------------ parameters
    @property
    def global_inhibition(self):
        return self._gi_host if self._gi_host.size > 1 else float(self._gi_host[0])

    @global_inhibition.setter
    def global_inhibition(self, value):
        g = np.broadcast_to(np.asarray(value, dtype=np.float64), (self.n_networks,)).copy()
        self._gi_host = g
        self._gi.copy_(torch.from_numpy(g).to(self.torch_dtype))

    @property
    def path(self):
        """``"pair"`` (fused SMEM-resident kernel, one network per 2-CTA cluster), ``"resident"`` (the same with one
        CTA per network), ``"cluster"`` (one network spread over a large thread-block cluster: lowest latency),
        ``"tiled"`` (large-grid kernels) or ``"generic"``."""
        return _PATHS[nat.lib().prs_pc_path(self._h)]

    def force_path(self, name):
        """Choose the kernel family (``"auto"`` or one of the ``path`` names); ``ValueError`` if the plan's shape
        or dtype is not supported by it.  For tests and profiling."""
        code = {v: k for k, v in _PATHS.items()}.get(name, -1 if name == "auto" else None)
        if code is None:
            raise ValueError("unknown path %r" % (name,))
        if nat.lib().prs_pc_set_path(self._h, code) != 0:
            raise ValueError(nat.lib().prs_last_error().decode())

    def set_option(self, name, value):
        """The per-plan option of the kernels, ``"active_set"`` -- 0 / 1 / 2: the sparsity-aware update of
        csrc/posecell_active.cu (off / the state is scanned for its non-zero cells every update / the list of non-zero
        cells is carried from update to update), same results, a cost that follows the size of the activity packet
        instead of the grid."""
        code = {"active_set": 2}[name]
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_set_option(self._h, code, int(value)), "prs_pc_set_option")

    def invalidate_active(self):
        """``active_set=2`` keeps the list of non-zero cells from one update to the next; whoever writes ``state`` other
        than through this class (a torch operation on the tensor) calls this afterwards."""
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_invalidate_active(self._h, nat.stream_ptr()), "prs_pc_invalidate_active")

    # ------------------------------------------------------------------ state access
    @property
    def state(self):
        """The device tensor ``[B, Th, X, Y]`` (theta-major)."""
        return self._state

    @property
    def posecells(self):
        """Host copy in the reference's layout and dtype: float64 ``[B, X, Y, Th]``."""
        with torch.cuda.device(self.device):
            out = torch.empty((self.n_networks,) + self.shape, dtype=self.torch_dtype, device=self.device)
            nat.check(nat.lib().prs_pc_export_xyt(self._h, self._state.data_ptr(), out.data_ptr(), nat.stream_ptr()),
                      "prs_pc_export_xyt")
            return out.cpu().numpy().astype(np.float64)

    @posecells.setter
    def posecells(self, value):
        self._state_gen += 1
        v = np.asarray(value, dtype=self.np_dtype).reshape((self.n_networks,) + self.shape)
        with torch.cuda.device(self.device):
            src = torch.from_numpy(np.ascontiguousarray(v)).to(self.device)
            nat.check(nat.lib().prs_pc_import_xyt(self._h, self._state.data_ptr(), src.data_ptr(), nat.stream_ptr()),
                      "prs_pc_import_xyt")
            torch.cuda.current_stream().synchronize()

    def inject(self, energy, loc, network=None):
        """``posecells[loc] += energy`` on one network or on all of them (posecell_network.py:322-324)."""
        self._state_gen += 1
        x, y, th = (int(v) for v in loc)  # py2 callers pass math.floor() floats; old numpy truncated them
        X, Y, Th = self.shape
        x, y, th = (v + n if -n <= v < 0 else v for v, n in ((x, X), (y, Y), (th, Th)))  # numpy negative indices
        if not (0 <= x < X and 0 <= y < Y and 0 <= th < Th):
            raise IndexError("index %r is out of bounds for shape %r" % (tuple(loc), self.shape))
        b = -1 if network is None else int(network)
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_inject(self._h, self._state.data_ptr(), b, x, y, th, float(energy),
                                              nat.stream_ptr()), "prs_pc_inject")

    def active_cells(self, threshold=0.002, network=0, max_cells=None):
        """Cells with activity above ``threshold`` as ``(index int64[n, 3], value float64[n])`` in the reference's
        C order -- ``nonzero(pc > threshold)`` and ``pc[...]`` of ``simulate.py:60-62`` without moving the whole
        grid to the host (compaction runs on the device)."""
        N = int(np.prod(self.shape))
        cap = N if max_cells is None else int(max_cells)
        with torch.cuda.device(self.device):
            idx = torch.empty(cap, dtype=torch.int32, device=self.device)
            val = torch.empty(cap, dtype=self.torch_dtype, device=self.device)
            cnt = torch.zeros(1, dtype=torch.int32, device=self.device)
            work = torch.empty(int(nat.lib().prs_pc_active_work_bytes(self._h)), dtype=torch.uint8, device=self.device)
            nat.check(nat.lib().prs_pc_active_cells(self._h, self._state.data_ptr(), int(network), float(threshold), cap,
                                                    idx.data_ptr(), val.data_ptr(), cnt.data_ptr(), work.data_ptr(),
                                                    nat.stream_ptr()), "prs_pc_active_cells")
            n = min(int(cnt.item()), cap)
            flat = idx[:n].cpu().numpy().astype(np.int64)
            return self._unravel(flat), val[:n].cpu().numpy().astype(np.float64)

    def _unravel(self, flat):
        X, Y, Th = self.shape
        flat = np.asarray(flat, dtype=np.int64)
        return np.stack([flat // (Y * Th), (flat // Th) % Y, flat % Th], axis=-1)

    def get_pc_max(self):
        """Arg-max cell of every network, ``int64[B, 3]`` (first maximum in the reference's C order)."""
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_argmax(self._h, self._state.data_ptr(), self._argmax.data_ptr(),
                                              nat.stream_ptr()), "prs_pc_argmax")
            return self._unravel(self._argmax.cpu().numpy())

    # ------------------------------------------------------------------ stepping
    def update_async(self, odom_dev=None):
        """One update of all networks with device odometry ``float64[B, 2]``; no host synchronisation.

        Results land in ``self._argmax`` (flat indices), ``self._total`` and ``self._err`` on the device.
        """
        self._state_gen += 1
        od = self._odom if odom_dev is None else odom_dev
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_step(self._h, self._state.data_ptr(), od.data_ptr(), self._gi.data_ptr(),
                                            self._argmax.data_ptr(), self._total.data_ptr(), self._err.data_ptr(),
                                            nat.stream_ptr()), "prs_pc_step")

    def update(self, v):
        """One ``update`` per network with host odometry ``[B, 2]``; returns ``int64[B, 3]`` arg-max cells.

        Raises ``KeyError`` / ``ValueError`` if any network hit the conditions under which the reference
        raises or reads unwritten memory (see PRS_ERR_* in the header).
        """
        self._state_gen += 1
        self._odom_np[...] = np.asarray(v, dtype=np.float64).reshape(self.n_networks, 2)
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_step_host_xyz(self._h, self._state.data_ptr(), self._odom_pin.data_ptr(),
                                                     self._gi.data_ptr(), self._res_pin.data_ptr(), nat.stream_ptr()),
                      "prs_pc_step_host_xyz")
        res = self._res_np
        if res[:, 3].any():
            self._raise_on_err(res[:, 3])
        self.max_pc = res[:, :3].astype(np.int64)
        return self.max_pc

    # Overlapped host stepping: ``update_submit`` stages one step (pinned odometry in, kernels, packed result out) on
    # the current stream without waiting; ``update_result`` returns the oldest outstanding step's arg-max cells.  With
    # one step kept in flight the copies and the launch overhead of step t+1 hide behind the kernel of step t.
    def update_submit(self, v):
        self._state_gen += 1
        if not hasattr(self, "_pipe"):
            B = self.n_networks
            self._pipe = [{"odom": torch.zeros((B, 2), dtype=torch.float64).pin_memory(),
                           "res": torch.zeros((B, 4), dtype=torch.int32).pin_memory(),
                           "slot": ctypes.c_int(0)} for _ in range(2)]
            for sl in self._pipe:
                sl["odom_np"], sl["res_np"] = sl["odom"].numpy(), sl["res"].numpy()
            self._pipe_head = self._pipe_tail = 0
        if self._pipe_head - self._pipe_tail >= 2:
            raise RuntimeError("update_submit: two steps are already in flight; call update_result() first")
        sl = self._pipe[self._pipe_head % 2]
        sl["odom_np"][...] = np.asarray(v, dtype=np.float64).reshape(self.n_networks, 2)
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_step_host_xyz_async(self._h, self._state.data_ptr(), sl["odom"].data_ptr(),
                                                           self._gi.data_ptr(), sl["res"].data_ptr(), nat.stream_ptr(),
                                                           ctypes.byref(sl["slot"])), "prs_pc_step_host_xyz_async")
        self._pipe_head += 1

    def update_result(self):
        if not hasattr(self, "_pipe") or self._pipe_head == self._pipe_tail:
            raise RuntimeError("update_result: no step in flight")
        sl = self._pipe[self._pipe_tail % 2]
        self._pipe_tail += 1
        nat.check(nat.lib().prs_pc_host_result_wait(self._h, sl["slot"].value), "prs_pc_host_result_wait")
        res = sl["res_np"]
        if res[:, 3].any():
            self._raise_on_err(res[:, 3])
        self.max_pc = res[:, :3].astype(np.int64)
        return self.max_pc

    def update_stream(self, odom_seq):
        """Generator over ``update`` results for a sequence of host odometry arrays, one step kept in flight."""
        first = True
        for v in odom_seq:
            self.update_submit(v)
            if not first:
                yield self.update_result()
            first = False
        if not first:
            yield self.update_result()

    def path_integration(self, v):
        """Path integration only (no DoG / inhibition / normalisation) with host odometry ``[B, 2]``."""
        self._state_gen += 1
        vv = np.asarray(v, dtype=np.float64).reshape(self.n_networks, 2)
        self._odom.copy_(torch.from_numpy(vv))
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_path_integration(self._h, self._state.data_ptr(), self._odom.data_ptr(),
                                                        self._err.data_ptr(), nat.stream_ptr()),
                      "prs_pc_path_integration")
        self._raise_on_err(self._err.cpu().numpy())

    def run(self, odom, return_totals=False):
        """``T`` consecutive updates from ``odom[T, B, 2]`` (host or device); returns ``int64[T, B, 3]``."""
        self._state_gen += 1
        if isinstance(odom, torch.Tensor):
            od = odom.to(self.device, torch.float64).contiguous()
        else:
            od = torch.from_numpy(np.ascontiguousarray(np.asarray(odom, dtype=np.float64))).to(self.device)
        T = od.shape[0]
        od = od.reshape(T, self.n_networks, 2)
        amax = torch.empty((T, self.n_networks), dtype=torch.int64, device=self.device)
        tot = torch.empty((T, self.n_networks), dtype=self.torch_dtype, device=self.device)
        with torch.cuda.device(self.device):
            nat.check(nat.lib().prs_pc_run(self._h, self._state.data_ptr(), od.data_ptr(), T, self._gi.data_ptr(),
                                           amax.data_ptr(), tot.data_ptr(), self._err.data_ptr(), nat.stream_ptr()),
                      "prs_pc_run")
        self._raise_on_err(self._err.cpu().numpy())
        out = self._unravel(amax.cpu().numpy())
        if T:
            self.max_pc = out[-1]
        return (out, tot.cpu().numpy().astype(np.float64)) if return_totals else out

    @staticmethod
    def _raise_on_err(err):
        if not err.any():
            return
        bad = np.flatnonzero(err)
        e = int(np.bitwise_or.reduce(err))
        if e & nat.ERR_LUT_KEY:
            raise KeyError((5, 5))  # posecell_network.py:249: the LUT has no key 5
        if e & nat.ERR_RADIUS:
            raise ValueError("translation exceeds the grid: 3 + ceil|vtrans/%.3g| > min(X, Y) for network(s) %s"
                             % (K.PC_CELL_X_SIZE, bad[:8].tolist()))
        raise ValueError("rotation beyond the theta filter table for network(s) %s" % bad[:8].tolist())


class PoseCellNetwork:
    """Drop-in for ``ratslam/posecell_network.py:PoseCellNetwork`` (one network, B = 1).

    ``dtype=numpy.float32`` (default) is the fast mode; ``dtype=numpy.float64`` is the strict-parity
    mode in the reference's own precision.  Unknown keyword arguments are accepted and ignored like
    the reference's ``**kwargs`` (posecell_network.py:24).
    """

    def __init__(self, shape, dtype=np.float32, device=None, active_set=0, **kwargs):
        self._ens = PoseCellEnsemble(shape, 1, dtype=dtype, device=device, active_set=active_set)
        self.shape = self._ens.shape
        e = self._ens
        self.kernel_3d = e.kernel_3d
        self.kernel_2d = K.diff_gaussian(order=2)
        self.kernel_1d = K.diff_gaussian(order=1)
        self.kernel_1d_sep = K.diff_gaussian_separable()
        self.pc_vtrans_scale = e.pc_vtrans_scale
        self.pc_vrot_scale = e.pc_vrot_scale
        self.filter_dict_2d = e.filter_dict_2d
        self.filter_dict_2d_precision = e.filter_dict_2d_precision
        self.max_pc = (0, 0, 0)
        self._max_valid = False   # max_pc mirrors the device state (set by update, cleared by writes)

    # reference attribute: a plain float (posecell_network.py:34)
    @property
    def global_inhibition(self):
        return self._ens.global_inhibition

    @global_inhibition.setter
    def global_inhibition(self, v):
        self._ens.global_inhibition = float(v)

    @property
    def posecells(self):
        """float64 ``[X, Y, Th]`` host copy (synchronises); assignable."""
        return self._ens.posecells[0]

    @posecells.setter
    def posecells(self, value):
        self._ens.posecells = np.asarray(value)[None]
        self._max_valid = False

    @property
    def path(self):
        return self._ens.path

    # builder methods of the reference class surface (host, cheap)
    diff_gaussian = staticmethod(K.diff_gaussian)
    diff_gaussian_separable = staticmethod(K.diff_gaussian_separable)
    diff_gaussian_offset_2d = staticmethod(K.diff_gaussian_offset_2d)
    diff_gaussian_offset_1d = staticmethod(K.diff_gaussian_offset_1d)
    build_diff_gaussian_set_2d = staticmethod(K.build_diff_gaussian_set_2d)
    build_kernel = staticmethod(K.build_kernel)

    def filters_from_origins(self, origins, shape=(7, 7)):
        num = origins.shape[1]
        out = np.empty((shape[0], shape[1], num))
        for z in range(num):
            out[:, :, z] = K.diff_gaussian_offset_2d(shape=shape, origin=origins[:, z])
        return out

    def filters_from_origins_approx(self, origins, shape=(7, 7)):
        """LUT lookup of posecell_network.py:244-250 (both key parts come from the x offset)."""
        num = origins.shape[1]
        out = np.empty((shape[0], shape[1], num))
        for z in range(num):
            k = int(origins[0, z] * self.filter_dict_2d_precision)
            out[:, :, z] = self.filter_dict_2d[(k, k)]
        return out

    def inject(self, energy, loc):
        self._ens.inject(energy, loc, network=0)
        self._max_valid = False

    def active_cells(self, threshold=0.002, max_cells=None):
        """``(index[n, 3], value[n])`` of the cells above ``threshold`` (what ``simulate.py:60-62`` plots)."""
        return self._ens.active_cells(threshold, 0, max_cells)

    def get_pc_max(self):
        """Arg-max cell (posecell_network.py:317-319).  Right after ``update`` this is the value the step
        kernel already produced; otherwise it is recomputed on the device."""
        if self._max_valid:
            return self.max_pc
        x, y, th = self._ens.get_pc_max()[0]
        return (int(x), int(y), int(th))

    def _precheck(self, vtrans, vrot):
        """Raise what the reference raises (or would have to) *before* touching the device state."""
        e = self._ens
        vt = vtrans / e.pc_vtrans_scale
        ex = vt * e._cos
        d = ex - np.around(ex)
        if ((d * 10).astype(np.int64) >= 5).any():
            raise KeyError((5, 5))                          # posecell_network.py:249
        if 3 + math.ceil(abs(vt)) > min(self.shape[0], self.shape[1]):
            raise ValueError("translation of %.3g cells does not fit a %dx%d grid (convolution.py:661-675 would "
                             "read unwritten memory)" % (vt, self.shape[0], self.shape[1]))

    def update(self, v=(0.0, 0.0)):
        """One attractor update + path integration; returns the arg-max cell (posecell_network.py:326-353).

        One library call (``prs_pc_update_host``): the odometry is checked on the host for the cases in which the
        reference raises (``KeyError``) or reads unwritten memory (``ValueError``) *before* the device state is
        touched, then the step runs and the packed ``(x, y, th, err)`` result comes back through pinned memory."""
        vtrans, vrot = float(v[0]), float(v[1])
        e = self._ens
        if torch.cuda.current_device() != e._dev_index:
            with torch.cuda.device(e.device):
                return self.update((vtrans, vrot))
        e._state_gen += 1
        rc = e._update_host(e._h, e._state_ptr, vtrans, vrot, e._gi_ptr, e._odom_pin_ptr, e._res_pin_ptr,
                            _raw_stream(e._dev_index))
        if rc != 0:
            if rc == nat.E_LUT_KEY:
                raise KeyError((5, 5))                      # posecell_network.py:249
            if rc == nat.E_RADIUS:
                raise ValueError(nat.lib().prs_last_error().decode(errors="replace"))
            nat.check(rc, "prs_pc_update_host")
        res = e._res_np
        if res[0, 3]:
            e._raise_on_err(res[:, 3])
        self.max_pc = (int(res[0, 0]), int(res[0, 1]), int(res[0, 2]))
        e.max_pc = res[:, :3].astype(np.int64)
        self._max_valid = True
        return self.max_pc

    def path_integration(self, vtrans, vrot):
        """Shift the packet by the odometry without the attractor dynamics (posecell_network.py:252-314)."""
        vtrans, vrot = float(vtrans), float(vrot)
        self._precheck(vtrans, vrot)
        self._ens.path_integration(np.array([[vtrans, vrot]]))
        self._max_valid = False

    # north_star spellings
    get_pose = get_pc_max


PosecellNetwork = PoseCellNetwork
