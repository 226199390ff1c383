"""ctypes binding of the C ABI in include/cwr.h (libcwr_b200.so, hand-written sm_100a CUDA).

There is deliberately no CPU fallback: if the shared library is missing or no CUDA
device is present, construction raises.  Everything crosses the boundary as plain
pointers and sizes in the reference's cell / edge numbering.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional, Sequence

import numpy as np

from .kinetics import DEFAULT_MIN_DEPTH

_LIB_NAME = "libcwr_b200.so"
_lib = None

CWR_OK, CWR_EINVAL, CWR_ECUDA, CWR_ENOTCONVERGED, CWR_EBREAKDOWN, CWR_ENAN, CWR_ESINGULAR, CWR_ENOMEM = 0, -1, -2, -3, -4, -5, -6, -7
STATUS_NAMES = {0: "CWR_OK", -1: "CWR_EINVAL", -2: "CWR_ECUDA", -3: "CWR_ENOTCONVERGED", -4: "CWR_EBREAKDOWN",
                -5: "CWR_ENAN", -6: "CWR_ESINGULAR", -7: "CWR_ENOMEM"}


class CwrOptions(C.Structure):
    _fields_ = [("rtol", C.c_double), ("max_iter", C.c_int), ("reorder", C.c_int), ("keep_history", C.c_int),
                ("hydro_capacity", C.c_int), ("mass_flux", C.c_int), ("solver_path", C.c_int),
                ("solver", C.c_int), ("check_every", C.c_int), ("precond_steps", C.c_int),
                ("precond_precision", C.c_int), ("precond_sweep", C.c_int), ("precond_colors", C.c_int),
                ("dd_rank", C.c_int), ("dd_world", C.c_int), ("dd_halo_per_colour", C.c_int), ("precond_sync", C.c_int)]


class CwrStepInfo(C.Structure):
    _fields_ = [("iterations", C.c_int), ("restarts", C.c_int), ("status", C.c_int),
                ("max_relres", C.c_double), ("n_launches", C.c_int), ("sweeps", C.c_int)]


class CwrDdInfo(C.Structure):
    _fields_ = [("rank", C.c_int), ("world", C.c_int), ("rows_owned", C.c_int), ("rows_sent", C.c_int),
                ("neighbour_mask", C.c_int), ("n_colors", C.c_int), ("n_levels", C.c_int)]


IPC_HANDLE_BYTES = 64


class CwrMassTotals(C.Structure):
    _fields_ = [("vol_start", C.c_double), ("mass_start", C.c_double), ("vol_end", C.c_double), ("mass_end", C.c_double)]


class CwrError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


class SolverWarning(UserWarning):
    """The iterative solve ended without meeting rtol (results are stored, like scipy's
    MatrixRankWarning path in the reference, transport.py:249)."""


def library_path() -> Path:
    return Path(__file__).resolve().parent / _LIB_NAME


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("CWR_B200_LIB", library_path()))
    if not path.is_file():
        raise RuntimeError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  clearwater_riverine_b200 has no CPU fallback.")
    lib = C.CDLL(str(path))
    H = C.c_void_p
    dp, fp, ip = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_int32)
    sigs = {
        "cwr_default_options": ([C.POINTER(CwrOptions)], C.c_int),
        "cwr_create": ([C.POINTER(H), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, ip, C.c_double,
                        C.POINTER(CwrOptions)], C.c_int),
        "cwr_create_with_hint": ([C.POINTER(H), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, ip, C.c_double,
                                  C.POINTER(CwrOptions), fp], C.c_int),
        "cwr_destroy": ([H], None),
        "cwr_last_error": ([H], C.c_char_p),
        "cwr_set_hydro": ([H, C.c_int, C.c_int, fp, dp, fp, fp, dp], C.c_int),
        "cwr_set_geometry": ([H, dp, dp], C.c_int),
        "cwr_set_flow_hint": ([H, fp], C.c_int),
        "cwr_set_hydro_raw": ([H, C.c_int, C.c_int, fp, fp, fp, dp], C.c_int),
        "cwr_prefetch_hydro_raw": ([H, C.c_int, C.c_int, fp, fp, fp, dp], C.c_int),
        "cwr_set_inputs": ([H, C.c_int, dp], C.c_int),
        "cwr_set_state": ([H, C.c_int, C.c_int, dp], C.c_int),
        "cwr_set_state_all": ([H, C.c_int, dp, C.POINTER(C.c_uint8)], C.c_int),
        "cwr_step": ([H, C.c_int, C.POINTER(CwrStepInfo)], C.c_int),
        "cwr_run": ([H, C.c_int, C.c_int, C.POINTER(CwrStepInfo)], C.c_int),
        "cwr_get_state": ([H, C.c_int, C.c_int, dp], C.c_int),
        "cwr_get_state_all": ([H, C.c_int, dp], C.c_int),
        "cwr_get_state_rows": ([H, C.c_int, C.POINTER(C.c_void_p)], C.c_int),
        "cwr_fetch_async": ([H, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)], C.c_int),
        "cwr_fetch_wait": ([H], C.c_int),
        "cwr_host_register": ([C.c_void_p, C.c_size_t], C.c_int),
        "cwr_host_unregister": ([C.c_void_p], C.c_int),
        "cwr_get_mass_flux": ([H, C.c_int, C.c_int, dp, dp, dp], C.c_int),
        "cwr_mass_totals_at": ([H, C.c_int, C.c_int, C.c_int, C.POINTER(CwrMassTotals)], C.c_int),
        "cwr_get_flux_sums": ([H, C.c_int, dp, dp, dp], C.c_int),
        "cwr_get_volume_sums": ([H, dp, dp, dp], C.c_int),
        "cwr_set_kinetics": ([H, dp, dp, dp, C.c_int, C.c_double], C.c_int),
        "cwr_set_kinetics_sources": ([H, dp, dp, dp, dp, dp, ip], C.c_int),
        "cwr_set_kinetics_limits": ([H, C.c_int, ip, ip, ip, ip, dp], C.c_int),
        "cwr_set_kinetics_depth": ([H, dp, C.c_double, ip, ip, ip], C.c_int),
        "cwr_get_reaction_mass": ([H, C.c_int, dp], C.c_int),
        "cwr_get_lhs": ([H, C.POINTER(C.c_int64), ip, ip, dp], C.c_int),
        "cwr_get_rhs": ([H, C.c_int, dp], C.c_int),
        "cwr_get_permutation": ([H, ip], C.c_int),
        "cwr_strip_layout": ([C.c_int, C.c_int, C.c_int, ip, ip, C.c_int, fp, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                              ip, ip, ip, ip, C.POINTER(C.c_uint8), C.c_int], C.c_int),
        "cwr_get_options": ([H, C.POINTER(CwrOptions)], C.c_int),
        "cwr_dd_export": ([H, C.c_void_p], C.c_int),
        "cwr_dd_attach": ([H, C.c_void_p], C.c_int),
        "cwr_dd_layout": ([H, C.POINTER(CwrDdInfo), C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)], C.c_int),
        "cwr_stream": ([H, C.POINTER(C.c_void_p)], C.c_int),
        "cwr_order_cells": ([C.c_int, C.c_int, C.c_int, ip, ip, C.c_int, C.c_int, fp, C.c_int, ip, ip, C.POINTER(C.c_int),
                             C.POINTER(C.c_int), ip, ip], C.c_int),
        "cwr_counters": ([H, C.POINTER(C.c_int64), C.POINTER(C.c_int64)], C.c_int),
        "cwr_solver_stats": ([H, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int)], C.c_int),
        "cwr_time_spmm": ([H, C.c_int, dp, dp], C.c_int),
        "cwr_profile": ([H, C.c_int, dp, C.POINTER(C.c_int64)], C.c_int),
    }
    for name, (argtypes, restype) in sigs.items():
        fn = getattr(lib, name)      # AttributeError here = the .so does not export what cwr.h declares
        fn.argtypes, fn.restype = argtypes, restype
    lib._cwr_symbols = tuple(sigs)
    _lib = lib
    return lib


def _ptr(a: Optional[np.ndarray], ctype):
    return None if a is None else a.ctypes.data_as(C.POINTER(ctype))


def _arr(a, dtype, shape=None, name="array") -> np.ndarray:
    out = np.ascontiguousarray(a, dtype=dtype)
    if shape is not None and tuple(out.shape) != tuple(shape):
        raise ValueError(f"{name}: expected shape {tuple(shape)}, got {tuple(out.shape)}")
    return out


def pin_host_array(a: np.ndarray) -> bool:
    """Page-lock a numpy array in place (cudaHostRegister); False if that is not possible (no device...)."""
    try:
        return load_library().cwr_host_register(a.ctypes.data, a.nbytes) == CWR_OK
    except Exception:
        return False


def unpin_host_array(a: np.ndarray) -> None:
    try:
        load_library().cwr_host_unregister(a.ctypes.data)
    except Exception:
        pass


def bind_to_gpu_numa(device: int = 0) -> Optional[list]:
    """Restrict this process to the CPUs next to GPU `device` (NVML affinity), so that the host arrays it allocates and
    page-locks afterwards are first-touched on the GPU's NUMA node -- with one process per GPU, device->host copies into
    remote-node memory share the inter-socket link (round 1: 13 GB/s per GPU with 8 ranks).  Returns the CPU list, or None
    when NVML or the affinity call is unavailable (the process is left as it was).  Host-side only; optional."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(int(device))
        n_words = (os.cpu_count() + 63) // 64
        mask = nv.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = [w * 64 + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return allowed
    except Exception:
        return None


def order_cells(f1, f2, n_face: int, reorder: bool = True, n_colors: int = 0, flow_hint=None, n_parts: int = 1):
    """Host-only: the ordering the library builds (cwr_order_cells).  Returns (new_of_old, color_ptr, n_levels) for
    n_parts == 1, with color_ptr of shape (n_colors+1,); for n_parts > 1 returns
    (new_of_old, color_ptr (n_parts, n_colors+1), n_levels, part_ptr (n_parts+1,), n_send (n_parts,))."""
    lib = load_library()
    f1 = _arr(f1, np.int32); f2 = _arr(f2, np.int32, f1.shape, "f2")
    n = int(f1.max()) + 1
    hint = None if flow_hint is None else _arr(flow_hint, np.float32, f1.shape, "flow_hint")
    new_of_old = np.empty(n, np.int32); cptr = np.zeros(8 * 65, np.int32)
    part_ptr = np.zeros(9, np.int32); n_send = np.zeros(8, np.int32)
    nc, nl = C.c_int(), C.c_int()
    rc = lib.cwr_order_cells(n, int(n_face), len(f1), _ptr(f1, C.c_int32), _ptr(f2, C.c_int32), int(reorder), int(n_colors),
                             _ptr(hint, C.c_float), int(n_parts), _ptr(new_of_old, C.c_int32), _ptr(cptr, C.c_int32),
                             C.byref(nc), C.byref(nl), _ptr(part_ptr, C.c_int32), _ptr(n_send, C.c_int32))
    if rc != CWR_OK:
        raise CwrError(rc, lib.cwr_last_error(None).decode())
    if nc.value == 0:
        colours = np.array([0, n], np.int32) if n_parts == 1 else part_ptr[: n_parts + 1].copy()
    else:
        colours = cptr[: n_parts * (nc.value + 1)].reshape(n_parts, nc.value + 1).copy()
    if n_parts == 1:
        return new_of_old, (colours[0] if nc.value else colours), nl.value
    return new_of_old, colours, nl.value, part_ptr[: n_parts + 1].copy(), n_send[:n_parts].copy()


def strip_layout(f1, f2, n_face: int, n_colors: int, flow_hint, n_strips: int, n_parts: int = 1, strip_cap: int = 0):
    """Host-only: the strips of the neighbour-synchronised sweep kernel (cwr_strip_layout) as a dict of numpy arrays."""
    lib = load_library()
    f1 = _arr(f1, np.int32); f2 = _arr(f2, np.int32, f1.shape, "f2")
    n = int(f1.max()) + 1
    hint = None if flow_hint is None else _arr(flow_hint, np.float32, f1.shape, "flow_hint")
    nc, nb = C.c_int(), C.c_int()
    args = (n, int(n_face), len(f1), _ptr(f1, C.c_int32), _ptr(f2, C.c_int32), int(n_colors), _ptr(hint, C.c_float),
            int(n_parts), int(n_strips), C.byref(nc), C.byref(nb))
    rc = lib.cwr_strip_layout(*args, None, None, None, None, None, int(strip_cap))
    if rc != CWR_OK:
        raise CwrError(rc, lib.cwr_last_error(None).decode())
    NS = n_parts * n_strips
    out = {"new_of_old": np.empty(n, np.int32), "strip_cptr": np.empty((NS, nc.value + 1), np.int32),
           "strip_nptr": np.empty(NS + 1, np.int32), "strip_nbr": np.empty(max(1, nb.value), np.int32), "color_of": np.empty(n, np.uint8)}
    rc = lib.cwr_strip_layout(*args, _ptr(out["new_of_old"], C.c_int32), _ptr(out["strip_cptr"], C.c_int32),
                              _ptr(out["strip_nptr"], C.c_int32), _ptr(out["strip_nbr"], C.c_int32), _ptr(out["color_of"], C.c_uint8),
                              int(strip_cap))
    if rc != CWR_OK:
        raise CwrError(rc, lib.cwr_last_error(None).decode())
    out["strip_nbr"] = out["strip_nbr"][: nb.value]
    out.update(n_colors=nc.value, n_strips=n_strips, n_parts=n_parts)
    return out


class TransportBackend:
    """One model on one GPU: fixed topology, K constituents, T time slices."""

    def __init__(self, f1, f2, n_face: int, n_time: int, n_constituents: int, diffusion_coefficient: float,
                 device: int = 0, flow_hint=None, **options):
        self._lib = load_library()
        self._h = C.c_void_p()
        f1 = _arr(f1, np.int32); f2 = _arr(f2, np.int32, f1.shape, "f2")
        self.n_edge = int(f1.shape[0]); self.n_face = int(n_face); self.n_time = int(n_time)
        self.n_real = int(f1.max()) + 1            # reference: nreal = max(edges_face1)  (io/hdf.py:268-269)
        self.K = int(n_constituents)
        self.diffusion_coefficient = float(diffusion_coefficient)
        opt = CwrOptions()
        self._lib.cwr_default_options(C.byref(opt))
        for key, val in options.items():
            if not hasattr(opt, key):
                raise TypeError(f"unknown option {key!r}")
            setattr(opt, key, val)
        self.options = opt
        hint = None if flow_hint is None else _arr(flow_hint, np.float32, (self.n_edge,), "flow_hint")
        rc = self._lib.cwr_create_with_hint(C.byref(self._h), device, self.n_real, self.n_face, self.n_edge, self.n_time,
                                            self.K, _ptr(f1, C.c_int32), _ptr(f2, C.c_int32), self.diffusion_coefficient,
                                            C.byref(opt), _ptr(hint, C.c_float))
        if rc != CWR_OK:
            msg = self._lib.cwr_last_error(None).decode()
            self._h = C.c_void_p()
            raise CwrError(rc, msg)
        self._lib.cwr_get_options(self._h, C.byref(self.options))     # autos resolved
        self.last_info = CwrStepInfo()

    # -- plumbing ------------------------------------------------------------------------------
    def _check(self, rc: int, allow_solver_status: bool = False) -> int:
        if rc == CWR_OK:
            return rc
        if allow_solver_status and rc in (CWR_ENOTCONVERGED, CWR_EBREAKDOWN, CWR_ENAN, CWR_ESINGULAR):
            return rc
        raise CwrError(rc, self._lib.cwr_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.cwr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- inputs ----------------------------------------------------------------------------------
    def set_hydro(self, t0: int, adv, cdiff, vel, vol, dt):
        adv = _arr(adv, np.float32); nt = adv.shape[0] if adv.ndim == 2 else 1
        adv = adv.reshape(nt, self.n_edge)
        cdiff = _arr(cdiff, np.float64).reshape(nt, self.n_edge)
        vel = _arr(vel, np.float32).reshape(nt, self.n_edge)
        vol = _arr(vol, np.float32).reshape(nt, self.n_face)
        dt = _arr(dt, np.float64).reshape(nt)
        self._check(self._lib.cwr_set_hydro(self._h, t0, nt, _ptr(adv, C.c_float), _ptr(cdiff, C.c_double),
                                            _ptr(vel, C.c_float), _ptr(vol, C.c_float), _ptr(dt, C.c_double)))

    def set_flow_hint(self, face_flow):
        q = _arr(face_flow, np.float32, (self.n_edge,), "face_flow")
        self._check(self._lib.cwr_set_flow_hint(self._h, _ptr(q, C.c_float)))

    def set_geometry(self, face_x, face_y):
        fx = _arr(face_x, np.float64, (self.n_face,), "face_x"); fy = _arr(face_y, np.float64, (self.n_face,), "face_y")
        self._check(self._lib.cwr_set_geometry(self._h, _ptr(fx, C.c_double), _ptr(fy, C.c_double)))

    def set_hydro_raw(self, t0: int, face_flow, edge_velocity, volume, dt):
        q = _arr(face_flow, np.float32); nt = q.shape[0] if q.ndim == 2 else 1
        q = q.reshape(nt, self.n_edge)
        u = _arr(edge_velocity, np.float32).reshape(nt, self.n_edge)
        v = _arr(volume, np.float32).reshape(nt, self.n_face)
        dt = _arr(dt, np.float64).reshape(nt)
        self._check(self._lib.cwr_set_hydro_raw(self._h, t0, nt, _ptr(q, C.c_float), _ptr(u, C.c_float),
                                                _ptr(v, C.c_float), _ptr(dt, C.c_double)))

    def prefetch_hydro_raw(self, t0: int, face_flow, edge_velocity, volume, dt):
        """set_hydro_raw on the upload stream (overlaps the next device->host copy); the arrays must be float32 /
        float64 contiguous already (no conversion copy is kept alive here) and stay valid until the next step."""
        q, u, v, d = face_flow, edge_velocity, volume, dt
        for a, ty in ((q, np.float32), (u, np.float32), (v, np.float32), (d, np.float64)):
            assert a.dtype == ty and a.flags.c_contiguous
        nt = q.shape[0] if q.ndim == 2 else 1
        self._check(self._lib.cwr_prefetch_hydro_raw(self._h, t0, nt, _ptr(q, C.c_float), _ptr(u, C.c_float),
                                                     _ptr(v, C.c_float), _ptr(d, C.c_double)))

    def set_inputs(self, k: int, input_array):
        a = _arr(input_array, np.float64, (self.n_time, self.n_face), "input_array")
        self._check(self._lib.cwr_set_inputs(self._h, k, _ptr(a, C.c_double)))

    def set_state(self, k: int, t: int, c):
        a = _arr(np.asarray(c)[: self.n_real], np.float64, (self.n_real,), "c")
        self._check(self._lib.cwr_set_state(self._h, k, t, _ptr(a, C.c_double)))

    def set_state_all(self, t: int, c, mask: Optional[Sequence[bool]] = None):
        a = _arr(c, np.float64, (self.K, self.n_real), "c")
        m = None if mask is None else _arr(mask, np.uint8, (self.K,), "mask")
        self._check(self._lib.cwr_set_state_all(self._h, t, _ptr(a, C.c_double), _ptr(m, C.c_uint8)))

    # -- stepping ----------------------------------------------------------------------------------
    def step(self, t: int) -> CwrStepInfo:
        info = CwrStepInfo()
        self._check(self._lib.cwr_step(self._h, t, C.byref(info)), allow_solver_status=True)
        self.last_info = info
        return info

    def run(self, t_begin: int, t_end: int) -> CwrStepInfo:
        info = CwrStepInfo()
        self._check(self._lib.cwr_run(self._h, t_begin, t_end, C.byref(info)), allow_solver_status=True)
        self.last_info = info
        return info

    # -- outputs -----------------------------------------------------------------------------------
    def get_state(self, k: int, t: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        out = np.empty(self.n_face) if out is None else out
        assert out.dtype == np.float64 and out.flags.c_contiguous and out.shape == (self.n_face,)
        self._check(self._lib.cwr_get_state(self._h, k, t, _ptr(out, C.c_double)))
        return out

    def get_state_all(self, t: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        out = np.empty((self.K, self.n_real)) if out is None else out
        assert out.dtype == np.float64 and out.flags.c_contiguous and out.shape == (self.K, self.n_real)
        self._check(self._lib.cwr_get_state_all(self._h, t, _ptr(out, C.c_double)))
        return out

    def get_state_rows(self, t: int, rows: Sequence[Optional[np.ndarray]]):
        """c[t] of constituent k (real cells) straight into rows[k][:n] -- e.g. row t of each constituent's (T,F) array."""
        ptrs = (C.c_void_p * self.K)()
        for k, r in enumerate(rows):
            if r is None:
                continue
            assert r.dtype == np.float64 and r.flags.c_contiguous and r.shape[0] >= self.n_real
            ptrs[k] = r.ctypes.data
        self._check(self._lib.cwr_get_state_rows(self._h, t, ptrs))

    def _row_pointers(self, rows, length):
        if rows is None:
            return None
        ptrs = (C.c_void_p * self.K)()
        for k, r in enumerate(rows):
            if r is None:
                continue
            assert r.dtype == np.float64 and r.flags.c_contiguous and r.shape[0] >= length
            ptrs[k] = r.ctypes.data
        return ptrs

    def fetch_async(self, t: int, state_rows=None, adv_rows=None, diff_rows=None, tot_rows=None):
        """c[t] into state_rows[k][:n] and the mass fluxes of step t - 1 into *_rows[k][:E], copied on a separate
        stream while the next step runs; call fetch_wait() before reading them."""
        self._check(self._lib.cwr_fetch_async(self._h, t, self._row_pointers(state_rows, self.n_real),
                                              self._row_pointers(adv_rows, self.n_edge), self._row_pointers(diff_rows, self.n_edge),
                                              self._row_pointers(tot_rows, self.n_edge)))

    def fetch_wait(self):
        self._check(self._lib.cwr_fetch_wait(self._h))

    def get_mass_flux(self, k: int, t: int, advection=None, diffusion=None, total=None):
        outs = []
        for a in (advection, diffusion, total):
            if a is None:
                a = np.empty(self.n_edge)
            assert a.dtype == np.float64 and a.flags.c_contiguous and a.shape == (self.n_edge,)
            outs.append(a)
        self._check(self._lib.cwr_get_mass_flux(self._h, k, t, *[_ptr(a, C.c_double) for a in outs]))
        return tuple(outs)

    def flux_sums(self, k: int):
        outs = [np.empty(self.n_edge) for _ in range(3)]
        self._check(self._lib.cwr_get_flux_sums(self._h, k, *[_ptr(a, C.c_double) for a in outs]))
        return tuple(outs)

    def volume_sums(self):
        outs = [np.empty(self.n_edge) for _ in range(3)]
        self._check(self._lib.cwr_get_volume_sums(self._h, *[_ptr(a, C.c_double) for a in outs]))
        return tuple(outs)

    def mass_totals(self, k: int, t_start: int, t_end: int) -> CwrMassTotals:
        m = CwrMassTotals()
        self._check(self._lib.cwr_mass_totals_at(self._h, k, t_start, t_end, C.byref(m)))
        return m

    # -- kinetics --------------------------------------------------------------------------------
    def set_kinetics(self, decay_per_day=None, theta=None, yields=None, temperature_k: int = -1, temperature_c: float = 20.0):
        """First-order decay / transformations applied on the device in every later step (cwr_set_kinetics):
        decay_per_day (K,) or None = off; theta (K,) or None = all 1; yields (K, K), yields[j, k] = mass of j formed per
        mass of k decayed, or None; temperature_k = temperature constituent or -1 for the constant temperature_c (deg C).
        An invalid set raises ValueError; any call clears set_kinetics_sources, set_kinetics_limits and set_kinetics_depth.
        kinetics.compile_kinetics builds the arrays from a by-name spec."""
        if decay_per_day is None:
            self._check(self._lib.cwr_set_kinetics(self._h, None, None, None, -1, 20.0))
            return
        d = _arr(decay_per_day, np.float64, (self.K,), "decay_per_day")
        th = None if theta is None else _arr(theta, np.float64, (self.K,), "theta")
        y = None if yields is None else _arr(yields, np.float64, (self.K, self.K), "yields")
        rc = self._lib.cwr_set_kinetics(self._h, _ptr(d, C.c_double), _ptr(th, C.c_double), _ptr(y, C.c_double),
                                        int(temperature_k), float(temperature_c))
        if rc == CWR_EINVAL:
            raise ValueError(self._lib.cwr_last_error(self._h).decode())
        self._check(rc)

    def set_kinetics_sources(self, source_per_day=None, source_theta=None, exchange_per_day=None, exchange_theta=None,
                             equilibrium=None, equilibrium_kind=None):
        """Zero-order sources and relaxation toward an equilibrium, applied after the first-order chain of the kinetics set
        last (cwr_set_kinetics_sources): dc/dt = s + r (ceq - c) per column, solved exactly over each step.
        source_per_day (K,) or None; exchange_per_day (K,) 1/day or None (both None: sources off); a theta (K,) or None =
        all 1; equilibrium (K,) the constant targets; equilibrium_kind (K,) 0 = constant, 1 = oxygen saturation at T, or
        None = all 0.  set_kinetics clears them; any call clears set_kinetics_limits and set_kinetics_depth.  An invalid
        set raises ValueError."""
        K = (self.K,)
        f = lambda a, name: None if a is None else _arr(a, np.float64, K, name)
        arrs = [f(source_per_day, "source_per_day"), f(source_theta, "source_theta"), f(exchange_per_day, "exchange_per_day"),
                f(exchange_theta, "exchange_theta"), f(equilibrium, "equilibrium")]
        kind = None if equilibrium_kind is None else _arr(equilibrium_kind, np.int32, K, "equilibrium_kind")
        rc = self._lib.cwr_set_kinetics_sources(self._h, *[_ptr(a, C.c_double) for a in arrs], _ptr(kind, C.c_int32))
        if rc == CWR_EINVAL:
            raise ValueError(self._lib.cwr_last_error(self._h).decode())
        self._check(rc)

    def set_kinetics_limits(self, process=None, column=None, factor_column=None, factor_kind=None, half_saturation=None):
        """Monod limitation and inhibition of the kinetics and sources set last (cwr_set_kinetics_limits); (n,) arrays:
        factor i scales process[i] (0 = the decay of column[i], 1 = its source) by c+/(K + c+) (factor_kind 0) or
        K/(K + c+) (1) of constituent factor_column[i], K = half_saturation[i], c+ = max(c, 0).  process None = limits
        off.  set_kinetics and set_kinetics_sources clear them.  An invalid set raises ValueError."""
        if process is None:
            self._check(self._lib.cwr_set_kinetics_limits(self._h, 0, None, None, None, None, None))
            return
        pr = _arr(process, np.int32).reshape(-1)
        n = (pr.shape[0],)
        ints = [pr] + [_arr(a, np.int32, n, name) for a, name in ((column, "column"), (factor_column, "factor_column"),
                                                                  (factor_kind, "factor_kind"))]
        hs = _arr(half_saturation, np.float64, n, "half_saturation")
        rc = self._lib.cwr_set_kinetics_limits(self._h, n[0], *[_ptr(a, C.c_int32) for a in ints], _ptr(hs, C.c_double))
        if rc == CWR_EINVAL:
            raise ValueError(self._lib.cwr_last_error(self._h).decode())
        self._check(rc)

    def set_kinetics_depth(self, cell_area=None, min_depth: float = DEFAULT_MIN_DEPTH, decay_per_depth=None, source_per_depth=None,
                           exchange_per_depth=None):
        """Depth-scaled processes of the kinetics and sources set last (cwr_set_kinetics_depth): a flag (K,) of 1 divides
        that process's rate of column k by the cell's depth h = max(V[t] / cell_area, min_depth), making the decay a
        settling velocity, the source an areal flux and the exchange a transfer velocity (mesh length units).  cell_area
        (F,) plan areas; every flag None or 0 = depth off.  set_kinetics and set_kinetics_sources clear it;
        set_kinetics_limits does not.  An invalid set raises ValueError."""
        K = (self.K,)
        flags = [None if a is None else _arr(a, np.int32, K, name) for a, name in
                 ((decay_per_depth, "decay_per_depth"), (source_per_depth, "source_per_depth"),
                  (exchange_per_depth, "exchange_per_depth"))]
        area = None if cell_area is None else _arr(cell_area, np.float64, (self.n_face,), "cell_area")
        rc = self._lib.cwr_set_kinetics_depth(self._h, _ptr(area, C.c_double), float(min_depth),
                                              *[_ptr(a, C.c_int32) for a in flags])
        if rc == CWR_EINVAL:
            raise ValueError(self._lib.cwr_last_error(self._h).decode())
        self._check(rc)

    def reaction_mass(self, k: int) -> float:
        """Sum over the steps taken of sum_i V[t]_i (c~'_ik - c~_ik): the mass the reactions added to constituent k."""
        out = C.c_double()
        self._check(self._lib.cwr_get_reaction_mass(self._h, k, C.byref(out)))
        return out.value

    # -- domain decomposition (one TransportBackend per GPU/process; see domain.py) -----------------------
    def dd_export(self) -> bytes:
        buf = C.create_string_buffer(IPC_HANDLE_BYTES)
        self._check(self._lib.cwr_dd_export(self._h, buf))
        return buf.raw

    def dd_attach(self, handles: bytes):
        buf = C.create_string_buffer(handles, len(handles))
        self._check(self._lib.cwr_dd_attach(self._h, buf))

    def dd_layout(self):
        info = CwrDdInfo()
        cells = np.zeros(self.n_real, np.uint8); edges = np.zeros(self.n_edge, np.uint8)
        self._check(self._lib.cwr_dd_layout(self._h, C.byref(info), _ptr(cells, C.c_uint8), _ptr(edges, C.c_uint8)))
        return info, cells.astype(bool), edges.astype(bool)

    # -- introspection ---------------------------------------------------------------------------------
    def get_lhs(self):
        """scipy CSR of A(t) as last assembled, reference numbering."""
        from scipy.sparse import csr_matrix
        nnz = C.c_int64()
        self._check(self._lib.cwr_get_lhs(self._h, C.byref(nnz), None, None, None))
        indptr = np.empty(self.n_real + 1, np.int32); indices = np.empty(nnz.value, np.int32); data = np.empty(nnz.value)
        self._check(self._lib.cwr_get_lhs(self._h, C.byref(nnz), _ptr(indptr, C.c_int32), _ptr(indices, C.c_int32),
                                          _ptr(data, C.c_double)))
        return csr_matrix((data, indices, indptr), shape=(self.n_real, self.n_real))

    def get_rhs(self, k: int) -> np.ndarray:
        b = np.empty(self.n_real)
        self._check(self._lib.cwr_get_rhs(self._h, k, _ptr(b, C.c_double)))
        return b

    def permutation(self) -> np.ndarray:
        p = np.empty(self.n_real, np.int32)
        self._check(self._lib.cwr_get_permutation(self._h, _ptr(p, C.c_int32)))
        return p

    def counters(self):
        a, b = C.c_int64(), C.c_int64()
        self._check(self._lib.cwr_counters(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def solver_stats(self):
        """(Gauss-Seidel sweeps so far, solves that fell back to BiCGSTAB, strips of the sweep kernel, max strip neighbours)."""
        a, b, c, d = C.c_int64(), C.c_int64(), C.c_int(), C.c_int()
        self._check(self._lib.cwr_solver_stats(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value

    def stream(self) -> int:
        s = C.c_void_p()
        self._check(self._lib.cwr_stream(self._h, C.byref(s)))
        return s.value or 0

    PROFILE_FAMILIES = ("assemble", "rhs", "spmm_init", "spmm_v", "update_s", "spmm_t", "update_xrp", "mass_flux", "precond", "solve_small", "dc_update")

    def profile(self, enable: int = -1):
        """enable = 1/0 switches per-kernel-family event timing on/off; returns {family: (ms, launches)}."""
        ms = np.zeros(len(self.PROFILE_FAMILIES)); cnt = np.zeros(len(self.PROFILE_FAMILIES), np.int64)
        self._check(self._lib.cwr_profile(self._h, enable, _ptr(ms, C.c_double), cnt.ctypes.data_as(C.POINTER(C.c_int64))))
        return {f: (float(ms[i]), int(cnt[i])) for i, f in enumerate(self.PROFILE_FAMILIES)}

    def time_spmm(self, reps: int = 20):
        ms, nbytes = C.c_double(), C.c_double()
        self._check(self._lib.cwr_time_spmm(self._h, reps, C.byref(ms), C.byref(nbytes)))
        return ms.value, nbytes.value
