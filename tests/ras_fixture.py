"""HEC-RAS 2D plan files for the reader tests, written from the stored golden arrays.

The HDF5 writer covers what HEC-RAS 6.x "classic" files use and io/hdf5_mini.py reads: superblock v0, object
header v1, symbol-table groups (v1 B-tree + SNOD + local heap), dataspace v1, integer / float / string / compound
datatypes, contiguous layout (message v3) and attribute messages v1.  The plan file holds the datasets io/ras.py
reads, at the paths the reference's reader uses (reference io/hdf.py).
"""
from __future__ import annotations

import struct
from pathlib import Path

import numpy as np
import pandas as pd

_UNDEF = 0xFFFFFFFFFFFFFFFF
_TS = "Results/Unsteady/Output/Output Blocks/Base Output/Unsteady Time Series"


def _pad8(b: bytes) -> bytes:
    return b + b"\0" * (-len(b) % 8)


def _datatype(dt: np.dtype) -> bytes:
    dt = np.dtype(dt)
    if dt.names:                                            # compound, version 1
        body = b""
        for name in dt.names:
            sub, off = dt.fields[name][:2]
            body += _pad8(name.encode() + b"\0") + struct.pack("<IB3xI4x16x", off, 0, 0) + _datatype(sub)
        n = len(dt.names)
        return struct.pack("<BBBBI", 0x16, n & 0xFF, n >> 8, 0, dt.itemsize) + body
    if dt.kind in "iu":
        return struct.pack("<BBBBIHH", 0x10, 0x08 if dt.kind == "i" else 0, 0, 0, dt.itemsize, 0, 8 * dt.itemsize)
    if dt.kind == "f":
        exp, mant, bias = {4: (8, 23, 127), 8: (11, 52, 1023)}[dt.itemsize]
        return struct.pack("<BBBBIHHBBBBI", 0x11, 0x20, 8 * dt.itemsize - 1, 0, dt.itemsize, 0, 8 * dt.itemsize, mant, exp, 0, mant, bias)
    if dt.kind == "S":
        return struct.pack("<BBBBI", 0x13, 0, 0, 0, dt.itemsize)
    raise TypeError(dt)


def _dataspace(shape) -> bytes:
    return struct.pack("<BBBB4x", 1, len(shape), 0, 0) + b"".join(struct.pack("<Q", d) for d in shape)


class _Writer:
    def __init__(self):
        self.buf = bytearray(96)                            # superblock + root symbol-table entry, filled in last

    def _put(self, data: bytes) -> int:
        self.buf += b"\0" * (-len(self.buf) % 8)
        addr = len(self.buf)
        self.buf += data
        return addr

    def _header(self, messages) -> int:
        body = b"".join(struct.pack("<HHB3x", t, len(_pad8(m)), 0) + _pad8(m) for t, m in messages)
        return self._put(struct.pack("<BBHII4x", 1, 0, len(messages), 1, len(body)) + body)

    def dataset(self, a: np.ndarray, attrs=None) -> int:
        a = np.ascontiguousarray(a)
        a = a.astype(a.dtype.newbyteorder("<")) if a.dtype.byteorder == ">" else a
        addr = self._put(a.tobytes())
        msgs = [(0x01, _dataspace(a.shape)), (0x03, _datatype(a.dtype)), (0x08, struct.pack("<BBQQ", 3, 1, addr, a.nbytes))]
        for name, v in (attrs or {}).items():
            v = np.ascontiguousarray(v)
            nm, dt, ds = name.encode() + b"\0", _datatype(v.dtype), _dataspace(v.shape)
            msgs.append((0x0C, struct.pack("<BBHHH", 1, 0, len(nm), len(dt), len(ds)) + _pad8(nm) + _pad8(dt) + _pad8(ds) + v.tobytes()))
        return self._header(msgs)

    def group(self, children: dict) -> int:
        """children: {name: dict (a subgroup) | (array, attrs)}; returns the group's object header address."""
        addrs = {name: self.group(c) if isinstance(c, dict) else self.dataset(*c) for name, c in children.items()}
        heap, offsets = bytearray(8), {}
        for name in sorted(addrs):
            offsets[name] = len(heap)
            heap += _pad8(name.encode() + b"\0")
        data = self._put(bytes(heap))
        heap_addr = self._put(b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap), _UNDEF, data))
        snod = self._put(b"SNOD" + struct.pack("<BBH", 1, 0, len(addrs)) +
                         b"".join(struct.pack("<QQI4x16x", offsets[nm], addrs[nm], 0) for nm in sorted(addrs)))
        last = offsets[max(addrs)] if addrs else 0
        btree = self._put(b"TREE" + struct.pack("<BBHQQ", 0, 0, 1, _UNDEF, _UNDEF) + struct.pack("<QQQ", 0, snod, last))
        self._btree_heap = (btree, heap_addr)
        return self._header([(0x11, struct.pack("<QQ", btree, heap_addr))])

    def write(self, path, tree: dict):
        root = self.group(tree)
        btree, heap = self._btree_heap
        sb = b"\x89HDF\r\n\x1a\n" + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, 64, 16, 0)
        sb += struct.pack("<QQQQ", 0, _UNDEF, len(self.buf), _UNDEF) + struct.pack("<QQI4xQQ", 0, root, 1, btree, heap)
        self.buf[:96] = sb
        Path(path).write_bytes(bytes(self.buf))


def write_plan(path, g: dict, extra_times: int = 0, area: str = "2D Area"):
    """A HEC-RAS 2D plan file holding the golden case g's mesh, hydrodynamics and boundary lines.  extra_times rows
    of NaN hydrodynamics are appended after the golden time range (what a datetime_range has to cut off).  Every
    boundary line gets one more external face that is not in its "Flow per Face" list (the reader must drop it)."""
    T, E = g["face_flow"].shape
    start = pd.Timestamp("2020-01-01")
    times = start + pd.to_timedelta(np.append(g["time_seconds"], g["time_seconds"][-1] + 60.0 * np.arange(1, extra_times + 1)), unit="s")
    stamps = np.array([t.strftime("%d%b%Y %H:%M:%S").upper() for t in times], dtype="S19")

    def series(a):
        return np.concatenate([a, np.full((extra_times, a.shape[1]), np.nan, a.dtype)])

    names = list(dict.fromkeys(str(x) for x in g["bc_names"]))
    faces = {nm: [int(f) for x, f in zip(g["bc_names"], g["bc_faces"]) if str(x) == nm] for nm in names}
    spare = [e for e in range(E) if e not in {f for fs in faces.values() for f in fs}]
    ext_dt = np.dtype([("BC Line ID", "<i4"), ("Face Index", "<i4"), ("Station Start", "<f4"), ("Station End", "<f4")])
    ext = np.array([(i, f, 0.0, 1.0) for i, nm in enumerate(names) for f in faces[nm] + [spare[i]]], dtype=ext_dt)
    att = np.array([(nm.encode(), b"2D Flow Area", area.encode()) for nm in names],
                   dtype=[("Name", "S32"), ("Type", "S16"), ("SA-2D", "S16")])
    flow_per_face = {f"{nm} - Flow per Face": (np.zeros((len(times), len(faces[nm])), "<f4"), {"Faces": np.array(faces[nm], "<i4")})
                     for nm in names}
    fc = np.stack([g["f1"], g["f2"]], axis=1).astype("<i4")
    xy = np.stack([g["face_x"], g["face_y"]], axis=1).astype("<f8")
    ts = {"Time Date Stamp": (stamps, None),
          "2D Flow Areas": {area: {"Face Velocity": (series(g["edge_velocity"]), None), "Face Flow": (series(g["face_flow"]), None),
                                   "Cell Volume": (series(g["volume"]), None)}},
          "Boundary Conditions": flow_per_face}
    tree = {"Geometry": {"2D Flow Areas": {"Attributes": (np.array([(area.encode(),)], dtype=[("Name", "S16")]), None),
                                           area: {"Faces Cell Indexes": (fc, None), "Cells Center Coordinate": (xy, None)}},
                         "Boundary Condition Lines": {"External Faces": (ext, None), "Attributes": (att, None)}}}
    node = tree
    for part in _TS.split("/")[:-1]:
        node = node.setdefault(part, {})
    node[_TS.split("/")[-1]] = ts
    _Writer().write(path, tree)
    return times[:T]
