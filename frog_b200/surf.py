"""ctypes face of libfrogsurf.so (include/frogsurf.h): the SURF3D producer on one B200.

Mirrors how surf3d.cxx drives vtk3DSURF (surf3d.cxx:258-328): set the volume, detect, keep the
strongest `number_of_points`, describe.  Volumes are numpy arrays indexed [z, y, x].
There is no CPU path: `Producer()` raises FrogSurfError when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build

PUBLIC_SYMBOLS = [
    "fs_device_count", "fs_create", "fs_destroy", "fs_last_error", "fs_version", "fs_set_volume", "fs_detect",
    "fs_select", "fs_set_points", "fs_describe", "fs_num_points", "fs_get_points", "fs_get_points_as_read", "fs_get_stats",
    "fs_get_cast_volume", "fs_get_integral", "fs_num_layers", "fs_get_layer",
]

VOXEL_TYPES = {np.dtype(np.uint8): 0, np.dtype(np.int16): 1, np.dtype(np.uint16): 2, np.dtype(np.int32): 3,
               np.dtype(np.float32): 4, np.dtype(np.int8): 5, np.dtype(np.uint32): 6, np.dtype(np.float64): 7}

POINT_DTYPE = np.dtype([("x", np.float32), ("y", np.float32), ("z", np.float32), ("scale", np.float32),
                        ("response", np.float32), ("laplacian", np.int32)])


class Stats(C.Structure):
    _fields_ = [("ms_integral", C.c_float), ("ms_response_map", C.c_float), ("ms_extrema", C.c_float),
                ("ms_describe", C.c_float), ("n_layers", C.c_uint32), ("n_candidates", C.c_uint32),
                ("n_points", C.c_uint32), ("n_clamped", C.c_uint32), ("response_voxels", C.c_uint64)]


class FrogSurfError(RuntimeError):
    pass


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(build.SURF_LIB):
        raise FrogSurfError(f"{build.SURF_LIB} is not built (python -m frog_b200.build); there is no fallback")
    L = C.CDLL(build.SURF_LIB)
    L.fs_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.fs_destroy.argtypes = [C.c_void_p]
    L.fs_last_error.restype = C.c_char_p
    L.fs_last_error.argtypes = [C.c_void_p]
    L.fs_version.restype = C.c_char_p
    L.fs_set_volume.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    L.fs_detect.argtypes = [C.c_void_p, C.c_float, C.POINTER(C.c_uint32)]
    L.fs_select.argtypes = [C.c_void_p, C.c_int]
    L.fs_set_points.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    L.fs_describe.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.fs_num_points.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.fs_get_points.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.fs_get_points_as_read.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.fs_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.fs_get_cast_volume.argtypes = [C.c_void_p, C.c_void_p]
    L.fs_get_integral.argtypes = [C.c_void_p, C.c_void_p]
    L.fs_num_layers.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    L.fs_get_layer.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    # host-side pieces (include/frogsurf_debug.h)
    L.fs_debug_expf.restype = C.c_float
    L.fs_debug_expf.argtypes = [C.c_float]
    L.fs_debug_expf_many.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.fs_debug_solve_offsets.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.fs_debug_layers.restype = C.c_int
    L.fs_debug_layers.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.fs_debug_keep_cast_volume.argtypes = [C.c_void_p, C.c_int]
    L.fs_debug_set_option.argtypes = [C.c_char_p, C.c_int]
    L.fs_debug_sort_keys.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    L.fs_debug_as_read.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    L.fs_debug_select.restype = C.c_uint32
    L.fs_debug_select.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_void_p]
    _lib = L
    return L


class Producer:
    def __init__(self, device: int = 0):
        self._L = load()
        h = C.c_void_p()
        rc = self._L.fs_create(device, C.byref(h))
        if rc != 0:
            raise FrogSurfError(self._L.fs_last_error(None).decode())
        self._h = h
        self.shape = None

    def close(self):
        if self._h:
            self._L.fs_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def keep_cast_volume(self, on: bool = True):
        self._L.fs_debug_keep_cast_volume(self._h, int(on))

    def _check(self, rc):
        if rc != 0:
            raise FrogSurfError(f"{rc}: {self._L.fs_last_error(self._h).decode()}")

    def set_volume(self, volume: np.ndarray):
        v = np.ascontiguousarray(volume)
        self.shape = v.shape
        self._check(self._L.fs_set_volume(self._h, v.ctypes.data, VOXEL_TYPES[v.dtype], v.shape[2], v.shape[1], v.shape[0]))

    def set_volume_device(self, ptr: int, dtype, shape):
        self.shape = tuple(shape)
        self._check(self._L.fs_set_volume(self._h, C.c_void_p(ptr), VOXEL_TYPES[np.dtype(dtype)], shape[2], shape[1], shape[0]))

    def detect(self, threshold: float = 0.0) -> int:
        n = C.c_uint32()
        self._check(self._L.fs_detect(self._h, threshold, C.byref(n)))
        return n.value

    def select(self, number_of_points: int):
        self._check(self._L.fs_select(self._h, number_of_points))

    def set_points(self, xyzs: np.ndarray):
        a = np.ascontiguousarray(xyzs, np.float32).reshape(-1, 4)
        self._check(self._L.fs_set_points(self._h, a.ctypes.data, a.shape[0]))

    def describe(self, descriptor_type: int = 0, radius: int = 5, normalize: bool = True):
        self._check(self._L.fs_describe(self._h, descriptor_type, radius, int(normalize)))

    def points(self, with_descriptors: bool = True):
        n, d = C.c_uint32(), C.c_uint32()
        self._check(self._L.fs_num_points(self._h, C.byref(n), C.byref(d)))
        pts = np.zeros(n.value, POINT_DTYPE)
        desc = np.zeros((n.value, d.value), np.float32) if with_descriptors and d.value else None
        self._check(self._L.fs_get_points(self._h, pts.ctypes.data, desc.ctypes.data if desc is not None and n.value else None))
        return pts, desc

    def points_as_read(self, precision: int = -1, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0)):
        """(head [n, 6], desc [n, d]) float32: the keypoints exactly as the .csv.gz reader returns them from the file
        surf3d writes for a volume of this spacing / origin at -precision `precision` (converted on the device)."""
        n, d = C.c_uint32(), C.c_uint32()
        self._check(self._L.fs_num_points(self._h, C.byref(n), C.byref(d)))
        head = np.zeros((n.value, 6), np.float32)
        desc = np.zeros((n.value, d.value), np.float32)
        sp = np.asarray(spacing, np.float64)
        org = np.asarray(origin, np.float64)
        self._check(self._L.fs_get_points_as_read(self._h, precision, sp.ctypes.data, org.ctypes.data, head.ctypes.data,
                                                  desc.ctypes.data))
        return head, desc

    def stats(self) -> dict:
        s = Stats()
        self._check(self._L.fs_get_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def cast_volume(self) -> np.ndarray:
        out = np.zeros(self.shape, np.int32)
        self._check(self._L.fs_get_cast_volume(self._h, out.ctypes.data))
        return out

    def integral(self) -> np.ndarray:
        out = np.zeros(self.shape, np.uint64)
        self._check(self._L.fs_get_integral(self._h, out.ctypes.data))
        return out

    def layers(self):
        n = C.c_uint32()
        self._check(self._L.fs_num_layers(self._h, C.byref(n)))
        out = []
        for i in range(n.value):
            info = (C.c_int32 * 5)()
            self._check(self._L.fs_get_layer(self._h, i, info, None, None, None))
            w, h, d, step, filt = list(info)
            r = np.zeros((d, h, w), np.float32)
            lp = np.zeros((d, h, w), np.uint8)
            ib = np.zeros((d, h, w), np.uint8)
            self._check(self._L.fs_get_layer(self._h, i, info, r.ctypes.data, lp.ctypes.data, ib.ctypes.data))
            out.append(dict(width=w, height=h, depth=d, step=step, filter=filt, responses=r, laplacian=lp, isblob=ib))
        return out


def run(volume: np.ndarray, threshold=0.0, number_of_points=-1, descriptor_type=0, radius=5, normalize=True, device=0):
    """surf3d's pipeline on one volume: (points, descriptors, stats)."""
    p = Producer(device)
    try:
        p.set_volume(volume)
        p.detect(threshold)
        p.select(number_of_points)
        p.describe(descriptor_type, radius, normalize)
        pts, desc = p.points()
        return pts, desc, p.stats()
    finally:
        p.close()


# ---- host-side pieces (CPU tests) ------------------------------------------------------------------
def debug_set_option(name: str, value: int) -> None:
    if load().fs_debug_set_option(name.encode(), value) != 0:
        raise FrogSurfError(f"unknown option {name}")


def debug_sort_keys(keys: np.ndarray) -> np.ndarray:
    k = np.ascontiguousarray(keys, np.uint64)
    order = np.zeros(max(k.size, 1), np.uint32)
    load().fs_debug_sort_keys(k.ctypes.data, k.size, order.ctypes.data)
    return order[:k.size]


def debug_expf(x: np.ndarray) -> np.ndarray:
    L = load()
    x = np.ascontiguousarray(x, np.float32)
    y = np.zeros_like(x)
    L.fs_debug_expf_many(x.ctypes.data, y.ctypes.data, x.size)
    return y


def debug_solve_offsets(dD, H10) -> np.ndarray:
    L = load()
    a = np.ascontiguousarray(dD, np.float64)
    h = np.ascontiguousarray(H10, np.float64)
    x = np.zeros(4)
    L.fs_debug_solve_offsets(a.ctypes.data, h.ctypes.data, x.ctypes.data)
    return x


def debug_layers(nx, ny, nz) -> np.ndarray:
    L = load()
    out = np.zeros((16, 6), np.int32)
    n = L.fs_debug_layers(nx, ny, nz, out.ctypes.data, 16)
    return out[:n]


def debug_as_read(values: np.ndarray, precision: int) -> np.ndarray:
    """fs_get_points_as_read's conversion of float64 values on device 0 (float32 results; needs a GPU)."""
    v = np.ascontiguousarray(values, np.float64)
    out = np.zeros(v.shape, np.float32)
    rc = load().fs_debug_as_read(v.ctypes.data, v.size, precision, out.ctypes.data)
    if rc != 0:
        raise FrogSurfError(f"fs_debug_as_read: status {rc}")
    return out


def debug_select(response: np.ndarray, number_of_points: int) -> np.ndarray:
    L = load()
    r = np.ascontiguousarray(response, np.float32)
    order = np.zeros(max(r.size, 1), np.uint32)
    n = L.fs_debug_select(r.ctypes.data, r.size, number_of_points, order.ctypes.data)
    return order[:n]


# ---- host I/O of bin/surf3d (frog_b200/libfsio.so, no CUDA) ---------------------------------------------
_fsio = None


def _io():
    global _fsio
    if _fsio is None:
        if not os.path.exists(build.FSIO):
            raise FrogSurfError(f"{build.FSIO} is not built (python -m frog_b200.build)")
        L = C.CDLL(build.FSIO)
        L.fsio_write_points.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.c_size_t, C.c_void_p, C.c_void_p]
        L.fsio_read_metaimage.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_size_t, C.c_void_p, C.c_void_p]
        L.fsio_last_error.restype = C.c_char_p
        L.fsio_last_error.argtypes = []
        L.fsio_write_bounds_json.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.fsio_debug_as_read.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_void_p]
        L.fsio_read_points.restype = C.c_long
        L.fsio_read_points.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
        _fsio = L
    return _fsio


def write_points(path: str, fmt: str, pts: np.ndarray, desc: np.ndarray, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0),
                 gz_opts=None, precision=-1) -> None:
    """vtk3DSURF::WritePointsCSV / CSVGZ / Binary (vtk3DSURF.cxx:405-525) on voxel-unit keypoints."""
    pts = np.ascontiguousarray(pts, POINT_DTYPE)
    desc = np.ascontiguousarray(desc, np.float32).reshape(len(pts), -1)
    sp = np.asarray(spacing, np.float64)
    org = np.asarray(origin, np.float64)
    rc = _io().fsio_write_points(path.encode(), {"csv": 0, "csv.gz": 1, "bin": 2}[fmt], gz_opts.encode() if gz_opts else None,
                                 precision, pts.ctypes.data, desc.ctypes.data, len(pts), desc.shape[1], sp.ctypes.data,
                                 org.ctypes.data)
    if rc != 0:
        raise FrogSurfError(f"cannot write {path}")


def as_read_host(values: np.ndarray, precision: int) -> np.ndarray:
    """strtof of each float64 value as the .csv.gz writer formats it at -precision `precision` (host, no CUDA)."""
    v = np.ascontiguousarray(values, np.float64)
    out = np.zeros(v.shape, np.float32)
    _io().fsio_debug_as_read(v.ctypes.data, v.size, precision, out.ctypes.data)
    return out


def read_points_file(path: str, spacing, origin, shape):
    """vtk3DSURF::ReadIPoints (surf3d -p): (xyzs [n, 4] float32 in voxel units, number of points outside the image);
    `shape` is the volume's [z, y, x] shape."""
    sp = np.asarray(spacing, np.float64)
    org = np.asarray(origin, np.float64)
    dims = np.asarray([shape[2], shape[1], shape[0]], np.int32)
    outside = C.c_long()
    n = _io().fsio_read_points(path.encode(), sp.ctypes.data, org.ctypes.data, dims.ctypes.data, None, 0, C.byref(outside))
    if n < 0:
        raise FrogSurfError(f"cannot read points from {path}")
    out = np.zeros((n, 4), np.float32)
    if n:
        _io().fsio_read_points(path.encode(), sp.ctypes.data, org.ctypes.data, dims.ctypes.data, out.ctypes.data, n, C.byref(outside))
    return out, outside.value


_MET = {0: np.uint8, 1: np.int16, 2: np.uint16, 3: np.int32, 4: np.float32, 5: np.int8, 6: np.uint32, 7: np.float64}
_MET_NAME = {np.dtype(np.uint8): "MET_UCHAR", np.dtype(np.int16): "MET_SHORT", np.dtype(np.uint16): "MET_USHORT",
             np.dtype(np.int32): "MET_INT", np.dtype(np.float32): "MET_FLOAT", np.dtype(np.int8): "MET_CHAR",
             np.dtype(np.uint32): "MET_UINT", np.dtype(np.float64): "MET_DOUBLE"}


def read_metaimage(path: str, phases: dict | None = None):
    """(volume [z, y, x] in native byte order, spacing, origin) through bin/surf3d's own reader.  `phases`, when given,
    receives the seconds spent on the header, reading, inflating and byte swaps / axis flips."""
    dims = (C.c_int * 3)()
    sp = (C.c_double * 3)()
    org = (C.c_double * 3)()
    vt = C.c_int()
    nbytes = C.c_size_t()
    L = _io()
    if L.fsio_read_metaimage(path.encode(), dims, sp, org, C.byref(vt), None, 0, C.byref(nbytes), None) != 0:
        raise FrogSurfError(f"cannot read {path}: {L.fsio_last_error().decode()}")
    vol = np.empty((dims[2], dims[1], dims[0]), _MET[vt.value])
    secs = (C.c_double * 4)()
    if L.fsio_read_metaimage(path.encode(), dims, sp, org, C.byref(vt), vol.ctypes.data, vol.nbytes, C.byref(nbytes), secs) != 0:
        raise FrogSurfError(f"cannot read {path}: {L.fsio_last_error().decode()}")
    if phases is not None:
        phases.update(zip(("header_s", "read_s", "inflate_s", "swap_s"), secs))
    return vol, tuple(sp), tuple(org)


def write_metaimage(path: str, volume: np.ndarray, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0), transform=None, *,
                    compress: int | None = None, gzip: bool = False, compressed_size: bool = True, byte_order: str = "<",
                    data_file: str | None = None, header_size: int | None = None) -> None:
    """MetaImage of a [z, y, x] volume, for feeding bin/surf3d and bin/match.

    compress: zlib level (CompressedData = True), the stream wrapped as zlib or, with `gzip`, as a gzip member;
    compressed_size: write CompressedDataSize.  byte_order: "<" or ">" (BinaryDataByteOrderMSB = True).
    data_file: the data goes to this file (a name next to the header, usually .raw or .zraw) instead of after the
    header; header_size: HeaderSize of that file, as many filler bytes written before the data (-1: 61 filler bytes,
    HeaderSize = -1, the data ends the file)."""
    import zlib
    v = np.ascontiguousarray(volume)
    data = v.astype(v.dtype.newbyteorder(byte_order)).tobytes()
    if compress is not None:
        z = zlib.compressobj(compress, zlib.DEFLATED, 31 if gzip else 15)
        data = z.compress(data) + z.flush()
    hdr = "ObjectType = Image\nNDims = 3\nBinaryData = True\n"
    hdr += "BinaryDataByteOrderMSB = %s\n" % ("True" if byte_order == ">" else "False")
    hdr += "CompressedData = %s\n" % ("True" if compress is not None else "False")
    if compress is not None and compressed_size:
        hdr += "CompressedDataSize = %d\n" % len(data)
    if transform is not None:
        hdr += "TransformMatrix = " + " ".join(repr(float(t)) for t in transform) + "\n"
    hdr += "Offset = %r %r %r\n" % tuple(float(o) for o in origin)
    hdr += "ElementSpacing = %r %r %r\n" % tuple(float(s) for s in spacing)
    hdr += "DimSize = %d %d %d\n" % (v.shape[2], v.shape[1], v.shape[0])
    hdr += "ElementType = %s\n" % _MET_NAME[np.dtype(v.dtype)]
    if data_file is None:
        with open(path, "wb") as f:
            f.write((hdr + "ElementDataFile = LOCAL\n").encode())
            f.write(data)
        return
    if header_size is not None:
        hdr += "HeaderSize = %d\n" % header_size
    with open(path, "wb") as f:
        f.write((hdr + "ElementDataFile = %s\n" % data_file).encode())
    filler = 61 if header_size == -1 else (header_size or 0)
    with open(os.path.join(os.path.dirname(path), data_file), "wb") as f:
        f.write(bytes((i * 37 + 11) & 255 for i in range(filler)))
        f.write(data)
