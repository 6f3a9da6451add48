"""Host-side mirror of the decaf377 crate surface over the C ABI.

Names, argument meaning and error behaviour follow the reference
(src/lib.rs:7-29): ``Encoding.vartime_decompress`` raises
``EncodingError("InvalidEncoding")`` where the crate returns
``Err(EncodingError::InvalidEncoding)`` (src/error.rs:2-5), and so on.  Scalar
``Fq`` / ``Fr`` values are plain host integers (host logic, as in the crate);
every group operation and every batch goes to the GPU.  Batch functions take
and return ``numpy`` ``uint8`` arrays in the wire formats of
``include/decaf377_b200.h``.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (OUT_ELEMENT, OUT_ENCODING, OUT_WIDTH, PT_AFFINE, PT_BASES, PT_ELEMENT,  # noqa: F401
                   PT_ENCODING, PT_WIDTH, PT_XYZ, SCALARS_MONTGOMERY, D377Error, check)

# moduli: src/fields/fq.rs:29-34, src/fields/fr.rs:29-34
Q_MODULUS = 0x12AB655E9A2CA55660B44D1E5C37B00159AA76FED00000010A11800000000001
R_MODULUS = 0x04AAD957A68B2955982D1347970DEC005293A3AFC43C8AFEB95AEE9AC33FD9FF
_MONT = 1 << 256
_MONT_INV_Q = pow(_MONT, -1, Q_MODULUS)

_initialised_device: Optional[int] = None


def init(device: int = 0) -> None:
    """d377_init: bind this process to one GPU.  Raises if none is usable."""
    global _initialised_device
    check(_lib.load().d377_init(int(device)))
    _initialised_device = int(device)


def init_multi(devices: Sequence[int]) -> None:
    """d377_init_multi: one engine per listed GPU (devices[0] becomes the default and the
    gathering device of msm_multi)."""
    global _initialised_device
    devs = [int(d) for d in devices]
    arr = (C.c_int * len(devs))(*devs)
    check(_lib.load().d377_init_multi(arr, len(devs)))
    _initialised_device = devs[0]


def set_device(device: int) -> None:
    """d377_set_device: the initialised GPU the CALLING THREAD's calls act on (-1: default)."""
    check(_lib.load().d377_set_device(int(device)))


def get_device() -> int:
    return int(_lib.load().d377_get_device())


def device_list() -> list:
    arr = (C.c_int * 64)()
    k = int(_lib.load().d377_device_list(arr, 64))
    return [int(arr[i]) for i in range(min(k, 64))]


def _ensure_init() -> None:
    if _initialised_device is None:
        init(0)


def shutdown() -> None:
    global _initialised_device
    check(_lib.load().d377_shutdown())
    _initialised_device = None


def sync() -> None:
    """d377_sync: waits for the engine stream; raises the status of any asynchronous MSM
    enqueued since the last sync."""
    check(_lib.load().d377_sync())


def join() -> None:
    """d377_join: order the engine stream behind the result stream (no host wait)."""
    check(_lib.load().d377_join())


def msm_set_tail_overlap(on: bool) -> None:
    check(_lib.load().d377_msm_set_tail_overlap(1 if on else 0))


def debug_build() -> int:
    """0 = release library, 1 / 2 = on-curve (and order) predicate compiled into the kernels."""
    return int(_lib.load().d377_debug_build())


def debug_counts() -> Tuple[int, int]:
    """(failures, points checked) of the debug predicate since the library was loaded."""
    f, c = C.c_uint64(0), C.c_uint64(0)
    check(_lib.load().d377_debug_counts(C.byref(f), C.byref(c)))
    return int(f.value), int(c.value)


def launch_count() -> int:
    return int(_lib.load().d377_launch_count())


def msm_set_window(c: int) -> None:
    check(_lib.load().d377_msm_set_window(int(c)))


def msm_set_normalize(mode: int) -> None:
    """d377_msm_set_normalize: batch-normalise Element inputs first (1), never (-1), auto (0)."""
    check(_lib.load().d377_msm_set_normalize(int(mode)))


def msm_set_groups(groups: int) -> None:
    """d377_msm_set_groups: window groups of the sort/accumulate pipeline (0 = automatic)."""
    check(_lib.load().d377_msm_set_groups(int(groups)))


def msm_set_host_chunks(k: int) -> None:
    """d377_msm_set_host_chunks: sub-MSMs per host-buffer MSM (0 = automatic)."""
    check(_lib.load().d377_msm_set_host_chunks(int(k)))


class _PinnedBlock:
    """Owner of one d377_host_alloc block; frees it when the last array view dies."""

    def __init__(self, nbytes: int):
        lib = _lib.load()
        self.ptr = lib.d377_host_alloc(nbytes)
        if not self.ptr:
            raise D377Error(_lib.ERR_CUDA, lib.d377_last_error().decode(errors="replace"))
        self.nbytes = nbytes

    def __del__(self):
        try:
            if self.ptr:
                _lib.load().d377_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def pinned_empty(shape, dtype=np.uint8) -> np.ndarray:
    """Page-locked numpy array (d377_host_alloc).  Passing pinned inputs and ``out=``
    buffers to the batch functions lets upload, kernel and download overlap."""
    _ensure_init()
    dt = np.dtype(dtype)
    shape = (shape,) if isinstance(shape, int) else tuple(shape)
    nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
    blk = _PinnedBlock(max(nbytes, 1))
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(blk.ptr)
    buf._d377_owner = blk            # keeps the block alive as long as any view exists
    return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)


def pinned_copy(a) -> np.ndarray:
    a = np.asarray(a)
    out = pinned_empty(a.shape, a.dtype)
    out[...] = a
    return out


MSM_STAGES = ("points", "count", "scan", "scatter", "accumulate", "stitch", "bucket_reduce", "tail")


def msm_stage_info() -> dict:
    """Per-stage device times (ms) and geometry of the most recent MSM ("windowed": it ran
    over a windowed MsmBases set; c and W are then the set's)."""
    ms = (C.c_float * 8)()
    c, w, n = C.c_int(0), C.c_int(0), C.c_uint64(0)
    check(_lib.load().d377_msm_stage_info(ms, C.byref(c), C.byref(w), C.byref(n)))
    mixed, windowed = C.c_int(0), C.c_int(0)
    check(_lib.load().d377_msm_last_mode(C.byref(mixed)))
    check(_lib.load().d377_msm_last_windowed(C.byref(windowed)))
    return {"ms": dict(zip(MSM_STAGES, [float(x) for x in ms])), "c": c.value, "W": w.value,
            "n": int(n.value), "mixed": bool(mixed.value), "windowed": bool(windowed.value)}


def msm_timeline() -> list:
    """Per window group (processing order) of the most recent MSM: ms after its start at which
    the sorted list was ready, the accumulation started / ended, and the group's tail ended."""
    ms = (C.c_float * 32)()
    ng = C.c_int(0)
    check(_lib.load().d377_msm_timeline(ms, 32, C.byref(ng)))
    return [{"sorted": float(ms[4 * k]), "acc_start": float(ms[4 * k + 1]), "acc_end": float(ms[4 * k + 2]),
             "tail_end": float(ms[4 * k + 3])} for k in range(ng.value)]


def imad_peak() -> float:
    """Measured IMAD.WIDE.U32 issue rate in G multiply-adds / s."""
    _ensure_init()
    v = C.c_double(0.0)
    check(_lib.load().d377_imad_peak(C.byref(v)))
    return float(v.value)


class EncodingError(ValueError):
    """src/error.rs:2-5.  ``kind`` is 'InvalidEncoding' or 'InvalidSliceLength'."""

    def __init__(self, kind: str = "InvalidEncoding"):
        super().__init__(kind)
        self.kind = kind


# ---------------------------------------------------------------------------
# numpy helpers
# ---------------------------------------------------------------------------
def _arr(a, width: int, name: str) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.ndim == 1:
        if a.size % width:
            raise EncodingError("InvalidSliceLength")
        a = a.reshape(-1, width)
    if a.ndim != 2 or a.shape[1] != width:
        raise ValueError("%s must have shape [n, %d], got %r" % (name, width, a.shape))
    return a


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _out(out: Optional[np.ndarray], shape, name: str = "out") -> np.ndarray:
    """Result buffer: a fresh (pageable) array, or the caller's -- e.g. a pinned one."""
    if out is None:
        return np.empty(shape, np.uint8)
    if out.dtype != np.uint8 or tuple(out.shape) != tuple(shape) or not out.flags.c_contiguous:
        raise ValueError("%s must be a C-contiguous uint8 array of shape %r" % (name, tuple(shape)))
    return out


def _mont(flag: bool) -> int:
    return SCALARS_MONTGOMERY if flag else 0


# ---------------------------------------------------------------------------
# batch entry points (host buffers)
# ---------------------------------------------------------------------------
def batch_decompress(enc, out: Optional[np.ndarray] = None, ok: Optional[np.ndarray] = None
                     ) -> Tuple[np.ndarray, np.ndarray]:
    """Encoding::vartime_decompress over a batch -> (elements [n,128], ok [n])."""
    _ensure_init()
    enc = _arr(enc, 32, "enc")
    n = enc.shape[0]
    out = _out(out, (n, 128))
    ok = _out(ok, (n,), "ok")
    check(_lib.load().d377_batch_decompress(_ptr(enc), n, _ptr(out), _ptr(ok)))
    return out, ok


def batch_compress(elements, out: Optional[np.ndarray] = None) -> np.ndarray:
    """Element::vartime_compress over a batch -> encodings [n,32]."""
    _ensure_init()
    el = _arr(elements, 128, "elements")
    n = el.shape[0]
    out = _out(out, (n, 32))
    check(_lib.load().d377_batch_compress(_ptr(el), n, _ptr(out)))
    return out


def batch_affine_deserialize(enc, out: Optional[np.ndarray] = None, ok: Optional[np.ndarray] = None
                             ) -> Tuple[np.ndarray, np.ndarray]:
    """CanonicalDeserialize for AffinePoint (ark_curve/serialize.rs:8-28) over a batch:
    encodings [n,32] -> (x||y montgomery [n,64], ok [n])."""
    _ensure_init()
    enc = _arr(enc, 32, "enc")
    n = enc.shape[0]
    out = _out(out, (n, 64))
    ok = _out(ok, (n,), "ok")
    check(_lib.load().d377_batch_decompress_fmt(_ptr(enc), n, PT_AFFINE, _ptr(out), _ptr(ok)))
    return out, ok


def batch_compress_fmt(points, point_format: int, out: Optional[np.ndarray] = None) -> np.ndarray:
    """vartime_compress of points held as Element (128 B), AffinePoint (64 B:
    CanonicalSerialize for AffinePoint, ark_curve/serialize.rs:30-46) or X||Y||Z (96 B)."""
    _ensure_init()
    if point_format not in (PT_ELEMENT, PT_AFFINE, PT_XYZ):
        raise ValueError("point_format must be PT_ELEMENT, PT_AFFINE or PT_XYZ")
    pts = _arr(points, PT_WIDTH[point_format], "points")
    n = pts.shape[0]
    out = _out(out, (n, 32))
    check(_lib.load().d377_batch_compress_fmt(_ptr(pts), point_format, n, _ptr(out)))
    return out


def batch_affine_serialize(affine, out: Optional[np.ndarray] = None) -> np.ndarray:
    return batch_compress_fmt(affine, PT_AFFINE, out)


def _wide(a, name: str) -> np.ndarray:
    """[n, width] uint8 input of the Elligator entry points (any width 1..256)."""
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.ndim == 1:
        a = _arr(a, 32, name)
    if a.ndim != 2 or not (1 <= a.shape[1] <= 256):
        raise ValueError("%s must have shape [n, width], 1 <= width <= 256" % name)
    return a


def batch_encode_to_curve(r, out_format: int = OUT_ELEMENT, out: Optional[np.ndarray] = None
                          ) -> np.ndarray:
    """Element::encode_to_curve(Fq::from_le_bytes_mod_order(r[i])); r is [n, width] bytes
    (32 as in the reference's tests, 64 for hash outputs, any width up to 256)."""
    _ensure_init()
    r = _wide(r, "r")
    n, w = r.shape
    out = _out(out, (n, OUT_WIDTH[out_format]))
    check(_lib.load().d377_batch_encode_to_curve_wide(_ptr(r), w, n, _ptr(out), out_format))
    return out


def batch_hash_to_curve(r1, r2, out_format: int = OUT_ELEMENT, out: Optional[np.ndarray] = None
                        ) -> np.ndarray:
    _ensure_init()
    r1 = _wide(r1, "r1")
    r2 = _wide(r2, "r2")
    if r1.shape != r2.shape:
        raise ValueError("r1 and r2 differ in shape")
    n, w = r1.shape
    out = _out(out, (n, OUT_WIDTH[out_format]))
    check(_lib.load().d377_batch_hash_to_curve_wide(_ptr(r1), _ptr(r2), w, n, _ptr(out), out_format))
    return out


def fq_batch_from_le_bytes_mod_order(data) -> np.ndarray:
    """Fq::from_le_bytes_mod_order over [n, width] bytes (any width) -> montgomery [n, 32]."""
    _ensure_init()
    data = _wide(data, "data")
    n, w = data.shape
    out = np.empty((n, 32), np.uint8)
    check(_lib.load().d377_fq_batch_from_le_bytes_mod_order(_ptr(data), w, n, _ptr(out)))
    return out


def batch_scalar_mul(points, scalars, point_format: int = PT_ELEMENT,
                     out_format: int = OUT_ELEMENT, return_ok: bool = False,
                     out: Optional[np.ndarray] = None, ok: Optional[np.ndarray] = None,
                     scalars_montgomery: bool = False):
    """out[i] = scalars[i] * points[i].  `scalars_montgomery`: the scalars are the in-memory
    Montgomery limbs of the reference's Fr (D377_SCALARS_MONTGOMERY), converted on the GPU."""
    _ensure_init()
    pts = _arr(points, PT_WIDTH[point_format], "points")
    sc = _arr(scalars, 32, "scalars")
    if pts.shape[0] != sc.shape[0]:
        raise ValueError("points and scalars differ in length")
    n = pts.shape[0]
    out = _out(out, (n, OUT_WIDTH[out_format]))
    ok = _out(ok, (n,), "ok")
    check(_lib.load().d377_batch_scalar_mul(_ptr(pts), point_format | _mont(scalars_montgomery), _ptr(sc),
                                            n, _ptr(out), out_format, _ptr(ok)))
    return (out, ok) if return_ok else out


def fixed_base_mul(scalars, out_format: int = OUT_ELEMENT, out: Optional[np.ndarray] = None,
                   scalars_montgomery: bool = False) -> np.ndarray:
    """Element::GENERATOR * s for a batch of scalars."""
    _ensure_init()
    sc = _arr(scalars, 32, "scalars")
    n = sc.shape[0]
    out = _out(out, (n, OUT_WIDTH[out_format]))
    check(_lib.load().d377_fixed_base_mul(_ptr(sc), n, _ptr(out), out_format | _mont(scalars_montgomery)))
    return out


def batch_add(a, b) -> np.ndarray:
    _ensure_init()
    a = _arr(a, 128, "a")
    b = _arr(b, 128, "b")
    if a.shape != b.shape:
        raise ValueError("a and b differ in length")
    out = np.empty_like(a)
    check(_lib.load().d377_batch_add(_ptr(a), _ptr(b), a.shape[0], _ptr(out)))
    return out


def batch_sub(a, b) -> np.ndarray:
    _ensure_init()
    a = _arr(a, 128, "a")
    b = _arr(b, 128, "b")
    if a.shape != b.shape:
        raise ValueError("a and b differ in length")
    out = np.empty_like(a)
    check(_lib.load().d377_batch_sub(_ptr(a), _ptr(b), a.shape[0], _ptr(out)))
    return out


def batch_neg(a) -> np.ndarray:
    _ensure_init()
    a = _arr(a, 128, "a")
    out = np.empty_like(a)
    check(_lib.load().d377_batch_neg(_ptr(a), a.shape[0], _ptr(out)))
    return out


def batch_double(a) -> np.ndarray:
    _ensure_init()
    a = _arr(a, 128, "a")
    out = np.empty_like(a)
    check(_lib.load().d377_batch_double(_ptr(a), a.shape[0], _ptr(out)))
    return out


def batch_on_curve(elements, check_order: bool = False) -> np.ndarray:
    """OnCurve::is_on_curve over a batch (ark_curve/on_curve.rs:17-38) -> ok [n]."""
    _ensure_init()
    el = _arr(elements, 128, "elements")
    ok = np.empty((el.shape[0],), np.uint8)
    check(_lib.load().d377_batch_on_curve(_ptr(el), el.shape[0], 1 if check_order else 0, _ptr(ok)))
    return ok


def batch_element_eq(a, b) -> np.ndarray:
    _ensure_init()
    a = _arr(a, 128, "a")
    b = _arr(b, 128, "b")
    if a.shape != b.shape:
        raise ValueError("a and b differ in length")
    out = np.empty((a.shape[0],), np.uint8)
    check(_lib.load().d377_batch_element_eq(_ptr(a), _ptr(b), a.shape[0], _ptr(out)))
    return out


def element_sum(elements) -> Tuple[np.ndarray, np.ndarray]:
    """Sum<Element>: returns (element [128], encoding [32])."""
    _ensure_init()
    el = _arr(elements, 128, "elements")
    oe = np.empty((128,), np.uint8)
    oc = np.empty((32,), np.uint8)
    check(_lib.load().d377_element_sum(_ptr(el), el.shape[0], _ptr(oe), _ptr(oc)))
    return oe, oc


class MsmBases:
    """Long-lived MSM bases (d377_msm_bases_create): ScalarMul::batch_convert_to_mul_base once
    (ark_curve/element.rs:27-34), then VariableBaseMSM::msm(&bases, &scalars) many times.
    Pass the object as `points` to vartime_multiscalar_mul / msm_submit / device.msm: only
    the scalars cross the link and the normalisation is skipped.

    ``windowed=True`` (d377_msm_bases_create_windowed) also stores 2^(c j) * P_i for every
    window j: n * W * 128 bytes of device memory, and every MSM over the set adds all windows
    into one bucket set and skips the Horner tail.  ``c`` is the window width of such a set
    (0: chosen from n; 4..22 otherwise).  ``.c``, ``.windows`` and ``.nbytes`` describe the
    set (c = 0 and windows = 1 for a plain one)."""

    def __init__(self, points=None, point_format: int = PT_ELEMENT, *, device_ptr: int = 0, n: int = 0,
                 windowed: bool = False, c: int = 0):
        _ensure_init()
        lib = _lib.load()
        out = C.c_void_p(0)
        if points is not None:
            pts = _arr(points, PT_WIDTH[point_format], "points")
            n = pts.shape[0]
            if windowed:
                check(lib.d377_msm_bases_create_windowed(_ptr(pts), point_format, n, int(c), C.byref(out)))
            else:
                check(lib.d377_msm_bases_create(_ptr(pts), point_format, n, C.byref(out)))
        elif windowed:
            check(lib.d377_msm_bases_create_windowed_dev(C.c_void_p(device_ptr), point_format, n, int(c),
                                                         C.byref(out)))
        else:
            check(lib.d377_msm_bases_create_dev(C.c_void_p(device_ptr), point_format, n, C.byref(out)))
        self.ptr = out.value or 0
        self.n = n
        nn, cc, ww, nb = C.c_size_t(0), C.c_int(0), C.c_int(0), C.c_size_t(0)
        check(lib.d377_msm_bases_info(C.c_void_p(self.ptr), C.byref(nn), C.byref(cc), C.byref(ww), C.byref(nb)))
        self.c = int(cc.value)
        self.windows = int(ww.value)
        self.nbytes = int(nb.value)

    def close(self) -> None:
        if self.ptr:
            check(_lib.load().d377_msm_bases_destroy(C.c_void_p(self.ptr)))
            self.ptr = 0

    def __len__(self) -> int:
        return self.n

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _bases_ptr(b: "MsmBases"):
    if not b.ptr:
        raise ValueError("MsmBases has been closed")
    return C.c_void_p(b.ptr)


class FixedBases:
    """Prepared fixed bases (d377_fixed_bases_create): window tables of k caller-chosen points
    B_0..B_{k-1}, 48 MiB of device memory per base, built once.  ``mul(scalars)`` then computes
    out[i] = sum_j scalars[i, j] * B_j for every row -- with k = 1, fixed-base multiplication by
    an arbitrary point; with k = 2, e.g. Pedersen commitments v * G_a + r * H.  ``points``: k
    inputs in `point_format` (host memory), or ``device_ptr`` / ``k`` for device memory.
    ``.k``, ``.nbytes`` and ``len()`` describe the set; ``close()`` releases it."""

    def __init__(self, points=None, point_format: int = PT_ELEMENT, *, device_ptr: int = 0, k: int = 0):
        _ensure_init()
        lib = _lib.load()
        out = C.c_void_p(0)
        if points is not None:
            pts = _arr(points, PT_WIDTH[point_format], "points")
            k = pts.shape[0]
            check(lib.d377_fixed_bases_create(_ptr(pts), point_format, k, C.byref(out)))
        else:
            check(lib.d377_fixed_bases_create_dev(C.c_void_p(device_ptr), point_format, int(k), C.byref(out)))
        self.ptr = out.value or 0
        kk, nb = C.c_size_t(0), C.c_size_t(0)
        check(lib.d377_fixed_bases_info(C.c_void_p(self.ptr), C.byref(kk), C.byref(nb)))
        self.k = int(kk.value)
        self.nbytes = int(nb.value)

    def _handle(self):
        if not self.ptr:
            raise ValueError("FixedBases has been closed")
        return C.c_void_p(self.ptr)

    def _scalars(self, scalars) -> np.ndarray:
        """`scalars` as the [n, k, 32] uint8 array mul() passes on; [n, 32] is accepted for k = 1."""
        sc = np.ascontiguousarray(scalars, dtype=np.uint8)
        if sc.ndim == 2 and self.k == 1 and sc.shape[1] == 32:
            sc = sc.reshape(-1, 1, 32)
        if sc.ndim != 3 or sc.shape[1:] != (self.k, 32):
            raise ValueError("scalars must have shape [n, %d, 32]%s, got %r"
                             % (self.k, " or [n, 32]" if self.k == 1 else "", sc.shape))
        return sc

    def mul(self, scalars, out_format: int = OUT_ELEMENT, out: Optional[np.ndarray] = None,
            scalars_montgomery: bool = False) -> np.ndarray:
        """out[i] = sum_j scalars[i, j] * B_j -> [n, 128] Elements or [n, 32] encodings.  Each
        scalar is any 256-bit little-endian integer; `scalars_montgomery`: the in-memory
        Montgomery limbs of the reference's Fr (D377_SCALARS_MONTGOMERY)."""
        sc = self._scalars(scalars)
        n = sc.shape[0]
        out = _out(out, (n, OUT_WIDTH[out_format]))
        check(_lib.load().d377_fixed_bases_mul(self._handle(), _ptr(sc), n, _ptr(out),
                                               out_format | _mont(scalars_montgomery)))
        return out

    def close(self) -> None:
        if self.ptr:
            check(_lib.load().d377_fixed_bases_destroy(C.c_void_p(self.ptr)))
            self.ptr = 0

    def __len__(self) -> int:
        return self.k

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def vartime_multiscalar_mul(scalars, points, point_format: int = PT_ELEMENT,
                            scalars_montgomery: bool = False) -> Tuple[np.ndarray, np.ndarray]:
    """Element::vartime_multiscalar_mul: returns (element [128], encoding [32]).

    Like the reference (element/projective.rs:110) the two sequences are
    zipped: the longer one is truncated.  `points` may be an MsmBases object.
    """
    _ensure_init()
    sc = _arr(scalars, 32, "scalars")
    oe = np.empty((128,), np.uint8)
    oc = np.empty((32,), np.uint8)
    if isinstance(points, MsmBases):
        n = min(sc.shape[0], points.n)
        check(_lib.load().d377_msm(_ptr(sc), _bases_ptr(points), PT_BASES | _mont(scalars_montgomery), n,
                                   _ptr(oe), _ptr(oc)))
        return oe, oc
    pts = _arr(points, PT_WIDTH[point_format], "points")
    n = min(sc.shape[0], pts.shape[0])
    check(_lib.load().d377_msm(_ptr(sc), _ptr(pts), point_format | _mont(scalars_montgomery), n,
                               _ptr(oe), _ptr(oc)))
    return oe, oc


def msm_multi(scalars, points, point_format: int = PT_ELEMENT, ngpu: Optional[int] = None,
              scalars_montgomery: bool = False) -> Tuple[np.ndarray, np.ndarray]:
    """d377_msm_multi: one MSM over the first `ngpu` GPUs of init_multi (host buffers; every
    GPU takes a contiguous slice, partial sums meet on the first GPU)."""
    _ensure_init()
    sc = _arr(scalars, 32, "scalars")
    pts = _arr(points, PT_WIDTH[point_format], "points")
    n = min(sc.shape[0], pts.shape[0])
    ngpu = len(device_list()) if ngpu is None else int(ngpu)
    oe = np.empty((128,), np.uint8)
    oc = np.empty((32,), np.uint8)
    check(_lib.load().d377_msm_multi(_ptr(sc), _ptr(pts), point_format | _mont(scalars_montgomery), n, ngpu,
                                     _ptr(oe), _ptr(oc)))
    return oe, oc


def batch_msm(scalars, points, offsets, point_format: int = PT_ELEMENT, out_format: int = OUT_ELEMENT,
              return_ok: bool = False, scalars_montgomery: bool = False):
    """d377_batch_msm: many independent small MSMs; MSM j covers pairs offsets[j]..offsets[j+1]
    (Element::vartime_multiscalar_mul called in a loop).  Returns [nmsm, 128 | 32] (and ok [nmsm])."""
    _ensure_init()
    sc = _arr(scalars, 32, "scalars")
    pts = _arr(points, PT_WIDTH[point_format], "points")
    off = np.ascontiguousarray(offsets, dtype=np.uint32)
    if off.ndim != 1 or off.size < 1:
        raise ValueError("offsets must hold nmsm + 1 entries")
    nmsm = off.size - 1
    if int(off[-1]) > min(sc.shape[0], pts.shape[0]):
        raise ValueError("offsets reach past the end of the inputs")
    out = np.empty((nmsm, OUT_WIDTH[out_format]), np.uint8)
    ok = np.empty((nmsm,), np.uint8)
    check(_lib.load().d377_batch_msm(_ptr(sc), _ptr(pts), point_format | _mont(scalars_montgomery),
                                     off.ctypes.data_as(C.c_void_p), nmsm, _ptr(out), out_format, _ptr(ok)))
    return (out, ok) if return_ok else out


def msm_segmented(scalars, points, offsets, point_format: int = PT_ELEMENT, out_format: int = OUT_ELEMENT,
                  return_ok: bool = False, scalars_montgomery: bool = False):
    """d377_msm_segmented: the results of ``batch_msm`` (MSM j covers pairs
    offsets[j]..offsets[j+1]) from one segmented Pippenger over all segments -- the call for
    many MSMs of tens to tens of thousands of pairs.  Returns [nmsm, 128 | 32] (and ok [nmsm])."""
    _ensure_init()
    sc = _arr(scalars, 32, "scalars")
    pts = _arr(points, PT_WIDTH[point_format], "points")
    off = np.ascontiguousarray(offsets, dtype=np.uint32)
    if off.ndim != 1 or off.size < 1:
        raise ValueError("offsets must hold nmsm + 1 entries")
    nmsm = off.size - 1
    if int(off[-1]) > min(sc.shape[0], pts.shape[0]):
        raise ValueError("offsets reach past the end of the inputs")
    out = np.empty((nmsm, OUT_WIDTH[out_format]), np.uint8)
    ok = np.empty((nmsm,), np.uint8)
    check(_lib.load().d377_msm_segmented(_ptr(sc), _ptr(pts), point_format | _mont(scalars_montgomery),
                                         off.ctypes.data_as(C.c_void_p), nmsm, _ptr(out), out_format, _ptr(ok)))
    return (out, ok) if return_ok else out


def msm_segmented_last() -> Tuple[int, int, int]:
    """d377_msm_segmented_last: (c, W, chunks) of the most recent segmented MSM."""
    c, w, k = C.c_int(), C.c_int(), C.c_size_t()
    check(_lib.load().d377_msm_segmented_last(C.byref(c), C.byref(w), C.byref(k)))
    return c.value, w.value, k.value


def msm_submit(scalars, points, point_format: int = PT_ELEMENT, slot: int = 0,
               scalars_montgomery: bool = False) -> None:
    """d377_msm_submit: start an MSM over host buffers without waiting (slots 0..3).
    The arrays must stay alive and unmodified until ``msm_wait(slot)``.  `points` may be an
    MsmBases object."""
    _ensure_init()
    sc = _arr(scalars, 32, "scalars")
    if isinstance(points, MsmBases):
        n = min(sc.shape[0], points.n)
        check(_lib.load().d377_msm_submit(_ptr(sc), _bases_ptr(points), PT_BASES | _mont(scalars_montgomery), n, slot))
        return
    pts = _arr(points, PT_WIDTH[point_format], "points")
    n = min(sc.shape[0], pts.shape[0])
    check(_lib.load().d377_msm_submit(_ptr(sc), _ptr(pts), point_format | _mont(scalars_montgomery), n, slot))


def msm_wait(slot: int = 0) -> Tuple[np.ndarray, np.ndarray]:
    """d377_msm_wait: (element [128], encoding [32]) of the MSM submitted on `slot`."""
    oe = np.empty((128,), np.uint8)
    oc = np.empty((32,), np.uint8)
    check(_lib.load().d377_msm_wait(slot, _ptr(oe), _ptr(oc)))
    return oe, oc


def fq_batch_op(op: int, a, b=None) -> np.ndarray:
    _ensure_init()
    a = _arr(a, 32, "a")
    bb = None if b is None else _arr(b, 32, "b")
    out = np.empty_like(a)
    check(_lib.load().d377_fq_batch_op(op, _ptr(a), _ptr(bb), a.shape[0], _ptr(out)))
    return out


def fq_batch_isqrt(x) -> Tuple[np.ndarray, np.ndarray]:
    _ensure_init()
    x = _arr(x, 32, "x")
    out = np.empty_like(x)
    ws = np.empty((x.shape[0],), np.uint8)
    check(_lib.load().d377_fq_batch_isqrt(_ptr(x), x.shape[0], _ptr(out), _ptr(ws)))
    return out, ws


def fq_batch_sqrt_ratio_zeta(num, den) -> Tuple[np.ndarray, np.ndarray]:
    """Fq::sqrt_ratio_zeta over a batch (montgomery in / out) -> (roots [n,32], was_square [n])."""
    _ensure_init()
    num = _arr(num, 32, "num")
    den = _arr(den, 32, "den")
    if num.shape != den.shape:
        raise ValueError("num and den differ in length")
    out = np.empty_like(num)
    ws = np.empty((num.shape[0],), np.uint8)
    check(_lib.load().d377_fq_batch_sqrt_ratio_zeta(_ptr(num), _ptr(den), num.shape[0], _ptr(out),
                                                    _ptr(ws)))
    return out, ws


FIELD_FQ, FIELD_FR = 0, 1


def field_batch_deserialize(field: int, data) -> Tuple[np.ndarray, np.ndarray]:
    """CanonicalDeserialize for Fq (-> montgomery) / Fr (-> canonical) over a batch of
    32-byte LE values -> (out [n,32], ok [n]); ok = 0 marks a value >= the modulus."""
    _ensure_init()
    data = _arr(data, 32, "data")
    out = np.empty_like(data)
    ok = np.empty((data.shape[0],), np.uint8)
    check(_lib.load().d377_field_batch_deserialize(int(field), _ptr(data), data.shape[0], _ptr(out),
                                                   _ptr(ok)))
    return out, ok


def batch_normalize(elements, out: Optional[np.ndarray] = None) -> np.ndarray:
    """CurveGroup::normalize_batch / batch_convert_to_mul_base: [n,128] -> affine [n,64]."""
    _ensure_init()
    el = _arr(elements, 128, "elements")
    out = _out(out, (el.shape[0], 64))
    check(_lib.load().d377_batch_normalize(_ptr(el), el.shape[0], _ptr(out)))
    return out


# ---------------------------------------------------------------------------
# scalar types mirroring the crate
# ---------------------------------------------------------------------------
class _PrimeField:
    MODULUS = 0
    __slots__ = ("v",)

    def __init__(self, v: int = 0):
        self.v = int(v) % self.MODULUS

    # fields/fq.rs:90-119 (host integer arithmetic; the batch form on the GPU is
    # fq_batch_from_le_bytes_mod_order)
    @classmethod
    def from_le_bytes_mod_order(cls, b: bytes):
        return cls(int.from_bytes(bytes(b), "little"))

    @classmethod
    def from_bytes_checked(cls, b: bytes):
        b = bytes(b)
        if len(b) != 32:
            raise EncodingError("InvalidSliceLength")
        v = int.from_bytes(b, "little")
        if v >= cls.MODULUS:
            raise EncodingError("InvalidEncoding")
        return cls(v)

    def to_bytes(self) -> bytes:
        return self.v.to_bytes(32, "little")

    def to_montgomery_bytes(self) -> bytes:
        """The in-memory form of the reference's field types: x * 2^256 mod p, little-endian."""
        return (self.v * _MONT % self.MODULUS).to_bytes(32, "little")

    def __add__(self, o): return type(self)(self.v + type(self)._c(o))
    def __sub__(self, o): return type(self)(self.v - type(self)._c(o))
    def __mul__(self, o):
        if isinstance(o, Element):
            return o.__rmul__(self)
        return type(self)(self.v * type(self)._c(o))
    def __neg__(self): return type(self)(-self.v)
    def __eq__(self, o): return isinstance(o, type(self)) and self.v == o.v
    def __hash__(self): return hash((type(self).__name__, self.v))
    def __int__(self): return self.v
    def __repr__(self): return "%s(0x%064x)" % (type(self).__name__, self.v)
    def square(self): return type(self)(self.v * self.v)
    def is_zero(self): return self.v == 0

    def inverse(self):
        return None if self.v == 0 else type(self)(pow(self.v, -1, self.MODULUS))

    @classmethod
    def _c(cls, o) -> int:
        if isinstance(o, cls):
            return o.v
        if isinstance(o, int):
            return o
        raise TypeError("cannot combine %s with %r" % (cls.__name__, type(o)))


class Fq(_PrimeField):
    """fields/fq.rs: element of GF(q)."""
    MODULUS = Q_MODULUS

    # sign.rs:3-23
    def is_nonnegative(self) -> bool: return (self.v & 1) == 0
    def is_negative(self) -> bool: return (self.v & 1) == 1
    def abs(self): return -self if self.is_negative() else self

    @classmethod
    def from_montgomery_bytes(cls, b: bytes):
        return cls(int.from_bytes(bytes(b), "little") * _MONT_INV_Q)

    @staticmethod
    def sqrt_ratio_zeta(num: "Fq", den: "Fq") -> Tuple[bool, "Fq"]:
        """ark_curve/invsqrt.rs:75-166 on the GPU (same root as the reference)."""
        out, ws = fq_batch_sqrt_ratio_zeta(np.frombuffer(num.to_montgomery_bytes(), np.uint8),
                                           np.frombuffer(den.to_montgomery_bytes(), np.uint8))
        return bool(ws[0]), Fq.from_montgomery_bytes(out[0].tobytes())

    # CanonicalSerialize / CanonicalDeserialize (fq/arkworks.rs:189-277): 32 canonical LE bytes
    def serialize_compressed(self) -> bytes:
        return self.to_bytes()

    @classmethod
    def deserialize_compressed(cls, b: bytes):
        return cls.from_bytes_checked(b)


class Fr(_PrimeField):
    """fields/fr.rs: scalar mod the group order r."""
    MODULUS = R_MODULUS


ZETA = Fq(2841681278031794617739547238867782961338435681360110683443920362658525667816)


class Encoding:
    """ark_curve/encoding.rs:14-15 ``Encoding(pub [u8; 32])``."""
    __slots__ = ("bytes",)

    def __init__(self, b: bytes):
        b = bytes(b)
        if len(b) != 32:
            raise EncodingError("InvalidSliceLength")     # encoding.rs:181-188
        self.bytes = b

    def vartime_decompress(self) -> "Element":
        el, ok = batch_decompress(np.frombuffer(self.bytes, np.uint8))
        if not ok[0]:
            raise EncodingError("InvalidEncoding")
        return Element(el[0].tobytes())

    def __eq__(self, o): return isinstance(o, Encoding) and self.bytes == o.bytes
    def __hash__(self): return hash(self.bytes)
    def __repr__(self): return "Encoding(%s)" % self.bytes.hex()


class Element:
    """ark_curve/element/projective.rs:13-16: a decaf377 group element, held as its
    128-byte wire image X||Y||Z||T."""
    __slots__ = ("wire",)

    def __init__(self, wire: bytes):
        wire = bytes(wire)
        if len(wire) != 128:
            raise ValueError("Element wire image must be 128 bytes")
        self.wire = wire

    @classmethod
    def _from_coords(cls, x, y, z, t):
        return cls(b"".join(Fq(c).to_montgomery_bytes() for c in (x, y, z, t)))

    def _np(self):
        return np.frombuffer(self.wire, np.uint8).reshape(1, 128)

    def vartime_compress(self) -> Encoding:
        return Encoding(batch_compress(self._np())[0].tobytes())

    def vartime_compress_to_field(self) -> Fq:
        return Fq.from_bytes_checked(self.vartime_compress().bytes)

    # CanonicalSerialize / CanonicalDeserialize, ark_curve/encoding.rs:158-176,272-292
    def serialize_compressed(self) -> bytes:
        return self.vartime_compress().bytes

    @staticmethod
    def deserialize_compressed(b: bytes) -> "Element":
        return Encoding(b).vartime_decompress()

    def into_affine(self) -> "AffinePoint":
        """CurveGroup::into_affine (ark_curve/element.rs:83-85)."""
        return AffinePoint(batch_normalize(self._np())[0].tobytes())

    @staticmethod
    def normalize_batch(elements: Sequence["Element"]) -> list:
        """CurveGroup::normalize_batch (ark_curve/element.rs:74-81)."""
        if not elements:
            return []
        el = np.frombuffer(b"".join(e.wire for e in elements), np.uint8).reshape(-1, 128)
        aff = batch_normalize(el)
        return [AffinePoint(aff[i].tobytes()) for i in range(aff.shape[0])]

    batch_convert_to_mul_base = normalize_batch      # ark_curve/element.rs:27-34

    @staticmethod
    def encode_to_curve(r: Fq) -> "Element":
        return Element(batch_encode_to_curve(np.frombuffer(r.to_bytes(), np.uint8))[0].tobytes())

    @staticmethod
    def hash_to_curve(r1: Fq, r2: Fq) -> "Element":
        return Element(batch_hash_to_curve(np.frombuffer(r1.to_bytes(), np.uint8),
                                           np.frombuffer(r2.to_bytes(), np.uint8))[0].tobytes())

    def __add__(self, o: "Element") -> "Element":
        return Element(batch_add(self._np(), o._np())[0].tobytes())

    def __neg__(self) -> "Element":
        return Element(batch_neg(self._np())[0].tobytes())

    def __sub__(self, o: "Element") -> "Element":
        return Element(batch_sub(self._np(), o._np())[0].tobytes())

    def double(self) -> "Element":
        return Element(batch_double(self._np())[0].tobytes())

    def is_on_curve(self) -> bool:
        """OnCurve::is_on_curve (ark_curve/on_curve.rs:17-38), including the [2r]P test."""
        return bool(batch_on_curve(self._np(), check_order=True)[0])

    def __rmul__(self, s: Fr) -> "Element":
        if not isinstance(s, Fr):
            return NotImplemented
        out = batch_scalar_mul(self._np(), np.frombuffer(s.to_bytes(), np.uint8))
        return Element(out[0].tobytes())

    __mul__ = __rmul__

    def __eq__(self, o) -> bool:
        return isinstance(o, Element) and bool(batch_element_eq(self._np(), o._np())[0])

    def __hash__(self):
        return hash(self.vartime_compress().bytes)

    def is_identity(self) -> bool:
        return Fq.from_montgomery_bytes(self.wire[:32]).v == 0

    @staticmethod
    def vartime_multiscalar_mul(scalars: Iterable[Fr], points: Iterable["Element"]) -> "Element":
        sc = [s.to_bytes() for s in scalars]
        pt = [p.wire for p in points]
        n = min(len(sc), len(pt))
        sc_np = np.frombuffer(b"".join(sc[:n]), np.uint8).reshape(n, 32)
        pt_np = np.frombuffer(b"".join(pt[:n]), np.uint8).reshape(n, 128)
        el, _ = vartime_multiscalar_mul(sc_np, pt_np)
        return Element(el.tobytes())

    def __repr__(self):
        return "Element(%s)" % self.wire.hex()


class AffinePoint:
    """ark_curve/element/affine.rs:12-15: affine (x, y), held as its 64-byte wire image
    x||y (montgomery); the D377_PT_AFFINE input format of the MSM."""
    __slots__ = ("wire",)

    def __init__(self, wire: bytes):
        wire = bytes(wire)
        if len(wire) != 64:
            raise ValueError("AffinePoint wire image must be 64 bytes")
        self.wire = wire

    def into_element(self) -> Element:
        x = Fq.from_montgomery_bytes(self.wire[:32])
        y = Fq.from_montgomery_bytes(self.wire[32:])
        return Element._from_coords(x.v, y.v, 1, (x * y).v)

    def __eq__(self, o) -> bool:                      # affine.rs:41-46
        return isinstance(o, AffinePoint) and self.into_element() == o.into_element()

    def __hash__(self):
        return hash(self.serialize_compressed())

    # ark_curve/serialize.rs:8-46
    def serialize_compressed(self) -> bytes:
        return batch_affine_serialize(np.frombuffer(self.wire, np.uint8))[0].tobytes()

    @staticmethod
    def deserialize_compressed(b: bytes) -> "AffinePoint":
        xy, ok = batch_affine_deserialize(np.frombuffer(Encoding(b).bytes, np.uint8))
        if not ok[0]:
            raise EncodingError("InvalidEncoding")
        return AffinePoint(xy[0].tobytes())

    def __repr__(self):
        return "decaf377::AffinePoint(%s)" % self.serialize_compressed().hex()


# ark_curve/constants.rs:61-79, element/projective.rs:20-27
Element.IDENTITY = Element._from_coords(0, 1, 1, 0)
_BX = 0x0AF6F264422A797BDF65D3E521D79000CB029727F00000009C432AAAAAAAAAAB
_BY = 0x0D661B0655477AE2E9C1817E3B1BC4D94DBB532F4E32AD8B963CADFA16D9E2B8
Element.GENERATOR = Element._from_coords(_BX, _BY, 1, _BX * _BY % Q_MODULUS)
Element.default = staticmethod(lambda: Element.IDENTITY)
