"""Device-resident entry points: the `_dev` half of the C ABI over torch CUDA
tensors (torch is used for device memory, streams and torch.distributed only).

All kernels run on the engine's own stream.  ``engine_stream()`` exposes it as a
``torch.cuda.ExternalStream`` so that callers can order work against it and
record CUDA events on the stream the kernels are actually launched on.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib, api
from ._lib import OUT_ELEMENT, OUT_WIDTH, PT_ELEMENT, PT_WIDTH, SCALARS_MONTGOMERY, check

_ext_streams = {}


def _wrap(ptr: int) -> "torch.cuda.ExternalStream":
    dev = api.get_device()
    key = (dev, ptr)
    if key not in _ext_streams:
        _ext_streams[key] = torch.cuda.ExternalStream(ptr, device=torch.device("cuda", dev))
    return _ext_streams[key]


def engine_stream() -> "torch.cuda.ExternalStream":
    api._ensure_init()
    return _wrap(_lib.load().d377_stream())


def result_stream() -> "torch.cuda.ExternalStream":
    """d377_result_stream: where the results of asynchronous MSMs become complete.  Asking
    for it tells the engine that work is about to be enqueued there (the next join orders
    the engine stream behind it)."""
    api._ensure_init()
    return _wrap(_lib.load().d377_result_stream())


def reset_stream_cache() -> None:
    _ext_streams.clear()


def _chk(t: torch.Tensor, width: int, name: str) -> int:
    if not (t.is_cuda and t.dtype == torch.uint8 and t.is_contiguous()):
        raise ValueError("%s must be a contiguous CUDA uint8 tensor" % name)
    if t.dim() != 2 or t.shape[1] != width:
        raise ValueError("%s must have shape [n, %d]" % (name, width))
    return t.shape[0]


def _after_torch() -> None:
    """Make the engine stream wait for work already queued on torch's stream."""
    engine_stream().wait_stream(torch.cuda.current_stream())


def _then_torch() -> None:
    """Order torch's current stream after the engine stream, so that torch ops issued
    next see the results (no host synchronisation either way)."""
    torch.cuda.current_stream().wait_stream(engine_stream())




def decompress(enc: torch.Tensor, out: Optional[torch.Tensor] = None,
               ok: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    n = _chk(enc, 32, "enc")
    out = torch.empty((n, 128), dtype=torch.uint8, device=enc.device) if out is None else out
    ok = torch.empty((n,), dtype=torch.uint8, device=enc.device) if ok is None else ok
    _after_torch()
    check(_lib.load().d377_batch_decompress_dev(enc.data_ptr(), n, out.data_ptr(), ok.data_ptr()))
    _then_torch()
    return out, ok


def compress(elements: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    n = _chk(elements, 128, "elements")
    out = torch.empty((n, 32), dtype=torch.uint8, device=elements.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_batch_compress_dev(elements.data_ptr(), n, out.data_ptr()))
    _then_torch()
    return out


def decompress_fmt(enc: torch.Tensor, out_format: int, out: Optional[torch.Tensor] = None,
                   ok: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """d377_batch_decompress_fmt_dev: Element (128 B) or AffinePoint (64 B) outputs."""
    n = _chk(enc, 32, "enc")
    out = torch.empty((n, PT_WIDTH[out_format]), dtype=torch.uint8, device=enc.device) if out is None else out
    ok = torch.empty((n,), dtype=torch.uint8, device=enc.device) if ok is None else ok
    _after_torch()
    check(_lib.load().d377_batch_decompress_fmt_dev(enc.data_ptr(), n, out_format, out.data_ptr(),
                                                    ok.data_ptr()))
    _then_torch()
    return out, ok


def compress_fmt(points: torch.Tensor, point_format: int,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """d377_batch_compress_fmt_dev: Element, AffinePoint or X||Y||Z inputs."""
    n = _chk(points, PT_WIDTH[point_format], "points")
    out = torch.empty((n, 32), dtype=torch.uint8, device=points.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_batch_compress_fmt_dev(points.data_ptr(), point_format, n, out.data_ptr()))
    _then_torch()
    return out


def encode_to_curve(r: torch.Tensor, out_format: int = OUT_ELEMENT,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    n = _chk(r, 32, "r")
    out = torch.empty((n, OUT_WIDTH[out_format]), dtype=torch.uint8,
                      device=r.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_batch_encode_to_curve_dev(r.data_ptr(), n, out.data_ptr(), out_format))
    _then_torch()
    return out


def hash_to_curve(r1: torch.Tensor, r2: torch.Tensor, out_format: int = OUT_ELEMENT,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    n = _chk(r1, 32, "r1")
    _chk(r2, 32, "r2")
    out = torch.empty((n, OUT_WIDTH[out_format]), dtype=torch.uint8,
                      device=r1.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_batch_hash_to_curve_dev(r1.data_ptr(), r2.data_ptr(), n, out.data_ptr(),
                                                   out_format))
    _then_torch()
    return out


def scalar_mul(points: torch.Tensor, scalars: torch.Tensor, point_format: int = PT_ELEMENT,
               out_format: int = OUT_ELEMENT, out: Optional[torch.Tensor] = None,
               ok: Optional[torch.Tensor] = None) -> torch.Tensor:
    n = _chk(points, PT_WIDTH[point_format], "points")
    _chk(scalars, 32, "scalars")
    out = torch.empty((n, OUT_WIDTH[out_format]), dtype=torch.uint8,
                      device=points.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_batch_scalar_mul_dev(points.data_ptr(), point_format, scalars.data_ptr(),
                                                n, out.data_ptr(), out_format,
                                                None if ok is None else ok.data_ptr()))
    _then_torch()
    return out


def fixed_base_mul(scalars: torch.Tensor, out_format: int = OUT_ELEMENT,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    n = _chk(scalars, 32, "scalars")
    out = torch.empty((n, OUT_WIDTH[out_format & ~SCALARS_MONTGOMERY]), dtype=torch.uint8,
                      device=scalars.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_fixed_base_mul_dev(scalars.data_ptr(), n, out.data_ptr(), out_format))
    _then_torch()
    return out


def fixed_bases_mul(bases, scalars: torch.Tensor, out_format: int = OUT_ELEMENT,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """d377_fixed_bases_mul_dev: out[i] = sum_j scalars[i, j] * B_j over an api.FixedBases set;
    `scalars` is a contiguous CUDA uint8 tensor of shape [n, k, 32] ([n, 32] for k = 1);
    OR SCALARS_MONTGOMERY into `out_format` for in-memory Fr limbs."""
    if not (scalars.is_cuda and scalars.dtype == torch.uint8 and scalars.is_contiguous()):
        raise ValueError("scalars must be a contiguous CUDA uint8 tensor")
    if scalars.dim() == 2 and bases.k == 1 and scalars.shape[1] == 32:
        n = scalars.shape[0]
    elif scalars.dim() == 3 and tuple(scalars.shape[1:]) == (bases.k, 32):
        n = scalars.shape[0]
    else:
        raise ValueError("scalars must have shape [n, %d, 32], got %r" % (bases.k, tuple(scalars.shape)))
    out = torch.empty((n, OUT_WIDTH[out_format & ~SCALARS_MONTGOMERY]), dtype=torch.uint8,
                      device=scalars.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_fixed_bases_mul_dev(bases._handle(), scalars.data_ptr(), n, out.data_ptr(), out_format))
    _then_torch()
    return out


def msm_segmented(scalars: torch.Tensor, points: torch.Tensor, offsets, point_format: int = PT_ELEMENT,
                  out_format: int = OUT_ELEMENT, out: Optional[torch.Tensor] = None,
                  ok: Optional[torch.Tensor] = None, scalars_montgomery: bool = False) -> torch.Tensor:
    """d377_msm_segmented_dev over device-resident scalars / points: MSM j covers pairs
    offsets[j]..offsets[j+1].  `offsets` stays on the host (a sequence, numpy array or CPU
    tensor of nmsm + 1 entries); `ok` (optional, [nmsm] uint8 on the device) receives the
    per-segment decode status."""
    import numpy as np
    n = _chk(scalars, 32, "scalars")
    if _chk(points, PT_WIDTH[point_format], "points") < n:
        raise ValueError("fewer points than scalars")
    if isinstance(offsets, torch.Tensor):
        if offsets.is_cuda:
            raise ValueError("offsets must be in host memory")
        offsets = offsets.numpy()
    off = np.ascontiguousarray(offsets, dtype=np.uint32)
    if off.ndim != 1 or off.size < 1:
        raise ValueError("offsets must hold nmsm + 1 entries")
    if int(off[-1]) > n:
        raise ValueError("offsets reach past the end of the inputs")
    nmsm = off.size - 1
    out = torch.empty((nmsm, OUT_WIDTH[out_format]), dtype=torch.uint8,
                      device=scalars.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_msm_segmented_dev(scalars.data_ptr(), points.data_ptr(),
                                             point_format | (SCALARS_MONTGOMERY if scalars_montgomery else 0),
                                             off.ctypes.data, nmsm, out.data_ptr(), out_format,
                                             None if ok is None else ok.data_ptr()))
    _then_torch()
    return out


def normalize(elements: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """CurveGroup::normalize_batch on device-resident elements -> affine [n, 64]."""
    n = _chk(elements, 128, "elements")
    out = torch.empty((n, 64), dtype=torch.uint8, device=elements.device) if out is None else out
    _after_torch()
    check(_lib.load().d377_batch_normalize_dev(elements.data_ptr(), n, out.data_ptr()))
    _then_torch()
    return out


def sqrt_ratio_zeta(num: torch.Tensor, den: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Fq::sqrt_ratio_zeta over device-resident montgomery operands -> (roots, was_square)."""
    n = _chk(num, 32, "num")
    _chk(den, 32, "den")
    out = torch.empty_like(num)
    ws = torch.empty((n,), dtype=torch.uint8, device=num.device)
    _after_torch()
    check(_lib.load().d377_fq_batch_sqrt_ratio_zeta_dev(num.data_ptr(), den.data_ptr(), n,
                                                        out.data_ptr(), ws.data_ptr()))
    _then_torch()
    return out, ws


def element_sum(elements: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    n = _chk(elements, 128, "elements")
    oe = torch.empty((128,), dtype=torch.uint8, device=elements.device)
    oc = torch.empty((32,), dtype=torch.uint8, device=elements.device)
    _after_torch()
    check(_lib.load().d377_element_sum_dev(elements.data_ptr(), n, oe.data_ptr(), oc.data_ptr()))
    _then_torch()
    return oe, oc


def element_sum_result(elements: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """d377_element_sum_result_dev: the sum runs on the result stream (after whatever torch's
    current stream has queued, e.g. an all-gather of partial sums) and leaves the engine
    stream free for the next MSM.  Results are complete on result_stream()."""
    n = _chk(elements, 128, "elements")
    oe = torch.empty((128,), dtype=torch.uint8, device=elements.device)
    oc = torch.empty((32,), dtype=torch.uint8, device=elements.device)
    rs = result_stream()
    rs.wait_stream(torch.cuda.current_stream())
    for t in (elements, oe, oc):       # used on a stream torch's allocator does not know about
        t.record_stream(rs)
    check(_lib.load().d377_element_sum_result_dev(elements.data_ptr(), n, oe.data_ptr(), oc.data_ptr()))
    return oe, oc


def msm_async(scalars: torch.Tensor, points: torch.Tensor, point_format: int = PT_ELEMENT,
              want_encoding: bool = True, out_element: Optional[torch.Tensor] = None,
              out_encoding: Optional[torch.Tensor] = None, inputs_ready: bool = False,
              scalars_montgomery: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """d377_msm_dev_async: enqueue only.  The outputs are complete on result_stream() (and
    for torch after ``api.join(); torch.cuda.current_stream().wait_stream(engine_stream())``);
    a bad scalar / encoding is raised by the next ``api.sync()``.  Back-to-back calls overlap
    the tail of one MSM with the head of the next.  ``inputs_ready=True`` (D377_MSM_INPUTS_READY)
    promises that `scalars` / `points` are complete already -- not still being written by
    work queued on torch's or the engine's stream -- which lets this MSM's counting sort run
    under the previous MSM's bucket accumulation."""
    n = _chk(scalars, 32, "scalars")
    if hasattr(points, "ptr") and hasattr(points, "n"):
        if points.n < n or not points.ptr:
            raise ValueError("fewer prepared bases than scalars")
        pptr, point_format = points.ptr, 4
    else:
        if _chk(points, PT_WIDTH[point_format], "points") != n:
            raise ValueError("scalars and points differ in length")
        pptr = points.data_ptr()
    oe = torch.empty((128,), dtype=torch.uint8, device=scalars.device) if out_element is None else out_element
    oc = out_encoding
    if oc is None and want_encoding:
        oc = torch.empty((32,), dtype=torch.uint8, device=scalars.device)
    if not inputs_ready:
        # (with inputs_ready the engine stream must NOT wait for torch's stream: in a sharded
        # loop that stream carries the previous step's all-gather, which waits for the previous
        # MSM's tail -- exactly the dependency the asynchronous form removes)
        _after_torch()
    rs = result_stream()
    for t in (oe, oc):
        if t is not None:
            t.record_stream(rs)
    check(_lib.load().d377_msm_dev_async(scalars.data_ptr(), pptr, point_format | (0x100 if scalars_montgomery else 0), n,
                                         oe.data_ptr(), None if oc is None else oc.data_ptr(),
                                         1 if inputs_ready else 0))
    return oe, oc


def msm_multi(scalars, points, point_format: int = PT_ELEMENT):
    """d377_msm_multi_dev: `scalars` / `points` are lists of CUDA tensors, entry k living on
    the k-th device of init_multi.  Returns host (element, encoding) numpy arrays."""
    import ctypes as C

    import numpy as np
    k = len(scalars)
    if len(points) != k:
        raise ValueError("one scalar and one point tensor per device")
    ns = []
    for s_k, p_k in zip(scalars, points):
        n_k = _chk(s_k, 32, "scalars")
        if _chk(p_k, PT_WIDTH[point_format], "points") != n_k:
            raise ValueError("scalars and points differ in length")
        ns.append(n_k)
    for s_k in scalars:                       # inputs produced by torch: wait for them
        torch.cuda.synchronize(s_k.device)
    sp = (C.c_void_p * k)(*[t.data_ptr() for t in scalars])
    pp = (C.c_void_p * k)(*[t.data_ptr() for t in points])
    nn = (C.c_size_t * k)(*ns)
    oe = np.empty((128,), np.uint8)
    oc = np.empty((32,), np.uint8)
    check(_lib.load().d377_msm_multi_dev(sp, pp, point_format, nn, k, oe.ctypes.data_as(C.c_void_p),
                                         oc.ctypes.data_as(C.c_void_p)))
    return oe, oc


def msm_multi_async(scalars, points, point_format: int = PT_ELEMENT,
                    out_element: Optional[torch.Tensor] = None, out_encoding: Optional[torch.Tensor] = None):
    """d377_msm_multi_dev_async: enqueue one MSM over the devices of init_multi (entry k of
    `scalars` / `points` lives on the k-th device; the inputs must be complete).  The outputs
    are tensors on the first device, complete after ``multi_sync()``."""
    import ctypes as C
    k = len(scalars)
    ns = [_chk(s_k, 32, "scalars") for s_k in scalars]
    for p_k, n_k in zip(points, ns):
        if _chk(p_k, PT_WIDTH[point_format], "points") != n_k:
            raise ValueError("scalars and points differ in length")
    dev0 = scalars[0].device
    oe = torch.empty((128,), dtype=torch.uint8, device=dev0) if out_element is None else out_element
    oc = torch.empty((32,), dtype=torch.uint8, device=dev0) if out_encoding is None else out_encoding
    sp = (C.c_void_p * k)(*[t.data_ptr() for t in scalars])
    pp = (C.c_void_p * k)(*[t.data_ptr() for t in points])
    nn = (C.c_size_t * k)(*ns)
    check(_lib.load().d377_msm_multi_dev_async(sp, pp, point_format, nn, k, oe.data_ptr(), oc.data_ptr()))
    return oe, oc


def multi_sync() -> None:
    """d377_multi_sync: wait for every initialised device; raises the status of any leg."""
    check(_lib.load().d377_multi_sync())


def msm(scalars: torch.Tensor, points: torch.Tensor, point_format: int = PT_ELEMENT,
        want_encoding: bool = True, scalars_montgomery: bool = False
        ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Pippenger MSM over device-resident inputs -> (element [128], encoding [32] | None)."""
    n = _chk(scalars, 32, "scalars")
    if hasattr(points, "ptr") and hasattr(points, "n"):          # api.MsmBases
        if points.n < n or not points.ptr:
            raise ValueError("fewer prepared bases than scalars")
        pptr, point_format = points.ptr, 4                        # D377_PT_BASES
    else:
        if _chk(points, PT_WIDTH[point_format], "points") != n:
            raise ValueError("scalars and points differ in length")
        pptr = points.data_ptr()
    oe = torch.empty((128,), dtype=torch.uint8, device=scalars.device)
    oc = torch.empty((32,), dtype=torch.uint8, device=scalars.device) if want_encoding else None
    _after_torch()
    check(_lib.load().d377_msm_dev(scalars.data_ptr(), pptr, point_format | (0x100 if scalars_montgomery else 0), n,
                                   oe.data_ptr(), None if oc is None else oc.data_ptr()))
    _then_torch()
    return oe, oc
