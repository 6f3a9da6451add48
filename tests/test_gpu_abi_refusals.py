"""The public ABI's argument checks, entry point by entry point, host-buffer and device-pointer
form alike: which format words each one takes (with and without D377_SCALARS_MONTGOMERY where
it takes scalars), input widths, null pointers, what n = 0 returns, and the order in which the
checks are made.  Every refusal must leave the caller's output buffers as they were."""
import ctypes as C
import random

import numpy as np
import pytest

from decaf377_b200 import _lib
from oracle import decaf377_ref as o
from tests.util import mont, np_bytes, oracle_points

pytestmark = pytest.mark.gpu

N = 4
MONT = _lib.SCALARS_MONTGOMERY
SENT = 0xA5                 # fill of every output buffer
HSENT = 0x5A5A5A5A00        # fill of every handle out-pointer
OK, INVALID = _lib.OK, _lib.ERR_INVALID_ARG
PT_W = {0: 128, 1: 32, 2: 64, 3: 96}


def _rejected(accepted, scalars):
    """Format words an entry point that takes `accepted` must refuse."""
    top = max(accepted)
    bad = {v for v in range(5) if v not in accepted} | {-1, top + 1, 5, 0x200}
    if scalars:
        bad |= {0x200 | MONT, (top + 1) | MONT, -1 & ~MONT}
    else:
        bad |= {a | MONT for a in accepted}
    return sorted(bad)


def _accepted(accepted, scalars):
    return list(accepted) + ([a | MONT for a in accepted] if scalars else [])


@pytest.fixture(scope="module")
def data(engine):
    rnd = random.Random(377)
    P = oracle_points("abi refusals", N)
    sc = [rnd.randrange(o.R) for _ in range(N)]
    d = {
        "pt0": np_bytes([o.point_to_wire(p) for p in P], 128),
        "pt1": np_bytes([o.compress(p) for p in P], 32),
        "pt2": np_bytes([o.fq_to_mont_bytes(x) + o.fq_to_mont_bytes(y) for x, y in (o.to_affine(p) for p in P)], 64),
        "sc": np_bytes([s.to_bytes(32, "little") for s in sc], 32),
        "scm": np_bytes([(s * (1 << 256) % o.R).to_bytes(32, "little") for s in sc], 32),
        "r": np_bytes([rnd.getrandbits(256).to_bytes(32, "little") for _ in range(N)], 32),
        "r64": np_bytes([rnd.getrandbits(512).to_bytes(64, "little") for _ in range(N)], 64),
        "fq": mont([rnd.randrange(1, 1 << 64) for _ in range(N)]),
    }
    d["pt3"] = np.ascontiguousarray(d["pt0"][:, :96])
    bases = engine.MsmBases(d["pt0"])
    fixed = engine.FixedBases(d["pt0"][:1])
    d["bases"], d["fixed"] = bases.ptr, fixed.ptr
    yield d
    bases.close()
    fixed.close()


class Call:
    """Buffers of one call: inputs as host arrays or device tensors, sentinel-filled outputs."""

    def __init__(self, data, dev):
        self.data, self.dev, self.keep, self.outs, self.hv = data, dev, [], [], None

    def _place(self, a):
        if self.dev:
            import torch
            a = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            self.keep.append(a)
            return C.c_void_p(a.data_ptr())
        a = np.ascontiguousarray(a)
        self.keep.append(a)
        return a.ctypes.data_as(C.c_void_p)

    def i(self, key):
        return self._place(self.data[key])

    def pts(self, fmt):
        """Points in format `fmt` (a refused format reads Elements; D377_PT_BASES the prepared set)."""
        f = fmt & ~MONT if fmt >= 0 else fmt
        if f == _lib.PT_BASES:
            return C.c_void_p(self.data["bases"])
        return self.i("pt%d" % f if f in PT_W else "pt0")

    def sc(self, fmt):
        return self.i("scm" if fmt >= 0 and fmt & MONT else "sc")

    def o(self, width, rows=N):
        if self.dev:
            import torch
            a = torch.full((rows, width), SENT, dtype=torch.uint8, device="cuda")
            self.outs.append(a)
            return C.c_void_p(a.data_ptr())
        a = np.full((rows, width), SENT, np.uint8)
        self.outs.append(a)
        return a.ctypes.data_as(C.c_void_p)

    def ho(self, width):
        """Host output (the multi-GPU calls return their sum in host memory)."""
        a = np.full((1, width), SENT, np.uint8)
        self.outs.append(a)
        return a.ctypes.data_as(C.c_void_p)

    def ow(self, fmt, rows=N):
        return self.o(32 if fmt >= 0 and fmt & ~MONT == 1 else 128, rows)

    def offsets(self, n):
        return self._place(np.arange(n + 1, dtype=np.uint32).view(np.uint8))

    def h(self):
        self.hv = C.c_void_p(HSENT)
        return C.byref(self.hv)

    def untouched(self):
        if self.dev:
            import torch
            torch.cuda.synchronize()
        return all(bool((a == SENT).all()) for a in self.outs) and (self.hv is None or self.hv.value == HSENT)


def _arr(ptr):
    return (C.c_void_p * 1)(ptr)


# name: (host form?, device form?, {word: (accepted, takes scalars)}, args(c, n, w), data pointers,
#        width argument index, handle destroyer)
# `w` maps each format-word name to its value; `n` is the batch size (segments for batch_msm).
SPECS = {
    "d377_batch_decompress": (True, True, {}, lambda c, n, w: [c.i("pt1"), n, c.o(128), c.o(1)], (0, 2), None, None),
    "d377_batch_compress": (True, True, {}, lambda c, n, w: [c.i("pt0"), n, c.o(32)], (0, 2), None, None),
    "d377_batch_decompress_fmt": (True, True, {"of": ((0, 2), False)},
                                  lambda c, n, w: [c.i("pt1"), n, w["of"], c.o(64 if w["of"] == 2 else 128), c.o(1)],
                                  (0, 3), None, None),
    "d377_batch_compress_fmt": (True, True, {"pf": ((0, 2, 3), False)},
                                lambda c, n, w: [c.pts(w["pf"]), w["pf"], n, c.o(32)], (0, 3), None, None),
    "d377_batch_encode_to_curve": (True, True, {"of": ((0, 1), False)},
                                   lambda c, n, w: [c.i("r"), n, c.ow(w["of"]), w["of"]], (0, 2), None, None),
    "d377_batch_encode_to_curve_wide": (True, True, {"of": ((0, 1), False)},
                                        lambda c, n, w: [c.i("r64"), 64, n, c.ow(w["of"]), w["of"]], (0, 3), 1, None),
    "d377_batch_hash_to_curve": (True, True, {"of": ((0, 1), False)},
                                 lambda c, n, w: [c.i("r"), c.i("r"), n, c.ow(w["of"]), w["of"]], (0, 1, 3), None,
                                 None),
    "d377_batch_hash_to_curve_wide": (True, True, {"of": ((0, 1), False)},
                                      lambda c, n, w: [c.i("r64"), c.i("r64"), 64, n, c.ow(w["of"]), w["of"]],
                                      (0, 1, 4), 2, None),
    "d377_fq_batch_from_le_bytes_mod_order": (True, True, {}, lambda c, n, w: [c.i("r64"), 64, n, c.o(32)], (0, 3), 1,
                                              None),
    "d377_batch_scalar_mul": (True, True, {"pf": ((0, 1, 2), True), "of": ((0, 1), False)},
                              lambda c, n, w: [c.pts(w["pf"]), w["pf"], c.sc(w["pf"]), n, c.ow(w["of"]), w["of"],
                                               c.o(1)], (0, 2, 4), None, None),
    "d377_fixed_base_mul": (True, True, {"of": ((0, 1), True)},
                            lambda c, n, w: [c.sc(w["of"]), n, c.ow(w["of"]), w["of"]], (0, 2), None, None),
    "d377_fixed_bases_mul": (True, True, {"of": ((0, 1), True)},
                             lambda c, n, w: [C.c_void_p(c.data["fixed"]), c.sc(w["of"]), n, c.ow(w["of"]), w["of"]],
                             (1, 3), None, None),
    "d377_batch_add": (True, True, {}, lambda c, n, w: [c.i("pt0"), c.i("pt0"), n, c.o(128)], (0, 1, 3), None, None),
    "d377_batch_sub": (True, True, {}, lambda c, n, w: [c.i("pt0"), c.i("pt0"), n, c.o(128)], (0, 1, 3), None, None),
    "d377_batch_neg": (True, True, {}, lambda c, n, w: [c.i("pt0"), n, c.o(128)], (0, 2), None, None),
    "d377_batch_double": (True, True, {}, lambda c, n, w: [c.i("pt0"), n, c.o(128)], (0, 2), None, None),
    "d377_batch_element_eq": (True, True, {}, lambda c, n, w: [c.i("pt0"), c.i("pt0"), n, c.o(1)], (0, 1, 3), None,
                              None),
    "d377_batch_on_curve": (True, True, {}, lambda c, n, w: [c.i("pt0"), n, 1, c.o(1)], (0, 3), None, None),
    "d377_element_sum": (True, True, {}, lambda c, n, w: [c.i("pt0"), n, c.o(128, 1), c.o(32, 1)], (0,), None, None),
    "d377_fq_batch_isqrt": (True, True, {}, lambda c, n, w: [c.i("fq"), n, c.o(32), c.o(1)], (0, 2, 3), None, None),
    "d377_fq_batch_sqrt_ratio_zeta": (True, True, {}, lambda c, n, w: [c.i("fq"), c.i("fq"), n, c.o(32), c.o(1)],
                                      (0, 1, 3, 4), None, None),
    "d377_field_batch_deserialize": (True, True, {"field": ((0, 1), False)},
                                     lambda c, n, w: [w["field"], c.i("fq"), n, c.o(32), c.o(1)], (1, 4), None, None),
    "d377_batch_normalize": (True, True, {}, lambda c, n, w: [c.i("pt0"), n, c.o(64)], (0, 2), None, None),
    "d377_batch_msm": (True, False, {"pf": ((0, 1, 2), True), "of": ((0, 1), False)},
                       lambda c, n, w: [c.sc(w["pf"]), c.pts(w["pf"]), w["pf"], c.offsets(n), n, c.ow(w["of"]),
                                        w["of"], c.o(1)], (0, 1, 3, 5), None, None),
    "d377_batch_msm_dev": (False, True, {"pf": ((0, 1, 2), True), "of": ((0, 1), False)},
                           lambda c, n, w: [c.sc(w["pf"]), c.pts(w["pf"]), w["pf"], c.offsets(n), n, n,
                                            c.ow(w["of"]), w["of"], c.o(1)], (0, 1, 3, 6), None, None),
    "d377_msm": (True, True, {"pf": ((0, 1, 2, 3, 4), True)},
                 lambda c, n, w: [c.sc(w["pf"]), c.pts(w["pf"]), w["pf"], n, c.o(128, 1), c.o(32, 1)], (0, 1), None,
                 None),
    "d377_msm_dev_async": (False, True, {"pf": ((0, 1, 2, 3, 4), True)},
                           lambda c, n, w: [c.sc(w["pf"]), c.pts(w["pf"]), w["pf"], n, c.o(128, 1), c.o(32, 1), 0],
                           (0, 1), None, None),
    "d377_msm_submit": (True, False, {"pf": ((0, 1, 2, 3, 4), True)},
                        lambda c, n, w: [c.sc(w["pf"]), c.pts(w["pf"]), w["pf"], n, 0], (0, 1), None, None),
    "d377_msm_multi": (True, False, {"pf": ((0, 1, 2, 3), True)},
                       lambda c, n, w: [c.sc(w["pf"]), c.pts(w["pf"]), w["pf"], n, 1, c.o(128, 1), c.o(32, 1)], (0, 1),
                       None, None),
    "d377_msm_multi_dev": (False, True, {"pf": ((0, 1, 2, 3), True)},
                           lambda c, n, w: [_arr(c.sc(w["pf"])), _arr(c.pts(w["pf"])), w["pf"], (C.c_size_t * 1)(n),
                                            1, c.ho(128), c.ho(32)], (), None,
                           None),
    "d377_msm_multi_dev_async": (False, True, {"pf": ((0, 1, 2, 3), True)},
                                 lambda c, n, w: [_arr(c.sc(w["pf"])), _arr(c.pts(w["pf"])), w["pf"],
                                                  (C.c_size_t * 1)(n), 1, c.o(128, 1), c.o(32, 1)], (), None, None),
    "d377_msm_bases_create": (True, True, {"pf": ((0, 1, 2, 3), False)},
                              lambda c, n, w: [c.pts(w["pf"]), w["pf"], n, c.h()], (0,), None, "d377_msm_bases_destroy"),
    "d377_msm_bases_create_windowed": (True, True, {"pf": ((0, 1, 2, 3), False)},
                                       lambda c, n, w: [c.pts(w["pf"]), w["pf"], n, 8, c.h()], (0,), None,
                                       "d377_msm_bases_destroy"),
    "d377_fixed_bases_create": (True, True, {"pf": ((0, 1, 2, 3), False)},
                                lambda c, n, w: [c.pts(w["pf"]), w["pf"], n, c.h()], (0,), None,
                                "d377_fixed_bases_destroy"),
}

# entry points that refuse n = 0 with null data pointers (k = 0 tables)
N0_REFUSED = {"d377_fixed_bases_create"}


def _forms():
    out = []
    for name, (host, dev, *_rest) in SPECS.items():
        if host:
            out.append((name, name, False))
        if dev:
            out.append((name, name if name.endswith(("_dev", "_async")) else name + "_dev", True))
    return out


FORMS = _forms()
IDS = [f[1] for f in FORMS]


def _call(lib, data, spec_name, fn_name, dev, n=N, words=None, null=(), patch=None):
    """One call; returns (rc, Call).  A call that succeeds is waited for and cleaned up."""
    _, _, slots, build, _, _, destroy = SPECS[spec_name]
    w = {k: v[0][0] for k, v in slots.items()}
    w.update(words or {})
    c = Call(data, dev)
    args = build(c, n, w)
    for k in null:
        args[k] = None
    for k, v in (patch or {}).items():
        args[k] = v
    rc = getattr(lib, fn_name)(*args)
    if rc == OK:
        if fn_name == "d377_msm_submit":
            assert lib.d377_msm_wait(0, None, None) == OK
        elif fn_name == "d377_msm_multi_dev_async":
            assert lib.d377_multi_sync() == OK
        if destroy and c.hv is not None:
            assert c.hv.value not in (None, HSENT)
            assert getattr(lib, destroy)(c.hv) == OK
        assert lib.d377_sync() == OK
    return rc, c


@pytest.fixture(scope="module")
def lib(engine):
    return _lib.load()


@pytest.mark.parametrize("spec,fn,dev", FORMS, ids=IDS)
def test_accepted_formats_succeed(lib, data, spec, fn, dev):
    slots = SPECS[spec][2]
    if not slots:
        assert _call(lib, data, spec, fn, dev)[0] == OK, (fn, lib.d377_last_error())
    for word, (acc, scalars) in slots.items():
        for v in _accepted(acc, scalars):
            rc, _ = _call(lib, data, spec, fn, dev, words={word: v})
            assert rc == OK, (fn, word, v, lib.d377_last_error())


@pytest.mark.parametrize("spec,fn,dev", [f for f in FORMS if SPECS[f[0]][2]], ids=[f[1] for f in FORMS if SPECS[f[0]][2]])
def test_refused_formats(lib, data, spec, fn, dev):
    """Every format word outside the accepted set is refused, before n = 0 is looked at,
    and leaves the outputs alone."""
    slots = SPECS[spec][2]
    for word, (acc, scalars) in slots.items():
        for v in _rejected(acc, scalars):
            for n in (N, 0):
                rc, c = _call(lib, data, spec, fn, dev, n=n, words={word: v})
                assert rc == INVALID, (fn, word, v, n, rc)
                assert c.untouched(), (fn, word, v, n)


@pytest.mark.parametrize("spec,fn,dev", FORMS, ids=IDS)
def test_null_pointers(lib, data, spec, fn, dev):
    """A null data pointer is refused when n > 0; with n = 0 the batch calls return D377_OK
    whatever their data pointers."""
    req = SPECS[spec][4]
    for k in req:
        rc, c = _call(lib, data, spec, fn, dev, null=(k,))
        assert rc == INVALID, (fn, k, rc)
        assert c.untouched(), (fn, k)
    rc, _ = _call(lib, data, spec, fn, dev, n=0, null=req)
    assert rc == (INVALID if spec in N0_REFUSED else OK), (fn, rc)


@pytest.mark.parametrize("spec,fn,dev", [f for f in FORMS if SPECS[f[0]][5] is not None],
                         ids=[f[1] for f in FORMS if SPECS[f[0]][5] is not None])
def test_input_width(lib, data, spec, fn, dev):
    at = SPECS[spec][5]
    for width in (0, 257):
        for n in (N, 0):
            rc, c = _call(lib, data, spec, fn, dev, n=n, patch={at: width})
            assert rc == INVALID, (fn, width, n, rc)
            assert c.untouched()
    for width in (1, 32, 64):
        assert _call(lib, data, spec, fn, dev, patch={at: width})[0] == OK


@pytest.mark.parametrize("spec,fn,dev", [f for f in FORMS if SPECS[f[0]][6]], ids=[f[1] for f in FORMS if SPECS[f[0]][6]])
def test_create_handle_slot(lib, data, spec, fn, dev):
    """The create calls refuse a null handle out-pointer even when n = 0; a plain or windowed
    set over no points is a valid (empty) set, a fixed-bases set needs k >= 1."""
    at = len(SPECS[spec][3](Call(data, dev), N, {"pf": 0})) - 1
    for n in (N, 0):
        assert _call(lib, data, spec, fn, dev, n=n, patch={at: None})[0] == INVALID
    rc, c = _call(lib, data, spec, fn, dev, n=0)
    assert rc == (INVALID if spec in N0_REFUSED else OK)
    if rc:
        assert c.untouched()


@pytest.mark.parametrize("fn,dev", [("d377_msm_bases_create_windowed", False),
                                    ("d377_msm_bases_create_windowed_dev", True)])
def test_window_width(lib, data, fn, dev):
    spec = "d377_msm_bases_create_windowed"
    for cw in (-1, 1, 3, 23, 64):
        for n in (N, 0):
            rc, c = _call(lib, data, spec, fn, dev, n=n, patch={3: cw})
            assert rc == INVALID and c.untouched(), (cw, n)
    for cw in (0, 4, 22):
        assert _call(lib, data, spec, fn, dev, patch={3: cw})[0] == OK


@pytest.mark.parametrize("fn,dev", [("d377_fixed_bases_mul", False), ("d377_fixed_bases_mul_dev", True)])
def test_foreign_fixed_bases_handle(lib, data, fn, dev):
    """A pointer that is not a live fixed-bases handle is refused before n = 0 is looked at,
    a prepared MSM set included."""
    for h in (None, HSENT, data["bases"]):
        for n in (N, 0):
            rc, c = _call(lib, data, "d377_fixed_bases_mul", fn, dev, n=n, patch={0: C.c_void_p(h)})
            assert rc == INVALID and c.untouched(), (h, n)


@pytest.mark.parametrize("fn,dev", [("d377_msm_multi_dev", True), ("d377_msm_multi_dev_async", True)])
def test_multi_pointer_arrays(lib, data, fn, dev):
    """Null pointer arrays are refused whatever n; a null slice pointer only with n > 0."""
    for k in (0, 1, 3):
        for n in (N, 0):
            rc, c = _call(lib, data, fn, fn, dev, n=n, null=(k,))
            assert rc == INVALID and c.untouched(), (k, n)
    for k in (0, 1):
        rc, c = _call(lib, data, fn, fn, dev, patch={k: _arr(None)})
        assert rc == INVALID and c.untouched(), k
        assert _call(lib, data, fn, fn, dev, n=0, patch={k: _arr(None)})[0] == OK


def test_msm_submit_slot(lib, data):
    for slot in (-1, 4):
        for n in (N, 0):
            assert _call(lib, data, "d377_msm_submit", "d377_msm_submit", False, n=n, patch={4: slot})[0] == INVALID
