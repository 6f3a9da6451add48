"""The quartic fixed-base kernel k_fixed_base_jq (scalar.cu) against the oracle, in every
per-thread variant and through each of its Edwards fallbacks.

fixed_base_mul(..., OUT_ENCODING) runs on the Jacobi quartic once the 1.6 GB quartic table
exists, or for a batch of at least 2^18 scalars.  The kernel then gives every thread 1, 4, 8
or 16 elements (n >= 2^16, 2^19, 2^22) that share one batched inversion, and recomputes on
the Edwards path every element whose scalar has a bit at or above 2^252, whose signed
21-bit recoding carries out of the 12th window, or whose quartic result the encoding
shortcut does not cover (Z = 0 on the way, S T Z = 0 at the end, s = +-1).  A fallback
element is left out of its thread's products; a slip in that bookkeeping leaves the
fallback element itself correct (it is recomputed) and breaks its good neighbours instead.

Which kernel runs depends on whether the table already exists in the process, so each half
runs in a fresh Python process: one that builds the table first and then runs every size
on the quartic kernel, and one that never reaches 2^18 scalars and so runs the same planted
scalars through the Edwards kernels k_fixed_base<true> and <false>.  The children write
their outputs to an .npz; the comparisons run here, so that a failure names the index and
the scalar.
"""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import decaf377_ref as o
from tests.test_jacobi_shortcuts_cpu import encoding_from_projective, inv, jq_dbl, jq_madd
from tests.util import canon

Q, R = o.Q, o.R
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK = 128                         # kCodecBlock
JQ_C, JQ_W, JQ_K = 21, 12, 1 << 20  # kJqC, kJqW, kJqK

# one size per per-thread variant <1>, <4>, <8>, <16>, each with a ragged last CTA
SIZES = [(1 << 16) - 3, (1 << 16) + 5, (1 << 19) + 7, (1 << 22) + 11]
EDWARDS_SIZES = SIZES[:2]           # below 2^18: the quartic table is never built
HOST_N = (1 << 19) + 7              # host-buffer entry: chunks of 2^18 and a ragged last one
FULL_ORACLE_MAX = (1 << 16) + 5     # every element against the oracle up to this size
ORACLE_SAMPLE = 4096

# ---- planted scalars -------------------------------------------------------------------------
# S = 0 at the end: G_J has order 2r, r G_J = 3r G_J = (0, -1) is the kernel point of the
# isogeny and 0 G_J = 2r G_J = (0, 1) the quartic identity
S_ZERO = [0, R, 2 * R, 3 * R]
# below 2^252, but the signed recoding carries out of the top window
CARRY = [(1 << 252) - 1, (1 << 251) + (1 << 231) + 1]
# a bit at or above 2^252: not covered by 12 windows
TOP_BIT = [1 << 252, (1 << 252) + 5, (1 << 256) - 1]
FALLBACK = S_ZERO + CARRY + TOP_BIT
# digits at their extremes, on the quartic path
EXTREMES = [
    sum(JQ_K << (JQ_C * w) for w in range(JQ_W)),                         # every digit +2^20: last entry
    (JQ_K + 1) + sum(JQ_K << (JQ_C * w) for w in range(1, JQ_W - 1)),     # -(2^20 - 1) in windows 0..10
    sum((JQ_K + 1) << (JQ_C * w) for w in range(JQ_W - 1)),               # -(2^20 - 1), then -(2^20 - 2)
    sum((-1) ** (w + 1) << (JQ_C * w) for w in range(JQ_W)),              # -1, +1, -1, ..., +1
    sum((-1) ** w << (JQ_C * w) for w in range(JQ_W - 1)),                # +1, -1, ..., +1, 0
]
BOUNDARY = [1, 2, R - 1, R - 2, (R - 1) // 2] + \
    [(1 << (JQ_C * k)) + d for k in range(1, JQ_W) for d in (-1, 1)]
EDGES = FALLBACK + EXTREMES + BOUNDARY


def per_thread(n):
    """Elements per thread of k_fixed_base_jq for a launch of n scalars (launch_fixed_base)."""
    return 16 if n >= 1 << 22 else 8 if n >= 1 << 19 else 4 if n >= 1 << 16 else 1


def slot_index(n, b, lane, e):
    """Index of element e of thread `lane` of CTA b."""
    return (b * per_thread(n) + e) * BLOCK + lane


def thread_indices(n, i):
    """Every in-range index of the thread that holds element i."""
    p = per_thread(n)
    b, lane = i // (p * BLOCK), i % BLOCK
    return [j for j in (slot_index(n, b, lane, e) for e in range(p)) if j < n]


@functools.lru_cache(maxsize=None)
def planted_batch(n):
    """Random canonical scalars with the edge scalars planted; returns (scalars, {index: k})."""
    p = per_thread(n)
    rng = np.random.default_rng(n)
    sc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x03                                   # < 2^250 < r
    planted = {}

    def plant(i, k):
        planted[i] = k
        sc[i] = np.frombuffer(k.to_bytes(32, "little"), np.uint8)

    # index 0 is what the padding lanes of the ragged last CTA re-read: a carry scalar makes
    # them fallback elements beside the good elements of the last threads
    plant(0, CARRY[1])
    plant(n - 1, TOP_BIT[2])
    # every slot of one thread: the edge list in order
    for e in range(p):
        plant(slot_index(n, 1, 5, e), EDGES[e % len(EDGES)])
    # the only fallback element in the last slot, good elements below it: the reverse walk
    # must leave it out of the running inverse (a carry and a top-bit scalar; with S = 0 a
    # slip would only zero the neighbours' inverse, and they would recompute correctly)
    plant(slot_index(n, 2, 77, p - 1), CARRY[1])
    plant(slot_index(n, 2, 78, p - 1), TOP_BIT[1])
    # one thread of nothing but fallback elements
    for e in range(p):
        plant(slot_index(n, 3, 100, e), FALLBACK[e % len(FALLBACK)])
    # lanes 0 and 31 of a warp
    plant(slot_index(n, 4, 32, 0), S_ZERO[1])
    plant(slot_index(n, 4, 63, 0), CARRY[0])
    # every edge scalar once more, each in its own thread among random neighbours
    for j, k in enumerate(EDGES):
        plant(slot_index(n, 8 + j, (37 * j) % BLOCK, j % p), k)
    return sc, planted


def _int(row):
    return int.from_bytes(row.tobytes(), "little")


@functools.lru_cache(maxsize=None)
def _full_oracle(n):
    sc, _ = planted_batch(n)
    return co.fixed_base(sc, out_enc=True, threads=co.threads_default())


def _oracle_indices(n):
    """Planted indices, every index of their threads, a strided sample; all for small n."""
    if n <= FULL_ORACLE_MAX:
        return np.arange(n)
    _, planted = planted_batch(n)
    idx = set(np.linspace(0, n - 1, ORACLE_SAMPLE, dtype=np.int64).tolist())
    for i in planted:
        idx.update(thread_indices(n, i))
    return np.array(sorted(idx))


def _assert_matches_oracle(n, got, idx, what):
    sc, planted = planted_batch(n)
    want = _full_oracle(n)[idx] if n <= FULL_ORACLE_MAX else \
        co.fixed_base(sc[idx], out_enc=True, threads=co.threads_default())
    bad = np.nonzero((got[idx] != want).any(axis=1))[0]
    if len(bad):
        i = int(idx[bad[0]])
        pytest.fail("%s, n = %d: %d of %d checked elements differ from the oracle; first at index %d "
                    "(scalar %#x%s)" % (what, n, len(bad), len(idx), i, _int(sc[i]),
                                        ", planted" if i in planted else ""))


def _run_child(script, path):
    r = subprocess.run([sys.executable, "-c", script % ROOT, str(path)], capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    return np.load(path)


# ---- CPU: the planted scalars and the oracle they are checked against ------------------------
def _model_fallback(k):
    """k_fixed_base_jq's decision for one scalar, restated with Python integers: True where
    the kernel recomputes the element on the Edwards path."""
    G = o.decompress((8).to_bytes(32, "little"))
    sG, tG = 8, 65 * inv(o.to_affine(G)[1]) % Q
    bases, P = [], (sG, tG, 1)
    for _ in range(JQ_W):
        iz = inv(P[2])
        bases.append((P[0] * iz % Q, P[1] * iz * iz % Q))
        for _ in range(JQ_C):
            P = jq_dbl(P)

    def entry(w, m):
        acc = (0, 1, 1)
        for i in reversed(range(JQ_C)):
            acc = jq_dbl(acc)
            if (m >> i) & 1:
                acc = jq_madd(acc, *bases[w])
        iz = inv(acc[2])
        return acc[0] * iz % Q, acc[1] * iz * iz % Q

    acc, carry, bad = (0, 1, 1), 0, k >> 252 != 0
    for w in range(JQ_W):
        raw = ((k >> (JQ_C * w)) & ((1 << JQ_C) - 1)) + carry
        carry = 1 if raw > JQ_K else 0
        d = raw - (carry << JQ_C)
        s2, t2 = (0, 1) if d == 0 else entry(w, abs(d))
        acc = jq_madd(acc, s2 if d >= 0 else (-s2) % Q, t2)
        bad = bad or acc[2] == 0
    bad = bad or carry != 0
    if not bad:
        enc = encoding_from_projective(*acc)
        if enc is not None:
            assert enc == o.compress_to_field(o.scalar_mul(o.GENERATOR, k)), hex(k)
    return bad or encoding_from_projective(*acc) is None


def test_planted_scalars_take_the_paths_they_are_planted_for():
    """Each fallback scalar makes the quartic kernel fall back, for the reason it is listed
    under; every other edge scalar stays on the quartic path and its quartic encoding is the
    oracle's.  The C oracle, which the GPU tests compare with, agrees with the Python oracle
    on every one of them, canonical or not."""
    for k in S_ZERO:
        assert k < 1 << 252 and _model_fallback(k), hex(k)
    for k in CARRY:
        assert k < 1 << 252 and _model_fallback(k), hex(k)
    for k in TOP_BIT:
        assert k >> 252 and _model_fallback(k), hex(k)
    for k in EXTREMES + BOUNDARY:
        assert not _model_fallback(k), hex(k)
    got = co.fixed_base(canon(EDGES), out_enc=True, threads=4)
    for i, k in enumerate(EDGES):
        assert got[i].tobytes() == o.compress(o.scalar_mul(o.GENERATOR, k)), hex(k)


def test_placement_covers_every_slot_and_the_edges_of_threads():
    for n in SIZES:
        p = per_thread(n)
        _, planted = planted_batch(n)
        assert 0 in planted and n - 1 in planted
        assert {i for i in planted if planted[i] in CARRY + TOP_BIT and
                (i // BLOCK) % p == p - 1 and
                all(j not in planted for j in thread_indices(n, i) if j != i)}, n
        whole = thread_indices(n, slot_index(n, 3, 100, 0))
        assert len(whole) == p and all(planted[j] in FALLBACK for j in whole)
        assert len(thread_indices(n, slot_index(n, 1, 5, 0))) == p
        assert n % (p * BLOCK) != 0                      # a ragged last CTA


# ---- GPU: the quartic kernel, table built first -------------------------------------------------
_QUARTIC_CHILD = r"""
import sys, numpy as np, torch
sys.path.insert(0, %r)
import decaf377_b200 as d
from decaf377_b200 import device as dev
from tests.test_gpu_quartic_paths import HOST_N, SIZES, planted_batch
d.init(0)
torch.cuda.synchronize()
free0, _ = torch.cuda.mem_get_info()
warm = torch.from_numpy(planted_batch(1 << 18)[0]).cuda()
dev.fixed_base_mul(warm, d.OUT_ENCODING)                # 2^18 scalars: builds the quartic table
torch.cuda.synchronize()
free1, _ = torch.cuda.mem_get_info()
out = {"grew_mib": np.int64((free0 - free1) >> 20)}
del warm
for n in SIZES:
    sc, _ = planted_batch(n)
    x = torch.from_numpy(sc).cuda()
    out["enc%%d" %% n] = dev.fixed_base_mul(x, d.OUT_ENCODING).cpu().numpy()
    out["elc%%d" %% n] = dev.compress(dev.fixed_base_mul(x, d.OUT_ELEMENT)).cpu().numpy()
    if n == HOST_N:
        out["host%%d" %% n] = d.fixed_base_mul(sc, d.OUT_ENCODING)
    del x
np.savez(sys.argv[1], **out)
"""


@pytest.fixture(scope="module")
def quartic_outputs(tmp_path_factory):
    return _run_child(_QUARTIC_CHILD, tmp_path_factory.mktemp("quartic") / "out.npz")


@pytest.mark.gpu
def test_quartic_table_is_built_before_the_checked_calls(quartic_outputs):
    grew = int(quartic_outputs["grew_mib"])
    assert grew > 1500, "a 2^18-scalar call should have built the 1.6 GB quartic table (%d MiB)" % grew


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_quartic_fixed_base_matches_element_path_and_oracle(quartic_outputs, n):
    sc, _ = planted_batch(n)
    enc, elc = quartic_outputs["enc%d" % n], quartic_outputs["elc%d" % n]
    assert enc.shape == (n, 32)
    # every element against the Edwards element kernel (it never reads the quartic table)
    diff = np.nonzero((enc != elc).any(axis=1))[0]
    assert not len(diff), "n = %d: %d elements differ from compress(OUT_ELEMENT); first at %d (scalar %#x)" \
        % (n, len(diff), diff[0], _int(sc[diff[0]]))
    _assert_matches_oracle(n, enc, _oracle_indices(n), "quartic kernel <%d>" % per_thread(n))


@pytest.mark.gpu
def test_quartic_host_buffer_entry_matches_device_entry(quartic_outputs):
    """fixed_base_mul over host buffers cuts 2^19 + 7 scalars into chunks of 2^18 and a ragged
    7, each launched with its own per-thread variant; the bytes are those of one launch."""
    host, dev_ = quartic_outputs["host%d" % HOST_N], quartic_outputs["enc%d" % HOST_N]
    diff = np.nonzero((host != dev_).any(axis=1))[0]
    assert not len(diff), "%d elements differ; first at %d" % (len(diff), diff[0])


# ---- GPU: the Edwards kernels, table never built --------------------------------------------------
_EDWARDS_CHILD = r"""
import sys, numpy as np, torch
sys.path.insert(0, %r)
import decaf377_b200 as d
from decaf377_b200 import device as dev
from tests.test_gpu_quartic_paths import EDWARDS_SIZES, planted_batch
d.init(0)
torch.cuda.synchronize()
free0, _ = torch.cuda.mem_get_info()
out = {}
for n in EDWARDS_SIZES:
    x = torch.from_numpy(planted_batch(n)[0]).cuda()
    out["enc%%d" %% n] = dev.fixed_base_mul(x, d.OUT_ENCODING).cpu().numpy()
    out["el%%d" %% n] = dev.fixed_base_mul(x, d.OUT_ELEMENT).cpu().numpy()
torch.cuda.synchronize()
free1, _ = torch.cuda.mem_get_info()
out["grew_mib"] = np.int64((free0 - free1) >> 20)
np.savez(sys.argv[1], **out)
"""


@pytest.fixture(scope="module")
def edwards_outputs(tmp_path_factory):
    return _run_child(_EDWARDS_CHILD, tmp_path_factory.mktemp("edwards") / "out.npz")


@pytest.mark.gpu
@pytest.mark.parametrize("n", EDWARDS_SIZES)
def test_edwards_fixed_base_planted_scalars_match_oracle(edwards_outputs, n):
    grew = int(edwards_outputs["grew_mib"])
    assert grew < 512, "calls below 2^18 scalars grew device memory by %d MiB" % grew
    _assert_matches_oracle(n, edwards_outputs["enc%d" % n], np.arange(n), "k_fixed_base<true>")
    # the element output, compressed by the C oracle
    elc = co.compress(edwards_outputs["el%d" % n], threads=co.threads_default())
    _assert_matches_oracle(n, elc, np.arange(n), "k_fixed_base<false>")
