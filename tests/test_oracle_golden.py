"""The CPU oracle (oracle/hnsw_oracle.c) against the fixtures generated FROM the compiled
reference (tests/golden/make_golden.py) and against the reference itself on fresh random inputs
(its outputs replayed from tests/golden/reference_replay/, see helpers.ReferenceReplay)."""
import ctypes as C

import numpy as np
import pytest

from helpers import GOLDEN_CASES, golden_key, reference  # noqa: F401  (reference: fixture)
from leann_b200.csr import read_compact_index
from oracle.binding import HERE, Oracle, Reference


@pytest.fixture(scope="module")
def fx(golden_dir):
    return dict(x=np.load(golden_dir / "hnsw_small_vectors.npy"), q=np.load(golden_dir / "hnsw_small_queries.npy"),
                exp=np.load(golden_dir / "hnsw_small_expected.npz"),
                g={t: read_compact_index(str(golden_dir / f"hnsw_small_{t}.index")) for t in ("ip", "l2")})


@pytest.mark.parametrize("tag", ["ip", "l2"])
@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_oracle_matches_reference_golden(fx, tag, case):
    ef, beam, batch, cr, k = case
    D, I, ndis, nhops = Oracle(fx["g"][tag], fx["x"]).search(fx["q"], k, ef=ef, beam=beam, batch_size=batch, check_rel=bool(cr))
    key = golden_key(tag, *case)
    assert np.array_equal(I, fx["exp"][key + "_I"])
    assert np.array_equal(D, fx["exp"][key + "_D"])  # bit-exact: same canonical summation order
    assert np.array_equal(ndis, fx["exp"][key + "_ndis"])
    assert np.array_equal(nhops, fx["exp"][key + "_nhops"])


def test_golden_has_distance_ties(fx):
    # the fixture plants duplicate vectors so that the tie rules of pop_min / the heaps are exercised
    D = fx["exp"][golden_key("ip", 64, 1, 0, 1, 10) + "_D"]
    assert any(len(np.unique(row)) < len(row) for row in D)


@pytest.mark.parametrize("metric_ip", [True, False])
def test_oracle_vs_compiled_reference_random(metric_ip, reference):
    rng = np.random.default_rng(7)
    n, d = 3000, 48
    x = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((40, d)).astype(np.float32)
    R = reference.proxy(Reference, d, M=8, metric_ip=metric_ip)
    R.build(x, ef_construction=40, nthreads=1)
    from oracle.binding import export_to_csr
    g = export_to_csr(R.export())
    O = Oracle(g, x)
    for (ef, beam, batch, cr, k) in [(64, 1, 0, 1, 10), (20, 3, 0, 1, 5), (40, 1, 50, 1, 10), (10, 2, 0, 0, 30)]:
        a = R.search(q, k, ef=ef, beam=beam, batch_size=batch, check_rel=bool(cr))
        b = O.search(q, k, ef=ef, beam=beam, batch_size=batch, check_rel=bool(cr))
        for u, v in zip(a, b):
            assert np.array_equal(u, v)


@pytest.mark.parametrize("seed", range(10))
def test_oracle_vs_compiled_reference_fuzz(seed, reference):
    """Randomised shapes and search parameters, on purpose degenerate: integer-valued coordinates (many exactly equal
    distances -> every tie-break of the heaps, the beam and the result handler matters), duplicate vectors, k above and below
    efSearch, more results requested than nodes reachable, beam / batch modes, both metrics, the relative-distance stop rule on
    and off.  The C restatement must return the compiled reference's ids, distances, ndis and nhops exactly."""
    from oracle.binding import export_to_csr
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.choice([12, 60, 400, 1500]))
    d = int(rng.choice([4, 16, 33]))
    M = int(rng.choice([4, 8, 16]))
    metric_ip = bool(rng.integers(0, 2))
    x = rng.integers(-3, 4, (n, d)).astype(np.float32)
    x[rng.integers(0, n, n // 10 + 1)] = x[0]                      # exact duplicates of one vector
    q = np.concatenate([rng.integers(-3, 4, (12, d)), x[:4]]).astype(np.float32)   # some queries ARE data points
    R = reference.proxy(Reference, d, M=M, metric_ip=metric_ip)
    R.build(x, ef_construction=int(rng.choice([16, 40])), nthreads=1)
    O = Oracle(export_to_csr(R.export()), x)
    for _ in range(5):
        ef = int(rng.choice([1, 3, 10, 32, 64]))
        beam = int(rng.choice([1, 1, 2, 5]))
        batch = int(rng.choice([0, 0, 7, 40]))
        cr = bool(rng.integers(0, 2))
        k = int(rng.choice([1, 5, 10, 40]))
        a = R.search(q, k, ef=ef, beam=beam, batch_size=batch, check_rel=cr)
        b = O.search(q, k, ef=ef, beam=beam, batch_size=batch, check_rel=cr)
        for name, u, v in zip(("D", "I", "ndis", "nhops"), a, b):
            assert np.array_equal(u, v), (name, dict(n=n, d=d, M=M, ip=metric_ip, ef=ef, beam=beam, batch=batch, cr=cr, k=k))


class MinimaxHeap:
    """The MinimaxHeap entry points of the compiled reference (which="ref": ref_mmh_* of oracle/_ref/libleann_ref.so) or
    of the C restatement (which="oracle": lbo_mmh_* of oracle/liboracle.so)."""

    def __init__(self, which):
        lib, prefix = {"ref": (HERE / "_ref" / "libleann_ref.so", "ref_mmh_"), "oracle": (HERE / "liboracle.so", "lbo_mmh_")}[which]
        lib = C.CDLL(str(lib))
        self.f = {f: getattr(lib, prefix + f) for f in ("new", "push", "pop_min", "count_below", "size", "free")}
        self.f["new"].restype = C.c_void_p
        for f, a in {"push": [C.c_void_p, C.c_int, C.c_float], "pop_min": [C.c_void_p, C.POINTER(C.c_float)],
                     "count_below": [C.c_void_p, C.c_float], "size": [C.c_void_p], "free": [C.c_void_p]}.items():
            self.f[f].argtypes = a

    def new(self, cap):
        return self.f["new"](cap)

    def push(self, h, i, v):
        self.f["push"](h, i, v)

    def pop_min(self, h):
        v = C.c_float()
        return self.f["pop_min"](h, C.byref(v)), v.value

    def count_below(self, h, t):
        return self.f["count_below"](h, t)

    def size(self, h):
        return self.f["size"](h)

    def free(self, h):
        self.f["free"](h)


def test_minimax_heap_vs_reference(reference):
    """Random push / pop_min / count_below traces incl. equal and infinite distances
    (shape of faiss/tests/test_hnsw.cpp:20-195)."""
    ref = reference.proxy(MinimaxHeap, "ref")
    ora = MinimaxHeap("oracle")
    rng = np.random.default_rng(3)
    for trial in range(30):
        cap = int(rng.integers(1, 40))
        hr, ho = ref.new(cap), ora.new(cap)
        vals = np.concatenate([rng.integers(0, 8, 200).astype(np.float32), [np.inf] * 5])
        for step in range(400):
            op = rng.random()
            if op < 0.6:
                i, v = int(rng.integers(0, 1000)), float(rng.choice(vals))
                ref.push(hr, i, v); ora.push(ho, i, v)
            elif op < 0.85:
                if ref.size(hr) > 0:
                    assert ref.pop_min(hr) == ora.pop_min(ho)
            else:
                t = float(rng.choice(vals))
                assert ref.count_below(hr, t) == ora.count_below(ho, t)
            assert ref.size(hr) == ora.size(ho)
        ref.free(hr); ora.free(ho)
