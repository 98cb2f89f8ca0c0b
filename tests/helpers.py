"""Shared helpers of the test-suite (test infrastructure; may use oracle/)."""
from __future__ import annotations

import glob
import hashlib
import json
import os
import tempfile
from pathlib import Path

import numpy as np
import pytest

from leann_b200 import csr, synth

GOLDEN_CASES = [  # (ef, beam, batch, check_rel, k) — keep in sync with tests/golden/make_golden.py
    (64, 1, 0, 1, 10), (16, 1, 0, 1, 10), (8, 1, 0, 1, 20), (32, 4, 0, 1, 10), (32, 16, 0, 1, 5),
    (32, 1, 24, 1, 10), (24, 2, 0, 0, 10), (128, 1, 0, 1, 1), (64, 3, 40, 0, 7),
]


def golden_key(tag, ef, beam, batch, cr, k):
    return f"{tag}_ef{ef}_b{beam}_bs{batch}_cr{cr}_k{k}"


from leann_b200.tooling import open_encoder_only, recall_at_k, stub_graph, write_leann_index  # noqa: E402,F401


VAMANA_GOLDEN_CASES = [(64, 1, 10), (32, 4, 5), (16, 2, 10), (100, 2, 10)]  # keep in sync with tests/golden/make_vamana_golden.py


def load_vamana_golden(golden_dir, metric):
    """The committed DiskANN-format fixture, read back with the format readers (not the builder)."""
    from leann_b200 import diskann_format as dfmt

    prefix = str(golden_dir / f"vamana_small_{metric}")
    coords, g = dfmt.read_disk_index(prefix + "_disk.index")
    pq = dfmt.read_pq_pivots(prefix + "_pq_pivots.bin")
    codes = dfmt.read_bin(prefix + "_pq_compressed.bin", np.uint8)
    mx = float(dfmt.read_bin(prefix + "_disk.index_max_base_norm.bin", np.float32)[0, 0]) if metric == "mips" else 0.0
    g.medoid = int(dfmt.read_bin(prefix + "_disk.index_medoids.bin", np.uint32)[0, 0])
    return dict(prefix=prefix, g=g, coords=coords, pq=pq, codes=codes, max_norm=mx,
                emb=np.load(golden_dir / "vamana_small_emb.npy"), q=np.load(golden_dir / "vamana_small_queries.npy"),
                exp=np.load(golden_dir / "vamana_small_expected.npz"))


def load_c1(golden_dir, n_queries=40, seed=5):
    """BASELINE config C1 (the reference's sample document) as a synth.Corpus: 254-token chunks at stride 127, each wrapped in
    [CLS]=101 / [SEP]=102, plus queries = random 12..30-token spans of the same text (wrapped the same way)."""
    stream = np.load(golden_dir / "c1_pride_tokens.npz")["tokens"]
    starts = np.arange(0, max(1, len(stream) - 127), 127)
    toks, offs = [], [0]
    for s in starts:
        body = stream[s:s + 254]
        toks.append(np.concatenate([[101], body, [102]]).astype(np.uint16))
        offs.append(offs[-1] + len(toks[-1]))
    corpus = synth.Corpus(np.concatenate(toks), np.asarray(offs, np.uint64), np.zeros(len(starts), np.int32))
    rng = np.random.default_rng(seed)
    qt, qo = [], [0]
    for _ in range(n_queries):
        a = int(rng.integers(0, len(stream) - 40))
        body = stream[a:a + int(rng.integers(12, 31))]
        qt.append(np.concatenate([[101], body, [102]]).astype(np.uint16))
        qo.append(qo[-1] + len(qt[-1]))
    queries = synth.Corpus(np.concatenate(qt), np.asarray(qo, np.uint64), np.zeros(n_queries, np.int32))
    return corpus, queries


# ---------------------------------------------------------------------------------------------------------------------
# The compiled reference (oracle/_ref/, built from the original project's sources, which are not part of this repository)
# recorded once and replayed in every run of the suite.
REPLAY_DIR = Path(__file__).resolve().parent / "golden" / "reference_replay"


def _digest(h, obj):
    """Feeds the value of a call argument into h.  A string naming a path prefix stands for the contents of the files
    that start with it (index prefixes, PQ files written into a temporary directory)."""
    if isinstance(obj, _Proxy):
        h.update(b"P" + obj._token.encode())
    elif isinstance(obj, np.ndarray):
        a = np.ascontiguousarray(obj)
        h.update(f"A{a.dtype.str}{a.shape}".encode() + a.tobytes())
    elif isinstance(obj, (list, tuple)):
        h.update(b"L%d" % len(obj))
        for o in obj:
            _digest(h, o)
    elif isinstance(obj, dict):
        for k in sorted(obj):
            h.update(b"K" + str(k).encode())
            _digest(h, obj[k])
    elif isinstance(obj, (str, Path)) and os.sep in str(obj):
        for f in sorted(glob.glob(glob.escape(str(obj)) + "*")):
            h.update(b"F" + f[len(str(obj)):].encode() + Path(f).read_bytes())
    elif obj is None or isinstance(obj, (str, bool, int, float, np.generic)):
        h.update(b"S" + repr(obj).encode())
    elif hasattr(obj, "__dict__"):                       # CSRGraph, PQTable, ... : their fields
        h.update(b"O" + type(obj).__name__.encode())
        _digest(h, {k: v for k, v in vars(obj).items() if not k.startswith("_")})
    else:
        raise TypeError(f"cannot digest a {type(obj).__name__} argument")


class _Proxy:
    """An object the reference returned (a handle, a queue): method calls on it go through the replay too."""

    def __init__(self, rr, live, token):
        self._rr, self._live, self._token = rr, live, token

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        fn = getattr(self._live, name) if self._live is not None else None
        return lambda *a, **kw: self._rr._call(f"{self._token}.{name}", fn, a, kw)


def _bulk(obj) -> bool:
    """An argument worth checking call by call: an array, files, or a structure holding arrays (not a scalar or a handle)."""
    if isinstance(obj, (list, tuple)):
        return any(_bulk(o) for o in obj)
    if isinstance(obj, dict):
        return any(_bulk(o) for o in obj.values())
    return isinstance(obj, np.ndarray) or (isinstance(obj, (str, Path)) and os.sep in str(obj)) or \
        (hasattr(obj, "__dict__") and not isinstance(obj, _Proxy))


class ReferenceReplay:
    """Stands in for the compiled reference in a test that compares against it.

    Every call the test makes on the reference is replayed, in order, from tests/golden/reference_replay/<module>.npz:
    its outputs are the reference's, stored when the call was recorded.  A running digest covers the inputs of all calls;
    it is checked at every call that takes arrays or files and at the end of the test, so a replayed call whose inputs
    differ from the recorded ones (the test, or the data it builds, changed) fails instead of passing on stale outputs.
    With LEANN_RECORD_REFERENCE=1 and oracle/_ref/ built, the calls go to the compiled reference and are recorded
    (tests/golden/make_reference_replay.py)."""

    def __init__(self, module: str, test: str):
        self.path, self.test = REPLAY_DIR / f"{module}.npz", test
        self.record = os.environ.get("LEANN_RECORD_REFERENCE") == "1"
        self.h = hashlib.sha1()
        self.n_obj = 0
        self.cursor = dict(i=0, f=0, a=0, d=0)
        if self.record:
            self.calls, self.dig, self.ints, self.floats, self.arrays, self.uniq, self.seen = [], [], [], [], [], [], {}
            return
        if not self.path.exists() or f"{test}/calls" not in np.load(self.path).files:
            raise AssertionError(f"no recorded reference outputs for {test} in {self.path} (see tests/golden/make_reference_replay.py)")
        z = np.load(self.path)
        self.calls = json.loads(z[f"{test}/calls"].tobytes())
        self.dig = z[f"{test}/digests"]
        self.ints, self.floats = z[f"{test}/ints"], z[f"{test}/floats"]
        self.bufs = {k[len(test) + 5:]: z[k] for k in z.files if k.startswith(f"{test}/buf:")}
        self.offsets, self.final = z[f"{test}/offsets"], int(z[f"{test}/final"])
        self.i = 0

    def proxy(self, factory, *args, **kw):
        """factory(*args, **kw) — a reference class, classmethod or function — through the replay."""
        return self._call(factory.__qualname__, factory if self.record else None, args, kw)

    def _d16(self):
        return int.from_bytes(self.h.digest()[:2], "little")

    def _call(self, name, fn, args, kw):
        self.h.update(b"C" + name.encode())
        _digest(self.h, (args, kw))
        bulk = _bulk((args, kw))
        if self.record:
            unwrap = lambda v: v._live if isinstance(v, _Proxy) else v  # noqa: E731
            out = fn(*[unwrap(a) for a in args], **{k: unwrap(v) for k, v in kw.items()})
            struct, value = self._encode(out)
            self.calls.append([name, struct])
            if bulk:
                self.dig.append(self._d16())
            return value
        i, self.i = self.i, self.i + 1
        ok = i < len(self.calls) and self.calls[i][0] == name
        if ok and bulk:
            ok = self.cursor["d"] < len(self.dig) and int(self.dig[self.cursor["d"]]) == self._d16()
            self.cursor["d"] += 1
        assert ok, f"{self.test}: reference call #{i} ({name}) is not the recorded one; record the reference outputs again"
        return self._decode(self.calls[i][1])

    def finish(self):
        if self.record:
            self.save()
            return
        assert self.i == len(self.calls), f"{self.test}: {len(self.calls) - self.i} recorded reference calls were not made"
        assert int.from_bytes(self.h.digest()[:8], "little", signed=True) == self.final, \
            f"{self.test}: the inputs of the reference calls are not the recorded ones; record the reference outputs again"

    def _encode(self, v):
        """(structure, value handed to the test).  Scalars and arrays are stored in call order, so the structure holds only
        their kinds; an array equal to one stored before is stored once."""
        if isinstance(v, (bool, int, np.integer, np.bool_)):
            b = isinstance(v, (bool, np.bool_))
            self.ints.append(int(v))
            return ("b" if b else "i"), (bool(v) if b else int(v))
        if isinstance(v, (float, np.floating)) and not isinstance(v, np.float32):
            self.floats.append(float(v))
            return "f", float(v)
        if isinstance(v, (np.ndarray, np.float32)):
            a = np.ascontiguousarray(v)
            key = (a.dtype.str, a.shape, hashlib.sha1(a.tobytes()).digest())
            if key not in self.seen:
                self.seen[key] = len(self.uniq)
                self.uniq.append(a)
            self.arrays.append(self.seen[key])
            return ["a", a.dtype.str, list(a.shape)], v
        if v is None or isinstance(v, str):
            return ["s", v], v
        if isinstance(v, (list, tuple, dict)):
            keys = list(v) if isinstance(v, dict) else None
            enc = [self._encode(x) for x in (v.values() if keys is not None else v)]
            s, vals = [e[0] for e in enc], [e[1] for e in enc]
            if keys is not None:
                return ["d", keys, s], dict(zip(keys, vals))
            return ["t" if isinstance(v, tuple) else "l", s], (tuple(vals) if isinstance(v, tuple) else vals)
        self.n_obj += 1
        p = _Proxy(self, v, f"o{self.n_obj}")
        return ["o", p._token], p

    def _next(self, kind):
        j = self.cursor[kind]
        self.cursor[kind] += 1
        return j

    def _decode(self, s):
        if s in ("i", "b"):
            v = int(self.ints[self._next("i")])
            return bool(v) if s == "b" else v
        if s == "f":
            return float(self.floats[self._next("f")])
        kind = s[0]
        if kind == "a":
            ds, shape = s[1], s[2]
            o = int(self.offsets[self._next("a")])
            a = self.bufs[ds][o:o + int(np.prod(shape))].astype(np.dtype(ds)).reshape(shape)
            return a if shape else a[()]
        if kind == "s":
            return s[1]
        if kind == "d":
            return {k: self._decode(x) for k, x in zip(s[1], s[2])}
        if kind in ("t", "l"):
            vals = [self._decode(x) for x in s[1]]
            return tuple(vals) if kind == "t" else vals
        return _Proxy(self, None, s[1])

    def save(self):
        """Record mode: replaces this test's entries in the module's file.  Arrays of one dtype are stored end to end in
        one buffer, integers in the narrowest type that holds them."""
        z = dict(np.load(self.path)) if self.path.exists() else {}
        z = {k: v for k, v in z.items() if not k.startswith(self.test + "/")}
        groups, start, filled = {}, [], {}
        for a in self.uniq:
            start.append(filled.get(a.dtype.str, 0))
            filled[a.dtype.str] = start[-1] + a.size
            groups.setdefault(a.dtype.str, []).append(a.ravel())
        for ds, g in groups.items():
            b = np.concatenate(g)
            if b.dtype.kind in "iu" and b.size:
                b = b.astype(next(t for t in (np.int8, np.uint8, np.int16, np.uint16, np.int32, np.uint32, np.int64, np.uint64)
                                  if np.iinfo(t).min <= b.min() and b.max() <= np.iinfo(t).max))
            z[f"{self.test}/buf:{ds}"] = b
        z[f"{self.test}/offsets"] = np.asarray([start[u] for u in self.arrays], np.int64)
        z[f"{self.test}/calls"] = np.frombuffer(json.dumps(self.calls, separators=(",", ":")).encode(), np.uint8)
        z[f"{self.test}/digests"] = np.asarray(self.dig, np.uint16)
        z[f"{self.test}/final"] = np.int64(int.from_bytes(self.h.digest()[:8], "little", signed=True))
        z[f"{self.test}/ints"] = np.asarray(self.ints, np.int64)
        z[f"{self.test}/floats"] = np.asarray(self.floats, np.float64)
        REPLAY_DIR.mkdir(exist_ok=True)
        np.savez_compressed(self.path, **z)


@pytest.fixture
def reference(request):
    """The compiled reference, replayed (see ReferenceReplay); keyed by test module and test name with its parameters."""
    rr = ReferenceReplay(Path(request.node.fspath).stem, request.node.name)
    yield rr
    rr.finish()
