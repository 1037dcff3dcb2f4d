"""Recorded results of the reference's own builds (oracle/_ref: its OSQP, kino_astar.cpp, a_star.cpp, rrt_star.cpp + kdtree.cpp).

oracle/_ref is compiled from the reference's sources, so it exists only where those sources are readable.  Everywhere else the tests
and smoke() compare against what those builds returned for the same inputs, stored in tests/golden/ref_record.json.gz and looked up
by a digest of every input of the call.  Scalars are stored exactly.  An array is stored as a digest of its bits, plus its values
unless the caller passed `like` arrays (the result it is about to compare with) that reproduced them bit for bit.  On lookup, an
array whose values were not stored is returned as the caller's `like` array when the bits match, and as NaN otherwise, so a
comparison against it fails.  Inputs that were never recorded raise LookupError.

Regenerating the record, where oracle/_ref is built (make -C oracle with the reference sources present):
    UAVMP_REF_RECORD=<dir> python -m pytest tests            (the GPU tests on a GPU machine, the others anywhere)
    UAVMP_REF_RECORD=<dir> python -c "import __graft_entry__ as g; g.smoke()"
    python tests/ref_record.py <dir> [<dir> ...]              (packs every <dir>/*.jsonl into the record file)
"""
import ctypes as C
import gzip
import hashlib
import json
import os
import sys

import numpy as np

RECORD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_record.json.gz")
_records = None


def _update(h, p):
    if p is None:
        h.update(b"N")
    elif isinstance(p, np.ndarray):
        a = np.ascontiguousarray(p)
        h.update(f"A{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    elif isinstance(p, C.Structure):
        h.update(repr([_item(getattr(p, f[0])) for f in p._fields_]).encode())
    elif isinstance(p, (list, tuple)):
        h.update(b"L")
        for x in p:
            _update(h, x)
    else:
        h.update(("S" + repr(_item(p))).encode())


def _item(v):
    return v.item() if isinstance(v, np.generic) else v


def digest(*parts):
    h = hashlib.sha256()
    for p in parts:
        _update(h, p)
    return h.hexdigest()[:24]


def _bits(a):
    a = np.ascontiguousarray(a)
    return digest(a)[:16]


def _encode(v, like):
    if isinstance(v, np.ndarray):
        e = {"dtype": v.dtype.str, "shape": list(v.shape), "bits": _bits(v)}
        if like is None or np.size(like) != v.size or _bits(np.asarray(like, v.dtype).reshape(v.shape)) != e["bits"]:
            e["data"] = v.ravel().tolist()
        return e
    if isinstance(v, dict):
        return {"fields": {k: _encode(x, (like or {}).get(k)) for k, x in v.items()}}
    return _item(v)


def _decode(e, like):
    if not isinstance(e, dict):
        return e
    if "fields" in e:
        return {k: _decode(x, (like or {}).get(k)) for k, x in e["fields"].items()}
    dt, shape = np.dtype(e["dtype"]), tuple(e["shape"])
    if "data" in e:
        return np.array(e["data"], dt).reshape(shape)
    if like is not None and np.size(like) == int(np.prod(shape)):
        cand = np.array(like, dt).reshape(shape)
        if _bits(cand) == e["bits"]:
            return cand
    return np.full(shape, np.nan, dt)


def _load():
    global _records
    if _records is None:
        _records = {}
        if os.path.exists(RECORD):
            with gzip.open(RECORD, "rt") as f:
                _records = json.load(f)
    return _records


def call(name, live, key, like=None):
    """The result of the reference build's `name` on inputs `key`: live() when the build is present (None when it is not), else
    the recorded result.  `like`: {field: array} the caller will compare the result with (see the module docstring)."""
    k = digest(name, key)
    if live is not None:
        out = live()
        rec_dir = os.environ.get("UAVMP_REF_RECORD")
        if rec_dir:
            os.makedirs(rec_dir, exist_ok=True)
            with open(os.path.join(rec_dir, f"{os.getpid()}.jsonl"), "a") as f:
                f.write(json.dumps({"key": k, "name": name, "out": _encode(out, like)}) + "\n")
        return out
    rec = _load().get(k)
    if rec is None:
        raise LookupError(f"{name}: the reference build (oracle/_ref) is not built here and no result is recorded for these inputs "
                          f"in {os.path.relpath(RECORD)}; see tests/ref_record.py to regenerate it")
    return _decode(rec, like)


def pack(dirs):
    """Merges the *.jsonl files of `dirs` into RECORD; of several records of one call, the one that keeps its values wins."""
    out = {}
    for d in dirs:
        for fn in sorted(os.listdir(d)):
            if fn.endswith(".jsonl"):
                for line in open(os.path.join(d, fn)):
                    r = json.loads(line)
                    old = out.get(r["key"])
                    if old is None or '"data"' in json.dumps(r["out"]) and '"data"' not in json.dumps(old):
                        out[r["key"]] = r["out"]
    data = json.dumps(out, sort_keys=True, separators=(",", ":")).encode()
    with open(RECORD, "wb") as f:
        f.write(gzip.compress(data, mtime=0))
    print(f"{len(out)} records, {os.path.getsize(RECORD)} bytes -> {RECORD}")


if __name__ == "__main__":
    pack(sys.argv[1:])
