"""TEST INFRASTRUCTURE — records what the reference's own test suite asks of `sparse_dot_topn`.

    python oracle/record_standin_calls.py <checkout of Bergvca/string_grouper>

Runs the UNMODIFIED reference's unittest suite (string_grouper/test/test_string_grouper.py) in this process with the
C oracle standing in for the absent `sparse_dot_topn` wheel (oracle/standin/), records the arguments and the result
of every distinct sp_matmul_topn / zip_sp_matmul_topn call, and writes them with the suite's outcome to
tests/golden/standin_calls.npz.  tests/test_oracle.py replays the calls through oracle.sdt, which keeps the stand-in
pinned to the answers under which the reference's suite passes without the reference tree at hand.

Layout: every matrix is {format, shape, dtype, index dtype, offsets} into two pools, `values` (float64; float32 data
widens exactly) and `ints` (int64 indices and indptr); `meta` is JSON.
"""
import json
import os
import sys
import unittest

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden", "standin_calls.npz")
# the one reference test the suite pin has always left out (pandas 3 removed Series._append, off the hot path)
DESELECTED = ("test_add_match_single_occurence",)


class Pools:
    def __init__(self):
        self.values, self.ints, self.nv, self.ni = [], [], 0, 0

    def put(self, m):
        """Store a scipy sparse matrix in its own format (the reference hands over CSC transposes)."""
        m = m if m.format in ("csr", "csc") else m.tocsr()
        rec = {"format": m.format, "shape": list(m.shape), "dtype": m.dtype.name, "index_dtype": m.indices.dtype.name,
               "values": [self.nv, len(m.data)], "indices": [self.ni, len(m.indices)],
               "indptr": [self.ni + len(m.indices), len(m.indptr)]}
        self.values.append(m.data.astype(np.float64))
        self.ints += [m.indices.astype(np.int64), m.indptr.astype(np.int64)]
        self.nv += len(m.data)
        self.ni += len(m.indices) + len(m.indptr)
        return rec

    def arrays(self):
        return {"values": np.concatenate(self.values or [np.zeros(0)]),
                "ints": np.concatenate(self.ints or [np.zeros(0, np.int64)])}


def _key(m):
    return (m.format, m.shape, m.dtype.str, m.indices.tobytes(), m.indptr.tobytes(), m.data.tobytes())


def _jsonable(v):
    if isinstance(v, type):
        return np.dtype(v).name
    if isinstance(v, np.generic):
        return v.item()
    raise TypeError("cannot store %r" % (v,))


def record(reference_dir):
    for p in (ROOT, reference_dir, os.path.join(HERE, "standin")):
        sys.path.insert(0, p)
    import string_grouper.string_grouper as ref

    pools, calls, seen = Pools(), [], {}
    mm, zipped = ref.sp_matmul_topn, ref.zip_sp_matmul_topn

    def keep(key, make):
        if key in seen:
            calls[seen[key]]["count"] += 1
        else:
            seen[key] = len(calls)
            calls.append(dict(make(), count=1))

    def rec_mm(A, B, *args, **kw):
        out = mm(A, B, *args, **kw)
        opts = json.loads(json.dumps({"args": list(args), "kwargs": kw}, default=_jsonable, sort_keys=True))
        keep(("mm", json.dumps(opts), _key(A), _key(B)),
             lambda: dict(opts, fn="sp_matmul_topn", A=pools.put(A), B=pools.put(B), out=pools.put(out)))
        return out

    def rec_zip(top_n, C_mats):
        out = zipped(top_n=top_n, C_mats=C_mats)
        keep(("zip", int(top_n)) + tuple(_key(c) for c in C_mats),
             lambda: {"fn": "zip_sp_matmul_topn", "top_n": int(top_n), "C_mats": [pools.put(c) for c in C_mats],
                      "out": pools.put(out)})
        return out

    ref.sp_matmul_topn, ref.zip_sp_matmul_topn = rec_mm, rec_zip
    suite = unittest.defaultTestLoader.loadTestsFromName("string_grouper.test.test_string_grouper")

    def flat(s):
        for t in s:
            yield from (flat(t) if isinstance(t, unittest.TestSuite) else [t])

    kept = unittest.TestSuite([t for t in flat(suite) if t.id().rsplit(".", 1)[-1] not in DESELECTED])
    result = unittest.TestResult()
    kept.run(result)
    failed = sorted(t.id().rsplit(".", 1)[-1] for t, _ in result.failures + result.errors)
    meta = {"calls": calls, "suite": {"ran": result.testsRun, "passed": result.testsRun - len(failed),
                                      "failed": failed, "deselected": list(DESELECTED)}}
    np.savez_compressed(OUT, meta=np.array(json.dumps(meta)), **pools.arrays())
    return meta


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    meta = record(os.path.abspath(sys.argv[1]))
    print("%d distinct calls recorded; suite %s" % (len(meta["calls"]), json.dumps(meta["suite"])))
