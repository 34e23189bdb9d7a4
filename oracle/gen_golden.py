"""oracle/gen_golden.py -- writes tests/golden/*.npz from the REFERENCE engine (oracle/_ref =
the reference's own libcuckoo, built by oracle/Makefile when the reference tree is present):
    python oracle/gen_golden.py [table_ops] [traces]      (both when no argument is given)
table_ops: tests/golden/table_ops_dim*.npz, op streams with every input and output.
traces:    tests/golden/ref_engine_traces.npz, digests of what the op streams of tests/helpers.py observe.
The fixtures are committed; machines without the reference replay them against the CUDA path
and against the C port.  TEST INFRASTRUCTURE ONLY.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle as O  # noqa: E402
from tests import helpers as H  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def op_stream(dim, seed, n0=2000, threads=1):
  """One deterministic op stream: insert, find(full default), accum, remove, find(broadcast default),
  insert(overwrite + new), export.  Keys include negatives, 0, -1 and both int64 extremes."""
  rng = np.random.default_rng(seed)
  t = O.RefTable(dim, 0, threads=threads)
  g = {"dim": np.int64(dim)}
  pool = rng.integers(-2**62, 2**62, size=3 * n0, dtype=np.int64)
  pool[:6] = [0, -1, 1, np.iinfo(np.int64).min, np.iinfo(np.int64).min + 1, np.iinfo(np.int64).max]
  pool = np.unique(pool)
  rng.shuffle(pool)
  k0 = pool[:n0].copy()
  v0 = rng.normal(0, 0.01, size=(n0, dim)).astype(np.float32)
  t.insert(k0, v0)
  g["k0"], g["v0"] = k0, v0
  g["size0"] = np.int64(t.size())
  # find, ~50% hits, full-size defaults
  q1 = np.concatenate([rng.choice(k0, n0 // 2, replace=False), pool[n0:n0 + n0 // 2]])
  rng.shuffle(q1)
  d1 = rng.normal(0, 1, size=(q1.shape[0], dim)).astype(np.float32)
  o1, e1 = t.find(q1, d1, True)
  g["q1"], g["d1"], g["o1"], g["e1"] = q1, d1, o1, e1
  # accum: exists flags mostly from the find, some flipped (the 4 cases of accumrase_fn)
  ex = e1.copy()
  flip = rng.random(q1.shape[0]) < 0.2
  ex[flip] = ~ex[flip]
  vod = rng.normal(0, 0.01, size=(q1.shape[0], dim)).astype(np.float32)
  t.accum(q1, vod, ex)
  g["acc_ex"], g["acc_vod"] = ex, vod
  g["size1"] = np.int64(t.size())
  # remove: some present, some absent
  r = np.concatenate([rng.choice(k0, n0 // 5, replace=False), pool[2 * n0:2 * n0 + 50]])
  t.remove(r)
  g["r"] = r
  g["size2"] = np.int64(t.size())
  # find with one broadcast default row
  q2 = np.concatenate([k0[::3], pool[n0:n0 + n0 // 6], r[:n0 // 20]])
  d2 = rng.normal(0, 1, size=(dim,)).astype(np.float32)
  o2, e2 = t.find(q2, d2, True)
  g["q2"], g["d2"], g["o2"], g["e2"] = q2, d2, o2, e2
  # insert: overwrite + brand new + previously removed
  k3 = np.unique(np.concatenate([k0[::4], pool[2 * n0 + 50:2 * n0 + 50 + n0 // 4], r[:40]]))
  v3 = rng.normal(0, 0.01, size=(k3.shape[0], dim)).astype(np.float32)
  t.insert(k3, v3)
  g["k3"], g["v3"] = k3, v3
  ke, ve = t.export()
  order = np.argsort(ke, kind="stable")
  g["export_keys"], g["export_vals"] = ke[order], ve[order]
  g["size3"] = np.int64(t.size())
  t.close()
  return g


def table_ops():
  for dim, n0 in ((1, 2000), (8, 1000), (16, 1000), (64, 400), (128, 250)):
    g = op_stream(dim, seed=1000 + dim, n0=n0)
    path = os.path.join(OUT, "table_ops_dim%d.npz" % dim)
    np.savez_compressed(path, **g)
    print(path, os.path.getsize(path) >> 10, "KiB", "final size", int(g["size3"]))


def _trace(stream, *args):
  rec = H.Trace()
  stream(*args, rec)
  return rec.array()


def traces():
  g = {}
  for dim in (1, 16, 64, 128):
    g["random_ops_dim%d" % dim] = _trace(H.stream_random_ops, O.RefTable(dim, 0, threads=1), dim)
  # the sharded launchers (cuckoo_hashtable_op.cc:39-182) over 4 threads give the same set as 1 thread
  g["set_semantics"] = _trace(H.stream_set_semantics, O.RefTable(16, 0, threads=4))
  assert np.array_equal(g["set_semantics"], _trace(H.stream_set_semantics, O.RefTable(16, 0, threads=1)))
  for c, (dim, init_size, ops) in enumerate(H.small_op_streams()):
    g["small_ops_%d" % c] = _trace(H.stream_small_ops, O.RefTable(dim, init_size, threads=1), dim, ops)
  np.savez_compressed(H.TRACES, **g)
  print(H.TRACES, os.path.getsize(H.TRACES) >> 10, "KiB", sum(v.shape[0] for v in g.values()), "digests")


def main():
  what = sys.argv[1:] or ["table_ops", "traces"]
  unknown = set(what) - {"table_ops", "traces"}
  if unknown:
    sys.exit("gen_golden.py: unknown fixture set(s) %s; expected table_ops and/or traces" % ", ".join(sorted(unknown)))
  O.build()
  assert O.have_ref(), "oracle/_ref not built: the reference tree is needed to generate goldens"
  os.makedirs(OUT, exist_ok=True)
  if "table_ops" in what:
    table_ops()
  if "traces" in what:
    traces()


if __name__ == "__main__":
  main()
