"""CPU tests of the oracle itself: the C port (and the reference's own libcuckoo, when built here) against the
reference's known-answer tests, and the port against what the reference engine computed on the same op streams
(tests/golden/ref_engine_traces.npz).  No GPU."""
import numpy as np
import pytest

from oracle import oracle as O
from tests import helpers as H
from tests.helpers import golden_files, replay_golden

ENGINES = ["port"] + (["ref"] if O.have_ref() else [])


def make(engine, dim, init_size=0, threads=1):
  return O.PortTable(dim, init_size) if engine == "port" else O.RefTable(dim, init_size, threads)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("dim", [1, 8, 16, 128])
def test_variable_known_answer(engine, dim):
  """dynamic_embedding_variable_test.py:394-468 test_variable."""
  t = make(engine, dim)
  assert t.size() == 0
  t.insert([0, 1, 2, 3], np.array([[0] * dim, [1] * dim, [2] * dim, [3] * dim], np.float32))
  assert t.size() == 4
  t.remove([1, 5])
  assert t.size() == 3
  out = t.find([0, 1, 5], np.full(dim, -1, np.float32))
  np.testing.assert_array_equal(out, np.array([[0] * dim, [-1] * dim, [-1] * dim], np.float32))
  k, v = t.export()
  np.testing.assert_array_equal(np.sort(k), [0, 2, 3])
  np.testing.assert_array_equal(np.sort(v, axis=0), np.array([[0] * dim, [2] * dim, [3] * dim], np.float32))


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("dim", [1, 8, 16, 128])
def test_find_with_exists_and_accum_known_answer(engine, dim):
  """dynamic_embedding_variable_test.py:470-563: golden {0->10, 2->2, 3->13, 100->99}."""
  t = make(engine, dim)
  f = np.float32
  t.insert([0, 1, 2, 3], np.array([[0] * dim, [1] * dim, [2] * dim, [3] * dim], f))
  _, exists = t.find([0, 1, 100, 3], np.full(dim, -1, f), True)
  np.testing.assert_array_equal(exists, [True, True, False, True])
  t.insert([100], np.array([[99] * dim], f))  # "other process" adds 100 ...
  t.remove([1])                               # ... and removes 1
  assert t.size() == 4
  old = np.array([[0] * dim, [1] * dim, [2] * dim, [3] * dim], f)
  new = np.array([[10] * dim, [11] * dim, [100] * dim, [13] * dim], f)
  t.accum([0, 1, 100, 3], O.variable_accum_values(old, new, exists), exists)
  k, v = t.export()
  np.testing.assert_array_equal(np.sort(k), [0, 2, 3, 100])
  np.testing.assert_array_equal(np.sort(v, axis=0), np.array([[2] * dim, [10] * dim, [13] * dim, [99] * dim], f))


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("path", golden_files())
def test_golden_streams(engine, path):
  g = np.load(path)
  replay_golden(make(engine, int(g["dim"])), g)


@pytest.mark.parametrize("dim", [1, 16, 64, 128])
def test_port_equals_reference_engine(dim):
  """Same random op stream into the port as into the reference's libcuckoo (recorded; replayed on it too when it is
  built here): identical results INCLUDING export (iteration) order, through several doublings and cuckoo displacements."""
  for engine in ENGINES:
    rec = H.Trace()
    H.stream_random_ops(make(engine, dim), dim, rec)
    H.assert_trace("random_ops_dim%d" % dim, rec, engine)


def test_reference_engine_multithreaded_set_semantics():
  """The sharded launchers (cuckoo_hashtable_op.cc:39-182) of the reference engine over 4 threads give the same find
  results and the same SET as one thread: the recorded one-thread result, which the reference engine over 4 threads
  (when it is built here) and the single-threaded port must both reproduce."""
  for engine in ENGINES:
    rec = H.Trace()
    H.stream_set_semantics(make(engine, 16, 0, threads=4), rec)
    H.assert_trace("set_semantics", rec, engine)


def test_default_partition_fn():
  """dynamic_embedding_variable.py:165-197."""
  k = np.array([0, 1, 7, -1, -8, 2**40 + 5, np.iinfo(np.int64).min, np.iinfo(np.int64).max], np.int64)
  np.testing.assert_array_equal(O.default_partition_fn(k, 1), np.zeros(8, np.int32))
  got = O.default_partition_fn(k, 3, gpu_mode=True)
  exp = np.array([(int(x) & 0x7fffffff) % 3 for x in k], np.int32)
  np.testing.assert_array_equal(got, exp)
  got = O.default_partition_fn(k, 3, gpu_mode=False)
  np.testing.assert_array_equal(got, np.array([int(x) % 3 for x in k], np.int32))  # python % is floor-mod


def test_unique_first_occurrence():
  """tf.unique contract: dynamic_embedding_ops_test.py:803-821 style."""
  ids = np.array([5, 3, 5, 9, 3, 3, 1], np.int64)
  u, idx = O.unique_first_occurrence(ids)
  np.testing.assert_array_equal(u, [5, 3, 9, 1])
  np.testing.assert_array_equal(idx, [0, 1, 0, 2, 1, 1, 3])
  np.testing.assert_array_equal(u[idx], ids)


def _embedding_result(params, id_vals, weight_vals=None):
  """The NumPy oracle of the reference's own test (dynamic_embedding_ops_test.py:150-184), restated."""
  values, weights, weights_squared = [], [], []
  for ids, wts in zip(id_vals, weight_vals if weight_vals is not None else [[1.0] * len(i) for i in id_vals]):
    va = wa = sa = None
    for i, w in zip(ids, wts):
      val = params[i]
      if va is None:
        va, wa, sa = val * np.float32(w), np.float32(w), np.float32(w) * np.float32(w)
      else:
        va = va + val * np.float32(w)
        wa = wa + np.float32(w)
        sa = sa + np.float32(w) * np.float32(w)
    values.append(va), weights.append(wa), weights_squared.append(sa)
  return np.array(values, np.float32), np.array(weights, np.float32), np.array(weights_squared, np.float32)


@pytest.mark.parametrize("combiner", ["sum", "mean", "sqrtn"])
@pytest.mark.parametrize("use_weights", [False, True])
@pytest.mark.parametrize("dim", [1, 5])
def test_embedding_lookup_sparse_vs_reference_test_oracle(combiner, use_weights, dim):
  """EmbeddingLookupSparseTest (dynamic_embedding_ops_test.py:875-969): grouped ids, 5 rows, rtol=atol=1e-6."""
  rng = np.random.default_rng(3)
  vocab = 13
  params = {i: rng.standard_normal(dim).astype(np.float32) for i in range(vocab)}
  t = O.PortTable(dim)
  t.insert(np.arange(vocab), np.stack([params[i] for i in range(vocab)]))
  grouped_ids = [[0, 1, 2], [3], [4, 5, 6, 7, 7], [8, 9], [10, 11, 12, 0]]
  grouped_w = [[rng.uniform(0.5, 2) for _ in g] for g in grouped_ids] if use_weights else None
  ids = np.array([i for g in grouped_ids for i in g], np.int64)
  seg = np.array([r for r, g in enumerate(grouped_ids) for _ in g], np.int32)
  w = None if not use_weights else np.array([x for g in grouped_w for x in g], np.float32)
  got = O.embedding_lookup_sparse(t, ids, seg, w, 5, combiner)
  v, ws, wsq = _embedding_result(params, grouped_ids, grouped_w)
  if combiner == "mean":
    v = v / ws[:, None]
  elif combiner == "sqrtn":
    v = v / np.sqrt(wsq)[:, None]
  np.testing.assert_allclose(got, v, rtol=1e-6, atol=1e-6)


def test_twin_adagrad_matches_dense():
  """Twin-model idea of dynamic_embedding_optimizer_test.py:349-440: a dense array trained with the plain
  rule == the table trained through find -> rule -> upsert."""
  dim, n = 4, 50
  rng = np.random.default_rng(0)
  p, a = O.PortTable(dim), O.PortTable(dim)
  dense_p = np.zeros((n, dim), np.float32)
  dense_a = np.full((n, dim), 0.1, np.float32)
  for step in range(10):
    keys = rng.permutation(n)[:20].astype(np.int64)
    g = rng.standard_normal((20, dim)).astype(np.float32)
    O.sparse_adagrad_step(p, a, keys, g, 0.1, np.zeros(dim, np.float32), np.full(dim, 0.1, np.float32))
    dense_p[keys], dense_a[keys] = O.adagrad_dense(dense_p[keys], dense_a[keys], g, 0.1)
  k, v = p.export()
  np.testing.assert_array_equal(v[np.argsort(k)], dense_p[np.sort(k)])


# ---- pinning of the C port against the reference's own engine on many small op streams ---------------------------
def test_port_vs_reference_engine_property():
  """60 seeded op streams over a tiny key universe and tiny initial tables (init_size 1/4/64 slots: every insert path
  runs -- last-empty-slot placement, BFS displacement, doubling): the C port and the reference's libcuckoo (recorded;
  replayed on it too when it is built here) agree on sizes, find results, exists masks and export ORDER after every op.
  Duplicate keys inside a call are allowed here (both engines are single-threaded, so the outcome is deterministic)."""
  for engine in ENGINES:
    for c, (dim, init_size, ops) in enumerate(H.small_op_streams()):
      rec = H.Trace()
      t = make(engine, dim, init_size)
      H.stream_small_ops(t, dim, ops, rec)
      t.close()
      H.assert_trace("small_ops_%d" % c, rec, engine)


def test_optimizer_rules_against_an_independent_implementation():
  """The absolute Adagrad / Adam numbers are unpinned by the reference tree (the rules are stock TensorFlow kernels,
  SURVEY 8c): besides restating TF's documented rules, check the restatement against an implementation written by
  someone else -- torch.optim -- over 10 steps, at the reference twin-model tests' fp32 tolerance (1e-6,
  dynamic_embedding_optimizer_test.py:387-440).  Adagrad: the same rule (eps placed like Keras').  Adam: torch adds
  epsilon after the bias correction of v, TF before it -- the same update when eps_torch = eps_tf / sqrt(1 - b2^t),
  which is set per step below."""
  import torch
  rng = np.random.default_rng(11)
  n, dim, lr = 64, 16, 0.05
  p0 = rng.normal(0, 0.01, (n, dim)).astype(np.float32)
  grads = rng.normal(0, 1e-2, (10, n, dim)).astype(np.float32)
  for eps in (0.0, 1e-7):
    tp = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    opt = torch.optim.Adagrad([tp], lr=lr, initial_accumulator_value=0.1, eps=eps)
    p, a = p0.copy(), np.full((n, dim), 0.1, np.float32)
    for g in grads:
      tp.grad = torch.from_numpy(g.copy())
      opt.step()
      p, a = O.adagrad_dense(p, a, g, lr, eps)
    np.testing.assert_allclose(p, tp.detach().numpy(), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(a, opt.state[tp]["sum"].numpy(), rtol=1e-6, atol=1e-6)
  b1, b2, eps = 0.9, 0.999, 1e-8
  tp = torch.nn.Parameter(torch.from_numpy(p0.copy()))
  opt = torch.optim.Adam([tp], lr=lr, betas=(b1, b2), eps=eps)
  p, m, v = p0.copy(), np.zeros((n, dim), np.float32), np.zeros((n, dim), np.float32)
  for t, g in enumerate(grads, 1):
    tp.grad = torch.from_numpy(g.copy())
    opt.param_groups[0]["eps"] = eps / float(np.sqrt(1.0 - b2 ** t))
    opt.step()
    p, m, v = O.adam_dense(p, m, v, g, O.adam_scalars(lr, b1, b2, t), b1, b2, eps)
  np.testing.assert_allclose(m, opt.state[tp]["exp_avg"].numpy(), rtol=1e-6, atol=1e-7)
  np.testing.assert_allclose(v, opt.state[tp]["exp_avg_sq"].numpy(), rtol=1e-6, atol=1e-9)
  np.testing.assert_allclose(p, tp.detach().numpy(), rtol=1e-5, atol=1e-6)


def test_segment_reduce_is_the_sequential_position_order_sum():
  """oracle.segment_reduce (np.add.at) against the literal loop of TF's CPU unsorted_segment_sum: for every position in
  order, out[idx[i]] += rows[i], one fp32 add per element; negative / too large ids dropped"""
  rng = np.random.default_rng(17)
  n, g, dim = 400, 9, 5
  rows = (rng.normal(0, 1, (n, dim)) * np.exp(rng.uniform(-8, 8, (n, 1)))).astype(np.float32)
  idx = rng.integers(-1, g + 1, size=n).astype(np.int32)
  exp = np.zeros((g, dim), np.float32)
  for i in range(n):
    if 0 <= idx[i] < g:
      for c in range(dim):
        exp[idx[i], c] = np.float32(exp[idx[i], c] + rows[i, c])
  np.testing.assert_array_equal(O.segment_reduce(rows, idx, g), exp)
