"""bench.py contract (CPU part): the reference arm runs here without a GPU and prints ONE JSON line with the
keys the driver reads; the Zipf generators of both arms agree."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
  p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                      "--cpu-resident", "200000", "--batch", "50000", "--dim", "16"], capture_output=True, text=True,
                     timeout=300, cwd=ROOT)
  assert p.returncode == 0, p.stderr[-2000:]
  lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "M keys/s" and d["value"] > 0
  for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype",
            "data", "config", "cpu_baseline", "e2e"):
    assert k in d, k
  assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
  assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
  assert d["steps"] >= 20 and d["warmup"] >= 5                       # enough timed steps for a stable median
  cores = d["cpu_baseline"]["host_cores"]
  assert d["cpu_baseline"]["cores"] == cores["used"] <= cores["affinity"]   # never more workers than usable cores
  assert d["cpu_baseline"]["parity_mismatches_first_batch"] == 0


def test_other_ranks_of_the_reference_arm_exit_quietly():
  env = dict(os.environ, RANK="1", WORLD_SIZE="2")
  p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env,
                     capture_output=True, text=True, timeout=120, cwd=ROOT)
  assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_writes_the_same_float32_sample_every_time(tmp_path):
  sys.path.insert(0, ROOT)
  import bench as B
  import torch
  dim = 256
  keep = B.DUMP_BYTES // (4 * dim)
  rows = torch.randn(3 * keep, dim, generator=torch.Generator().manual_seed(0))
  rows[:, 0] = torch.arange(rows.shape[0])                             # column 0 = the row's position
  B.dump_rows(str(tmp_path / "a"), "rows", rows)
  B.dump_rows(str(tmp_path / "b"), "rows", rows.clone())
  a, b = np.load(tmp_path / "a" / "rows.npy"), np.load(tmp_path / "b" / "rows.npy")
  assert a.dtype == np.float32 and a.shape == (keep, dim) and a.nbytes <= B.DUMP_BYTES
  np.testing.assert_array_equal(a, b)                                  # the same positions in every run
  pos = a[:, 0].astype(np.int64)
  assert np.unique(pos).shape[0] == pos.shape[0]
  np.testing.assert_array_equal(a, rows.numpy()[pos])                  # every dumped row is a row of the output
  B.dump_rows(str(tmp_path / "c"), "rows", rows, world=4)
  assert np.load(tmp_path / "c" / "rows.npy").shape == (keep // 4, dim)   # the ranks share the budget
  B.dump_rows(str(tmp_path / "d"), "rows", rows[:, :1].repeat(1, 2 * dim))   # wider rows: fewer of them, same bytes
  assert np.load(tmp_path / "d" / "rows.npy").nbytes <= B.DUMP_BYTES
  p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                     capture_output=True, text=True, timeout=120, cwd=ROOT)
  assert p.returncode != 0 and "--dump-outputs" in p.stderr              # never a silent run without the dump


def test_zipf_key_stream_helpers():
  sys.path.insert(0, ROOT)
  import bench as B
  import torch
  r = np.arange(0, 1000, dtype=np.int64)
  kn = B.rank_to_key_np(r)
  kt = B.rank_to_key_torch(torch.from_numpy(r)).numpy()
  np.testing.assert_array_equal(kn, kt)              # both arms draw the same key for the same rank
  assert (kn >= 0).all() and np.unique(kn).shape[0] == 1000
  # the closed-form rows both arms (and the in-bench parity check) use: exact in fp32, torch == numpy
  for gen in (0, 1):
    np.testing.assert_array_equal(B.rows_of_keys_np(kn, 16, gen), B.rows_of_keys_torch(torch.from_numpy(kn), 16, gen).numpy())
  assert not np.array_equal(B.rows_of_keys_np(kn, 16, 0), B.rows_of_keys_np(kn, 16, 1))
  cdf = B.zipf_cdf_np(10000)
  b = B.zipf_unique_batch_np(cdf, 2000, np.random.default_rng(0))
  assert b.shape[0] == 2000 and np.unique(b).shape[0] == 2000 and b.max() < 10000
  assert (b < 100).sum() > 60                        # the Zipf head is (almost) always present
