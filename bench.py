#!/usr/bin/env python
"""bench.py -- headline benchmark of the dynamic-embedding table hot path.

Metric (BASELINE.json): embedding lookup+insert M keys/s at dim 64 on 1/2/4/8 B200, with the fraction of the
HBM roofline.  Workload at N=1 = BASELINE.json configs[1]: an HKV-style table with 100M resident int64 keys,
dim-64 fp32 rows, Zipf(alpha=1.05) id stream, 1,048,576 unique keys per step.

One STEP = one pass of the hot path over one batch: Find (lookup) of the batch + Insert (upsert, the
optimizer write-back) of the batch.  `value` = keys per second, every key looked up AND upserted once per step,
inputs resident in HBM.  `e2e` = the same step through the host-buffer entry points of the plugin API
(pinned HOST keys/values in, HOST rows out, PCIe copies inside the timed region).

N>1 (launched by torchrun, one rank per GPU): the table is key-hash sharded (owner = (key & 0x7fffffff) % N,
the reference's default_partition_fn); every rank keeps a 100M-key shard (weak scaling) and drives batches of
keys owned by ANY rank.  --exchange peer (default): ONE kernel per call probes the owner's shard over NVLink peer
memory (det_peer_find / det_peer_insert).  --exchange nccl (the baseline): partition -> NCCL all-to-all of keys ->
local find -> all-to-all of rows back, and keys+rows to their owners -> local insert.

--impl reference : the reference's own CPU cuckoo path (oracle/_ref = its vendored libcuckoo compiled from
/root/reference, else the C port) on the host cores, same metric, bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIM = 64
ALPHA = 1.05
KEY_SALT = 0x9E3779B97F4A7C15


def parse_args():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=2000,
                  help="timed steps of every GPU measurement: the headline and the c3 line (embedded or --workload c3); "
                       "the CPU arms time a bounded sample of their own (--impl reference: 20-40 steps, the embedded "
                       "cpu_baseline: 15), reported as their own `steps`")
  ap.add_argument("--warmup", type=int, default=20)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--resident", type=int, default=100_000_000, help="resident keys per GPU")
  ap.add_argument("--batch", type=int, default=1 << 20, help="unique keys per step per GPU")
  ap.add_argument("--dim", type=int, default=DIM)
  ap.add_argument("--cpu-resident", type=int, default=0,
                  help="resident keys of the CPU arm (0 = the GPU arm's resident count when host RAM allows, else the largest power-of-two fraction that fits)")
  ap.add_argument("--cpu-threads", type=int, default=0, help="worker threads of the CPU arm (0 = usable host cores: affinity mask capped by the cgroup quota)")
  ap.add_argument("--no-hard-cases", action="store_true", help="N=1: skip find_hit90 / insert_new / lookup_insert_new")
  ap.add_argument("--no-c3", action="store_true", help="N=1: skip the embedded configs[2] line (fused sparse lookup + Adagrad)")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-e2e", action="store_true")
  ap.add_argument("--e2e-steps", type=int, default=10)
  ap.add_argument("--exchange", default="hybrid", choices=["hybrid", "push", "peer", "nccl"],
                  help="N>1: hybrid (default) = lookups through the owners with posted NVLink stores only (det_peer_xchg_find) + "
                       "one-sided inserts (det_peer_insert); push = owner-side exchange both ways (det_peer_xchg_*); peer = the "
                       "one-sided remote-probe kernels both ways (det_peer_find/insert); nccl = NCCL all-to-all")
  ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c5"],
                  help="c2 = headline lookup+insert (BASELINE configs[1]); c3 = fused embedding_lookup_sparse + Adagrad (configs[2]); "
                       "c4 = the c2 step on configs[3] (torchrun --gpus 8: 1B keys = 125M resident per GPU, dim 128); "
                       "c5 = sharded forward+backward (configs[4], torchrun)")
  ap.add_argument("--grad-reduce", default="det", choices=["det", "torch"],
                  help="c3 / c5: per-unique gradient sum by det_segment_reduce (position order, deterministic) or by "
                       "torch index_add (atomics); sets DET_GRAD_REDUCE for the sharded combine as well")
  ap.add_argument("--distinct-batches", type=int, default=64, help="distinct key batches cycled through")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="after the timed steps, write a fixed sample of the rows the last timed step returned as "
                       "DIR/<name>.npy (float32): lookup_rows (c2 / c4) and c3_lookup_sparse (c3, also embedded in c2)")
  a = ap.parse_args()
  if a.dump_outputs and (a.impl == "reference" or a.workload == "c5"):
    ap.error("--dump-outputs covers the c2, c3 and c4 workloads of --impl ours")
  if a.workload == "c4":   # BASELINE configs[3]: key-hash sharded table, 1B keys over 8 GPUs, dim 128 -- the c2 step
    a.dim, a.resident = 128, 125_000_000
  return a


# ------------------------------------------------------------------------------------------------
# synthetic Criteo-shaped id stream (SURVEY.md 8d): rank ~ Zipf(1.05) over the vocabulary, key = fmix64(rank+salt)
# ------------------------------------------------------------------------------------------------
def fmix64_np(x):
  x = x.astype(np.uint64)
  x ^= x >> np.uint64(33)
  x *= np.uint64(0xff51afd7ed558ccd)
  x ^= x >> np.uint64(33)
  x *= np.uint64(0xc4ceb9fe1a85ec53)
  x ^= x >> np.uint64(33)
  return x


def rank_to_key_np(rank):
  with np.errstate(over="ignore"):
    k = fmix64_np(rank.astype(np.uint64) + np.uint64(KEY_SALT)) & np.uint64(0x7fffffffffffffff)
  return k.astype(np.int64)


def zipf_cdf_np(vocab):
  w = np.arange(1, vocab + 1, dtype=np.float64) ** (-ALPHA)
  c = np.cumsum(w)
  return c / c[-1]


def zipf_unique_batch_np(cdf, batch, rng):
  """`batch` distinct ranks drawn Zipf(alpha) (duplicates of a draw are dropped, as tf.unique does before the
  table is touched), in random order."""
  got = np.zeros(0, dtype=np.int64)
  while got.shape[0] < batch:
    r = np.searchsorted(cdf, rng.random(2 * batch), side="left").astype(np.int64)
    got = np.unique(np.concatenate([got, r]))
  rng.shuffle(got)
  return got[:batch]


def torch_fmix64(x):
  import torch
  m1 = torch.tensor(-49064778989728563, dtype=torch.int64, device=x.device)
  m2 = torch.tensor(-4265267296055464877, dtype=torch.int64, device=x.device)
  s = lambda v: (v >> 33) & 0x7fffffff
  x = x ^ s(x)
  x = x * m1
  x = x ^ s(x)
  x = x * m2
  x = x ^ s(x)
  return x


def rank_to_key_torch(rank):
  import torch
  salt = torch.tensor(KEY_SALT - (1 << 64), dtype=torch.int64, device=rank.device)
  return torch_fmix64(rank + salt) & 0x7fffffffffffffff


def rows_of_keys_torch(keys, dim, gen):
  """The row every copy of `keys` carries in generation `gen` (0 = prefill, 1 = written by the timed steps): a closed
  form of the key, exact in fp32 (20-bit integers scaled by 2^-20), so that ANY rank can check ANY looked-up row."""
  import torch
  j = torch.arange(dim, dtype=torch.int64, device=keys.device) * 7919 + int(gen) * 104729
  v = ((keys.reshape(-1, 1) & 0xFFFFF) + j) & 0xFFFFF
  return v.to(torch.float32) * (1.0 / (1 << 20)) - 0.5


def rows_of_keys_np(keys, dim, gen):
  j = np.arange(dim, dtype=np.int64) * 7919 + int(gen) * 104729
  v = ((keys.reshape(-1, 1) & 0xFFFFF) + j) & 0xFFFFF
  return v.astype(np.float32) * np.float32(1.0 / (1 << 20)) - np.float32(0.5)


def zipf_cdf_torch(vocab, device):
  import torch
  c = torch.empty(vocab, dtype=torch.float64, device=device)
  chunk = 1 << 26
  carry = 0.0
  for b in range(0, vocab, chunk):
    e = min(vocab, b + chunk)
    w = torch.arange(b + 1, e + 1, dtype=torch.float64, device=device).pow_(-ALPHA)
    torch.cumsum(w, 0, out=c[b:e])
    c[b:e] += carry
    carry = float(c[e - 1])
  c /= carry
  return c


def zipf_unique_batch_torch(cdf, batch, gen):
  import torch
  got = torch.zeros(0, dtype=torch.int64, device=cdf.device)
  while got.numel() < batch:
    u = torch.rand(2 * batch, dtype=torch.float64, device=cdf.device, generator=gen)
    r = torch.searchsorted(cdf, u).clamp_(max=cdf.numel() - 1)
    got = torch.unique(torch.cat([got, r]))
  perm = torch.randperm(got.numel(), device=cdf.device, generator=gen)
  return got[perm[:batch]]


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own cuckoo path on the host cores
# ------------------------------------------------------------------------------------------------
def usable_host_cores():
  """Cores this process may really use: the affinity mask, capped by the cgroup CPU quota.  os.cpu_count() ignores both;
  a pool of that size on a lease that owns fewer cores leaves libcuckoo's spinning writers fighting for time slices
  (round 1: the same arm gave 4.7 and 26 M keys/s on two boxes)."""
  info = {"cpu_count": os.cpu_count() or 1}
  try:
    info["affinity"] = len(os.sched_getaffinity(0))
  except AttributeError:
    info["affinity"] = info["cpu_count"]
  quota = None
  try:
    with open("/sys/fs/cgroup/cpu.max") as f:        # cgroup v2: "<quota> <period>" or "max <period>"
      q, per = f.read().split()[:2]
      if q != "max":
        quota = float(q) / float(per)
  except Exception:
    try:
      with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
        q, per = float(f.read()), float(g.read())
        if q > 0:
          quota = q / per
    except Exception:
      pass
  info["cgroup_quota_cores"] = quota
  n = info["affinity"]
  if quota is not None:
    n = max(1, min(n, int(quota)))
  info["used"] = n
  return n, info


def cpu_resident_for(dim, want):
  """largest resident key count <= want whose libcuckoo table (4-slot buckets of 8 + dim*4 B entries, power-of-two
  bucket count, ~0.75 load at `want`) fits in 60 % of the available host RAM"""
  try:
    import psutil
    avail = psutil.virtual_memory().available
  except Exception:
    avail = 32 << 30
  r = want
  while r > (1 << 20):
    buckets = 1
    while buckets * 4 < r:
      buckets *= 2
    if buckets * 4 * (8 + dim * 4) * 1.1 + r * 8 * 3 < 0.6 * avail:
      break
    r //= 2
  return r, avail


def cpu_arm(dim, resident, batch, steps, warmup, threads=0, want_resident=100_000_000):
  """The reference's own CPU cuckoo path (oracle/_ref: its vendored libcuckoo behind the restated TableWrapper and
  sharded launchers) on the usable host cores: resident table, then `warmup` + `steps` steps of Find(batch) +
  Insert(batch) over fresh Zipf batches; median / min / max of the timed steps."""
  from oracle import oracle as O
  O.build()
  n_thr, cores = usable_host_cores()
  if threads:
    n_thr = cores["used"] = int(threads)
  why = None
  if not resident:
    resident, avail = cpu_resident_for(dim, want_resident)
    if resident < want_resident:
      why = "host RAM: %.0f GB available, a %d-key libcuckoo table at dim %d needs ~%.0f GB" % (
          avail / 2**30, want_resident, dim, 2**25 * 4 * (8 + dim * 4) / 2**30)
  if O.have_ref():
    # init_size = resident: libcuckoo reserves the smallest power-of-two bucket count holding it (2^25 buckets x 4 slots
    # at 100M keys, load 0.745) -- no resize during the run, same as the GPU arm's pre-sized table
    table, kind = O.RefTable(dim, resident, threads=n_thr), "reference"
  else:
    table, kind = O.PortTable(dim, resident), "port"
    n_thr = cores["used"] = 1   # the port is single-threaded
  rng = np.random.default_rng(42)
  cdf = zipf_cdf_np(resident)
  fill = 1 << 20
  t_fill = time.perf_counter()
  for b in range(0, resident, fill):
    r = np.arange(b, min(resident, b + fill), dtype=np.int64)
    k = rank_to_key_np(r)
    table.insert(k, rows_of_keys_np(k, dim, 0))
  t_fill = time.perf_counter() - t_fill
  default = np.zeros(dim, np.float32)
  out = np.zeros((batch, dim), np.float32)  # reused output buffer (TF's allocator pools outputs as well)
  times_find, times_ins = [], []
  mism = 0
  for it in range(warmup + steps):
    keys = rank_to_key_np(zipf_unique_batch_np(cdf, batch, rng))
    vals = rows_of_keys_np(keys, dim, 1)
    t0 = time.perf_counter()
    table.find(keys, default, out=out)
    t1 = time.perf_counter()
    table.insert(keys, vals)
    t2 = time.perf_counter()
    if it == 0:   # same closed-form rows as the GPU arm: the CPU arm is checked too
      e0 = rows_of_keys_np(keys[:4096], dim, 0)
      mism = int((out[:4096] != e0).any(1).sum())
    if it >= warmup:
      times_find.append(t1 - t0)
      times_ins.append(t2 - t1)
  tot = np.asarray(times_find) + np.asarray(times_ins)
  tf, ti, tt = float(np.median(times_find)), float(np.median(times_ins)), float(np.median(tot))
  table.close()
  return {
      "value": batch / tt / 1e6, "unit": "M keys/s", "cores": n_thr, "kind": kind,
      "sample": "resident %d keys%s, dim %d, batch %d unique Zipf(%.2f) keys, %d timed steps of find+insert after %d "
                "warm-ups (median; fill took %.0f s)" %
                (resident, "" if why is None else " (of the GPU arm's %d: %s)" % (want_resident, why), dim, batch, ALPHA, steps,
                 warmup, t_fill),
      "find_Mkeys_s": batch / tf / 1e6, "insert_Mkeys_s": batch / ti / 1e6,
      "value_min": batch / float(tot.max()) / 1e6, "value_max": batch / float(tot.min()) / 1e6,
      "host_cores": cores, "resident": resident, "same_resident_as_gpu_arm": resident >= want_resident,
      "parity_mismatches_first_batch": mism,
      "ms_per_step": tt * 1e3,
  }


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
  Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
       "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
       "clocks_event_reasons.sw_power_cap")

  def __init__(self, gpu_index):
    self.idx = gpu_index
    self.samples = []
    self.proc = None

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                   stderr=subprocess.DEVNULL, text=True)
      self.th = threading.Thread(target=self._read, daemon=True)
      self.th.start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.samples.append(line.strip())

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    time.sleep(0.25)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:
      self.proc.kill()
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for s in self.samples:
      f = [x.strip() for x in s.split(",")]
      if len(f) < 8:
        continue
      try:
        sm.append(float(f[1]))
        mx.append(float(f[2]))
      except ValueError:
        continue
      for nme, v in zip(names, f[4:8]):
        if v.lower().startswith("active"):
          reasons.add(nme)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(gpu_index):
  """Run the calling thread on the CPUs nearest to the GPU (so pinned staging buffers are first-touched on the
  GPU's NUMA node).  Returns the previous affinity mask, or None when nothing was changed."""
  try:
    import pynvml
    prev = os.sched_getaffinity(0)
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
    pynvml.nvmlDeviceSetCpuAffinity(h)
    return prev
  except Exception:
    return None


DUMP_BYTES = 16 << 20   # per output, all ranks together: a run writes at most two outputs, 32 MB in all


def dump_rows(out_dir, name, rows, world=1):
  """--dump-outputs: the rows at a fixed, seeded set of positions of `rows` ([n, dim], what a caller of the timed path
  received in its last step) as out_dir/<name>.npy in float32, at most DUMP_BYTES // world bytes of rows.  The
  benchmark's inputs are seeded, so two builds run with the same arguments can be compared output for output."""
  import torch
  n, dim = rows.shape
  keep = max(1, DUMP_BYTES // (4 * dim * world))
  idx = np.sort(np.random.default_rng(0).choice(n, min(n, keep), replace=False))
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, name + ".npy"), rows[torch.from_numpy(idx).to(rows.device)].float().cpu().numpy())


def measured_peak_gbs():
  p = os.path.join(ROOT, "MEASURED_PEAKS.json")
  try:
    with open(p) as f:
      return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
  except Exception:
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"



def src_sha():
  """hash of the kernel sources a committed ncu traffic figure belongs to"""
  import hashlib
  h = hashlib.sha256()
  for f in ("table.cu", "common.cuh"):
    with open(os.path.join(ROOT, "recommenders_addons_b200", "csrc", f), "rb") as fh:
      h.update(fh.read())
  return h.hexdigest()[:16]


def committed_traffic(kernel_key):
  """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel_key` on this workload, from the ncu capture
  committed in profiles/r02_traffic.json by scripts/ncu_traffic.py.  A capture taken from other kernel sources is STALE:
  it is reported as null with the reason, never silently."""
  path = os.path.join(ROOT, "profiles", "r02_traffic.json")
  try:
    with open(path) as f:
      rec = json.load(f)[kernel_key]
  except Exception as ex:
    return None, "no committed capture (%s)" % (ex,)
  if rec.get("src_sha") != src_sha():
    print("bench.py: profiles/r02_traffic.json is STALE for %s (kernel sources changed since the capture): "
          "roofline.traffic = null; re-run scripts/ncu_traffic.py under gpurun" % kernel_key, file=sys.stderr)
    return None, "stale capture (sources %s, capture %s)" % (src_sha(), rec.get("src_sha"))
  return int(rec["dram_read"] + rec["dram_write"]), "profiles/r02_traffic.json (%s)" % rec.get("when", "?")


def hard_cases(de, table, dev, dim, B, vocab, default, peak, key_batches):
  """SURVEY 8(d)'s sweep beyond the all-hits step (N=1): Find with 10 % misses on the headline table; inserts of
  BRAND-NEW keys at load 0.25 / 0.5 / 0.75 and a Find+Insert pair with 50 % new keys on a second, pre-sized table
  (2^26 slots, 17 GB of rows: far beyond L2 like the headline table).  CUDA events, median of the reps, every rep a
  different batch.  honest bytes = key + 64 B bucket + row in + row out."""
  import torch
  row = dim * 4
  res = {}

  def med_ms(fns):
    ts = []
    for fn in fns:
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record()
      fn()
      b.record()
      torch.cuda.synchronize()
      ts.append(a.elapsed_time(b))
    return float(np.median(ts[2:] if len(ts) > 4 else ts))

  def entry(ms, n, algo, honest, note):
    return {"Mkeys_s": n / ms / 1e3, "ms": ms, "algorithmic_frac": algo / (ms * 1e-3) / 1e9 / peak,
            "honest_frac": honest / (ms * 1e-3) / 1e9 / peak, "note": note}

  gen = torch.Generator(device=dev).manual_seed(99)
  # ---- find_hit90 -------------------------------------------------------------------------------------------
  nm = B // 10
  qs = []
  for i in range(8):
    hit = key_batches[i % len(key_batches)][:B - nm]
    miss = rank_to_key_torch(vocab + 1000 + i * nm + torch.arange(nm, device=dev))
    q = torch.cat([hit, miss])
    qs.append(q[torch.randperm(B, device=dev, generator=gen)].contiguous())
  ms = med_ms([(lambda q=q: table.lookup(q, dynamic_default_values=default)) for q in qs])
  res["find_hit90"] = entry(ms, B, (B - nm) * row, B * (8 + 64 + row) + (B - nm) * row,
                            "Find, 90 % resident Zipf keys + 10 % absent keys (default row written), headline table")
  # ---- second table for the new-key cases -----------------------------------------------------------------------
  cap = 1 << 26
  t2 = de.CuckooHashTable(torch.int64, torch.float32, default, name="bench_new_keys", init_size=cap, max_capacity=cap,
                          max_load_factor=0.95)
  base = 20 * vocab
  filled = 0

  def fresh(n):
    nonlocal filled
    k = rank_to_key_torch(base + filled + torch.arange(n, device=dev))
    filled += n
    return k

  def fill_to(load):
    while filled < int(cap * load):
      k = fresh(min(1 << 20, int(cap * load) - filled))
      t2.insert(k, rows_of_keys_torch(k, dim, 0))

  vals = rows_of_keys_torch(key_batches[0], dim, 1)
  for load in (0.25, 0.5, 0.75):
    fill_to(load)
    batches = [fresh(B) for _ in range(6)]
    ms = med_ms([(lambda k=k: t2.insert(k, vals)) for k in batches])
    res["insert_new_load%02d" % int(load * 100)] = entry(
        ms, B, B * row, B * (8 + 64 + 2 * row),
        "Insert of %d BRAND-NEW keys per launch, table pre-sized (2^26 slots), load %.2f -> %.2f" % (B, load, filled / cap))
    if load == 0.5:
      # Find + Insert pair, 50 % of every batch brand-new, 50 % resident in this table
      pairs = []
      for i in range(6):
        old = rank_to_key_torch(base + torch.randint(0, filled, (B // 2,), device=dev, generator=gen))
        old = torch.unique(old)
        new = fresh(B - old.numel())
        pairs.append(torch.cat([old, new])[torch.randperm(B, device=dev, generator=gen)].contiguous())

      def pair(k):
        t2.lookup(k, dynamic_default_values=default)
        t2.insert(k, vals)
      ms = med_ms([(lambda k=k: pair(k)) for k in pairs])
      res["lookup_insert_new"] = entry(
          ms, B, B // 2 * row + B * row, B * (8 + 64 + row) + B // 2 * row + B * (8 + 64 + 2 * row),
          "Find(batch) + Insert(batch), 50 % of the batch brand-new keys, load ~0.5; Mkeys_s counts every key once "
          "(looked up AND upserted), like the headline value")
  assert t2.stats()["error_flags"] == 0
  t2.close()
  del t2
  torch.cuda.empty_cache()
  return res


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def gpu_arm(args):
  import torch
  import torch.distributed as dist
  from recommenders_addons_b200 import dynamic_embedding as de

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
  torch.cuda.set_device(local_rank)
  dev = torch.device("cuda", local_rank)
  dim, B, resident = args.dim, args.batch, args.resident
  free = torch.cuda.mem_get_info()[0]
  while 2 * resident * (8 + dim * 4) * 1.1 + (12 << 30) > free and resident > (1 << 20):
    resident //= 2  # smaller GPU than a B200: shrink and say so in config
  if args.dump_outputs and resident != args.resident:
    # a smaller table is a different key stream: its outputs cannot be compared with a run at the requested size
    raise SystemExit("bench.py: %.1f GB free on cuda:%d holds %d resident keys, not the %d asked for; --dump-outputs "
                     "needs the requested workload" % (free / 1e9, local_rank, resident, args.resident))
  vocab = resident * world

  gen = torch.Generator(device=dev).manual_seed(42 + rank)
  gen_v = torch.Generator(device=dev).manual_seed(43 + rank)
  sharded, exchange = None, "none"
  if world > 1:
    exchange = args.exchange
    if exchange in ("hybrid", "push", "peer"):
      try:
        # the shard lives in a symmetric-memory region that every rank maps (CUDA VMM, 2 MB pages)
        sharded = de.PeerShardedVariable.create(dim, 2 * resident, initializer=0.0, name="bench_table")
        if exchange in ("push", "hybrid"):
          # mailbox: request / insert segments per source rank + the output ring
          sharded.attach_exchange(B, insert="push" if exchange == "push" else "pull")
      except Exception as ex:  # no symmetric memory in this sandbox: NCCL exchange instead, and say so
        print("symmetric-memory peer group failed (%r): falling back to NCCL all-to-all" % (ex,), file=sys.stderr)
        exchange = "nccl"
        sharded = None
  if sharded is not None:
    var = sharded.local
  else:
    var = de.Variable(dim=dim, init_size=2 * resident, initializer=0.0, name="bench_table",
                      kv_creator=de.HkvHashTableCreator(de.HkvHashTableConfig(init_capacity=2 * resident,
                                                                               max_capacity=2 * resident)))
  if world > 1 and exchange == "nccl":
    sharded = de.ShardedVariable(var)
  is_peer = exchange in ("peer", "hybrid")     # one-sided remote writes: reads and writes need phase barriers
  is_push = exchange in ("push", "hybrid")     # lookups through the owners, rows land in the output ring
  table = var.tables[0]
  # ---- prefill this rank's shard: all ranks r of the vocabulary with owner(key(r)) == rank; row = f(key, generation 0)
  chunk = min(1 << 20, B)
  if sharded is None:
    for b in range(0, vocab, chunk):
      k = rank_to_key_torch(torch.arange(b, min(vocab, b + chunk), dtype=torch.int64, device=dev))
      table.insert(k, rows_of_keys_torch(k, dim, 0))
  else:
    # every rank generates 1/N of the vocabulary (ranks [rank*resident, (rank+1)*resident)) and writes it THROUGH the
    # sharded table: the keys travel to their owners over the same exchange the timed steps use (N times less work per
    # rank than filtering the whole vocabulary, and the exchange has moved `resident` keys per rank before it is timed)
    for b in range(rank * resident, (rank + 1) * resident, chunk):
      k = rank_to_key_torch(torch.arange(b, min((rank + 1) * resident, b + chunk), dtype=torch.int64, device=dev))
      sharded.upsert(k, rows_of_keys_torch(k, dim, 0))
    if is_peer:
      sharded.phase_barrier()
    torch.cuda.synchronize()
    dist.barrier()
  local_size = int(table.size())
  cdf = zipf_cdf_torch(vocab, dev)
  n_batches = max(1, min(args.steps + args.warmup, args.distinct_batches if dim <= 64 else min(args.distinct_batches, 8)))
  key_batches = [rank_to_key_torch(zipf_unique_batch_torch(cdf, B, gen)) for _ in range(n_batches)]
  del cdf
  # the rows the timed steps write: f(key, generation 1) -- a function of the key, so any rank can check any row later
  val_batches = [rows_of_keys_torch(k, dim, 1) for k in key_batches]
  default = torch.zeros(dim, device=dev)

  def step(i, ev=None):
    k = key_batches[i % n_batches]
    v = val_batches[i % n_batches]
    if sharded is None:
      if ev:
        ev[0].record()
      rows = table.lookup(k, dynamic_default_values=default)
      if ev:
        ev[1].record()
      table.insert(k, v)
      if ev:
        ev[2].record()
      return rows
    if ev:
      ev[0].record()
    rows = sharded.lookup(k, copy=False) if is_push else sharded.lookup(k)
    if is_peer:
      sharded.phase_barrier()  # every rank has finished reading before any rank writes
    if ev:
      ev[1].record()
    sharded.upsert(k, v)
    if is_peer:
      sharded.phase_barrier()  # every rank has finished writing before the next step reads
    if ev:
      ev[2].record()
    return rows

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()  # sampled over warm-up + timed region (both run the same load)
  for i in range(args.warmup):
    step(i)
  barrier()
  evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
  t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  t_start.record()
  for s in range(args.steps):
    out = step(args.warmup + s, evs[s])
  t_end.record()
  barrier()
  clocks = sampler.stop() if rank == 0 else None
  if args.dump_outputs:
    dump_rows(args.dump_outputs, "lookup_rows" if world == 1 else "lookup_rows_rank%d" % rank, out.reshape(-1, dim), world)
  del out
  total_ms = t_start.elapsed_time(t_end)
  find_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
  ins_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in evs]))
  tt = torch.tensor([total_ms, find_ms, ins_ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
  total_ms, find_ms_max, ins_ms_max = [float(x) for x in tt.tolist()]
  ms_per_step = total_ms / args.steps
  value = world * B / (ms_per_step * 1e-3) / 1e6

  # ---- parity: a fixed sample looked up AFTER the timed region against the closed-form rows (every N) ------------
  # (a) keys this rank wrote in its last timed step -> generation 1; (b) keys the OTHER ranks wrote in theirs ->
  # generation 1; (c) random resident keys of any owner -> generation 0 or 1, never a mixture (a torn row);
  # (d) keys outside the vocabulary -> the default row, exists = False.
  ns = 16384
  last = key_batches[(args.warmup + args.steps - 1) % n_batches]
  qa = last[:ns].contiguous()
  if world > 1:
    gathered = [torch.empty_like(qa) for _ in range(world)]
    dist.all_gather(gathered, qa)
    qb = torch.cat([g for r_, g in enumerate(gathered) if r_ != rank])
  else:
    qb = key_batches[(args.warmup + max(0, args.steps - 2)) % n_batches][ns:2 * ns].contiguous()
  gen_p = torch.Generator(device=dev).manual_seed(7 + rank)
  qc = rank_to_key_torch(torch.randint(0, vocab, (ns,), device=dev, generator=gen_p))
  qd = rank_to_key_torch(vocab + 17 + torch.arange(ns, device=dev) * (rank + 1))
  q = torch.cat([qa, qb, qc, qd])
  if sharded is None:
    rows, ex = table.lookup(q, dynamic_default_values=default, return_exists=True)
  elif exchange == "nccl":
    rows, ex = sharded.lookup(q), None
  else:
    rows, ex = sharded.lookup(q, return_exists=True)
  rows = rows.reshape(-1, dim)
  e0, e1 = rows_of_keys_torch(q, dim, 0), rows_of_keys_torch(q, dim, 1)
  is0, is1, isd = (rows == e0).all(1), (rows == e1).all(1), (rows == default).all(1)
  na, nb_ = qa.numel(), qb.numel()
  good = torch.cat([is1[:na + nb_], (is0 | is1)[na + nb_:na + nb_ + ns], isd[na + nb_ + ns:]])
  if ex is not None:
    good &= torch.cat([ex[:na + nb_ + ns], ~ex[na + nb_ + ns:]])
  pm = torch.tensor([int((~good).sum()), q.numel()], dtype=torch.int64, device=dev)
  if world > 1:
    if is_peer:
      sharded.phase_barrier()
    dist.all_reduce(pm)
  parity = {"checked": int(pm[1]), "mismatches": int(pm[0]),
            "what": "after the timed region every rank looks up 16384 keys it wrote last step + 16384 per peer that the "
                    "peers wrote (generation-1 rows), 16384 random resident keys (generation 0 or 1, never torn) and "
                    "16384 absent keys (default row, exists false) and compares with the closed-form row of the key"}

  # ---- N>1: upper bound without the exchange (every rank only touches keys it owns: pure local kernels) -----
  no_exchange = None
  if world > 1:
    own_batches = []
    for kb in key_batches[:8]:
      mine = kb[de.default_partition_fn(kb, world, True) == rank]
      reps = (B + mine.numel() - 1) // max(1, mine.numel())
      own_batches.append(mine.repeat(reps)[:B].contiguous() if mine.numel() else kb)
    own_vals = [rows_of_keys_torch(kb, dim, 1) for kb in own_batches]
    for i in range(3):
      table.lookup(own_batches[i % 8], dynamic_default_values=default)
    barrier()
    n_ne = min(args.steps, 200)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for i in range(n_ne):
      table.lookup(own_batches[i % 8], dynamic_default_values=default)
      table.insert(own_batches[i % 8], own_vals[i % 8])
    a1.record()
    barrier()
    tne = torch.tensor([a0.elapsed_time(a1) / n_ne], dtype=torch.float64, device=dev)
    dist.all_reduce(tne, op=dist.ReduceOp.MAX)
    no_exchange = {"value": world * B / (float(tne.item()) * 1e-3) / 1e6, "unit": "M keys/s",
                   "note": "same step with every rank's keys pre-partitioned to the shard it owns (no NVLink traffic; "
                           "duplicate keys inside a batch because a rank owns only 1/N of a Zipf batch): separates kernel "
                           "scaling from the exchange cost"}

  # ---- e2e through the host-buffer plugin API (N=1: table ops on pinned host tensors) -------------------
  e2e = None
  if not args.no_e2e:
    prev_aff = bind_to_gpu_numa(local_rank)
    n_e2e = max(1, min(args.e2e_steps, args.steps))
    hk = [key_batches[(args.warmup + i) % n_batches].cpu().pin_memory() for i in range(n_e2e)]
    hvs = [val_batches[(args.warmup + i) % n_batches].cpu().pin_memory() for i in range(n_e2e)]
    hd = default.cpu().pin_memory()
    ho = torch.empty(B, dim).pin_memory()
    if sharded is None:
      def e2e_step(i):
        table.lookup_host(hk[i], hd, ho)
        table.insert_host(hk[i], hvs[i])
    else:
      def e2e_step(i):
        k = hk[i].to(dev, non_blocking=True)
        v = hvs[i].to(dev, non_blocking=True)
        rows = sharded.lookup(k)
        if is_peer:
          sharded.phase_barrier()
        ho.copy_(rows, non_blocking=True)
        sharded.upsert(k, v)
        if is_peer:
          sharded.phase_barrier()
        torch.cuda.synchronize()
    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(n_e2e):
      e2e_step(i)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    seq_value = world * B * n_e2e / float(dt.item()) / 1e6
    e2e = {"value": seq_value, "unit": "M keys/s",
           "h2d_bytes_per_step": int(B * (8 + 8 + dim * 4) + dim * 4), "d2h_bytes_per_step": int(B * dim * 4),
           "steps": n_e2e,
           "api": "CuckooHashTable.lookup_host + insert_host (det_find_host / det_insert_host), pinned host buffers"
                  if sharded is None else ("PeerShardedVariable" if exchange != "nccl" else "ShardedVariable") + ".lookup/upsert with pinned H2D/D2H copies"}
    if sharded is None:
      # software-pipelined flavour of the SAME per-step work: the lookup of batch i+1 (D2H-heavy) is issued
      # together with the write-back of batch i (H2D-heavy) -- input prefetch, as tf.data does for the reference
      ho2 = torch.empty(B, dim).pin_memory()
      table.lookup_host_async(hk[0], hd, ho)
      table.host_sync()
      torch.cuda.synchronize()
      t0 = time.perf_counter()
      for i in range(n_e2e):
        table.lookup_host_async(hk[(i + 1) % n_e2e], hd, ho2 if i % 2 == 0 else ho)  # D2H-heavy: rows of batch i+1
        table.insert_host_async(hk[i], hvs[i])                                      # H2D-heavy: write-back of batch i
        table.host_sync()
      dtp = time.perf_counter() - t0
      e2e["sequential_value"] = seq_value
      e2e["drained_every_step_value"] = B * n_e2e / dtp / 1e6
      e2e["value"] = e2e["drained_every_step_value"]
      e2e["api"] = ("CuckooHashTable.lookup_host_async(batch i+1) + insert_host_async(batch i) + host_sync per step "
                    "(det_insert_host_async / det_find_host_async, pinned host buffers, both PCIe directions busy); "
                    "sequential_value = lookup_host then insert_host of the same batch, back to back")
      # Same per-step work, but a step only waits for what it CONSUMES: the looked-up rows of batch i+1
      # (det_host_sync_pipe(0)); the write-back of batch i keeps draining while step i+1's copies start, everything has
      # landed before the clock stops (final host_sync).  Every step still uploads its keys / rows and downloads its
      # rows inside the timed region; no step boundary drains the link.
      try:
        table.host_sync()
        t0 = time.perf_counter()
        for i in range(n_e2e):
          table.lookup_host_async(hk[(i + 1) % n_e2e], hd, ho2 if i % 2 == 0 else ho)
          table.insert_host_async(hk[i], hvs[i])
          table.host_sync("lookup")
        table.host_sync()
        dtq = time.perf_counter() - t0
        chk = ho2 if (n_e2e - 1) % 2 == 0 else ho                   # rows of the last prefetched batch, on the host
        kq = hk[n_e2e % n_e2e]
        okq = bool(torch.equal(chk[:4096], rows_of_keys_torch(kq[:4096], dim, 1)))
        if okq and B * n_e2e / dtq / 1e6 > e2e["value"]:
          e2e["value"] = B * n_e2e / dtq / 1e6
          e2e["api"] = ("CuckooHashTable.lookup_host_async(batch i+1) + insert_host_async(batch i) per step, the step waits "
                        "for its looked-up rows only (host_sync('lookup') = det_host_sync_pipe(0)) while the write-back "
                        "drains behind; final host_sync inside the timed region; pinned host buffers, both PCIe directions "
                        "busy across steps.  drained_every_step_value = full host_sync per step; sequential_value = "
                        "lookup_host then insert_host of the same batch, back to back")
        e2e["prefetch_rows_checked"] = {"checked": 4096, "ok": okq}
      except Exception as ex:   # never lose the line over the optional flavour
        e2e["pipelined_error"] = repr(ex)

  if not args.no_e2e and prev_aff is not None:
    os.sched_setaffinity(0, prev_aff)  # the CPU baseline below must see every host core again
  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return
  peak, peak_src = measured_peak_gbs()
  find_ms_1 = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
  algo_bytes = B * dim * 4  # north_star roofline: keys x dim x 4 B per lookup launch
  achieved = algo_bytes / (find_ms_1 * 1e-3) / 1e9
  honest_bytes = B * (8 + 64 + 2 * dim * 4)  # key in + one 64 B bucket + row read + row written out
  kernels = {"none": "det::find_kernel_tma<16>",
             "hybrid": "det::xchg_route_kernel<false> + xchg_serve_find_kernel<16> (+ 2 flag waits, + peer barrier)",
             "push": "det::xchg_route_kernel<false> + xchg_serve_find_kernel<16> (+ 2 flag waits)",
             "peer": "det::peer_find_kernel<16> (+peer barrier)",
             "nccl": "partition+all_to_all+find_kernel+all_to_all+scatter"}
  launches = {"none": 2, "hybrid": 7, "push": 8, "peer": 4, "nccl": 10}
  traffic, traffic_src = (committed_traffic("find_kernel_tma<16>") if (world == 1 and B == (1 << 20) and dim == 64)
                          else (None, "only captured for the N=1 headline workload"))
  line = {
      "metric": "embedding lookup+insert M keys/s at dim%d" % dim, "value": value, "unit": "M keys/s", "n_gpus": world,
      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
      "scaling": "weak", "vs_baseline": None, "dtype": "int64 keys / f32 rows (copy; no arithmetic)",
      "data": "synthetic",
      "config": {
          "workload": "BASELINE configs[%d]: HKV-style table, %d resident keys/GPU, dim %d fp32, Zipf(%.2f) ids, "
                      "%d unique keys/step/GPU; step = Find(batch) + Insert(batch)" %
                      (3 if args.workload == "c4" else 1, resident, dim, ALPHA, B),
          "resident_keys_per_gpu": local_size, "capacity_slots": table.capacity(), "batch": B, "dim": dim,
          "l2": "inputs larger than L2: %d distinct batches are cycled, every step touches %.0f MB of rows + %.0f MB out + "
                "%.0f MB in of a %.1f GB table (no L2 flush; the Zipf head is hot by design)" %
                (n_batches, B * dim * 4 / 1e6, B * dim * 4 / 1e6, B * dim * 4 / 1e6, table.stats()["hbm_bytes"] / 1e9),
          "parallelism": ("key-hash sharded x%d, %s" % (world, {
              "hybrid": "lookups: ids pushed to the owner's mailbox, local probe, rows pushed back with posted NVLink stores "
                        "(det_peer_xchg_find); inserts: one-sided kernel, remote probe + posted row store (det_peer_insert); flag "
                        "barrier between the read and the write phase; no collective",
              "push": "owner-side exchange: ids pushed to the owner's mailbox, local probe, rows pushed back with posted "
                      "NVLink stores, flag words instead of barriers (det_peer_xchg_find/insert), no collective",
              "peer": "one-sided NVLink peer-memory kernels with remote probes (det_peer_find/insert), no collective",
              "nccl": "NCCL all-to-all of keys and rows"}[exchange])) if world > 1 else "single GPU",
      },
      "find_ms": find_ms_max, "insert_ms": ins_ms_max,
      "find_Mkeys_s": world * B / (find_ms_max * 1e-3) / 1e6, "insert_Mkeys_s": world * B / (ins_ms_max * 1e-3) / 1e6,
      "gpu_launches": launches[exchange] * args.steps,
      "clocks": clocks,
      "parity": parity,
      "roofline": {
          "bound": "hbm", "kernel": kernels[exchange], "achieved": achieved, "peak": peak, "unit": "GB/s",
          "frac": achieved / peak,
          "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_src,
          "peak_source": peak_src,
          "algorithmic_bytes_per_launch": algo_bytes,
          "honest_frac": honest_bytes / (find_ms_1 * 1e-3) / 1e9 / peak,
          "note": "algorithmic = keys x dim x 4 B (north_star definition); the kernel necessarily also moves the "
                  "gathered rows out (+%d B/key) and one 64 B bucket + 8 B key per probe: honest-traffic rate %.0f GB/s "
                  "(%.2f of peak)" % (dim * 4, honest_bytes / (find_ms_1 * 1e-3) / 1e9,
                                      honest_bytes / (find_ms_1 * 1e-3) / 1e9 / peak),
      },
  }
  if world > 1:
    # SURVEY 8e: at N > 1 the exchange is bounded by NVLink, not HBM.  Bytes one rank must SEND (= receive) per step:
    # push: (N-1)/N of its requests (8 B key + 4 B position), of the rows it serves (4*D) and of its insert pairs
    # (8 + 4*D); peer (remote probes): (N-1)/N x (64 B bucket + 4*D row) inbound per find, 64 B inbound + 4*D outbound per
    # insert.  Peak = measured peer copy, one direction (profiles/r01_peer_microbench_2gpu.jsonl 735 GB/s, 770 GB/s on
    # the 8-GPU box; nominal 900 GB/s).
    f = (world - 1) / world
    nv_bytes = f * B * {"push": 12 + dim * 4 + 8 + dim * 4, "hybrid": 12 + dim * 4 + dim * 4, "peer": 64 + dim * 4 + dim * 4,
                        "nccl": 8 + dim * 4 + 8 + dim * 4}[exchange]
    nv_peak = float(os.environ.get("DET_NVLINK_PEAK_GBS", "770"))
    line["roofline_nvlink"] = {"bound": "nvlink", "kernel": "whole step (%s)" % exchange,
                               "achieved": nv_bytes / (ms_per_step * 1e-3) / 1e9, "peak": nv_peak, "unit": "GB/s",
                               "frac": nv_bytes / (ms_per_step * 1e-3) / 1e9 / nv_peak,
                               "bytes_per_step_per_direction": nv_bytes,
                               "peak_source": "measured peer copy, one direction (DET_NVLINK_PEAK_GBS overrides)"}
  if e2e:
    if world == 1:
      # the host-buffer step moves h2d + d2h bytes over one PCIe link; measured on this pool's boxes
      # (scripts/pcie_probe.py): 55-57 GB/s per direction, 99 GB/s with both directions busy
      pcie_peak = float(os.environ.get("DET_PCIE_BIDIR_GBS", "99"))
      moved = e2e["h2d_bytes_per_step"] + e2e["d2h_bytes_per_step"]
      e2e["pcie_GBs"] = moved * e2e["value"] * 1e6 / B / 1e9
      e2e["pcie_frac"] = e2e["pcie_GBs"] / pcie_peak
      e2e["pcie_peak_source"] = "scripts/pcie_probe.py, both directions busy (DET_PCIE_BIDIR_GBS overrides)"
    line["e2e"] = e2e
  if no_exchange:
    line["no_exchange"] = no_exchange
  if world == 1 and not args.no_hard_cases:
    try:
      line["hard_cases"] = hard_cases(de, table, dev, dim, B, vocab, default, peak, key_batches)
    except Exception as ex:
      line["hard_cases"] = {"error": repr(ex)}
  if world == 1 and not args.no_c3 and dim == 64:
    # BASELINE configs[2] in the same run (the driver only records this line): free the headline table first
    try:
      table.close()
      del table, var, key_batches, val_batches
      torch.cuda.empty_cache()
      line["c3"] = c3_measure(args, steps=args.steps, warmup=5)
    except Exception as ex:
      if args.dump_outputs:
        raise   # the c3 output was asked for: no silent gap in the dump
      line["c3"] = {"error": repr(ex)}
  if world == 1 and not args.no_cpu_baseline:
    try:
      cb = cpu_arm(dim, args.cpu_resident, B, steps=15, warmup=3, threads=args.cpu_threads, want_resident=args.resident)
      cb.pop("ms_per_step", None)
      line["cpu_baseline"] = cb
    except Exception as ex:  # the checker is optional for the bench line; never hide the GPU number
      line["cpu_baseline"] = {"value": None, "unit": "M keys/s", "cores": 0, "kind": "unavailable", "sample": repr(ex)}
  print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


def reference_arm(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  steps = max(20, min(args.steps, 40))     # >= 20 timed steps after >= 5 warm-ups, bounded so the run ends in minutes
  warm = max(5, min(args.warmup, 10))
  cb = cpu_arm(args.dim, args.cpu_resident, args.batch, steps=steps, warmup=warm, threads=args.cpu_threads,
               want_resident=args.resident)
  ms = cb.pop("ms_per_step")
  line = {
      "impl": "reference", "metric": "embedding lookup+insert M keys/s at dim%d" % args.dim, "value": cb["value"],
      "unit": "M keys/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms,
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "int64 keys / f32 rows (copy; no arithmetic)", "data": "synthetic",
      "config": {"workload": "BASELINE configs[1] on the reference's CPU cuckoo path (TableWrapperOptimized over "
                             "libcuckoo): " + cb["sample"], "batch": args.batch, "dim": args.dim,
                 "resident_keys": cb["resident"], "same_resident_as_gpu_arm": cb["same_resident_as_gpu_arm"]},
      "find_Mkeys_s": cb["find_Mkeys_s"], "insert_Mkeys_s": cb["insert_Mkeys_s"],
      "value_min": cb["value_min"], "value_max": cb["value_max"],
      "cpu_baseline": cb,
      "e2e": {"value": cb["value"], "unit": "M keys/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "gpu_launches": 0,
  }
  print(json.dumps(line))


def c3_arm(args):
  print(json.dumps(c3_measure(args, args.steps, args.warmup)))


def c3_measure(args, steps, warmup):
  """Secondary workload, BASELINE configs[2]: fused embedding_lookup_sparse + Adagrad, 26 Criteo-shaped sparse
  features x batch 65536 (nnz = 1,703,936 ids/step, one id per (sample, feature)), dim 64, single GPU.
  Step = forward (det_lookup_sparse: ids -> [nnz, dim] rows, combiner sum) + tf.unique of the ids + per-unique
  gradient sum + fused find-or-insert Adagrad (det_apply_adagrad).  Not the headline metric."""
  import torch
  from recommenders_addons_b200 import dynamic_embedding as de
  from recommenders_addons_b200.dynamic_embedding.ops import lookup_sparse_fused
  dev = torch.device("cuda", 0)
  torch.cuda.set_device(0)
  dim, nfeat, batch = args.dim, 26, 65536
  rng = np.random.default_rng(45)
  vocab = np.exp(rng.uniform(np.log(1e3), np.log(4e7), nfeat))
  vocab = np.maximum(1000, (vocab / vocab.sum() * 1e8)).astype(np.int64)  # ~1e8 rows in total
  gen = torch.Generator(device=dev).manual_seed(42)
  total = int(vocab.sum())
  var = de.Variable(dim=dim, init_size=2 * total, initializer=0.0, num_slot_planes=1, name="c3_table")
  table = var.tables[0]
  offs = np.concatenate([[0], np.cumsum(vocab)])[:-1]
  for b in range(0, total, 1 << 20):  # resident: every (feature, rank) key
    r = torch.arange(b, min(total, b + (1 << 20)), dtype=torch.int64, device=dev)
    k = rank_to_key_torch(r)
    table.insert(k, rows_of_keys_torch(k, dim, 0))
  cdfs = [zipf_cdf_torch(int(v), dev) for v in vocab]
  nb = max(1, min(steps + warmup, 16))
  batches = []
  for _ in range(nb):
    cols = [torch.searchsorted(c, torch.rand(batch, dtype=torch.float64, device=dev, generator=gen)).clamp_(max=c.numel() - 1) + int(o)
            for c, o in zip(cdfs, offs)]
    batches.append(rank_to_key_torch(torch.stack(cols, 1).reshape(-1)))  # row-major (sample, feature)
  del cdfs
  nnz = batch * nfeat
  seg = torch.arange(nnz, device=dev, dtype=torch.int32)
  gout = torch.randn(nnz, dim, device=dev, generator=gen) * 0.01  # upstream gradient of every (sample, feature) row
  opt = de.FusedAdagrad(0.01, 0.1)

  def backward(ids):
    opt.iterations += 1
    if args.grad_reduce == "det":
      # ONE C call: unique -> position-order gradient sum -> fused find-or-insert Adagrad, count stays on the device
      opt.apply_sparse_duplicate_indices(var, ids, gout)
    else:   # A/B: eager composition with torch index_add (atomics) and a host-side unique count
      uniq, idx = de.unique(ids)
      g = torch.zeros((uniq.numel(), dim), device=dev).index_add_(0, idx.long(), gout)
      opt.apply_sparse(var, uniq, g)

  def step(i):
    ids = batches[i % nb]
    out = lookup_sparse_fused(var, ids, seg, None, nnz, "sum")
    backward(ids)
    return out

  # parity of the fused forward before any optimizer step: one id per output row and combiner sum, so row i of the
  # output must be the closed-form generation-0 row of ids[i], bit for bit
  o0 = lookup_sparse_fused(var, batches[0], seg, None, nnz, "sum")
  parity = {"checked": nnz, "mismatches": int((o0 != rows_of_keys_torch(batches[0], dim, 0)).any(1).sum()),
            "what": "det_lookup_sparse output of the first batch vs the closed-form rows of its ids (before any update)"}
  del o0
  for i in range(warmup):
    step(i)
  torch.cuda.synchronize()
  t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t0.record()
  for i in range(steps):
    out = step(warmup + i)
  t1.record()
  torch.cuda.synchronize()
  ms = t0.elapsed_time(t1) / steps
  if args.dump_outputs:
    dump_rows(args.dump_outputs, "c3_lookup_sparse", out)
  del out
  # where the step goes: the same step with CUDA events between its phases (outside the timed region)
  phases = {"lookup_sparse": [], "backward_unique_gradsum_apply": []}
  for i in range(5):
    ids = batches[i % nb]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    lookup_sparse_fused(var, ids, seg, None, nnz, "sum")
    ev[1].record()
    backward(ids)
    ev[2].record()
    torch.cuda.synchronize()
    for k, name in enumerate(phases):
      phases[name].append(ev[k].elapsed_time(ev[k + 1]))
  phases_ms = {k: float(np.median(v)) for k, v in phases.items()}
  # host synchronisations inside a step: torch raises on any synchronising call in this mode (.item(), blocking copies)
  host_syncs = None
  try:
    torch.cuda.set_sync_debug_mode("error")
    try:
      for i in range(3):
        step(i)
      host_syncs = 0
    except RuntimeError as ex:
      host_syncs = "at least one (%s)" % str(ex).splitlines()[0][:120]
    finally:
      torch.cuda.set_sync_debug_mode("default")
  except Exception:
    pass
  torch.cuda.synchronize()
  uniq = de.unique(batches[0])[0]
  # algorithmic traffic of the step (SURVEY 8d): forward rows + ids/segs + out, gradient rows read once + sums written,
  # 5 x dim x 4 B per unique key for the fused Adagrad
  n_u = int(uniq.numel())
  step_bytes = nnz * dim * 4 + nnz * 12 + nnz * dim * 4 + (nnz + n_u) * dim * 4 + 5 * n_u * dim * 4
  peak, peak_src = measured_peak_gbs()
  table.close()
  return ({"metric": "fused embedding_lookup_sparse + Adagrad step, M ids/s (BASELINE configs[2])",
                    "phases_ms": phases_ms, "parity": parity, "host_syncs_per_step": host_syncs,
                    "roofline": {"bound": "hbm", "kernel": "whole step (lookup_sparse + unique + grad_reduce + apply_adagrad)",
                                 "achieved": step_bytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                 "frac": step_bytes / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                                 "algorithmic_bytes_per_step": step_bytes},
                    "value": nnz / ms / 1e3, "unit": "M ids/s", "n_gpus": 1, "steps": steps, "warmup": warmup,
                    "ms_per_step": ms, "higher_is_better": True, "data": "synthetic",
                    "config": {"workload": "26 features x batch 65536, dim %d, %d resident rows, Zipf(1.05) per feature; "
                                           "includes tf.unique + the per-unique gradient sum (%s)" % (dim, total, "one det_apply_adagrad_dup call: det_unique + det_segment_reduce in position order + fused Adagrad, device-side count" if args.grad_reduce == "det" else "torch index_add, host-side unique count"),
                               "nnz": nnz, "unique_per_step": n_u}})


def c5_arm(args):
  """Secondary workload, BASELINE configs[4] (torchrun, N GPUs): DLRM-style forward + backward over ONE key-hash
  sharded table (26 features share it through salted keys), dim 128, global batch 131072, half-sync sparse update.
  Per step and rank: tf.unique of the rank's ids -> one-sided sharded lookup (det_peer_find) -> dense tower stubbed
  by an all-reduce of a fixed 50 MB buffer -> per-unique row gradients routed to their owners over NVLink
  (det_peer_route), duplicates combined, fused Adagrad on the owner (det_apply_adagrad).  Not the headline."""
  import torch
  import torch.distributed as dist
  from recommenders_addons_b200 import dynamic_embedding as de
  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
  os.environ["DET_GRAD_REDUCE"] = args.grad_reduce   # the owner-side combine of PeerShardedVariable.apply_gradients
  torch.cuda.set_device(local_rank)
  dev = torch.device("cuda", local_rank)
  dist.init_process_group("nccl", device_id=dev)
  dim, nfeat, gbatch = 128, 26, 131072
  # BASELINE configs[4] asks for 2B rows of dim 128 on 8 GPUs: 2e9 x 512 B = 1 TB of rows plus 1 TB of Adagrad
  # accumulators -- more than the 8 x 180 GB of the box at ANY load factor.  Resident here: the most that fits next to
  # the accumulator plane and the inboxes, 80M rows per GPU in 128M slots (load 0.625): 128M x (8 + 2 x 512) B = 132 GB.
  resident = min(args.resident, 80_000_000)          # rows per GPU actually resident (of the 2B-row key space)
  vocab = resident * world
  sv = de.PeerShardedVariable.create(dim, int(1.6 * resident), initializer=0.0, num_slot_planes=1, name="c5_table")
  table = sv.local.tables[0]
  gen = torch.Generator(device=dev).manual_seed(42 + rank)
  for b in range(rank * resident, (rank + 1) * resident, 1 << 20):   # every rank writes 1/N of the rows through the sharded table
    k = rank_to_key_torch(torch.arange(b, min((rank + 1) * resident, b + (1 << 20)), dtype=torch.int64, device=dev))
    sv.upsert(k, rows_of_keys_torch(k, dim, 0))
  sv.phase_barrier()
  torch.cuda.synchronize()
  dist.barrier()
  cdf = zipf_cdf_torch(vocab, dev)
  ids_per_rank = gbatch // world * nfeat
  owner_side = args.exchange in ("push", "hybrid")
  if owner_side:   # forward and backward through the owners: no inbox round trip, every count stays on the device
    sv.attach_exchange(ids_per_rank)
  else:            # round-1 path: remote-probe lookup, inbox + host-side split counts
    sv.attach_inbox(ids_per_rank)
  nb = max(1, min(args.steps + args.warmup, 16))
  batches = [rank_to_key_torch(torch.searchsorted(cdf, torch.rand(ids_per_rank, dtype=torch.float64, device=dev, generator=gen))
                               .clamp_(max=vocab - 1)) for _ in range(nb)]
  del cdf
  dense = torch.zeros(50 * 1024 * 1024 // 4, device=dev)
  opt = de.FusedAdagrad(0.01, 0.1)

  def step(i):
    ids = batches[i % nb]
    uniq, idx = de.unique(ids)
    rows = sv.lookup(uniq)                          # forward: sharded lookup of the unique ids
    sv.phase_barrier()
    emb = rows[idx.long()]                          # [ids, dim] activations handed to the dense tower
    dist.all_reduce(dense)                          # half-sync: only the dense tower is all-reduced
    gout = emb * 1e-3                               # stand-in for the tower's gradient w.r.t. the activations
    if args.grad_reduce == "det":
      g = de.segment_reduce(gout, idx, uniq.numel())
    else:
      g = torch.zeros_like(rows).index_add_(0, idx.long(), gout)
    sv.apply_gradients(opt, uniq, g)                # backward: route -> combine -> fused Adagrad on the owner

  for i in range(args.warmup):
    step(i)
  torch.cuda.synchronize()
  dist.barrier()
  t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t0.record()
  for i in range(args.steps):
    step(args.warmup + i)
  t1.record()
  torch.cuda.synchronize()
  dist.barrier()
  ms = torch.tensor([t0.elapsed_time(t1) / args.steps], dtype=torch.float64, device=dev)
  dist.all_reduce(ms, op=dist.ReduceOp.MAX)
  if rank == 0:
    print(json.dumps({"metric": "DLRM-style sharded forward+backward step, M ids/s (BASELINE configs[4])",
                      "value": gbatch * nfeat / float(ms.item()) / 1e3, "unit": "M ids/s", "n_gpus": world,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(ms.item()),
                      "higher_is_better": True, "scaling": "strong", "data": "synthetic",
                      "config": {"workload": "26 features x global batch %d, dim %d, %d resident rows/GPU (2B-row key space), "
                                             "Zipf(1.05); unique -> sharded lookup -> 50 MB dense all-reduce -> sharded optimizer step (%s)" %
                                             (gbatch, dim, resident, "det_peer_xchg_find + det_peer_xchg_apply_adagrad: owner-side, counts on the device"
                                              if owner_side else "det_peer_find + det_peer_route / inbox / host counts / det_apply_adagrad"),
                                 "grad_reduce": args.grad_reduce, "ids_per_rank": ids_per_rank, "unique_per_rank": int(de.unique(batches[0])[0].numel())}}))
  dist.destroy_process_group()


if __name__ == "__main__":
  a = parse_args()
  if a.impl == "reference":
    reference_arm(a)
  elif a.workload == "c3":
    c3_arm(a)
  elif a.workload == "c5":
    c5_arm(a)
  else:
    gpu_arm(a)
