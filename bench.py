#!/usr/bin/env python
"""bench.py — FID lookups/s of the embedding hot path on synthetic MovieLens-shaped batches.

Workload (BASELINE.json configs[1], SURVEY.md §8d C2): one table, dim 32, 10 M resident keys,
Adagrad(lr .05, init_acc .1); a batch = B samples x 2 slots (uid, movie), one FID per slot,
FID = (slot << 48) | rank, rank ~ truncated Zipf(1.05) over 5 M ids per slot.

One "step" = the whole sparse part of one training step for one batch:
    forward : fused probe + row gather + per-slot pool of the M = 2B FID occurrences -> pooled [B, 2*32]
    backward: group the occurrences by FID (scratch set + stable radix sort), deterministic per-FID sum of
              the pooled grads (no float atomics), fused Adagrad update + expiry-timestamp bump (upsert)
  N > 1 (torchrun, one rank per GPU, weak scaling): the same step sharded by fid mod N (ShardedStep): group by
  owner, FIDs / rows / row gradients exchanged through fixed NVLink peer-window regions by the kernels
  themselves (device-side counts, per-source flags, no host synchronisation inside the step: xstep.cu);
  owners apply the requesters' gradients in rank order.  --exchange peer|nccl select the older paths.
`value`  = FID occurrences (lookups) per second over all ranks, inputs resident in HBM; median of --repeats
           timed regions of --steps steps each.
`e2e`    = the same step through the public Python API with pinned HOST inputs: per step the FIDs and labels
           are copied H2D (prefetched on a copy stream), forward, a small bf16 tower (64-64-1) on the device
           produces the loss and the pooled gradients, backward, and the loss is read back D2H.
`parity_check` = before timing, every rank runs a few small steps through the same sharded path and rank 0
           compares all tables with ONE global oracle table fed the concatenated batches.
`--impl reference` times a multi-threaded CPU implementation of the same step (oracle/oracle.cc orc_fastps_*:
partition-parallel dedup, flat hash shards; checked against the plain restatement in tests) on the host
cores; the reference itself needs bazel + TensorFlow and cannot be built here.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIM = 32
SLOTS = 2
LR = 0.05
INIT_ACC = 0.1
ZIPF_S = 1.05
METRIC = "fid_lookups_per_sec"
UNIT = "lookups/s"


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--new-frac", type=float, default=0.05, help="c4: fraction of a step's FID occurrences that are never-seen FIDs")
  ap.add_argument("--evict-every", type=int, default=8, help="c4: steps between TTL eviction scans")
  ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c5"],
                  help="c2 (default; BASELINE.json configs[1], the metric's config): MovieLens-shaped, 1 table dim 32, 2 slots, 10 M keys; "
                       "c3: Criteo-shaped, 26 slots dim 16 in one table, 26 M keys, batch 65 536 per GPU; "
                       "c4: streaming insert+evict, 200 slots dim 16, 125 M keys per GPU, batch 8192 per GPU; "
                       "c5: table sweep dim 8..128 (lookup and lookup+Adagrad GB/s), single GPU")
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (default: 1 048 576 for c2, 65 536 for c3)")
  ap.add_argument("--keys", type=int, default=None, help="resident keys per GPU (default: 10 M for c2 / c5, 26 M for c3)")
  ap.add_argument("--cpu-batch", type=int, default=None,
                  help="samples per step of the CPU arm / cpu_baseline (default: --batch, so that both arms run the same config)")
  ap.add_argument("--cpu-threads", type=int, default=0,
                  help="threads (= PS shards) of the CPU arm; 0 = sweep {1, 8, 16, 32, 64, 128} <= host cores and keep the best")
  ap.add_argument("--repeats", type=int, default=5, help="the timed region of --steps steps is repeated this often; the median is reported")
  ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity check that precedes the timed region")
  ap.add_argument("--no-extras", action="store_true", help="skip the extra roofline lines (uniform FIDs, CSR pooling, small batch)")
  ap.add_argument("--zipf", type=float, default=ZIPF_S, help="Zipf exponent of the FID ranks (0 = uniform)")
  ap.add_argument("--ab", default="", help="tuning A/B after the main timing: ';'-separated option sets 'name=v,name=v' "
                  "(mono_set_option knobs), each timed like the main region; reported under roofline.ab")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-e2e", action="store_true")
  ap.add_argument("--e2e-chunks", type=int, default=8,
                  help="e2e leg: slices of the pooled-rows D2H / gradient H2D round trip (1 = sequential copies)")
  ap.add_argument("--no-prepare", action="store_true",
                  help="exchange=direct: do NOT build the next batch's grouping on a side stream under the step in flight")
  ap.add_argument("--sharded", action="store_true", help="run the sharded step (ShardedStep) even at N=1 (profiling)")
  ap.add_argument("--remote-frac", type=float, default=None,
                  help="experiment: fraction of a rank's FID occurrences owned by other ranks (default: natural 1 - 1/N)")
  ap.add_argument("--exchange", default=None, choices=["direct", "peer", "nccl"],
                  help="exchange of the sharded step: 'direct' = device-driven (fixed window regions, directional flags, no host "
                       "round trip), 'peer' = host-driven NVLink peer windows with flag barriers, 'nccl' = NCCL all-to-all")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, fixed seeded "
                       "samples, see dump_outputs) so that two builds can be compared output for output; c2 / c3 only")
  args = ap.parse_args()
  if args.dump_outputs and (args.impl == "reference" or args.workload in ("c4", "c5")):
    ap.error("--dump-outputs applies to the GPU step of workloads c2 and c3")
  global DIM, SLOTS
  if args.workload == "c3":
    DIM, SLOTS = 16, 26
    args.batch = args.batch or (1 << 16)
    args.keys = args.keys or 26_000_000
  elif args.workload == "c4":
    args.batch = args.batch or (1 << 13)
    args.keys = args.keys or 125_000_000
  else:
    args.batch = args.batch or (1 << 20)
    args.keys = args.keys or 10_000_000
  return args


# ---------------------------------------------------------------------------------------------
# synthetic inputs
# ---------------------------------------------------------------------------------------------
class Zipf:
  """Truncated Zipf(s) over ranks [0, n) by inverse CDF."""

  def __init__(self, n, s):
    w = np.arange(1, n + 1, dtype=np.float64)**(-s)
    self.cdf = np.cumsum(w)
    self.cdf /= self.cdf[-1]

  def sample(self, rng, size):
    return np.searchsorted(self.cdf, rng.random(size), side="left").astype(np.int64)


def make_batches(n_batches, batch, keys_per_slot, seed, zipf_s=ZIPF_S, remote=None):
  """remote = (frac, world, rank): experiment knob (--remote-frac) that re-draws the owner of every FID so
  that `frac` of a rank's occurrences belong to OTHER ranks (emulates the N=8 traffic volume on 2 GPUs)."""
  rng = np.random.default_rng(seed)
  z = Zipf(keys_per_slot, zipf_s)
  # rank -> id via a fixed permutation-free affine map so that hot ids are spread over the table
  out = []
  for _ in range(n_batches):
    cols = []
    for s in range(1, SLOTS + 1):
      rank = z.sample(rng, batch)
      ident = (rank * 2654435761) % keys_per_slot  # bijection on [0, keys_per_slot) only if coprime; fine: stays in range
      if remote is not None:
        frac, world, me = remote
        other = (me + 1 + rng.integers(0, max(world - 1, 1), batch)) % world
        owner = np.where(rng.random(batch) < frac, other, me)
        ident = np.minimum((ident // world) * world + owner, keys_per_slot - 1)
      cols.append((np.int64(s) << np.int64(48)) | ident)
    out.append(np.stack(cols, 1).reshape(-1))  # sample-major: fid index = b * SLOTS + slot
  return out


def fwd_bytes(M, U, D=None):
  """SURVEY.md §8(d): 8*M (FIDs) + U*(32 (bucket sector) + 4D (row)) + 4*D*R (pooled rows), R == M here."""
  D = DIM if D is None else D
  return 8 * M + U * (32 + 4 * D) + 4 * D * M


def bwd_bytes(M, U, D=None):
  """SURVEY.md §8(d) backward (scatter + Adagrad): 4*D*R + U*(32 + 16*D + 8)."""
  D = DIM if D is None else D
  return 4 * D * M + U * (32 + 16 * D + 8)


# ---------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------
class Clocks:

  def __init__(self, index):
    self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
    self.ok = False
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nv = pynvml
      self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
      self.ok = True
    except Exception:
      pass

  def _run(self):
    nv = self.nv
    names = {
        getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
        getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
        getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
        getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
    }
    while not self._stop.is_set():
      try:
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        try:
          r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
          r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for bit, name in names.items():
          if r & bit:
            self.reasons.add(name)
      except Exception:
        pass
      self._stop.wait(0.05)

  def __enter__(self):
    if self.ok:
      self.t = threading.Thread(target=self._run, daemon=True)
      self.t.start()
    return self

  def __exit__(self, *a):
    if self.ok:
      self._stop.set()
      self.t.join()

  def summary(self):
    if not self.samples:
      return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
    return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------
# CPU arm (reference PS path, oracle port)
# ---------------------------------------------------------------------------------------------
def _fastps(lib, keys, threads):
  import ctypes as C
  from monolith_b200 import entry
  seg = entry.CombineAsSegment(DIM, entry.RandomUniformInitializer(-0.05, 0.05),
                               entry.AdagradOptimizer(LR, INIT_ACC))
  cfg = {"item": entry.HashTableConfigInstance(entry.TableConfig([seg], initial_capacity=keys, init_seed=1), [LR])}
  arr, keep = entry.to_c_table_cfgs(cfg)
  ps = C.c_void_p()
  lib.orc_fastps_create(arr, threads, C.byref(ps))
  t0 = time.time()
  lib.orc_fastps_fill_slots(ps, SLOTS, C.c_int64(keys // SLOTS))
  return ps, time.time() - t0, keep


def cpu_arm(keys, batch, steps, warmup, threads, zipf_s=ZIPF_S, candidates=(1, 8, 16, 32, 64, 128)):
  """Times the tuned CPU restatement of the reference PS path (oracle/oracle.cc orc_fastps_train_step: persistent
  worker pool, flat per-shard tables, dedup / scatter partitioned by shard, reference AVX Adagrad, built
  -O3 -mavx -mavx2 -mfma) on the SAME workload as the GPU arm.  threads = PS shards = worker threads; 0 = sweep
  `candidates` (one timed step each after one warm-up step) and keep the fastest."""
  import ctypes as C
  from tests import orc
  lib = orc.lib()
  lib.orc_fastps_train_step.restype = C.c_int64
  cores = os.cpu_count() or 1
  keys_per_slot = keys // SLOTS
  batches = make_batches(4, batch, keys_per_slot, seed=2, zipf_s=zipf_s)
  M = batch * SLOTS
  rng = np.random.default_rng(5)
  pg = rng.standard_normal((M, DIM)).astype(np.float32)
  out = np.zeros((M, DIM), np.float32)
  lr = np.array([LR], np.float32)

  def one(ps, i):
    f = batches[i % len(batches)]
    t0 = time.perf_counter()
    u = lib.orc_fastps_train_step(ps, orc.p(f), C.c_int64(M), None, C.c_int64(M), 0, orc.p(pg), orc.p(out), orc.p(lr),
                                  C.c_int64(1000 + i))
    return time.perf_counter() - t0, u

  sweep = {}
  if threads <= 0:
    cand = sorted({min(c, cores) for c in candidates} | {cores})
    best = None
    for c in cand:
      ps, _, keep = _fastps(lib, keys, c)
      one(ps, 0)
      one(ps, 1)
      dt = min(one(ps, 2)[0], one(ps, 3)[0])
      lib.orc_fastps_destroy(ps)
      sweep[c] = M / dt
      if best is None or dt < best[0]:
        best = (dt, c)
    threads = best[1]
  ps, fill_s, keep = _fastps(lib, keys, threads)
  times, uniq = [], []
  warmup = max(warmup, 3)
  for i in range(warmup + steps):
    dt, u = one(ps, i)
    if i >= warmup:
      times.append(dt)
      uniq.append(u)
  lib.orc_fastps_destroy(ps)
  # the value is the BEST step: the host is shared with other tenants and its timing jitters by 2x; the minimum is the
  # number most favourable to the CPU baseline
  med = float(np.min(times))
  return {"value": M / med, "ms_per_step": 1e3 * med, "ms_per_step_mean": 1e3 * float(np.mean(times)), "fill_s": fill_s, "batch": batch,
          "M": M, "U_mean": float(np.mean(uniq)), "threads": threads, "host_cores": cores,
          "thread_sweep_lookups_per_s": {str(k): v for k, v in sweep.items()},
          "ms_per_step_min": 1e3 * float(np.min(times)), "ms_per_step_max": 1e3 * float(np.max(times))}


CPU_KIND_NOTE = ("tuned CPU restatement of the reference PS path (persistent pool, flat per-shard tables, shard-partitioned "
                 "dedup/scatter, reference AVX Adagrad, -O3 -mavx2 -mfma); the reference itself needs bazel + TensorFlow and "
                 "cannot be built here")


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  batch = args.cpu_batch or args.batch
  r = cpu_arm(args.keys, batch, args.steps, args.warmup, args.cpu_threads, args.zipf)
  line = {
      "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
      "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
      "config": workload_config(args, batch),
      "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["threads"], "host_cores": r["host_cores"], "kind": "port",
                       "thread_sweep_lookups_per_s": r["thread_sweep_lookups_per_s"],
                       "ms_per_step_min": r["ms_per_step_min"], "ms_per_step_max": r["ms_per_step_max"],
                       "sample": f"{args.steps} steps x {r['M']} FIDs (batch {batch} samples) on a {args.keys}-key "
                                 f"table; {CPU_KIND_NOTE}"},
      "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "gpu_launches": 0,
  }
  print(json.dumps(line), flush=True)


def workload_config(args, batch):
  head = ("C3 Criteo-shaped DeepFM sparse step: 26 slots dim 16 in one table, Adagrad, " if getattr(args, "workload", "c2") == "c3"
          else "C2 MovieLens-shaped DSSM sparse step: 1 table dim 32 Adagrad, 10M resident keys, 2 slots/sample, ")
  return {
      "workload": head + "Zipf(1.05) FIDs; step = fused lookup+pool fwd + fused backward (group FIDs, deterministic per-FID grad "
                  "reduce, Adagrad upsert with expiry bump)" + (
                      "; sharded: group by owner, FID/row/grad exchange over NVLink peer windows (fused lookup+send, reduce+send; device-driven: fixed per-source regions, directional flags, no host round trip)"
                      if (args.gpus > 1 or getattr(args, "sharded", False)) else ""),
      **({"remote_frac_experiment": args.remote_frac} if getattr(args, "remote_frac", None) is not None else {}),
      "zipf_s": args.zipf, "keys": args.keys, "dim": DIM, "slots": SLOTS, "batch_per_gpu": batch, "fids_per_step_per_gpu": batch * SLOTS,
      "l2_hygiene": "inputs larger than L2: 2.6 GB table + 4 rotating batches, 268 MB pooled output per step",
      "parallelism": (f"fid-hash sharding x{args.gpus}, exchange={getattr(args, 'exchange', None) or os.environ.get('MONO_EXCHANGE', 'direct')}"
                      if (args.gpus > 1 or getattr(args, "sharded", False)) else "single GPU"),
  }


# ---------------------------------------------------------------------------------------------
# parity check (oracle as the checker; runs before the timed region, on every rank)
# ---------------------------------------------------------------------------------------------
def _parity_batch(rank, step, n=6000):
  rng = np.random.default_rng(1000 * step + rank)
  ids = rng.integers(0, 900, n)
  ids[rng.random(n) < 0.25] = 3                    # hot FID shared by every rank (a > 64-occurrence run)
  new = rng.random(n) < 0.02                       # FIDs first seen in this step (upserts), a few occurrences each
  ids[new] = 2000 + 50 * step + rng.integers(0, 50, int(new.sum()))
  fids = (np.int64(5) << 48) | ids.astype(np.int64)
  g = rng.standard_normal((n, 16)).astype(np.float32)
  return fids, g


def parity_check(world, rank, dev, steps=3):
  """One small sparse train job (3 steps x 6000 FIDs per rank, one hot FID shared by all ranks, new FIDs every step)
  run through the SAME path the timed region uses (N = 1: lookup_pool + pool_backward; N > 1: ShardedStep over the
  NVLink peer windows), then compared on rank 0 with ONE global oracle table that applies the requesters' gradients
  in rank order (ref protocol: NT/distributed_ps_test.py:892-975): pooled rows and final entries [emb | Adagrad state |
  ts] bit for bit for FIDs whose gradient sums have <= 64 terms (reference summation order); the hot FID (1500-term
  sums: piecewise fp32 on the GPU, sequential fp32 on the CPU; tests/test_gpu_parity.py checks both against fp64)
  within `hot_tolerance`, with the measured error reported."""
  import torch
  import torch.distributed as dist
  from monolith_b200 import MultiHashTable, entry
  D = 16
  hot = (np.int64(5) << 48) | np.int64(3)

  def cfg():
    seg = entry.CombineAsSegment(D, entry.RandomUniformInitializer(-0.05, 0.05), entry.AdagradOptimizer(0.1, 0.1))
    return {"t": entry.HashTableConfigInstance(entry.TableConfig([seg], initial_capacity=64, init_seed=9), [0.1])}

  table = MultiHashTable(cfg(), device=dev)
  st = None
  if world > 1:
    from monolith_b200.distributed_ps import ShardedStep
    st = ShardedStep(table, "t", D, world, rank, dev)
  pooled_all = []
  for step in range(steps):
    fids, g = _parity_batch(rank, step)
    f_d, g_d = torch.from_numpy(fids).to(dev), torch.from_numpy(g).to(dev)
    out = torch.empty(fids.size, D, device=dev)
    if st is None:
      table.lookup_pool("t", f_d, None, "sum", out=out)
      table.pool_backward("t", f_d, g_d, None, "sum", req_time=20 + step)
    else:
      st.step(f_d, g_d, out, 20 + step)
    pooled_all.append(out.cpu().numpy())
  ks, rows = [], []
  for ids, raw in table.export("t", chunk=1 << 14):
    ks.append(ids.cpu().numpy())
    rows.append(raw.cpu().numpy())
  ks, rows = np.concatenate(ks), np.concatenate(rows)
  o = np.argsort(ks)
  mine = (pooled_all, ks[o], rows[o])
  if st is not None and st.window is not None:
    torch.cuda.synchronize(dev)
    st.window.close(None)
  table.close()
  if world > 1:
    got = [None] * world
    dist.all_gather_object(got, mine)
  else:
    got = [mine]
  if rank != 0:
    return None
  from tests import orc
  glob = orc.OracleMultiHashTable(cfg())
  res = {"ranks": world, "steps": steps, "fids_per_rank_per_step": 6000, "ok": True, "pooled_rows_bit_exact": 0,
         "pooled_rows_hot": 0, "entries_bit_exact": 0, "hot_max_rel_err": 0.0, "errors": []}

  def rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-3))) if a.size else 0.0

  try:
    for step in range(steps):
      batches = [_parity_batch(r, step) for r in range(world)]
      for r, (fids, g) in enumerate(batches):
        want = glob.lookup_pool("t", fids, None, "sum")
        cold = fids != hot
        np.testing.assert_array_equal(got[r][0][step][cold].view(np.uint32), want[cold].view(np.uint32))
        res["pooled_rows_bit_exact"] += int(cold.sum())
        res["pooled_rows_hot"] += int((~cold).sum())
        res["hot_max_rel_err"] = max(res["hot_max_rel_err"], rel(got[r][0][step][~cold], want[~cold]))
      for r, (fids, g) in enumerate(batches):      # owners apply requester 0's rows, then requester 1's, ...
        u, inv = orc.dedup(fids)
        ug = orc.gather_pool_grad(g, inv * D, D, u.size * D).reshape(-1, D)
        glob.apply_gradients({"t": (u, ug)}, req_time=20 + step)
    keys = glob.keys("t")
    for r in range(world):
      own = keys[(keys.view(np.uint64) % np.uint64(world)) == r]
      k_r, e_r = got[r][1], got[r][2]
      np.testing.assert_array_equal(k_r, own)
      want = glob.lookup_entry("t", own)
      cold = own != hot
      np.testing.assert_array_equal(e_r[cold].view(np.uint32), want[cold].view(np.uint32))
      res["entries_bit_exact"] += int(cold.sum())
      np.testing.assert_array_equal(e_r[~cold][:, -2:].view(np.uint32), want[~cold][:, -2:].view(np.uint32))
      res["hot_max_rel_err"] = max(res["hot_max_rel_err"], rel(e_r[~cold][:, :-2], want[~cold][:, :-2]))
    if res["hot_max_rel_err"] > 2e-3:
      raise AssertionError(f"hot FID differs by {res['hot_max_rel_err']:.3g} relative")
  except AssertionError as e:
    res["ok"] = False
    res["errors"].append(str(e)[:400])
  res["hot_tolerance"] = 2e-3
  return res


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def bind_numa(local):
  """Pin this process (and the pinned buffers it allocates afterwards) to the CPUs next to its GPU: 8 ranks driving
  PCIe from the wrong socket cost the e2e leg 2.9x per GPU in round 1."""
  try:
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(local)
    words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
    cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
    cpus &= set(os.sched_getaffinity(0))
    if cpus:
      os.sched_setaffinity(0, cpus)
      return len(cpus)
  except Exception:
    pass
  return None


class Tower:
  """Stand-in dense tower of the DSSM (ref model: markdown/demo/demo_model.py:47-84): pooled [B, 2*32] -> bf16 MLP
  64 -> 64 -> 1 -> logistic loss against labels; forward + backward produce the gradient w.r.t. the pooled rows.
  Dense layers are out of scope (SURVEY §8): plain torch / cuBLAS on tensor cores, used only to close the e2e loop on
  the device and as the thing the exchange overlaps with."""

  def __init__(self, dev, batch, seed=0, lib=None):
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    self.w1 = (torch.randn(SLOTS * DIM, 64, device=dev, generator=g) * 0.05).to(torch.bfloat16)
    self.w2 = (torch.randn(64, 1, device=dev, generator=g) * 0.05).to(torch.bfloat16)
    self.batch = batch
    self.lib = lib   # the engine library: the tower runs as ONE fused kernel (csrc/tower.cu); None: the torch formulation
    if lib is not None:
      self.scratch = torch.empty(int(lib.mono_bench_tower_scratch_floats()), device=dev)
      self.loss = torch.zeros(1, device=dev)
      self.w2v = self.w2[:, 0].contiguous()

  def grad(self, pooled, labels, grad_out):
    """loss (device scalar) and d loss / d pooled written into grad_out [M, DIM]."""
    import torch
    if self.lib is None:
      return self.grad_torch(pooled, labels, grad_out)
    rc = self.lib.mono_bench_tower_grad(pooled.data_ptr(), self.batch, labels.data_ptr(), self.w1.data_ptr(),
                                        self.w2v.data_ptr(), grad_out.data_ptr(), self.loss.data_ptr(),
                                        self.scratch.data_ptr(), self.scratch.numel(),
                                        torch.cuda.current_stream().cuda_stream)
    if rc != 0:
      raise RuntimeError(self.lib.mono_last_error().decode())
    return self.loss[0]

  def grad_torch(self, pooled, labels, grad_out):
    """The same tower through torch / cuBLAS with a hand-written backward (no autograd graph): 0.68 ms per 524288-sample
    batch on B200 — skinny GEMMs and a dozen elementwise passes — against one pass for the fused kernel."""
    import torch
    B = self.batch
    xb = pooled.view(B, SLOTS * DIM).to(torch.bfloat16)
    h = torch.relu_(xb @ self.w1)                                   # [B, 64] bf16
    logit = (h @ self.w2).float().squeeze(1)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(logit, labels)
    dlogit = ((torch.sigmoid(logit) - labels) * (1.0 / B)).to(torch.bfloat16)
    dh = torch.outer(dlogit, self.w2[:, 0])                          # d loss / d h before the ReLU mask
    dh.masked_fill_(h <= 0, 0)
    torch.mm(dh, self.w1.t(), out=self._gx(B, pooled.device))        # [B, 64] bf16
    grad_out.view(B, SLOTS * DIM).copy_(self.gx)                     # fp32 rows for the sparse backward
    return loss

  def _gx(self, B, dev):
    import torch
    if getattr(self, "gx", None) is None:
      self.gx = torch.empty(B, SLOTS * DIM, dtype=torch.bfloat16, device=dev)
    return self.gx

  def grad_autograd(self, pooled, labels):
    """Reference for tests: the same loss and input gradient through torch.autograd."""
    import torch
    x = pooled.view(self.batch, SLOTS * DIM).detach().requires_grad_(True)
    h = torch.relu(x.to(torch.bfloat16) @ self.w1)
    logit = (h @ self.w2).float().squeeze(1)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(logit, labels)
    gx, = torch.autograd.grad(loss, [x])
    return loss.detach(), gx


DUMP_ROWS = 1 << 17


def dump_outputs(out_dir, table, pooled, fids, world, rank):
  """Writes what the last timed step gave its caller: `pooled.npy`, a fixed sample of DUMP_ROWS rows of the forward's
  pooled output, and `embeddings.npy` / `adagrad_accumulators.npy`, the table rows the backward left behind for a
  fixed sample of DUMP_ROWS / 2 of the step's unique FIDs that this rank owns (both sorted by position / FID).  The
  samples depend only on the batch, which is seeded, so the same arguments dump the same positions on every build.
  c2: 16 + 8 + 8 MB."""
  import torch
  torch.cuda.synchronize()
  dev = pooled.device
  rng = np.random.default_rng(0)
  rows = np.sort(rng.choice(pooled.shape[0], min(pooled.shape[0], DUMP_ROWS), replace=False))
  own = np.unique(fids)
  own = own[own % world == rank]
  ids = np.sort(rng.choice(own, min(own.size, DUMP_ROWS // 2), replace=False))
  ent = table.lookup_entry("item", torch.from_numpy(ids).to(dev))
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "pooled.npy"), pooled[torch.from_numpy(rows).to(dev)].cpu().numpy())
  np.save(os.path.join(out_dir, "embeddings.npy"), ent["num"].cpu().numpy())
  np.save(os.path.join(out_dir, "adagrad_accumulators.npy"), ent["opt"].cpu().numpy())


def run_ours(args):
  import torch
  import torch.distributed as dist
  from monolith_b200 import MultiHashTable, _lib, entry

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if world != args.gpus:
    raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
  numa_cpus = bind_numa(local)
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  if not os.path.exists(_lib.LIB_PATH):  # a checkout without the (git-ignored) .so: build it, loudly, once
    if rank == 0:
      import subprocess
      subprocess.check_call(["bash", os.path.join(ROOT, "monolith_b200", "csrc", "build.sh")], stdout=sys.stderr)
    if world > 1:
      dist.barrier()
  lib = _lib.load()

  # ---- parity first: the same path as the timed region, against ONE global oracle table ----
  parity = None
  if not args.no_parity:
    parity = parity_check(world, rank, dev)
    if rank == 0 and not parity["ok"]:
      print(json.dumps({"metric": METRIC, "parity_check": parity, "error": "parity check failed"}), flush=True)
    if world > 1:
      flag = torch.tensor([1 if (rank != 0 or parity["ok"]) else 0], device=dev)
      dist.broadcast(flag, 0)
      bad = flag.item() == 0
    else:
      bad = not parity["ok"]
    if bad:
      if world > 1:
        dist.destroy_process_group()
      raise SystemExit(3)

  use_sharded = world > 1 or args.sharded
  if use_sharded:
    from monolith_b200.distributed_ps import ShardedStep
  keys_per_slot = args.keys // SLOTS
  seg = entry.CombineAsSegment(DIM, entry.RandomUniformInitializer(-0.05, 0.05), entry.AdagradOptimizer(LR, INIT_ACC))
  # weak scaling: every GPU owns args.keys keys (global table = N * keys), FID ranks span the global range
  gkeys_per_slot = keys_per_slot * world
  cap = int(args.keys * 1.05)
  table = MultiHashTable({"item": entry.HashTableConfigInstance(
      entry.TableConfig([seg], initial_capacity=cap, init_seed=1), [LR])}, device=dev)

  # prefill this rank's shard: keys with fid % world == rank
  for s in range(1, SLOTS + 1):
    for lo in range(0, gkeys_per_slot, 1 << 22):
      hi = min(gkeys_per_slot, lo + (1 << 22))
      ids = (torch.arange(lo, hi, device=dev, dtype=torch.int64)) | (s << 48)
      if world > 1:
        ids = ids[(ids % world) == rank]
      table.assign_add({"item": (ids, torch.zeros(ids.numel(), DIM, device=dev))}, req_time=1, ids_unique=True)
  torch.cuda.synchronize()

  NB = 4
  M = args.batch * SLOTS
  batches_np = make_batches(NB, args.batch, gkeys_per_slot, seed=2 + rank, zipf_s=args.zipf,
                            remote=None if args.remote_frac is None else (args.remote_frac, world, rank))
  fids_dev = [torch.from_numpy(b).to(dev) for b in batches_np]
  gen = torch.Generator(device=dev)
  gen.manual_seed(5 + rank)
  pgrad_dev = torch.randn(M, DIM, device=dev, generator=gen)
  pooled = torch.empty(M, DIM, device=dev)

  if use_sharded:
    sharded = ShardedStep(table, "item", DIM, world, rank, dev, exchange=args.exchange)

  def step(i, fids, pgrad, out):
    if not use_sharded:
      table.lookup_pool("item", fids, None, "sum", out=out)
      table.pool_backward("item", fids, pgrad() if callable(pgrad) else pgrad, None, "sum", req_time=1000 + i)
      return 0
    return sharded.step(fids, pgrad, out, 1000 + i)

  counter = [0]

  def timed(fn, steps, warmup, repeats=1):
    """`repeats` timed regions of exactly `steps` steps each (barrier + synchronize on both sides, CUDA events, max
    over ranks); returns (median ms of a region, launches of the last region, all region times)."""
    for _ in range(warmup):
      fn(counter[0])
      counter[0] += 1
    regions, launches = [], 0
    for _ in range(max(1, repeats)):
      torch.cuda.synchronize()
      if world > 1:
        dist.barrier()
      torch.cuda.synchronize()
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      l0 = lib.mono_kernel_launch_count()
      e0.record()
      for _ in range(steps):
        fn(counter[0])
        counter[0] += 1
      e1.record()
      torch.cuda.synchronize()
      if world > 1:
        dist.barrier()
      torch.cuda.synchronize()
      ms = e0.elapsed_time(e1)
      launches = lib.mono_kernel_launch_count() - l0
      if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
      regions.append(ms)
    return float(np.median(regions)), launches, regions

  overlap = use_sharded and sharded.exchange == "direct" and not args.no_prepare

  def dev_step(i):
    step(i, fids_dev[i % NB], pgrad_dev, pooled)
    if overlap:   # the input pipeline knows the next batch: its grouping is built under this step's exchange phases
      sharded.prepare(fids_dev[(i + 1) % NB])

  with Clocks(local) as clk:
    ms, launches, regions = timed(dev_step, args.steps, args.warmup, args.repeats)
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, table, pooled, batches_np[(counter[0] - 1) % NB], world, rank)
  ab = {}
  if args.ab:
    _l = lib
    for spec in args.ab.split(";"):
      kv = [x.split("=") for x in spec.split(",") if "=" in x]
      old_v = {k: _l.mono_get_option(k.encode()) for k, _ in kv}
      for k, v in kv:
        _l.mono_set_option(k.encode(), int(v))
      ab_ms, _, ab_regions = timed(dev_step, args.steps, args.warmup, args.repeats)
      for k, v in old_v.items():
        _l.mono_set_option(k.encode(), int(v))
      ab[spec] = {"ms_per_step": ab_ms / args.steps, "regions_ms": [round(r / args.steps, 5) for r in ab_regions]}
    ab_ms, _, ab_regions = timed(dev_step, args.steps, args.warmup, args.repeats)
    ab["defaults_again"] = {"ms_per_step": ab_ms / args.steps, "regions_ms": [round(r / args.steps, 5) for r in ab_regions]}
  # unique FIDs per batch (counted once, outside the timed region; the fused step never needs it on the host)
  U_mean = float(np.mean([np.unique(b).size for b in batches_np]))
  value = M * world * args.steps / (ms * 1e-3)

  # ---- e2e: host FIDs + labels in (pinned, H2D inside the timed region), loss out (D2H), public API ----------
  e2e = None
  if not args.no_e2e:
    fids_pin = [torch.from_numpy(b).pin_memory() for b in batches_np]
    labels_pin = (torch.rand(args.batch) < 0.3).float().pin_memory()
    loss_pin = torch.zeros(2).pin_memory()
    ev_loss = [torch.cuda.Event(), torch.cuda.Event()]
    d_f = [torch.empty(M, dtype=torch.int64, device=dev) for _ in range(2)]
    d_g = torch.empty(M, DIM, device=dev)
    tower = Tower(dev, args.batch, lib=lib)
    tower_torch = Tower(dev, args.batch)

    copy_stream = torch.cuda.Stream(device=dev)
    ev_in = [torch.cuda.Event(), torch.cuda.Event()]
    ev_free = [torch.cuda.Event(), torch.cuda.Event()]
    d_labs = [torch.empty(args.batch, device=dev) for _ in range(2)]
    state = {"primed": -1}

    def enqueue_inputs(i):
      """H2D of step i's inputs (pinned host FIDs + labels) on the copy stream: the input pipeline runs one step
      ahead of the trainer, as any data loader does; every step's copy is inside the timed region."""
      b = i & 1
      with torch.cuda.stream(copy_stream):
        copy_stream.wait_event(ev_free[b])            # the step that last used buffer b has consumed it
        if not state.get("nocopy"):   # "nocopy" is a diagnostic region only: what the copies cost the step
          d_f[b].copy_(fids_pin[i % NB], non_blocking=True)
          d_labs[b].copy_(labels_pin, non_blocking=True)
        ev_in[b].record(copy_stream)

    def e2e_step(i):
      """What a training job does per step: the input pipeline hands over HOST FIDs + labels (copied H2D while the
      previous step computes); forward, dense tower forward/backward on the device, sparse backward; the loss comes
      back to the host."""
      t_host0 = time.perf_counter()
      main = torch.cuda.current_stream()
      if state["primed"] != i:
        enqueue_inputs(i)                              # first step of a region: nothing was prefetched
      b = i & 1
      main.wait_event(ev_in[b])
      enqueue_inputs(i + 1)
      state["primed"] = i + 1
      f, lab = d_f[b], d_labs[b]
      loss = []

      tr = state.get("trace")                          # phase trace (one untimed region): CUDA events on the main stream
      if tr is not None:
        tr.append([torch.cuda.Event(enable_timing=True) for _ in range(4)])
        tr[-1][0].record(main)                         # inputs have arrived, the forward starts

      def grads():
        if tr is not None:
          tr[-1][1].record(main)                       # forward done
        loss.append(tower.grad(pooled, lab, d_g))
        if tr is not None:
          tr[-1][2].record(main)                       # tower done
        return d_g

      step(i, f, grads, pooled)
      if tr is not None:
        tr[-1][3].record(main)                         # backward done
      ev_free[b].record(main)
      loss_pin[b:b + 1].copy_(loss[0].reshape(1), non_blocking=True)   # D2H of this step's loss, every step
      ev_loss[b].record(main)
      state["host_s"] = state.get("host_s", 0.0) + (time.perf_counter() - t_host0)   # host time to queue one step
      state["host_n"] = state.get("host_n", 0) + 1
      # the host reads step i-1's loss while step i runs on the device (asynchronous logging): it never waits for the
      # step it has just queued, so the launch queue stays one step deep; the region's closing synchronize covers the last
      ev_loss[b ^ 1].synchronize()
      state["loss_host"] = float(loss_pin[b ^ 1])

    for e_ in ev_free + ev_loss:
      e_.record(torch.cuda.current_stream())

    es, ew = max(3, args.steps // 2), 3
    ems, _, eregions = timed(e2e_step, es, ew, max(1, min(3, args.repeats)))

    # where an e2e step's time goes on the device (separate untimed region; world 1 only: the sharded step takes the
    # gradient callable at a different point)
    phases = None
    if not use_sharded:
      state["trace"] = []
      timed(e2e_step, 12, 2)
      tr = state.pop("trace")[4:]
      torch.cuda.synchronize()
      phases = {"forward_ms": float(np.mean([t[0].elapsed_time(t[1]) for t in tr])),
                "tower_ms": float(np.mean([t[1].elapsed_time(t[2]) for t in tr])),
                "backward_ms": float(np.mean([t[2].elapsed_time(t[3]) for t in tr])),
                "between_steps_ms": float(np.mean([a[3].elapsed_time(b_[0]) for a, b_ in zip(tr[:-1], tr[1:])])),
                "host_queue_ms_per_step": 1e3 * state["host_s"] / max(1, state["host_n"])}
      state["trace"] = None

    # diagnostic: the same loop with the per-step H2D copies switched off (inputs of an earlier step stay in the device
    # buffers): the difference is what the copy engine's traffic costs the kernels that run beside it
    state["nocopy"] = True
    ncms, _, _ = timed(e2e_step, es, 2)
    state["nocopy"] = False

    def tower_only(i):  # context: how much of the e2e step is not the sparse path
      tower.grad(pooled, d_labs[0], d_g)

    tms, _, _ = timed(tower_only, 10, 3)
    ttms, _, _ = timed(lambda i: tower_torch.grad(pooled, d_labs[0], d_g), 5, 2)
    e2e = {"value": M * world * es / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 8 * M + 4 * args.batch,
           "d2h_bytes_per_step": 4, "ms_per_step": ems / es, "ms_per_step_regions": [r / es for r in eregions],
           "dense_tower_ms": tms / 10, "dense_tower_torch_ms": ttms / 5, "device_phases": phases,
           "ms_per_step_without_input_copies": ncms / es,
           "pipeline": "per step: H2D of the step's FIDs (pinned int64[M]) and labels on a copy stream one step ahead (input "
                       "prefetch), fused lookup+pool forward, stand-in "
                       "DSSM tower (bf16 MLP 64-64-1 + logistic loss; one fused mma.sync kernel, csrc/tower.cu) on the device, fused sparse "
                       "backward, D2H of the loss every step; the host reads step i-1's loss while step i runs"}

    # round-1 variant for continuity: a HOST-resident tower (pooled rows D2H, gradients H2D: 553 MB over PCIe per step)
    if world == 1 and not args.no_extras:
      pgrad_pin = pgrad_dev.cpu().pin_memory()
      pooled_pin = torch.empty(M, DIM).pin_memory()
      KCH = max(1, args.e2e_chunks)
      s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
      ev_fwd, ev_in = torch.cuda.Event(), torch.cuda.Event()
      ev_o = [torch.cuda.Event() for _ in range(KCH)]
      cs = (M + KCH - 1) // KCH

      def host_round_trip():
        main = torch.cuda.current_stream()
        ev_fwd.record(main)
        s_out.wait_event(ev_fwd)
        for c in range(KCH):
          sl = slice(c * cs, min(M, (c + 1) * cs))
          with torch.cuda.stream(s_out):
            pooled_pin[sl].copy_(pooled[sl], non_blocking=True)
            ev_o[c].record(s_out)
          with torch.cuda.stream(s_in):
            s_in.wait_event(ev_o[c])
            d_g[sl].copy_(pgrad_pin[sl], non_blocking=True)
        ev_in.record(s_in)
        main.wait_event(ev_in)
        return d_g

      def e2e_host_step(i):
        f = d_f[i & 1]
        f.copy_(fids_pin[i % NB], non_blocking=True)
        step(i, f, host_round_trip, pooled)
        torch.cuda.current_stream().synchronize()

      hms, _, _ = timed(e2e_host_step, 3, 2)
      e2e["host_tower_variant"] = {
          "value": M * 3 / (hms * 1e-3), "ms_per_step": hms / 3, "h2d_bytes_per_step": 8 * M + 4 * M * DIM,
          "d2h_bytes_per_step": 4 * M * DIM,
          "note": f"round-1 definition: pooled rows D2H and gradients H2D in {KCH} full-duplex slices (a host-resident tower)"}

  # ---- per-kernel timing for the roofline (dominant kernel: fused lookup+pool forward) --------
  roof = None
  if world == 1:
    peaks = {}
    try:
      peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
      pass
    peak, peak_src = (peaks.get("hbm_gbs"), "measured") if peaks.get("hbm_gbs") else (6650.0, "fallback")

    def only_fwd(i):
      table.lookup_pool("item", fids_dev[i % NB], None, "sum", out=pooled)

    fms, _, _ = timed(only_fwd, 20, 5, 3)
    fwd_s = fms * 1e-3 / 20
    A = fwd_bytes(M, U_mean) / fwd_s / 1e9
    traffic = None
    try:
      traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("lookup_pool_dram_bytes_per_launch")
    except Exception:
      pass

    def only_bwd(i):
      table.pool_backward("item", fids_dev[i % NB], pgrad_dev, None, "sum", req_time=6000 + i)

    bms, _, _ = timed(only_bwd, 20, 5, 3)
    bwd_s = bms * 1e-3 / 20
    roof = {
        "bound": "hbm", "kernel": "lookup_kernel<8,true> (fused probe + row gather + per-slot pool forward, 1 FID per pooled row)", "achieved": A,
        "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": A / peak, "frac_of_nominal_8000": A / 8000.0,
        "traffic": traffic, "algorithmic_bytes_per_launch": fwd_bytes(M, U_mean), "launch_ms": fwd_s * 1e3,
        "lookups_per_s_fwd_only": M / fwd_s,
        "backward": {"what": "fused backward, whole launch chain (group FIDs, per-FID grad reduce, Adagrad upsert)",
                     "ms": bwd_s * 1e3, "algorithmic_bytes": bwd_bytes(M, U_mean),
                     "achieved": bwd_bytes(M, U_mean) / bwd_s / 1e9, "frac": bwd_bytes(M, U_mean) / bwd_s / 1e9 / peak},
        "others": {"fused_backward_ms": bwd_s * 1e3, "fused_backward_GBps": bwd_bytes(M, U_mean) / bwd_s / 1e9},
    }
    if not args.no_extras:
      ex = {}
      # (1) uniform FIDs (no hot rows in L2): forward only
      ub = make_batches(2, args.batch, gkeys_per_slot, seed=77, zipf_s=0.0)
      uf = [torch.from_numpy(b).to(dev) for b in ub]
      Uu = float(np.mean([np.unique(b).size for b in ub]))

      def fwd_uniform(i):
        table.lookup_pool("item", uf[i % 2], None, "sum", out=pooled)

      ums, _, _ = timed(fwd_uniform, 20, 5, 3)
      ex["forward_uniform_fids"] = {"ms": ums / 20, "U": Uu, "achieved": fwd_bytes(M, Uu) / (ums * 1e-3 / 20) / 1e9,
                                    "frac": fwd_bytes(M, Uu) / (ums * 1e-3 / 20) / 1e9 / peak}
      # (2) the CSR pooling kernel (lookup_pool_kernel): 4 FIDs per pooled row, SUM and MEAN
      ro4 = torch.arange(0, M + 1, 4, device=dev, dtype=torch.int32)
      R4 = M // 4
      for pool in ("sum", "mean"):

        def fwd_csr(i, pool=pool):
          table.lookup_pool("item", fids_dev[i % NB], ro4, pool, out=pooled[:R4])

        cms, _, _ = timed(fwd_csr, 20, 5, 3)
        by = 8 * M + 4 * (R4 + 1) + U_mean * (32 + 4 * DIM) + 4 * DIM * R4
        ex[f"forward_csr_pool_4_{pool}"] = {"kernel": "lookup_pool_kernel<8,1,4>", "ms": cms / 20, "algorithmic_bytes": by,
                                            "achieved": by / (cms * 1e-3 / 20) / 1e9, "frac": by / (cms * 1e-3 / 20) / 1e9 / peak}
      # (3) the batch SURVEY 8(d) quotes (B = 65 536, M = 131 072): launch-bound regime of the same step
      sb = 1 << 16
      sf = [t[:sb * SLOTS].contiguous() for t in fids_dev]

      def small_step(i):
        table.lookup_pool("item", sf[i % NB], None, "sum", out=pooled[:sb * SLOTS])
        table.pool_backward("item", sf[i % NB], pgrad_dev[:sb * SLOTS], None, "sum", req_time=8000 + i)

      sms, _, _ = timed(small_step, 20, 5, 3)
      ex["step_batch_65536"] = {"ms": sms / 20, "lookups_per_s": sb * SLOTS / (sms * 1e-3 / 20)}
      roof["extras"] = ex

  cpu = None
  if world == 1 and rank == 0 and not args.no_cpu_baseline:
    cores = os.cpu_count() or 1
    r = cpu_arm(args.keys, args.cpu_batch or args.batch, 4, 1, args.cpu_threads, args.zipf,
                candidates=(max(1, cores // 4), max(1, cores // 2), cores))
    cpu = {"value": r["value"], "unit": UNIT, "cores": r["threads"], "host_cores": r["host_cores"], "kind": "port",
           "thread_sweep_lookups_per_s": r["thread_sweep_lookups_per_s"],
           "sample": f"4 steps x {r['M']} FIDs (batch {r['batch']} samples, the GPU arm's batch) on the full {args.keys}-key table; "
                     f"{CPU_KIND_NOTE}",
           "ms_per_step": r["ms_per_step"]}

  if rank == 0:
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, args.batch),
        "repeats": {"n": len(regions), "statistic": "median", "ms_per_step_min": min(regions) / args.steps,
                    "ms_per_step_max": max(regions) / args.steps},
        "samples_per_sec": args.batch * world * args.steps / (ms * 1e-3), "unique_fids_per_step": U_mean,
        "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
        "parity_check": parity, "numa_bound_cpus": numa_cpus,
    }
    if ab:
      line["ab"] = ab
    print(json.dumps(line), flush=True)
  if use_sharded and rank == 0 and sharded.phases.enabled:
    print("phase_ms", json.dumps(sharded.phases.report()), file=sys.stderr, flush=True)
  if world > 1:
    dist.destroy_process_group()


def run_c5(args):
  """Hash-table sweep (BASELINE.json configs[4], single GPU): dim 8..128, `keys` resident keys, uniform and Zipf FIDs;
  lookup-only and lookup + Adagrad update, as achieved algorithmic GB/s and fraction of the measured HBM peak."""
  import torch
  from monolith_b200 import MultiHashTable, _lib, entry
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  lib = _lib.load()
  try:
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs") or 6650.0
  except Exception:
    peak = 6650.0
  M = 1 << 21
  rows = []
  for dim in (8, 16, 32, 64, 128):
    seg = entry.CombineAsSegment(dim, entry.RandomUniformInitializer(-0.05, 0.05), entry.AdagradOptimizer(LR, INIT_ACC))
    table = MultiHashTable({"t": entry.HashTableConfigInstance(
        entry.TableConfig([seg], initial_capacity=int(args.keys * 1.05), init_seed=1), [LR])}, device=dev)
    for lo in range(0, args.keys, 1 << 22):
      ids = torch.arange(lo, min(args.keys, lo + (1 << 22)), device=dev, dtype=torch.int64) | (1 << 48)
      table.assign_add({"t": (ids, torch.zeros(ids.numel(), dim, device=dev))}, req_time=1, ids_unique=True)
    out = torch.empty(M, dim, device=dev)
    g = torch.randn(M, dim, device=dev)
    for name, zipf in (("uniform", 0.0), ("zipf1.05", ZIPF_S)):
      rng = np.random.default_rng(3)
      z = Zipf(args.keys, zipf)
      fl = [torch.from_numpy(((z.sample(rng, M) * 2654435761) % args.keys) | (1 << 48)).to(dev) for _ in range(2)]
      U = float(np.mean([torch.unique(f).numel() for f in fl]))

      def timeit(fn, n=10, w=3):
        for i in range(w):
          fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
          fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

      fms = timeit(lambda i: table.lookup_pool("t", fl[i & 1], None, "sum", out=out))
      sms = timeit(lambda i: (table.lookup_pool("t", fl[i & 1], None, "sum", out=out),
                              table.pool_backward("t", fl[i & 1], g, None, "sum", req_time=100 + i)))
      fb, sb = fwd_bytes(M, U, dim), fwd_bytes(M, U, dim) + bwd_bytes(M, U, dim)
      rows.append({"dim": dim, "fids": name, "U": U, "lookup_ms": fms, "lookup_GBps": fb / fms / 1e6, "lookup_frac": fb / fms / 1e6 / peak,
                   "lookup_update_ms": sms, "lookup_update_GBps": sb / sms / 1e6, "lookup_update_frac": sb / sms / 1e6 / peak,
                   "lookups_per_s": M / fms * 1e3, "updates_per_s": M / sms * 1e3})
    table.close()
  print(json.dumps({"metric": "table_sweep_GBps", "workload": "c5", "keys": args.keys, "fids_per_launch": M, "peak_GBps": peak,
                    "rows": rows, "gpu_launches": int(lib.mono_kernel_launch_count())}), flush=True)


def run_c4(args):
  """Streaming insert + evict (BASELINE.json configs[3], DCN-v2-shaped): 200 slots x dim 16 in one collisionless table,
  `--keys` resident keys PER GPU (default 125 M: the 1 B-key table over 8 GPUs), Adagrad.  Every step a fraction
  `--new-frac` of the occurrences are FIDs never seen before (inserted by the backward with their initial row), the rest
  are Zipf-distributed over the resident population; every `--evict-every` steps the table drops every key whose
  last-update time is older than the TTL window (ref: CuckooEmbeddingHashTable::Evict, a full-table scan).  The resident
  keys are prefilled with last-update times spread uniformly over the window, so the stream is in steady state:
  keys inserted per step ~= keys evicted per step.  N > 1: the same stream through the sharded step (FID-hash exchange);
  every rank owns keys/GPU resident keys and evicts its own shard."""
  import torch
  import torch.distributed as dist
  from monolith_b200 import MultiHashTable, _lib, entry
  global DIM, SLOTS
  DIM, SLOTS = 16, 200
  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  lib = _lib.load()
  keys = args.keys
  batch = args.batch
  M = batch * SLOTS
  n_new = int(M * args.new_frac)
  window = max(args.evict_every, int(round(keys / max(1, n_new))))       # TTL in steps: insert rate == evict rate
  seg = entry.CombineAsSegment(DIM, entry.RandomUniformInitializer(-0.05, 0.05), entry.AdagradOptimizer(LR, INIT_ACC))
  # time: the TTL is ONE DAY (SlotExpireTimeConfig counts days; the reference evicts entries with max_update_time - ts >=
  # expire days, cuckoo_embedding_hash_table.cc:251-264); a step advances the clock by dt seconds so that the window is a day
  DAY = 86400
  dt = max(1, int(round(DAY / window)))
  table = MultiHashTable({"item": entry.HashTableConfigInstance(
      entry.TableConfig([seg], initial_capacity=int(keys * 1.15), init_seed=1, default_expire_time=1), [LR])}, device=dev)
  gkeys = keys * world                                                     # global resident population
  t_fill0 = time.time()
  CH = 1 << 20   # fine-grained last-update times: every eviction scan finds about as many expired keys as were inserted
  n_ch = (gkeys + CH - 1) // CH
  for c in range(n_ch):                                                    # chunk c gets last-update time in [0, one day)
    ids = torch.arange(c * CH, min(gkeys, (c + 1) * CH), device=dev, dtype=torch.int64)
    ids = ((ids % SLOTS + 1) << 48) | (ids // SLOTS)
    if world > 1:
      ids = ids[(ids % world) == rank]
    table.assign_add({"item": (ids, torch.zeros(ids.numel(), DIM, device=dev))}, req_time=int(c * DAY / n_ch), ids_unique=True)
  torch.cuda.synchronize()
  fill_s = time.time() - t_fill0
  size0 = int(table.size("item"))

  use_sharded = world > 1
  if use_sharded:
    from monolith_b200.distributed_ps import ShardedStep
    sharded = ShardedStep(table, "item", DIM, world, rank, dev, exchange=args.exchange)

  rng = np.random.default_rng(11 + rank)
  per_slot = gkeys // SLOTS
  fresh_next = [per_slot + 1 + rank]                                       # fresh ranks, disjoint over the ranks

  def make_batch():
    # continuous-power-law approximation of Zipf(1.05) over the resident ranks of a slot (no 1 GB CDF for 1 B keys)
    u = rng.random(M)
    a = 1.0 - ZIPF_S
    r = np.floor(((per_slot ** a - 1.0) * u + 1.0) ** (1.0 / a)).astype(np.int64) - 1
    ident = (np.clip(r, 0, per_slot - 1) * 2654435761) % per_slot
    slots = np.tile(np.arange(1, SLOTS + 1, dtype=np.int64), batch)
    fid = (slots << np.int64(48)) | ident
    pos = rng.choice(M, n_new, replace=False)
    fid[pos] = (slots[pos] << np.int64(48)) | (fresh_next[0] + np.arange(n_new, dtype=np.int64) * world)
    fresh_next[0] += n_new * world
    return fid

  total_steps = args.warmup + args.steps * max(1, args.repeats)
  fids_dev = [torch.from_numpy(make_batch()).to(dev) for _ in range(total_steps)]   # every batch brings NEW fresh FIDs
  gen = torch.Generator(device=dev)
  gen.manual_seed(5 + rank)
  pgrad = torch.randn(M, DIM, device=dev, generator=gen)
  pooled = torch.empty(M, DIM, device=dev)
  ev = {"n": 0, "ms": 0.0}

  def step(i):
    now = DAY + (i + 1) * dt
    if use_sharded:
      sharded.step(fids_dev[i], pgrad, pooled, now)
    else:
      table.lookup_pool("item", fids_dev[i], None, "sum", out=pooled)
      table.pool_backward("item", fids_dev[i], pgrad, None, "sum", req_time=now)
    if (i + 1) % args.evict_every == 0:
      table.evict("item", now)              # drops every key not updated for a day
      ev["n"] += 1

  for i in range(args.warmup):
    step(i)
  i0 = args.warmup
  regions, sizes = [], []
  with Clocks(local) as clk:
    for r in range(max(1, args.repeats)):
      torch.cuda.synchronize()
      if world > 1:
        dist.barrier()
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      l0 = lib.mono_kernel_launch_count()
      e0.record()
      for k in range(args.steps):
        step(i0 + r * args.steps + k)
      e1.record()
      torch.cuda.synchronize()
      launches = lib.mono_kernel_launch_count() - l0
      ms = e0.elapsed_time(e1)
      if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
      regions.append(ms)
      sizes.append(int(table.size("item")))
  ms = float(np.median(regions))
  # one eviction scan alone (outside the timed regions), for the report
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  table.evict("item", 0)     # threshold 0: a pure scan, nothing qualifies any more
  e1.record()
  torch.cuda.synchronize()
  scan_ms = e0.elapsed_time(e1)
  try:
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs") or 6650.0
  except Exception:
    peak = 6650.0
  if rank == 0:
    print(json.dumps({
        "metric": METRIC, "value": M * world * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C4 streaming insert+evict: {SLOTS} slots x dim {DIM}, {keys} resident keys per GPU ({gkeys} global), "
                               f"batch {batch} samples ({M} FID occurrences) per GPU, {args.new_frac:.3f} of them never-seen FIDs "
                               f"({n_new} inserts per step and GPU), evict every {args.evict_every} steps, TTL one day = {window} steps of {dt} s; "
                               "inputs larger than L2 (every batch distinct)",
                   "exchange": (sharded.exchange if use_sharded else None)},
        "repeats": {"n": len(regions), "statistic": "median", "ms_per_step_all": [r / args.steps for r in regions]},
        "inserts_per_sec": n_new * world * args.steps / (ms * 1e-3),
        "table_size": {"after_fill": size0, "after_each_region": sizes},
        "evict": {"scans_in_timed_regions": ev["n"], "full_scan_ms": scan_ms,
                  "scan_GBps": 16.0 * table.size("item") / 0.5 / scan_ms / 1e6 if scan_ms > 0 else None,
                  "scan_note": "bucket array only (16 B per slot at ~50 % load) / scan time; peak " + str(peak)},
        "fill_s": fill_s, "clocks": clk.summary(), "gpu_launches": int(launches),
    }), flush=True)
  if world > 1:
    dist.destroy_process_group()


def main():
  args = parse()
  if args.workload == "c5" and args.impl != "reference":
    return run_c5(args)
  if args.workload == "c4" and args.impl != "reference":
    return run_c4(args)
  if args.impl == "reference":
    run_reference(args)
  else:
    run_ours(args)


if __name__ == "__main__":
  main()
