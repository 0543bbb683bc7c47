"""Pins the CPU oracle against the reference's own known-answer tests (transcribed, with file:line,
in tests/golden/make_golden.py) and against outputs of the real reference headers (oracle/_ref)."""
import json
import os

import numpy as np
import pytest

from tests import orc
from tests.helpers import sgd_table, table

G = os.path.join(os.path.dirname(__file__), "golden")
KNOWN = json.load(open(os.path.join(G, "reference_known_answers.json")))


@pytest.mark.parametrize("case", KNOWN["optimizers"], ids=lambda c: c["name"])
def test_optimizer_known_answers(case):
  t = orc.OracleMultiHashTable({"t": table([(case["dim"], case["opt"], case["params"])], [0.0])})
  ids = np.array([7], np.int64)
  for st in case["steps"]:
    t.configs["t"]._learning_rate_fns = list(st["lr"])
    t.apply_gradients({"t": (ids, np.array([st["grad"]], np.float32))})
    got = t.lookup({"t": ids})["t"][0]
    np.testing.assert_allclose(got, st["expect"], atol=case["tol"], rtol=0)


def test_optimizer_combination():
  c = KNOWN["combination"]
  segs = [(s["dim"], s["opt"], s["params"]) for s in c["segments"]]
  t = orc.OracleMultiHashTable({"t": table(segs, c["lr"])})
  ids = np.array([1], np.int64)
  t.apply_gradients({"t": (ids, np.array([c["grad"]], np.float32))})
  np.testing.assert_allclose(t.lookup({"t": ids})["t"][0], c["expect_step1"], atol=c["tol"], rtol=0)
  # the reference restores the optimizer dump into an entry whose num is zero, then steps again
  t.assign({"t": (ids, np.zeros((1, 3), np.float32))})
  t.apply_gradients({"t": (ids, np.array([c["grad"]], np.float32))})
  np.testing.assert_allclose(t.lookup({"t": ids})["t"][0], c["expect_step2_from_zero_num"], atol=c["tol"], rtol=0)


@pytest.mark.parametrize("case", KNOWN["fused_reorder_by_indices"], ids=lambda c: str(c["ids"])[:40])
def test_fused_reorder_golden(case):
  dims = case.get("dims", [2] * len(case["ids"]))
  out, shard_sizes, slot_sizes, _, offs = orc.reorder_by_indices(case["ids"], case["N"], dims)
  assert out.tolist() == case["output"]
  assert shard_sizes.tolist() == case["shard_sizes"]
  assert slot_sizes.tolist() == case["sharded_slot_sizes"]
  if "offsets" in case:
    assert offs.tolist() == case["offsets"]


def _tables(dims, lrs=None):
  return {f"t{i}": sgd_table(d, (lrs or [1.0] * len(dims))[i]) for i, d in enumerate(dims)}


def test_fused_lookup_golden():
  c = KNOWN["fused_lookup"]
  t = orc.OracleMultiHashTable(_tables(c["dims"]))
  for i, a in enumerate(c["assign"]):
    t.assign({f"t{i}": (a["ids"], np.full((len(a["ids"]), c["dims"][i]), a["value"], np.float32))})
  emb, es, ko, eo = t.fused_lookup(c["ids"], c["fused_slot_size"], c["N"])
  assert emb.tolist() == c["embeddings"]
  assert es.tolist() == c["recv_splits"] and ko.tolist() == c["id_offsets"] and eo.tolist() == c["emb_offsets"]


def test_fused_optimize_golden():
  c = KNOWN["fused_optimize"]
  t = orc.OracleMultiHashTable(_tables(c["dims"], c["lr"]))
  for i, a in enumerate(c["assign"]):
    t.assign({f"t{i}": (a["ids"], np.full((len(a["ids"]), c["dims"][i]), a["value"], np.float32))})
  t.fused_apply_gradient(c["ids"], c["fused_slot_size"], c["grads"], c["N"])
  emb, es, ko, eo = t.fused_lookup(c["ids"], c["fused_slot_size"], c["N"])
  np.testing.assert_allclose(emb, c["embeddings_after"], rtol=1e-6)
  assert es.tolist() == c["recv_splits"] and ko.tolist() == c["id_offsets"] and eo.tolist() == c["emb_offsets"]


def test_basic_assign_add_and_assign():
  b = KNOWN["basic"]
  t = orc.OracleMultiHashTable({"t": sgd_table(1)})
  t.assign_add({"t": ([0, 1], np.ones((2, 1), np.float32))})
  assert t.lookup({"t": [0, 1, 2]})["t"].tolist() == b["assign_add"]["expect"]
  assert t.size("t") == b["assign_add"]["size"]
  t2 = orc.OracleMultiHashTable({"t": sgd_table(1)})
  t2.assign({"t": ([0, 1], np.ones((2, 1), np.float32))})
  assert t2.lookup({"t": [0, 1, 2]})["t"].tolist() == b["assign_overwrite"]["first"]
  t2.assign({"t": ([1], np.full((1, 1), 5, np.float32))})
  assert t2.lookup({"t": [0, 1, 2]})["t"].tolist() == b["assign_overwrite"]["second"]


@pytest.mark.parametrize("case", KNOWN["gradients"], ids=lambda c: c["name"])
def test_gradient_semantics(case):
  t = orc.OracleMultiHashTable({"t": sgd_table(case["dim"], case["lr"])})
  n = len(case["ids"])
  grads = -np.ones((n, case["dim"]), np.float32) if case["grads"] == "minus_ones" else np.array(case["grads"], np.float32)
  t.apply_gradients({"t": (case["ids"], grads)}, enable_dedup=case["dedup"])
  got = t.lookup({"t": case["lookup"]})["t"]
  if "expect" in case:
    np.testing.assert_allclose(got, case["expect"], rtol=1e-6)
  else:
    for row, v in zip(got, case["expect_scalar"]):
      np.testing.assert_allclose(row, np.full(case["dim"], v), rtol=1e-6)


def test_single_thread_semantics():
  s = KNOWN["single_thread"]
  t = orc.OracleMultiHashTable({"t": sgd_table(1, 0.01)})
  assert t.lookup({"t": [s["miss"]["id"]]})["t"].tolist() == [s["miss"]["expect"]]
  assert t.size("t") == 0  # lookup never inserts
  t.assign_add({"t": ([s["assign_add"]["id"]], [s["assign_add"]["value"]])}, req_time=s["assign_add"]["ts"])
  assert t.lookup({"t": [-10]})["t"].tolist() == [s["assign_add"]["expect"]]
  t.apply_gradients({"t": ([13], [s["optimize_fresh"]["grad"]])})
  np.testing.assert_allclose(t.lookup({"t": [13]})["t"], [s["optimize_fresh"]["expect"]], rtol=1e-6)
  e = t.lookup_entry("t", [-10, 99])
  assert e[0, -2:].view(np.uint32).tolist() == [1, 100] and e[1].tolist() == [0, 0, 0]


def test_evict_golden():
  e = KNOWN["evict"]
  cfg = sgd_table(1, default_expire_time=e["default_expire_days"],
                  slot_expire_times={int(k): v for k, v in e["slot_expire"].items()})
  t = orc.OracleMultiHashTable({"t": cfg})
  fids = [(r["slot"] << 48) | r["sig"] for r in e["rows"]]
  t.assign({"t": (fids, np.array([[r["value"]] for r in e["rows"]], np.float32))}, req_time=e["write_ts"])
  t.evict("t", e["evict_at"])
  assert t.lookup({"t": fids})["t"].reshape(-1).tolist() == e["expect_after"]
  assert t.size("t") == 2


def test_multi_hash_table_golden():
  m = KNOWN["multi_hash_table"]
  t = orc.OracleMultiHashTable({"slot0": sgd_table(1), "not_used": sgd_table(2), "slot1": sgd_table(2),
                                "slot2": sgd_table(2)})
  t.assign_add({"slot0": ([0], [[1]]), "slot1": ([1], [[2, 2]]), "slot2": ([2, 3], [[4, 4], [8, 8]])})
  got = t.lookup({"slot0": [0], "slot1": [1], "slot2": [2, 3]})
  assert got["slot0"].tolist() == [[1]] and got["slot1"].tolist() == [[2, 2]]
  assert got["slot2"].tolist() == [[4, 4], [8, 8]]
  assert t.reinitialize("slot2", [1, 2, 3]).tolist() == m["reinitialize"]["known_status"]
  assert t.reinitialize("slot3", [1, 2, 3]).tolist() == m["reinitialize"]["unknown_status"]
  assert t.lookup({"slot2": [1, 2, 3]})["slot2"].tolist() == [[0, 0]] * 3
  t2 = orc.OracleMultiHashTable({"slot0": sgd_table(1), "slot1": sgd_table(2)})
  t2.apply_gradients({"slot0": ([0], [[2.0]]), "slot1": ([1, 2], [[1.0, 3.0], [2.0, 4.0]])})
  got = t2.lookup({"slot0": [0], "slot1": [1, 2]})
  assert got["slot0"].tolist() == m["apply_gradients_sgd"]["slot0"]
  assert got["slot1"].tolist() == m["apply_gradients_sgd"]["slot1"]


# ---- vectors produced by the REAL reference code (oracle/_ref), committed as fixtures ------------
def test_adagrad_bit_exact_vs_reference_header_fixture():
  z = np.load(os.path.join(G, "ref_adagrad.npz"))
  import ctypes as C
  for ci in range(int(z["n_cases"])):
    dim, wd = int(z[f"c{ci}_dim"]), float(z[f"c{ci}_wd"])
    num, norm = z[f"c{ci}_num0"].copy(), np.full(dim, 0.1, np.float32)
    for step in range(z[f"c{ci}_grads"].shape[0]):
      g = np.ascontiguousarray(z[f"c{ci}_grads"][step])
      orc.lib().orc_adagrad(orc.p(num), orc.p(norm), orc.p(g), C.c_int64(dim), C.c_float(0.05), C.c_float(wd))
      # avx_utils.h AVX lanes are restated with explicit fma: bit-exact.  The scalar tail
      # (dim % 8 lanes) may differ in the last ulp depending on the reference compiler's contraction.
      d8 = dim - dim % 8
      assert np.array_equal(num[:d8], z[f"c{ci}_num"][step][:d8]), (ci, step)
      assert np.array_equal(norm[:d8], z[f"c{ci}_norm"][step][:d8]), (ci, step)
      np.testing.assert_allclose(num, z[f"c{ci}_num"][step], rtol=2e-6, atol=1e-8)
      np.testing.assert_allclose(norm, z[f"c{ci}_norm"][step], rtol=2e-6, atol=1e-8)


def test_first_occurrence_ordinals_vs_reference_uniq_hashtable_fixture():
  z = np.load(os.path.join(G, "ref_uniq_fid.npz"))
  for ci in range(int(z["n_cases"])):
    fids, N = z[f"c{ci}_fids"], int(z[f"c{ci}_shards"])
    out, shard_sizes, slot_sizes, _, offs = orc.reorder_by_indices([fids], N, [1])
    assert shard_sizes.tolist() == z[f"c{ci}_sizes"].tolist()
    # reference ordinal is local to the shard list; the oracle's offset is global (dim 1):
    base = np.concatenate([[0], np.cumsum(shard_sizes)[:-1]])
    shard = (fids.view(np.uint64) % np.uint64(N)).astype(np.int64)
    assert (offs - base[shard]).tolist() == z[f"c{ci}_uniq_idx"].tolist()


def test_adagrad_avx_lanes_bit_exact_vs_reference_header_fixture():
  """Rows of 8, 24 and 64 floats (every lane on the AVX path of avx_utils.h), unit-normal state and gradients, lr 0.01:
  the oracle's Adagrad equals the reference header's bit for bit after every one of five steps."""
  import ctypes as C
  z = np.load(os.path.join(G, "ref_adagrad_avx_lanes.npz"))
  for ci in range(int(z["n_cases"])):
    num, norm = z[f"c{ci}_num0"].copy(), z[f"c{ci}_norm0"].copy()
    for step in range(z[f"c{ci}_grads"].shape[0]):
      g = np.ascontiguousarray(z[f"c{ci}_grads"][step])
      orc.lib().orc_adagrad(orc.p(num), orc.p(norm), orc.p(g), C.c_int64(num.size), C.c_float(z["lr"]), C.c_float(0.0))
      assert np.array_equal(num, z[f"c{ci}_num"][step]) and np.array_equal(norm, z[f"c{ci}_norm"][step]), (ci, step)


def test_layout_pooling_vs_reference_numpy_oracle_fixture():
  """orc_embedding_to_layout (GatherEmb + pooling, fused_embedding_to_layout.cc:26-59,468-540) against the
  reference's own numpy pooling oracle (fused_embedding_to_layout_test.py:91-116), run by
  tests/golden/make_layout_golden.py.  SUM and FIRSTN are exact; MEAN is sum/n in the numpy oracle but
  sum of x_i/n in the op (SURVEY appendix A): 1e-6 relative."""
  from monolith_b200._lib import POOL_FIRSTN, POOL_MEAN, POOL_SUM
  from monolith_b200.distribution_ops import SliceTask
  z = np.load(os.path.join(G, "ref_layout_pooling.npz"))
  code = {0: POOL_SUM, 1: POOL_MEAN, 2: POOL_FIRSTN}
  for ci in range(int(z["n_cases"])):
    pt, max_len = int(z[f"c{ci}_pooling"]), int(z[f"c{ci}_max_len"])
    tab, idx, offs, want = z[f"c{ci}_table"], z[f"c{ci}_idx"], z[f"c{ci}_offs"], z[f"c{ci}_expect"]
    B, dim = offs.size - 1, tab.shape[1]
    # v3 encoding of ONE feature over one embedding list (parse_sparse_feature.cc:259-330)
    fid_offset = (idx * dim).astype(np.uint64)                      # list 0 << 32 | float offset of the row
    feature_offset = np.concatenate([offs[:-1], [idx.size]]).astype(np.int32)
    nfl_offset = np.array([0, feature_offset.size], np.uint32)
    if code[pt] == POOL_FIRSTN:
      task, shape = SliceTask(0, 0, dim, POOL_FIRSTN, max_len, 0, max_len * dim, 0, 0), (B, max_len, dim)
    else:
      task, shape = SliceTask(0, 0, dim, code[pt], 0, 0, dim, 0, 0), (B, dim)
    got = orc.embedding_to_layout([tab], [1], fid_offset, feature_offset, nfl_offset, B, [task], [shape])[0]
    if code[pt] == POOL_MEAN:
      np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)
    else:
      np.testing.assert_array_equal(got, want)


def test_distributed_ps_closed_form_ftrl_bias_adagrad_vec():
  """Closed-form expectation of the reference's sharded fwd+bwd test (NT/distributed_ps_test.py:787-882): rows
  [bias: FTRL dim 1 | vec: Adagrad], every value assigned 3.0, gradient 2.0 on every element, lr 1.0,
  initial_accumulator_value 0.1, beta 0 -> bias = -lr*z/(sqrt(n)+beta), vec = 3 - lr/sqrt(g^2+0.1)*g (1e-6)."""
  import math
  init_val, g, lr, acc, beta = 3.0, 2.0, 1.0, 0.1, 0.0
  ada_grad = lr / math.sqrt(g * g + acc) * g
  n = acc + g * g
  sigma = (math.sqrt(n) - math.sqrt(acc)) / lr
  z = g - sigma * init_val
  ftrl_val = -lr * z / (math.sqrt(n) + beta)
  cfg = {"uid": table([(1, "ftrl", {"initial_accumulator_value": acc, "beta": beta, "l1": 0.0, "l2": 0.0}),
                       (4, "adagrad", {"initial_accumulator_value": acc})], [lr, lr])}
  t = orc.OracleMultiHashTable(cfg)
  fids = np.arange(18, dtype=np.int64)                      # the test's FIDs 0..17, owners = fid mod 2
  t.assign({"uid": (fids, np.full((18, 5), init_val, np.float32))})
  t.apply_gradients({"uid": (fids, np.full((18, 5), g, np.float32))})
  got = t.lookup({"uid": fids})["uid"]
  np.testing.assert_allclose(got[:, 0], ftrl_val, atol=1e-6, rtol=0)
  np.testing.assert_allclose(got[:, 1:], init_val - ada_grad, atol=1e-6, rtol=0)
  assert sorted(fids[fids % 2 == 0].tolist()) == [0, 2, 4, 6, 8, 10, 12, 14, 16]   # uid:0/cid:0/gid:0 shards of the test


def test_sharding_sparse_fids_vs_reference_python_model_fixture():
  """distribution_ops.sharding_sparse_fids (row a2: ShardingSparseFids outputs) against the reference's own Python
  model of the op (parse_sparse_feature_test.py:87-240, run by tests/golden/make_sharding_golden.py): per-(table,
  shard) FID lists, fid_offset (index << 32 | float offset, per-feature dims_sum), feature_offset, nfl_offset with the
  shared flag — all exact.  The dedup / shard step is served by the oracle's FusedReorderByIndices here (CPU); on
  the GPU the same adapter runs on mono_reorder_by_indices, which is bit-exact with it (tests/test_gpu_parity.py)."""
  import torch
  from monolith_b200 import distribution_ops as dops

  def reorder_fn(lists, n, dims):
    out, ss, sl, _, offs = orc.reorder_by_indices([l.numpy() for l in lists], n, dims)
    return torch.from_numpy(out), ss.tolist(), sl.tolist(), None, torch.from_numpy(offs)

  z = np.load(os.path.join(G, "ref_sharding_sparse_fids.npz"))
  for ci in range(int(z["n_cases"])):
    names = [str(n) for n in z[f"c{ci}_names"]]
    N = int(z[f"c{ci}_N"])
    feats = {n: (torch.from_numpy(z[f"c{ci}_fids_{n}"]), torch.from_numpy(z[f"c{ci}_splits_{n}"])) for n in names}
    table_of = {n: str(t) for n, t in zip(names, z[f"c{ci}_tables"])}
    dims_sum = {n: int(d) for n, d in zip(names, z[f"c{ci}_dims_sum"])}
    shared = [n for n, s in zip(names, z[f"c{ci}_shared"]) if s]
    r = dops.sharding_sparse_fids(feats, table_of, dims_sum, N, shared, reorder_fn=reorder_fn)
    assert r["nfl_offset"].numpy().astype(np.uint32).tolist() == z[f"c{ci}_nfl_offset"].tolist()
    assert r["feature_offset"].numpy().tolist() == z[f"c{ci}_feature_offset"].tolist()
    assert r["fid_offset"].numpy().view(np.uint64).tolist() == z[f"c{ci}_fid_offset_unique"].tolist()
    K = int(z[f"c{ci}_n_tables"])
    assert len(r["fid_list"]) == K * N
    for k in range(K):
      for n in range(N):
        assert r["fid_list"][k * N + n].numpy().tolist() == z[f"c{ci}_list_{k}_{n}"].tolist(), (ci, k, n)


def test_sharding_sparse_fids_negative_fids_use_unsigned_shard():
  """shard = (uint64)fid % N also for FIDs with the top bit set (parse_sparse_feature.cc:205 `value % ps_num_` on
  uint64): the adapter's signed-remainder arithmetic must agree with numpy's uint64 arithmetic."""
  import torch
  from monolith_b200 import distribution_ops as dops

  def reorder_fn(lists, n, dims):
    out, ss, sl, _, offs = orc.reorder_by_indices([l.numpy() for l in lists], n, dims)
    return torch.from_numpy(out), ss.tolist(), sl.tolist(), None, torch.from_numpy(offs)

  rng = np.random.default_rng(5)
  fids = rng.integers(-2**63, 2**63 - 1, 500).astype(np.int64)
  fids[:4] = [-1, np.iinfo(np.int64).min, np.iinfo(np.int64).max, 0]
  for N in (1, 2, 3, 5, 8, 64):
    r = dops.sharding_sparse_fids({"f": (torch.from_numpy(fids), torch.tensor([0, fids.size]))}, {"f": "t"}, {"f": 4}, N,
                                  reorder_fn=reorder_fn)
    shard = (fids.view(np.uint64) % np.uint64(N)).astype(np.int64)
    assert ((r["fid_offset"].numpy() >> 32) == shard).all()                    # table index 0: index1 == shard
    for n in range(N):
      want = fids[shard == n]
      _, first = np.unique(want, return_index=True)
      assert r["fid_list"][n].numpy().tolist() == want[np.sort(first)].tolist()  # first-occurrence order


def test_hash_filter_threshold_schedule_golden():
  """Counting hash filter, oracle side (next-row prep, SURVEY §8(f) row 2): the reference's
  test_gradients_with_hash_filter (NT/hash_table_ops_test.py:223-260): dim 1, SGD lr 0.1, occurrence_threshold 3,
  ids [0, 0, 1] with gradient -1 applied four times -> lookups of [0, 1] after each step."""
  t = orc.OracleMultiHashTable({"t": sgd_table(1, 0.1)})
  t.set_hash_filter("t", capacity=1000, default_threshold=3)
  ids = np.array([0, 0, 1], np.int64)
  expected = [[[0.0], [0.0]], [[0.1], [0.0]], [[0.3], [0.0]], [[0.5], [0.1]]]
  for want in expected:
    t.apply_gradients({"t": (ids, -np.ones((3, 1), np.float32))})
    np.testing.assert_allclose(t.lookup({"t": np.array([0, 1], np.int64)})["t"], want, rtol=1e-6, atol=1e-7)
  # threshold 0 (and tables without a filter) never filter; per-slot thresholds override the default
  t2 = orc.OracleMultiHashTable({"t": sgd_table(1, 0.1)})
  t2.set_hash_filter("t", capacity=1000, default_threshold=0, slot_thresholds={2: 2})
  a, b = np.int64(5), (np.int64(2) << 48) | np.int64(5)
  t2.apply_gradients({"t": (np.array([a, b], np.int64), -np.ones((2, 1), np.float32))})
  np.testing.assert_allclose(t2.lookup({"t": np.array([a, b], np.int64)})["t"], [[0.1], [0.0]], rtol=1e-6)
  t2.apply_gradients({"t": (np.array([a, b], np.int64), -np.ones((2, 1), np.float32))})
  t2.apply_gradients({"t": (np.array([a, b], np.int64), -np.ones((2, 1), np.float32))})
  np.testing.assert_allclose(t2.lookup({"t": np.array([a, b], np.int64)})["t"], [[0.3], [0.1]], rtol=1e-6)
  # the dedup path passes the occurrence count to the filter (tf_bridge.cc:296-310): [7,7,7] counts 3 at once
  t3 = orc.OracleMultiHashTable({"t": sgd_table(1, 0.1)})
  t3.set_hash_filter("t", capacity=1000, default_threshold=3)
  for want in ([[0.0]], [[0.3]]):   # first call: previous count 0 < 3 -> filtered (counter becomes 3); second: 3 !< 3
    t3.apply_gradients({"t": (np.array([7, 7, 7], np.int64), -np.ones((3, 1), np.float32))}, enable_dedup=True)
    np.testing.assert_allclose(t3.lookup({"t": np.array([7], np.int64)})["t"], want, rtol=1e-6, atol=1e-7)


def test_fastps_baseline_equals_oracle_ps_step():
  """The tuned CPU baseline timed by bench.py (orc_fastps_*: persistent pool, flat tables, partitioned dedup and
  scatter) computes exactly what the plain oracle PS step (orc_ps_train_step over the oracle tables) computes:
  pooled rows bit for bit, and every touched entry [emb | Adagrad state] bit for bit, over several steps with
  hot FIDs, unseen FIDs (upserts) and CSR mean pooling."""
  import ctypes as C
  from monolith_b200 import entry
  lib = orc.lib()
  lib.orc_ps_train_step.restype = C.c_int64
  lib.orc_fastps_train_step.restype = C.c_int64
  D = 16
  seg = entry.CombineAsSegment(D, entry.RandomUniformInitializer(-0.05, 0.05), entry.AdagradOptimizer(0.05, 0.1))
  cfg = {"t": entry.HashTableConfigInstance(entry.TableConfig([seg], initial_capacity=1000, init_seed=3), [0.05])}
  arr, keep = entry.to_c_table_cfgs(cfg)
  T = 5
  a, b = C.c_void_p(), C.c_void_p()
  lib.orc_ps_create(arr, T, C.byref(a))
  lib.orc_fastps_create(arr, T, C.byref(b))
  lib.orc_ps_fill_slots(a, 2, C.c_int64(300))
  lib.orc_fastps_fill_slots(b, 2, C.c_int64(300))
  rng = np.random.default_rng(11)
  lr = np.array([0.05], np.float32)
  seen = set()
  for step in range(4):
    for csr in (False, True):
      M = 4000
      ids = rng.integers(0, 500, M)            # 300..499 are not pre-filled: upserted by the optimizer
      ids[rng.random(M) < 0.2] = 7             # hot FID
      fids = ((rng.integers(1, 3, M).astype(np.int64)) << 48) | ids.astype(np.int64)
      seen.update(fids.tolist())
      if csr:
        cuts = np.sort(rng.choice(np.arange(1, M), 900, replace=False))
        ro = np.concatenate([[0], cuts, [M]]).astype(np.int32)
        pooling = 1
      else:
        ro, pooling = None, 0
      R = M if ro is None else ro.size - 1
      pg = rng.standard_normal((R, D)).astype(np.float32)
      o1, o2 = np.zeros((R, D), np.float32), np.zeros((R, D), np.float32)
      u1 = lib.orc_ps_train_step(a, orc.p(fids), C.c_int64(M), orc.p(ro), C.c_int64(R), pooling, orc.p(pg), orc.p(o1),
                                 orc.p(lr), C.c_int64(100 + step))
      u2 = lib.orc_fastps_train_step(b, orc.p(fids), C.c_int64(M), orc.p(ro), C.c_int64(R), pooling, orc.p(pg),
                                     orc.p(o2), orc.p(lr), C.c_int64(100 + step))
      assert u1 == u2 == np.unique(fids).size
      np.testing.assert_array_equal(o1.view(np.uint32), o2.view(np.uint32))
  lib.orc_fastps_size.restype = C.c_int64
  assert lib.orc_ps_size(a) == lib.orc_fastps_size(b)
  # entries: one more forward over every FID ever seen reads the rows both implementations hold
  allf = np.array(sorted(seen), np.int64)
  o1, o2 = np.zeros((allf.size, D), np.float32), np.zeros((allf.size, D), np.float32)
  lib.orc_ps_lookup_pool(a, orc.p(allf), None, C.c_int64(allf.size), C.c_int64(allf.size), 0, orc.p(o1))
  ent = np.zeros(2 * D, np.float32)
  for i, f in enumerate(allf):
    assert lib.orc_fastps_entry(b, C.c_int64(int(f)), orc.p(ent)) == 1
    o2[i] = ent[:D]
  np.testing.assert_array_equal(o1.view(np.uint32), o2.view(np.uint32))
  lib.orc_ps_destroy(a)
  lib.orc_fastps_destroy(b)
