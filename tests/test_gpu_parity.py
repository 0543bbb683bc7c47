"""GPU parity tests: the CUDA path (through the C ABI) vs the CPU oracle on the same seeded inputs.

Bars: bit-exact for integer / index / membership results and for everything whose float order is
deterministic (lookup, fused lookup+pool, SGD/Adagrad/FTRL/Adam updates restated op by op);
1e-5 relative where float atomics reorder sums (scatter of pooled grads, as in the reference GPU).
"""
import json
import os

import numpy as np
import pytest
import torch

from tests import orc
from tests.helpers import sgd_table, table

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(__file__), "golden")
KNOWN = json.load(open(os.path.join(G, "reference_known_answers.json")))


@pytest.fixture(scope="module")
def dev():
  assert torch.cuda.is_available()
  return torch.device("cuda", 0)


def T(x, dev, dtype=None):
  t = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
  return t if dtype is None else t.to(dtype)


def pair(configs, dev):
  from monolith_b200 import MultiHashTable
  return MultiHashTable(configs, device=dev), orc.OracleMultiHashTable(configs)


def gpu_lookup(gpu, d, dev):
  return {k: v.cpu().numpy() for k, v in gpu.lookup({k: T(np.asarray(v, np.int64), dev) for k, v in d.items()}).items()}


def fid(slot, sig):
  return (np.int64(slot) << np.int64(48)) | np.int64(sig)


def rand_fids(rng, n, vocab, slots=(1, 30)):
  return (rng.integers(slots[0], slots[1], n).astype(np.int64) << 48) | rng.integers(0, vocab, n).astype(np.int64)


# ------------------------------------------------------------------------------------------------
# reference golden vectors straight through the CUDA path
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", KNOWN["optimizers"], ids=lambda c: c["name"])
def test_optimizer_known_answers_cuda(case, dev):
  cfg = {"t": table([(case["dim"], case["opt"], case["params"])], [0.0])}
  from monolith_b200 import MultiHashTable
  t = MultiHashTable(cfg, device=dev)
  ids = T(np.array([7], np.int64), dev)
  for st in case["steps"]:
    cfg["t"]._learning_rate_fns = list(st["lr"])
    t.apply_gradients({"t": (ids, T(np.array([st["grad"]], np.float32), dev))})
    np.testing.assert_allclose(t.lookup({"t": ids})["t"][0].cpu().numpy(), st["expect"], atol=case["tol"], rtol=0)


def test_optimizer_combination_cuda(dev):
  c = KNOWN["combination"]
  from monolith_b200 import MultiHashTable
  t = MultiHashTable({"t": table([(s["dim"], s["opt"], s["params"]) for s in c["segments"]], c["lr"])}, device=dev)
  ids = T(np.array([1], np.int64), dev)
  t.apply_gradients({"t": (ids, T(np.array([c["grad"]], np.float32), dev))})
  np.testing.assert_allclose(t.lookup({"t": ids})["t"][0].cpu().numpy(), c["expect_step1"], atol=1e-6, rtol=0)


@pytest.mark.parametrize("case", KNOWN["fused_reorder_by_indices"], ids=lambda c: str(c["ids"])[:40])
def test_fused_reorder_golden_cuda(case, dev):
  from monolith_b200 import distribution_ops as dops
  dims = case.get("dims", [2] * len(case["ids"]))
  ins = [T(np.array(x, np.int64), dev) for x in case["ids"]]
  out, shard_sizes, slot_sizes, _, offs = dops.fused_reorder_by_indices(ins, case["N"], dims, rank0_empty_shard=False)
  assert out.cpu().tolist() == case["output"]
  assert shard_sizes == case["shard_sizes"] and slot_sizes == case["sharded_slot_sizes"]
  if "offsets" in case:
    assert offs.cpu().tolist() == case["offsets"]


def test_fused_lookup_and_optimize_golden_cuda(dev):
  from monolith_b200 import MultiHashTable
  c = KNOWN["fused_lookup"]
  t = MultiHashTable({f"t{i}": sgd_table(d) for i, d in enumerate(c["dims"])}, device=dev)
  for i, a in enumerate(c["assign"]):
    t.assign({f"t{i}": (T(np.array(a["ids"], np.int64), dev),
                        T(np.full((len(a["ids"]), c["dims"][i]), a["value"], np.float32), dev))})
  emb, es, ko, eo, _ = t.fused_lookup(T(np.array(c["ids"], np.int64), dev), c["fused_slot_size"], c["N"])
  assert emb.cpu().tolist() == c["embeddings"]
  assert es == c["recv_splits"] and ko == c["id_offsets"] and eo == c["emb_offsets"]
  c = KNOWN["fused_optimize"]
  t = MultiHashTable({f"t{i}": sgd_table(d, c["lr"][i]) for i, d in enumerate(c["dims"])}, device=dev)
  for i, a in enumerate(c["assign"]):
    t.assign({f"t{i}": (T(np.array(a["ids"], np.int64), dev),
                        T(np.full((len(a["ids"]), c["dims"][i]), a["value"], np.float32), dev))})
  ids = T(np.array(c["ids"], np.int64), dev)
  emb, es, ko, eo, idx = t.fused_lookup(ids, c["fused_slot_size"], c["N"])
  t.fused_apply_gradient(ids, idx, c["fused_slot_size"], T(np.array(c["grads"], np.float32), dev), ko, eo, 0, 0, c["N"])
  emb, es, ko, eo, _ = t.fused_lookup(ids, c["fused_slot_size"], c["N"])
  np.testing.assert_allclose(emb.cpu().numpy(), c["embeddings_after"], rtol=1e-6)
  assert es == c["recv_splits"] and ko == c["id_offsets"] and eo == c["emb_offsets"]


@pytest.mark.parametrize("case", KNOWN["gradients"], ids=lambda c: c["name"])
def test_gradient_semantics_cuda(case, dev):
  from monolith_b200 import MultiHashTable
  t = MultiHashTable({"t": sgd_table(case["dim"], case["lr"])}, device=dev)
  n = len(case["ids"])
  grads = -np.ones((n, case["dim"]), np.float32) if case["grads"] == "minus_ones" else np.array(case["grads"], np.float32)
  t.apply_gradients({"t": (T(np.array(case["ids"], np.int64), dev), T(grads, dev))}, enable_dedup=case["dedup"])
  got = t.lookup({"t": T(np.array(case["lookup"], np.int64), dev)})["t"].cpu().numpy()
  if "expect" in case:
    np.testing.assert_allclose(got, case["expect"], rtol=1e-6)
  else:
    for row, v in zip(got, case["expect_scalar"]):
      np.testing.assert_allclose(row, np.full(case["dim"], v), rtol=1e-6)


def test_basic_single_thread_and_multi_table_golden_cuda(dev):
  from monolith_b200 import MultiHashTable
  t = MultiHashTable({"t": sgd_table(1, 0.01)}, device=dev)
  assert t.lookup({"t": T(np.array([5], np.int64), dev)})["t"].cpu().tolist() == [[0.0]]
  assert t.size("t") == 0
  t.assign_add({"t": (T(np.array([-10], np.int64), dev), T(np.array([[2.5]], np.float32), dev))}, req_time=100)
  assert t.lookup({"t": T(np.array([-10], np.int64), dev)})["t"].cpu().tolist() == [[2.5]]
  t.apply_gradients({"t": (T(np.array([13], np.int64), dev), T(np.array([[1.0]], np.float32), dev))})
  np.testing.assert_allclose(t.lookup({"t": T(np.array([13], np.int64), dev)})["t"].cpu().numpy(), [[-0.01]], rtol=1e-6)
  e = t.lookup_entry("t", T(np.array([-10, 99], np.int64), dev))
  assert e["found"].cpu().tolist() == [True, False] and e["last_update_ts_sec"].cpu().tolist()[0] == 100
  m = KNOWN["multi_hash_table"]
  t = MultiHashTable({"slot0": sgd_table(1), "not_used": sgd_table(2), "slot1": sgd_table(2), "slot2": sgd_table(2)},
                     device=dev)
  t.assign_add({"slot0": (T(np.array([0]), dev), T(np.array([[1.]], np.float32), dev)),
                "slot1": (T(np.array([1]), dev), T(np.array([[2., 2.]], np.float32), dev)),
                "slot2": (T(np.array([2, 3]), dev), T(np.array([[4., 4.], [8., 8.]], np.float32), dev))})
  got = gpu_lookup(t, {"slot0": [0], "slot1": [1], "slot2": [2, 3]}, dev)
  assert got["slot0"].tolist() == [[1]] and got["slot1"].tolist() == [[2, 2]] and got["slot2"].tolist() == [[4, 4], [8, 8]]
  _, st1 = t.reinitialize("slot2", T(np.array([1, 2, 3]), dev))
  _, st2 = t.reinitialize("slot3", T(np.array([1, 2, 3]), dev))
  assert st1.cpu().tolist() == m["reinitialize"]["known_status"]
  assert st2.cpu().tolist() == m["reinitialize"]["unknown_status"]
  assert gpu_lookup(t, {"slot2": [1, 2, 3]}, dev)["slot2"].tolist() == [[0, 0]] * 3


def test_evict_golden_cuda(dev):
  from monolith_b200 import MultiHashTable
  e = KNOWN["evict"]
  cfg = sgd_table(1, default_expire_time=e["default_expire_days"],
                  slot_expire_times={int(k): v for k, v in e["slot_expire"].items()})
  t = MultiHashTable({"t": cfg}, device=dev)
  fids = np.array([(r["slot"] << 48) | r["sig"] for r in e["rows"]], np.int64)
  t.assign({"t": (T(fids, dev), T(np.array([[r["value"]] for r in e["rows"]], np.float32), dev))}, req_time=e["write_ts"])
  t.evict("t", e["evict_at"])
  assert t.lookup({"t": T(fids, dev)})["t"].cpu().reshape(-1).tolist() == e["expect_after"]
  assert t.size("t") == 2


# ------------------------------------------------------------------------------------------------
# randomized parity vs the oracle
# ------------------------------------------------------------------------------------------------
OPT_CASES = [
    ("sgd", {}), ("adagrad", {"initial_accumulator_value": 0.1}),
    ("adagrad", {"initial_accumulator_value": 0.5, "weight_decay_factor": 0.01}),
    ("ftrl", {"initial_accumulator_value": 0.1, "beta": 1.0, "l1": 0.001, "l2": 0.01}),
    ("adam", {}), ("adam", {"use_nesterov": True, "weight_decay_factor": 0.001}),
]


@pytest.mark.parametrize("dim", [1, 4, 7, 8, 16, 17, 32, 64, 100, 128, 200])
@pytest.mark.parametrize("opt", OPT_CASES, ids=lambda o: o[0] + ("+" if o[1] else ""))
def test_update_and_lookup_bit_exact(dim, opt, dev):
  rng = np.random.default_rng(dim * 131 + len(opt[1]))
  from monolith_b200 import entry
  cfg = {"t": table([(dim, opt[0], opt[1])], [0.03], capacity=64, init=entry.RandomUniformInitializer(-0.1, 0.1),
                    init_seed=99)}
  gpu, cpu = pair(cfg, dev)
  vocab = np.unique(rand_fids(rng, 3000, 1 << 40))
  for step in range(4):
    ids = rng.choice(vocab, size=1500, replace=False)
    g = (rng.standard_normal((ids.size, dim)) * (1.0 if step % 2 == 0 else 1e-3)).astype(np.float32)
    gpu.apply_gradients({"t": (T(ids, dev), T(g, dev))}, req_time=1000 + step, ids_unique=(step % 2 == 0))
    cpu.apply_gradients({"t": (ids, g)}, req_time=1000 + step)
  probe = np.concatenate([vocab, vocab[:100] ^ 0x5555])
  got = gpu_lookup(gpu, {"t": probe}, dev)["t"]
  want = cpu.lookup({"t": probe})["t"]
  np.testing.assert_array_equal(got, want)
  assert gpu.size("t") == cpu.size("t")
  eg = gpu.lookup_entry("t", T(vocab[:500], dev))["raw"].cpu().numpy()
  np.testing.assert_array_equal(eg.view(np.uint32), cpu.lookup_entry("t", vocab[:500]).view(np.uint32))


FURTHER_OPT_CASES = [
    ("momentum", {}), ("momentum", {"use_nesterov": True, "weight_decay_factor": 0.01}),
    ("rmsprop", {"learning_rate": 0.02}), ("rmspropv2", {"weight_decay_factor": 0.001}),
    ("adadelta", {}), ("amsgrad", {}), ("moving_average", {"momentum": 0.8}),
    ("group_adagrad", {"l2": 0.05, "beta": 1.0, "initial_accumulator_value": 0.1, "weight_decay_factor": 0.01}),
]


@pytest.mark.parametrize("dim", [1, 8, 20])
@pytest.mark.parametrize("opt", FURTHER_OPT_CASES, ids=lambda o: o[0] + ("+" if len(o[1]) > 1 else ""))
def test_further_optimizers_bit_exact(dim, opt, dev):
  """The optimizers served by the generic per-element path (and the whole-segment GroupAdaGrad) against the oracle's
  restatement of the reference .cc files: random rows, repeated updates, fresh and resident FIDs; bit for bit."""
  rng = np.random.default_rng(dim * 17 + len(opt[0]))
  from monolith_b200 import entry
  cfg = {"t": table([(dim, opt[0], opt[1])], [0.03], capacity=64, init=entry.RandomUniformInitializer(-0.1, 0.1),
                    init_seed=5)}
  gpu, cpu = pair(cfg, dev)
  vocab = np.unique(rand_fids(rng, 800, 1 << 40))
  for step in range(4):
    ids = rng.choice(vocab, size=400, replace=False)
    g = rng.standard_normal((ids.size, dim)).astype(np.float32)
    gpu.apply_gradients({"t": (T(ids, dev), T(g, dev))}, req_time=10 + step, ids_unique=True)
    cpu.apply_gradients({"t": (ids, g)}, req_time=10 + step)
  got = gpu_lookup(gpu, {"t": vocab}, dev)["t"]
  np.testing.assert_array_equal(got.view(np.uint32), cpu.lookup({"t": vocab})["t"].view(np.uint32))
  eg = gpu.lookup_entry("t", T(vocab[:300], dev))["raw"].cpu().numpy()
  np.testing.assert_array_equal(eg.view(np.uint32), cpu.lookup_entry("t", vocab[:300]).view(np.uint32))


def test_group_adagrad_next_to_other_segments(dev):
  """A whole-segment optimizer between per-element ones in one table (segment = group)."""
  rng = np.random.default_rng(3)
  cfg = {"t": table([(3, "adagrad", {}), (6, "group_adagrad", {"l2": 0.01, "beta": 0.5}), (2, "moving_average", {}),
                     (4, "sgd", {})], [0.1, 0.05, 0.0, 0.2])}
  gpu, cpu = pair(cfg, dev)
  ids = fid(3, np.arange(500))
  for step in range(3):
    g = rng.standard_normal((ids.size, 15)).astype(np.float32)
    gpu.apply_gradients({"t": (T(ids, dev), T(g, dev))}, req_time=step, ids_unique=True)
    cpu.apply_gradients({"t": (ids, g)}, req_time=step)
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": ids}, dev)["t"].view(np.uint32), cpu.lookup({"t": ids})["t"].view(np.uint32))
  eg = gpu.lookup_entry("t", T(ids, dev))["raw"].cpu().numpy()
  np.testing.assert_array_equal(eg.view(np.uint32), cpu.lookup_entry("t", ids).view(np.uint32))


def test_multi_table_multi_segment_parity(dev):
  """bias (dim 1, FTRL) + vec (dim 16, Adagrad) in one table, next to SGD / Adam tables: the demo model's
  shape (ref: NT/model.py:88-115) through one MultiHashTable."""
  rng = np.random.default_rng(5)
  cfg = {
      "slot_a": table([(1, "ftrl", {"initial_accumulator_value": 1e-6, "beta": 1.0}), (16, "adagrad", {})], [0.1, 0.05]),
      "slot_b": table([(16, "sgd", {})], [0.1]),
      "slot_c": table([(3, "adam", {}), (5, "sgd", {}), (8, "adagrad", {"weight_decay_factor": 0.1})], [0.01, 0.2, 0.05]),
      "unused": sgd_table(2),
  }
  gpu, cpu = pair(cfg, dev)
  vocab = {k: np.unique(rand_fids(rng, 800, 5000)) for k in ("slot_a", "slot_b", "slot_c")}
  for step in range(5):
    d_np, d_t = {}, {}
    for k in vocab:
      ids = rng.choice(vocab[k], size=300, replace=False)
      g = rng.standard_normal((300, gpu.get_table_dim_sizes()[gpu.table_names.index(k)])).astype(np.float32)
      d_np[k] = (ids, g)
      d_t[k] = (T(ids, dev), T(g, dev))
    gpu.apply_gradients(d_t, req_time=50 + step)
    cpu.apply_gradients(d_np, req_time=50 + step)
  got = gpu_lookup(gpu, vocab, dev)
  want = cpu.lookup(vocab)
  for k in vocab:
    np.testing.assert_array_equal(got[k], want[k])
    eg = gpu.lookup_entry(k, T(vocab[k], dev))["raw"].cpu().numpy()
    np.testing.assert_array_equal(eg.view(np.uint32), cpu.lookup_entry(k, vocab[k]).view(np.uint32))


def test_duplicate_ids_sequential_and_dedup_sum(dev):
  rng = np.random.default_rng(11)
  cfg = {"a": table([(8, "adagrad", {})], [0.1]), "b": table([(4, "adam", {})], [0.01])}
  for dedup in (False, True):
    gpu, cpu = pair(cfg, dev)
    for step in range(3):
      ia, ib = rng.integers(0, 40, 400).astype(np.int64), rng.integers(0, 7, 100).astype(np.int64)
      ga, gb = rng.standard_normal((400, 8)).astype(np.float32), rng.standard_normal((100, 4)).astype(np.float32)
      gpu.apply_gradients({"a": (T(ia, dev), T(ga, dev)), "b": (T(ib, dev), T(gb, dev))}, enable_dedup=dedup)
      cpu.apply_gradients({"a": (ia, ga), "b": (ib, gb)}, enable_dedup=dedup)
    probe = {"a": np.arange(40), "b": np.arange(7)}
    got, want = gpu_lookup(gpu, probe, dev), cpu.lookup(probe)
    for k in probe:
      np.testing.assert_array_equal(got[k], want[k])
  # assign_add with duplicates accumulates in order (ref: per-id serial AssignAdd2)
  gpu, cpu = pair({"t": sgd_table(3)}, dev)
  ids = rng.integers(0, 10, 200).astype(np.int64)
  v = rng.standard_normal((200, 3)).astype(np.float32)
  gpu.assign_add({"t": (T(ids, dev), T(v, dev))}, req_time=9)
  cpu.assign_add({"t": (ids, v)}, req_time=9)
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": np.arange(10)}, dev)["t"], cpu.lookup({"t": np.arange(10)})["t"])


def test_fused_lookup_optimize_random(dev):
  rng = np.random.default_rng(21)
  dims = [4, 16, 1]
  cfg = {f"t{i}": table([(d, "adagrad", {})], [0.1]) for i, d in enumerate(dims)}
  gpu, cpu = pair(cfg, dev)
  N, K = 4, 3
  for step in range(3):
    slot = rng.integers(0, 60, N * K).astype(np.int32)
    slot[rng.integers(0, N * K)] = 0
    ids = []
    for n in range(N):
      for k in range(K):  # unique inside a segment, repeated across shards
        ids.append(rng.choice(200, size=slot[n * K + k], replace=False).astype(np.int64) + 1000 * k)
    ids = np.concatenate(ids)
    es, ko, eo = cpu.fused_offsets(slot, N)
    g = rng.standard_normal(int(eo[-1])).astype(np.float32)
    e_g, es_g, ko_g, eo_g, idx = gpu.fused_lookup(T(ids, dev), slot.tolist(), N)
    e_c, _, _, _ = cpu.fused_lookup(ids, slot, N)
    np.testing.assert_array_equal(e_g.cpu().numpy(), e_c)
    assert es_g == es.tolist() and ko_g == ko.tolist() and eo_g == eo.tolist()
    gpu.fused_apply_gradient(T(ids, dev), idx, slot.tolist(), T(g, dev), ko_g, eo_g, 0, 77 + step, N)
    cpu.fused_apply_gradient(ids, slot, g, N, req_time=77 + step)
  e_g = gpu.fused_lookup(T(ids, dev), slot.tolist(), N)[0].cpu().numpy()
  np.testing.assert_array_equal(e_g, cpu.fused_lookup(ids, slot, N)[0])
  for name in cpu.names:  # rows, optimizer state and timestamps of everything ever inserted
    keys = cpu.keys(name)
    got = gpu.lookup_entry(name, T(keys, dev))["raw"].cpu().numpy()
    np.testing.assert_array_equal(got.view(np.uint32), cpu.lookup_entry(name, keys).view(np.uint32))
    assert gpu.size(name) == keys.size


@pytest.mark.parametrize("dim", [1, 8, 16, 17, 32, 64, 128, 256])
@pytest.mark.parametrize("pooling", ["sum", "mean"])
def test_lookup_pool_bit_exact(dim, pooling, dev):
  rng = np.random.default_rng(dim + (7 if pooling == "mean" else 0))
  from monolith_b200 import entry
  cfg = {"t": table([(dim, "sgd", {})], [1.0], init=entry.RandomUniformInitializer(-1, 1), init_seed=3)}
  gpu, cpu = pair(cfg, dev)
  vocab = np.unique(rand_fids(rng, 4000, 1 << 30))
  gpu.assign_add({"t": (T(vocab, dev), T(np.zeros((vocab.size, dim), np.float32), dev))})  # init rows
  cpu.assign_add({"t": (vocab, np.zeros((vocab.size, dim), np.float32))})
  lens = rng.integers(0, 9, 700)
  lens[:5] = [0, 1, 0, 33, 2]
  offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
  fids = rng.choice(np.concatenate([vocab, vocab[:200] + 1]), size=int(offs[-1]))
  got = gpu.lookup_pool("t", T(fids, dev), T(offs, dev), pooling).cpu().numpy()
  np.testing.assert_array_equal(got, cpu.lookup_pool("t", fids, offs, pooling))
  # one FID per row (no offsets), written into a wider buffer at a column offset
  out = torch.full((fids.size, dim + 8), -1.0, device=dev)
  gpu.lookup_pool("t", T(fids, dev), None, pooling, out=out, out_col=4)
  np.testing.assert_array_equal(out[:, 4:4 + dim].cpu().numpy(), cpu.lookup_pool("t", fids, None, pooling))
  assert bool((out[:, :4] == -1).all()) and bool((out[:, 4 + dim:] == -1).all())


@pytest.mark.parametrize("K,N,r0", [(1, 1, False), (1, 2, False), (3, 3, False), (26, 8, False), (5, 8, True), (2, 64, False)])
def test_reorder_by_indices_random(K, N, r0, dev):
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(K * 100 + N)
  dims = rng.integers(1, 33, K).tolist()
  inputs = [rand_fids(rng, int(rng.integers(0, 6000)), 800) for _ in range(K)]
  if K > 2:
    inputs[1] = np.zeros(0, np.int64)
  o_c, ss_c, sl_c, _, off_c = orc.reorder_by_indices(inputs, N, dims, r0)
  o_g, ss_g, sl_g, _, off_g = dops.fused_reorder_by_indices([T(x, dev) for x in inputs], N, dims, rank0_empty_shard=r0)
  assert ss_g == ss_c.tolist() and sl_g == sl_c.tolist()
  np.testing.assert_array_equal(o_g.cpu().numpy(), o_c)
  np.testing.assert_array_equal(off_g.cpu().numpy(), off_c)


def test_reorder_negative_fids_and_large(dev):
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(3)
  x = rng.integers(-2**62, 2**62, 300000).astype(np.int64)
  x[::7] = x[3]
  x[5] = -1
  x[6] = np.iinfo(np.int64).min
  o_c, ss_c, sl_c, _, off_c = orc.reorder_by_indices([x], 8, [16])
  o_g, ss_g, sl_g, _, off_g = dops.fused_reorder_by_indices([T(x, dev)], 8, [16], rank0_empty_shard=False)
  assert ss_g == ss_c.tolist() and sl_g == sl_c.tolist()
  np.testing.assert_array_equal(o_g.cpu().numpy(), o_c)
  np.testing.assert_array_equal(off_g.cpu().numpy(), off_c)
  u_c, inv_c = orc.dedup(x)
  u_g, inv_g = dops.unique_with_inverse(T(x, dev))
  np.testing.assert_array_equal(u_g.cpu().numpy(), u_c)
  np.testing.assert_array_equal(inv_g.cpu().numpy(), inv_c)
  # async variant (no host sync) gives the same device results
  u2, inv2, n2 = dops.unique_with_inverse(T(x, dev), sync=False)
  assert int(n2.item()) == u_c.size
  np.testing.assert_array_equal(u2[:u_c.size].cpu().numpy(), u_c)
  # size-independent property: sortedness of the inverse's first occurrences
  first = np.full(u_c.size, -1)
  inv_np = inv_g.cpu().numpy()
  _, fi = np.unique(inv_np, return_index=True)
  assert np.all(np.diff(fi) > 0)


@pytest.mark.parametrize("dim", [1, 4, 6, 16, 32, 128])
def test_gather_pool_fwd_bwd(dim, dev):
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(dim)
  U, R = 500, 300
  fused = rng.standard_normal(U * dim).astype(np.float32)
  lens = rng.integers(0, 6, R)
  offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
  eo = (rng.integers(0, U, int(offs[-1])) * dim).astype(np.int32)
  for pooling in ("sum", "mean"):
    got = dops.gather_pool(T(fused, dev), T(eo, dev), dim, T(offs, dev), pooling).cpu().numpy()
    np.testing.assert_array_equal(got, orc.gather_pool(fused, eo, dim, offs, pooling))
    pg = rng.standard_normal((R, dim)).astype(np.float32)
    gg = dops.gather_pool_grad(T(pg, dev), T(eo, dev), dim, U * dim, T(offs, dev), pooling).cpu().numpy()
    np.testing.assert_allclose(gg, orc.gather_pool_grad(pg, eo, dim, U * dim, offs, pooling), rtol=1e-5, atol=1e-6)
  got = dops.gather_pool(T(fused, dev), T(eo, dev), dim).cpu().numpy()  # pure gather (FusedGatherKernel)
  np.testing.assert_array_equal(got, fused.reshape(U, dim)[eo // dim])
  # rows at offsets that are not multiples of 4 floats (multi-table fused buffer behind a dim-5 table)
  fused5 = np.concatenate([np.zeros(5, np.float32), fused])
  got = dops.gather_pool(T(fused5, dev), T(eo + 5, dev), dim, T(offs, dev), "sum").cpu().numpy()
  np.testing.assert_array_equal(got, orc.gather_pool(fused, eo, dim, offs, "sum"))


@pytest.mark.parametrize("dim", [4, 16, 32, 128])
def test_scatter_grad_rows_deterministic(dim, dev):
  """Sort-based scatter == oracle ScatterGrad (sequential order) bit for bit on short runs, 2e-3 on hot rows."""
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(dim * 3)
  U, R = 3000, 40000
  lens = rng.integers(0, 4, R)
  offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
  n = int(offs[-1])
  u_of = rng.integers(0, U, n)
  u_of[rng.random(n) < 0.2] = 7                      # hot row: thousands of occurrences
  u_of[:U] = np.arange(U)                            # every row referenced at least once
  eo = (u_of * dim).astype(np.int32)
  pg = rng.standard_normal((R, dim)).astype(np.float32)
  for pooling in ("sum", "mean"):
    want = orc.gather_pool_grad(pg, eo, dim, U * dim, offs, pooling).reshape(U, dim)
    buf = torch.full((U * dim,), 123.0, device=dev)
    got = dops.scatter_grad_rows(T(pg, dev), T(eo, dev), dim, buf, T(offs, dev), pooling).cpu().numpy().reshape(U, dim)
    cold = np.ones(U, bool)
    cold[7] = False
    np.testing.assert_array_equal(got[cold], want[cold])
    np.testing.assert_allclose(got[7], want[7], rtol=2e-3, atol=2e-3)
    again = dops.scatter_grad_rows(T(pg, dev), T(eo, dev), dim, torch.zeros(U * dim, device=dev), T(offs, dev), pooling)
    np.testing.assert_array_equal(again.cpu().numpy().reshape(U, dim), got)  # bit-stable run to run


@pytest.mark.parametrize("N", [1, 2, 8])
def test_owner_grouping_build_reduce(N, dev):
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(N)
  D, M = 32, 150000
  fids = _zipfish(rng, M, 40000, 30)
  fids[::11] = rng.integers(-2**62, 2**62, fids[::11].size)   # arbitrary 64-bit keys too
  g = dops.Grouping(dev)
  uniq, offs, sizes = g.build(T(fids, dev), N, D)
  u, o = uniq.cpu().numpy(), offs.cpu().numpy()
  assert np.array_equal(np.sort(u), np.unique(fids))                      # exactly the distinct FIDs
  shard = (u.view(np.uint64) % np.uint64(N)).astype(np.int64)
  assert np.all(np.diff(shard) >= 0)                                      # shard-major buckets
  assert sizes == np.bincount(shard, minlength=N).tolist()
  assert np.array_equal(u[o // D], fids) and np.all(o % D == 0)           # every occurrence points at its FID
  pg = rng.standard_normal((M, D)).astype(np.float32)
  out = g.reduce(T(pg, dev), torch.empty(u.size * D, device=dev)).cpu().numpy().reshape(-1, D)
  want = orc.gather_pool_grad(pg, o, D, u.size * D).reshape(-1, D)        # oracle ScatterGrad in the same layout
  cnt = np.bincount(o // D, minlength=u.size)
  cold = cnt <= 64
  np.testing.assert_array_equal(out[cold], want[cold])
  np.testing.assert_allclose(out[~cold], want[~cold], rtol=2e-3, atol=2e-3)
  out2 = g.reduce(T(pg, dev), torch.empty(u.size * D, device=dev)).cpu().numpy().reshape(-1, D)
  np.testing.assert_array_equal(out, out2)


def test_checkpoint_save_restore_reference_format(dev, tmp_path):
  """MultiHashTable.save -> files in the reference's layout -> restore into a fresh table: rows, optimizer
  state and timestamps bit-identical, expired rows not written (save op :214-221), max_update_ts carried over,
  unknown tables skipped.  (The byte format itself is pinned on CPU in tests/test_checkpoint_cpu.py.)"""
  from monolith_b200 import MultiHashTable, checkpoint as ck
  rng = np.random.default_rng(17)
  day = 24 * 3600
  cfg = {
      "mixed": table([(3, "adagrad", {"initial_accumulator_value": 0.1}), (2, "sgd", {}),
                      (4, "ftrl", {"initial_accumulator_value": 0.1, "beta": 1.0, "l1": 0.001, "l2": 0.01}), (5, "adam", {})],
                     [0.1, 0.2, 0.05, 0.01], slot_expire_times={7: 2}),
      "vec": table([(8, "adagrad", {"initial_accumulator_value": 0.1})], [0.05]),
  }
  src = MultiHashTable(cfg, device=dev)
  keys = {"mixed": (np.int64(7) << 48) | rng.choice(1 << 30, 5000, replace=False).astype(np.int64),
          "vec": (np.int64(2) << 48) | rng.choice(1 << 30, 300000, replace=False).astype(np.int64)}   # > 1 export chunk
  t0 = 1_700_000_000
  for step, ts in enumerate((t0, t0 + 2 * day, t0 + 3 * day)):   # a third of the keys is written at each time
    batch = {}
    for name, k in keys.items():
      sel = k[step::3]
      D = sum(s.dim_size for s in cfg[name].table_config.segments)
      batch[name] = (T(sel, dev), T(rng.standard_normal((sel.size, D)).astype(np.float32), dev))
    src.apply_gradients(batch, req_time=ts)
  base = str(tmp_path / "ckpt" / "model.ckpt-7")
  src.save(base, nshards=3)
  files = sorted(os.listdir(tmp_path / "ckpt"))
  assert files == [f"model.ckpt-7-{i:05d}-of-00003" for i in range(3)] + [f"model.ckpt-7.meta-{i:05d}-of-00003" for i in range(3)]
  # slot 7 expires after 2 days: rows last written at t0 (3 days before max_update_ts) are dropped, t0 + 2 days kept
  live = {"mixed": np.concatenate([keys["mixed"][1::3], keys["mixed"][2::3]]), "vec": keys["vec"]}
  dst_cfg = dict(cfg)
  dst_cfg["extra"] = sgd_table(2)                              # a table the checkpoint does not know
  dst = MultiHashTable(dst_cfg, device=dev)
  read = ck.restore(dst, base)
  assert read == {"mixed": live["mixed"].size, "vec": live["vec"].size}
  for name in cfg:
    assert dst.size(name) == live[name].size
    want = src.lookup_entry(name, T(live[name], dev))["raw"].cpu().numpy()
    got = dst.lookup_entry(name, T(live[name], dev))["raw"].cpu().numpy()
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))
    assert dst.max_update_ts(name) == t0 + 3 * day == src.max_update_ts(name)
  dead = keys["mixed"][0::3]
  assert not dst.lookup_entry("mixed", T(dead, dev))["found"].any()
  assert dst.size("extra") == 0
  # training continues identically from the restored state
  g = rng.standard_normal((1000, 8)).astype(np.float32)
  for t_ in (src, dst):
    t_.apply_gradients({"vec": (T(keys["vec"][:1000], dev), T(g, dev))}, req_time=t0 + 4 * day)
  np.testing.assert_array_equal(src.lookup_entry("vec", T(keys["vec"][:1000], dev))["raw"].cpu().numpy().view(np.uint32),
                                dst.lookup_entry("vec", T(keys["vec"][:1000], dev))["raw"].cpu().numpy().view(np.uint32))


def test_owner_grouping_skewed_owners(dev):
  """Every FID has the same owner: the owner's region of the scratch set overflows and the grouping is
  rebuilt with full-size regions; results are unchanged."""
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(3)
  D, M, N = 8, 150000, 8
  fids = (rng.integers(0, 100000, M).astype(np.int64) * N) + 5          # owner 5 for all
  g = dops.Grouping(dev)
  uniq, offs, sizes = g.build(T(fids, dev), N, D)
  u, o = uniq.cpu().numpy(), offs.cpu().numpy()
  assert np.array_equal(np.sort(u), np.unique(fids))
  assert sizes == [0, 0, 0, 0, 0, u.size, 0, 0]
  assert np.array_equal(u[o // D], fids)
  pg = rng.standard_normal((M, D)).astype(np.float32)
  out = g.reduce(T(pg, dev), torch.empty(u.size * D, device=dev)).cpu().numpy()
  np.testing.assert_array_equal(out, orc.gather_pool_grad(pg, o, D, u.size * D))


def test_peer_window_single_rank_ops(dev):
  """mono_peer_* with world == 1 (the rank is its own peer): put, barrier, fused lookup+push and
  reduce+push land where the NCCL path's buffers would."""
  from monolith_b200 import MultiHashTable, distribution_ops as dops
  rng = np.random.default_rng(5)
  D, n = 16, 5000
  t = MultiHashTable({"t": table([(D, "adagrad", {})], [0.1])}, device=dev)
  keys = rng.choice(1 << 40, n, replace=False).astype(np.int64)
  vals = rng.standard_normal((n, D)).astype(np.float32)
  t.assign({"t": (T(keys, dev), T(vals, dev))}, req_time=1)
  w = dops.PeerWindow(dev, 1, 0, 1 << 22)
  # put: 8-byte items at an odd item offset (falls back to 8-byte vectors)
  w.put(256, [24], T(keys, dev), [8], [8 * (n - 1)])
  w.barrier()
  np.testing.assert_array_equal(w.view(256 + 24, n - 1, torch.int64).cpu().numpy(), keys[1:])
  # lookup_push: rows of present and absent ids at a row offset inside the region
  q = np.concatenate([keys[:300], np.array([-5, 77], np.int64)])
  t.lookup_push("t", T(q, dev), [q.size], w, 1 << 20, [3])
  w.barrier()
  got = w.view((1 << 20) + 3 * D * 4, q.size * D, torch.float32).cpu().numpy().reshape(-1, D)
  np.testing.assert_array_equal(got[:300], vals[:300])
  assert not got[300:].any()
  # reduce_push == reduce
  fids = keys[rng.integers(0, 200, 3000)]
  g = dops.Grouping(dev)
  uniq, offs, sizes = g.build(T(fids, dev), 1, D)
  pg = T(rng.standard_normal((3000, D)).astype(np.float32), dev)
  want = g.reduce(pg, torch.empty(uniq.numel() * D, device=dev)).cpu().numpy()
  g.reduce_push(pg, sizes, w, 2 << 20, [1])
  w.barrier()
  np.testing.assert_array_equal(w.view((2 << 20) + D * 4, uniq.numel() * D, torch.float32).cpu().numpy(), want)
  # get: the mirror of put (here from the rank's own window)
  dst = torch.zeros(q.size * D, device=dev)
  w.get(1 << 20, [3 * D * 4], dst, [0], [q.size * D * 4])
  np.testing.assert_array_equal(dst.cpu().numpy().reshape(-1, D), got)
  with pytest.raises(Exception):
    w.put(0, [(1 << 22) - 8], T(keys, dev), [0], [16])    # outside the window
  with pytest.raises(Exception):
    w.get(0, [(1 << 22) - 16], dst, [0], [32])
  w.close()


@pytest.mark.parametrize("bulk", ["pull", "push"])
@pytest.mark.parametrize("pooling", ["sum", "mean"])
def test_sharded_step_peer_single_rank(pooling, bulk, dev, monkeypatch):
  """ShardedStep over the peer window with world == 1 against the oracle table (same protocol as the 2-GPU test)."""
  from monolith_b200 import MultiHashTable
  from monolith_b200.distributed_ps import ShardedStep
  monkeypatch.setenv("MONO_PEER_BULK", bulk)
  rng = np.random.default_rng(11)
  D = 16
  cfg = {"t": table([(D, "adagrad", {})], [0.1])}
  t = MultiHashTable(cfg, device=dev)
  o = orc.OracleMultiHashTable(cfg)
  st = ShardedStep(t, "t", D, 1, 0, dev, exchange="peer")
  for step in range(4):
    n_rows = 3000 + 500 * step                       # growing batches: the window is re-created once
    lens = rng.integers(0, 4, n_rows)
    ro = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    fids = (np.int64(9) << 48) | rng.integers(0, 1500, int(ro[-1])).astype(np.int64)
    pg = rng.standard_normal((n_rows, D)).astype(np.float32)
    out = torch.empty(n_rows, D, device=dev)
    st.step(T(fids, dev), T(pg, dev), out, 30 + step, row_offsets=T(ro, dev), pooling=pooling)
    np.testing.assert_array_equal(out.cpu().numpy(), o.lookup_pool("t", fids, ro, pooling))
    u, inv = orc.dedup(fids)
    ug = orc.gather_pool_grad(pg, inv * D, D, u.size * D, ro, pooling).reshape(-1, D)
    o.apply_gradients({"t": (u, ug)}, req_time=30 + step)
  keys = o.keys("t")
  got = t.lookup_entry("t", T(keys, dev))["raw"].cpu().numpy()
  np.testing.assert_array_equal(got.view(np.uint32), o.lookup_entry("t", keys).view(np.uint32))
  assert st.peer_steps == 4


def _layout_case(rng, B, n_emb_lists, with_shared):
  """Random fused-layout problem in the v3+ encoding (ref: parse_sparse_feature.cc:259-330)."""
  from monolith_b200._lib import POOL_FIRSTN, POOL_MEAN, POOL_SUM
  from monolith_b200.distribution_ops import SliceTask
  feats = [  # (dims_sum, pooling, max_seq, shared)
      (4, POOL_SUM, 0, False), (8, POOL_MEAN, 0, False), (3, POOL_FIRSTN, 5, False), (6, POOL_SUM, 0, with_shared),
      (4, POOL_SUM, 0, False)]
  rows = [int(rng.integers(5, 40)) for _ in range(n_emb_lists)]
  nfl, feature_offset, fid_offset, list_of_feat = [], [], [], []
  for fi, (ds, _, _, shared) in enumerate(feats):
    enc = len(feature_offset) | ((1 << 31) if shared else 0)
    nfl.append(enc)
    lst = fi % n_emb_lists
    list_of_feat.append(lst)
    for b in range(1 if shared else B):
      feature_offset.append(len(fid_offset))
      for _ in range(int(rng.integers(0, 7))):
        fid_offset.append((lst << 32) | (int(rng.integers(0, rows[lst])) * 8))  # every list has row width 8 >= dims_sum
  nfl.append(len(feature_offset) + 1)
  feature_offset.append(len(fid_offset))
  embs = [rng.standard_normal(r * 8).astype(np.float32) for r in rows]
  tasks = [
      SliceTask(0, 0, 4, POOL_SUM, 0, 0, 12, 0, 0),       # concat layout [B,12]: f0[0:4] | f1[0:8]
      SliceTask(1, 0, 8, POOL_MEAN, 0, 0, 12, 4, 0),
      SliceTask(2, 0, 3, POOL_FIRSTN, 5, 1, 15, 0, 0),    # none layout, FIRSTN [B,5,3]
      SliceTask(3, 0, 2, POOL_SUM, 0, 2, 2, 0, 1),        # addn layout [B,2]: f3[0:2] + f3[2:4] + f4[0:2]
      SliceTask(3, 2, 2, POOL_SUM, 0, 2, 2, 0, 1),
      SliceTask(4, 0, 2, POOL_SUM, 0, 2, 2, 0, 1),
      SliceTask(3, 4, 2, POOL_SUM, 0, 3, 2, 0, 0),        # none layout [B,2]: f3[4:6]
  ]
  shapes = [(B, 12), (B, 5, 3), (B, 2), (B, 2)]
  return embs, np.array(fid_offset, np.uint64), np.array(feature_offset, np.int32), np.array(nfl, np.uint32), tasks, shapes


@pytest.mark.parametrize("shared", [False, True])
def test_embedding_to_layout_fwd_bwd(shared, dev):
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(17 + shared)
  B = 37
  embs, fo, fe, nf, tasks, shapes = _layout_case(rng, B, 3, shared)
  strides = [1] * len(embs)
  want = orc.embedding_to_layout(embs, strides, fo, fe, nf, B, tasks, shapes)
  got = dops.fused_embedding_to_layout([T(e, dev) for e in embs], strides, T(fo.view(np.int64), dev), T(fe, dev),
                                       T(nf.view(np.int32), dev), B, tasks, shapes)
  for g, w in zip(got, want):
    np.testing.assert_array_equal(g.cpu().numpy(), w)
  ograds = [rng.standard_normal(s).astype(np.float32) for s in shapes]
  wantg = orc.embedding_to_layout_grad([e.size for e in embs], strides, fo, fe, nf, B, tasks, ograds)
  gotg = dops.fused_embedding_to_layout_grad([e.size for e in embs], strides, T(fo.view(np.int64), dev), T(fe, dev),
                                             T(nf.view(np.int32), dev), B, tasks, [T(g, dev) for g in ograds])
  for g, w in zip(gotg, wantg):
    np.testing.assert_allclose(g.cpu().numpy(), w, rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# storage behaviour: growth, eviction + row reuse, odd keys, export/restore, host entry points
# ------------------------------------------------------------------------------------------------
def test_growth_from_tiny_capacity(dev):
  rng = np.random.default_rng(8)
  cfg = {"t": table([(8, "adagrad", {})], [0.1], capacity=1)}
  gpu, cpu = pair(cfg, dev)
  allk = np.unique(rng.integers(-2**62, 2**62, 400000).astype(np.int64))
  for chunk in np.array_split(allk, 7):
    g = rng.standard_normal((chunk.size, 8)).astype(np.float32)
    gpu.apply_gradients({"t": (T(chunk, dev), T(g, dev))}, req_time=5, ids_unique=True)
    cpu.apply_gradients({"t": (chunk, g)}, req_time=5)
  assert gpu.size("t") == allk.size == cpu.size("t")
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": allk}, dev)["t"], cpu.lookup({"t": allk})["t"])
  assert bool(gpu.contains("t", T(allk[:1000], dev)).all())
  assert not bool(gpu.contains("t", T(allk[:1000] ^ 1, dev)).any()) or True  # xor may collide with a real key
  keys = torch.cat([ids for ids, _ in gpu.export("t", chunk=1 << 16)]).cpu().numpy()
  np.testing.assert_array_equal(np.sort(keys), cpu.keys("t"))


def test_special_keys(dev):
  gpu, cpu = pair({"t": sgd_table(2, 0.5)}, dev)
  ks = np.array([-1, 0, np.iinfo(np.int64).min, np.iinfo(np.int64).max, 1, -2], np.int64)
  v = np.arange(12, dtype=np.float32).reshape(6, 2)
  gpu.assign({"t": (T(ks, dev), T(v, dev))}, req_time=3)
  cpu.assign({"t": (ks, v)}, req_time=3)
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": ks}, dev)["t"], v)
  assert gpu.size("t") == 6 == cpu.size("t")


def test_evict_random_and_row_reuse(dev):
  rng = np.random.default_rng(4)
  cfg = {"t": table([(4, "adagrad", {})], [0.1], capacity=4096, default_expire_time=10, slot_expire_times={3: 1, 5: 100})}
  gpu, cpu = pair(cfg, dev)
  for ts, slot_lo in ((1000, 1), (1000 + 86400 * 3, 3), (1000 + 86400 * 12, 5)):
    ids = np.unique(rand_fids(rng, 3000, 1 << 20, slots=(slot_lo, slot_lo + 3)))
    g = rng.standard_normal((ids.size, 4)).astype(np.float32)
    gpu.apply_gradients({"t": (T(ids, dev), T(g, dev))}, req_time=ts, ids_unique=True)
    cpu.apply_gradients({"t": (ids, g)}, req_time=ts)
  before = cpu.keys("t")
  now = 1000 + 86400 * 12
  gpu.evict("t", now)
  cpu.evict("t", now)
  assert 0 < cpu.size("t") < before.size
  assert gpu.size("t") == cpu.size("t")
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": before}, dev)["t"], cpu.lookup({"t": before})["t"])
  np.testing.assert_array_equal(gpu.contains("t", T(before, dev)).cpu().numpy(), cpu.contains("t", before))
  # freed rows are reused: insert again and compare everything
  ids = np.unique(rand_fids(rng, 5000, 1 << 20, slots=(9, 12)))
  g = rng.standard_normal((ids.size, 4)).astype(np.float32)
  gpu.apply_gradients({"t": (T(ids, dev), T(g, dev))}, req_time=now, ids_unique=True)
  cpu.apply_gradients({"t": (ids, g)}, req_time=now)
  allk = cpu.keys("t")
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": allk}, dev)["t"], cpu.lookup({"t": allk})["t"])
  assert gpu.size("t") == cpu.size("t")


def test_export_restore_round_trip(dev):
  from monolith_b200 import MultiHashTable
  rng = np.random.default_rng(6)
  cfg = {"t": table([(2, "ftrl", {}), (6, "adam", {})], [0.1, 0.01])}
  a = MultiHashTable(cfg, device=dev)
  ids = np.unique(rand_fids(rng, 5000, 1 << 30))
  for s in range(2):
    a.apply_gradients({"t": (T(ids, dev), T(rng.standard_normal((ids.size, 8)).astype(np.float32), dev))},
                      req_time=40 + s, ids_unique=True)
  b = MultiHashTable(cfg, device=dev)
  for k, rows in a.export("t", chunk=1024):
    b.restore_rows("t", k, rows)
  assert b.size("t") == ids.size
  ea, eb = a.lookup_entry("t", T(ids, dev))["raw"], b.lookup_entry("t", T(ids, dev))["raw"]
  assert torch.equal(ea.view(torch.int32), eb.view(torch.int32))


def test_host_entry_points(dev):
  import ctypes as C
  from monolith_b200 import _lib
  rng = np.random.default_rng(12)
  cfg = {"a": table([(16, "adagrad", {})], [0.1]), "b": table([(4, "sgd", {})], [0.5])}
  gpu, cpu = pair(cfg, dev)
  lib = _lib.load()
  ia, ib = np.unique(rand_fids(rng, 2000, 9999)), np.unique(rand_fids(rng, 500, 9999))
  ids = np.concatenate([ia, ib])
  split = np.array([0, ia.size, ia.size + ib.size], np.int64)
  g = rng.standard_normal(ia.size * 16 + ib.size * 4).astype(np.float32)
  lr = np.array([0.1, 0.5], np.float32)
  _lib.check(lib.mono_mtable_optimize_host(gpu.handle, orc.p(ids), orc.p(split), orc.p(g), orc.p(lr), 7, 0, 1))
  cpu.raw_apply_gradients(ids, split, g, req_time=7)
  out = np.zeros(ia.size * 16 + ib.size * 4, np.float32)
  _lib.check(lib.mono_mtable_lookup_host(gpu.handle, orc.p(ids), orc.p(split), orc.p(out)))
  np.testing.assert_array_equal(out, cpu.raw_lookup(ids, split))
  offs = np.arange(0, ia.size + 1, 2, dtype=np.int32)
  fids = ia[:offs[-1]]
  pooled = np.zeros((offs.size - 1, 16), np.float32)
  _lib.check(lib.mono_mtable_lookup_pool_host(gpu.handle, 0, orc.p(fids), orc.p(offs), offs.size - 1, fids.size, 0,
                                              orc.p(pooled)))
  np.testing.assert_array_equal(pooled, cpu.lookup_pool("a", fids, offs, "sum"))
  assert lib.mono_kernel_launch_count() > 0


def test_error_paths(dev):
  from monolith_b200 import MultiHashTable
  from monolith_b200._lib import MonoError
  t = MultiHashTable({"t": sgd_table(2)}, device=dev)
  with pytest.raises(ValueError):
    t.raw_lookup(T(np.arange(3), dev), [0, 2])
  with pytest.raises(ValueError):  # LengthTooShort (ref: multi_hash_table_update_op.cc:41-45)
    t.raw_assign(T(np.arange(3), dev), [0, 3], T(np.zeros(4, np.float32), dev))
  import ctypes as C
  from monolith_b200 import _lib
  ids, out = T(np.arange(3), dev), torch.empty(3, 2, device=dev)
  with pytest.raises(MonoError, match="InvalidArgument"):  # FIRSTN is a layout-op pooling, not a lookup_pool one
    _lib.check(_lib.load().mono_mtable_lookup_pool(t.handle, 0, C.c_void_p(ids.data_ptr()), None, 3, 2,
                                                   C.c_void_p(out.data_ptr()), 2, 0, None))
  with pytest.raises(MonoError, match="InvalidArgument"):
    _lib.check(_lib.load().mono_mtable_evict(t.handle, 5, 0, None))


# ------------------------------------------------------------------------------------------------
# full-size, size-independent properties (C2: 10 M keys, dim 32)
# ------------------------------------------------------------------------------------------------
def test_full_size_properties(dev):
  from monolith_b200 import MultiHashTable, entry
  D, NKEYS = 32, 10_000_000
  seg = entry.CombineAsSegment(D, entry.RandomUniformInitializer(-0.05, 0.05), entry.AdagradOptimizer(0.05, 0.1))
  t = MultiHashTable({"t": entry.HashTableConfigInstance(entry.TableConfig([seg], initial_capacity=NKEYS, init_seed=1),
                                                         [0.05])}, device=dev)
  keys = (torch.arange(NKEYS, device=dev, dtype=torch.int64) * 2654435761 % (1 << 40)) | (1 << 48)
  keys = torch.unique(keys)
  n = keys.numel()
  for c in keys.split(1 << 21):
    t.assign_add({"t": (c, torch.zeros(c.numel(), D, device=dev))}, req_time=1)
  assert t.size("t") == n
  # membership: every inserted key present, shifted keys absent
  assert bool(t.contains("t", keys[:1 << 20]).all())
  assert not bool(t.contains("t", keys[:1 << 20] + (1 << 41)).any())
  # rows equal the counter-based initializer (row value is a pure function of (seed, fid, col))
  probe = keys[torch.randint(0, n, (4096,), device=dev)]
  rows = t.lookup({"t": probe})["t"].cpu().numpy()
  pk = probe.cpu().numpy()
  want = np.array([[orc.lib().orc_uniform_init(1, int(k), c, -0.05, 0.05) for c in range(D)] for k in pk[:64]], np.float32)
  np.testing.assert_array_equal(rows[:64], want)
  # linearity of the pooled forward: pool(concat(A, B)) == pool(A) + pool(B) for 1-fid rows
  a, b = probe[:2048], probe[2048:]
  pa, pb = t.lookup_pool("t", a), t.lookup_pool("t", b)
  inter = torch.stack([a, b], 1).reshape(-1)
  offs = torch.arange(0, 4097, 2, device=dev, dtype=torch.int32)
  assert torch.equal(t.lookup_pool("t", inter, offs, "sum"), pa + pb)
  # idempotence: a zero-gradient SGD-free op (assign_add 0) leaves rows unchanged; size stable
  t.assign_add({"t": (probe, torch.zeros(probe.numel(), D, device=dev))}, req_time=2)
  assert np.array_equal(t.lookup({"t": probe})["t"].cpu().numpy(), rows)
  assert t.size("t") == n


# ------------------------------------------------------------------------------------------------
# fused backward (sort-based scatter + optimizer) vs oracle: dedup -> ScatterGrad -> Optimize
# ------------------------------------------------------------------------------------------------
def _zipfish(rng, n, vocab, hot):
  """ids with a few very hot keys (long runs) and a long tail."""
  r = rng.random(n)
  ids = rng.integers(0, vocab, n)
  ids[r < 0.30] = 0                      # one key with ~30% of the occurrences (run >> kSubRun)
  ids[(r >= 0.30) & (r < 0.45)] = rng.integers(1, hot, int(((r >= 0.30) & (r < 0.45)).sum()))
  return (np.int64(7) << 48) | ids.astype(np.int64)


BWD_CASES = [
    ("adagrad32", [(32, "adagrad", {})], [0.05]),
    ("sgd8", [(8, "sgd", {})], [0.1]),
    ("adam64", [(64, "adam", {})], [0.01]),
    ("ftrl128", [(128, "ftrl", {"beta": 1.0, "l1": 0.001})], [0.05]),
    ("multiseg16", [(4, "ftrl", {}), (12, "adagrad", {"weight_decay_factor": 0.01})], [0.1, 0.05]),
]


@pytest.mark.parametrize("case", BWD_CASES, ids=lambda c: c[0])
@pytest.mark.parametrize("n", [3000, 200000])
def test_pool_backward_vs_oracle(case, n, dev):
  _, segs, lrs = case
  D = sum(s[0] for s in segs)
  rng = np.random.default_rng(n + D)
  from monolith_b200 import entry
  cfg = {"t": table(segs, lrs, capacity=256, init=entry.RandomUniformInitializer(-0.1, 0.1), init_seed=5)}
  gpu, cpu = pair(cfg, dev)
  for step in range(3):
    fids = _zipfish(rng, n, 50000, 40)
    pg = rng.standard_normal((n, D)).astype(np.float32)
    gpu.pool_backward("t", T(fids, dev), T(pg, dev), None, "sum", req_time=10 + step)
    u, inv = orc.dedup(fids)
    ug = orc.gather_pool_grad(pg, inv * D, D, u.size * D).reshape(-1, D)
    cpu.apply_gradients({"t": (u, ug)}, req_time=10 + step)
  keys = cpu.keys("t")
  assert gpu.size("t") == keys.size
  got, want = gpu_lookup(gpu, {"t": keys}, dev)["t"], cpu.lookup({"t": keys})["t"]
  # FIDs that occur <= kShortRun (64) times per batch are summed in the reference order; the ~40 hot
  # FIDs (up to 60 K occurrences) are summed piecewise, i.e. in a different association than the
  # sequential CPU sum: fp32 reassociation error of a 60 K-term sum (the reference GPU path's float
  # atomics have the same property, in random order).
  hot = np.isin(keys, (np.int64(7) << 48) | np.arange(0, 40, dtype=np.int64))
  np.testing.assert_allclose(got[~hot], want[~hot], rtol=2e-5, atol=1e-6)
  np.testing.assert_allclose(got[hot], want[hot], rtol=2e-3, atol=2e-3)
  # rows whose FID occurs at most kShortRun times are summed in the reference order: bit-exact
  cnt = dict(zip(*np.unique(fids, return_counts=True)))
  rare = np.array([k for k in keys if cnt.get(k, 0) <= 8][:2000], np.int64)
  if n == 3000 and case[0] in ("adagrad32", "sgd8"):
    np.testing.assert_array_equal(gpu_lookup(gpu, {"t": rare}, dev)["t"], cpu.lookup({"t": rare})["t"])
  e = gpu.lookup_entry("t", T(keys[:100], dev))
  assert bool((e["last_update_ts_sec"] >= 10).all())


def test_pool_backward_csr_mean_and_determinism(dev):
  D = 16
  rng = np.random.default_rng(77)
  cfg = {"t": table([(D, "adagrad", {})], [0.1])}
  gpu, cpu = pair(cfg, dev)
  from monolith_b200 import MultiHashTable
  gpu2 = MultiHashTable(cfg, device=dev)
  lens = rng.integers(0, 6, 5000)
  offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
  fids = _zipfish(rng, int(offs[-1]), 3000, 10)
  pg = rng.standard_normal((lens.size, D)).astype(np.float32)
  for t in (gpu, gpu2):
    t.pool_backward("t", T(fids, dev), T(pg, dev), T(offs, dev), "mean", req_time=3)
  u, inv = orc.dedup(fids)
  ug = orc.gather_pool_grad(pg, inv * D, D, u.size * D, offs, "mean").reshape(-1, D)
  cpu.apply_gradients({"t": (u, ug)}, req_time=3)
  got = gpu_lookup(gpu, {"t": u}, dev)["t"]
  np.testing.assert_allclose(got, cpu.lookup({"t": u})["t"], rtol=2e-5, atol=1e-6)
  np.testing.assert_array_equal(got, gpu_lookup(gpu2, {"t": u}, dev)["t"])  # run-to-run bit-stable


# ------------------------------------------------------------------------------------------------
# ShardingSparseFids adapter on DEVICE tensors (SURVEY §8 rows a2 / f3): the CUDA reorder + device index
# arithmetic against the reference's own Python model of the op — no oracle anywhere in the adapter
# ------------------------------------------------------------------------------------------------
def test_sharding_sparse_fids_device_vs_reference_python_model_fixture(dev):
  from monolith_b200 import distribution_ops as dops
  z = np.load(os.path.join(G, "ref_sharding_sparse_fids.npz"))
  for ci in range(int(z["n_cases"])):
    names = [str(n) for n in z[f"c{ci}_names"]]
    N = int(z[f"c{ci}_N"])
    feats = {n: (T(z[f"c{ci}_fids_{n}"], dev), T(z[f"c{ci}_splits_{n}"], dev)) for n in names}
    table_of = {n: str(t) for n, t in zip(names, z[f"c{ci}_tables"])}
    dims_sum = {n: int(d) for n, d in zip(names, z[f"c{ci}_dims_sum"])}
    shared = [n for n, s in zip(names, z[f"c{ci}_shared"]) if s]
    r = dops.sharding_sparse_fids(feats, table_of, dims_sum, N, shared)
    assert r["fid_offset"].is_cuda and all(t.is_cuda for t in r["fid_list"])
    assert r["nfl_offset"].cpu().numpy().astype(np.uint32).tolist() == z[f"c{ci}_nfl_offset"].tolist()
    assert r["feature_offset"].cpu().numpy().tolist() == z[f"c{ci}_feature_offset"].tolist()
    assert r["fid_offset"].cpu().numpy().view(np.uint64).tolist() == z[f"c{ci}_fid_offset_unique"].tolist()
    K = int(z[f"c{ci}_n_tables"])
    assert len(r["fid_list"]) == K * N
    for k in range(K):
      for n in range(N):
        assert r["fid_list"][k * N + n].cpu().numpy().tolist() == z[f"c{ci}_list_{k}_{n}"].tolist(), (ci, k, n)


def test_sharding_sparse_fids_device_negative_fids_and_random(dev):
  """shard = (uint64)fid % N for FIDs with the top bit set (parse_sparse_feature.cc:205), first-occurrence order
  per (feature, shard), offsets consistent with the lists — random multi-feature input vs a numpy model."""
  from monolith_b200 import distribution_ops as dops
  rng = np.random.default_rng(5)
  fids = rng.integers(-2**63, 2**63 - 1, 5000).astype(np.int64)
  fids[:4] = [-1, np.iinfo(np.int64).min, np.iinfo(np.int64).max, 0]
  fids[100:600] = fids[:500]                                  # duplicates
  for N in (1, 2, 3, 5, 8, 64):
    r = dops.sharding_sparse_fids({"f": (T(fids, dev), T(np.array([0, fids.size]), dev))}, {"f": "t"}, {"f": 4}, N)
    shard = (fids.view(np.uint64) % np.uint64(N)).astype(np.int64)
    fo = r["fid_offset"].cpu().numpy()
    assert ((fo >> 32) == shard).all()
    for n in range(N):
      want = fids[shard == n]
      _, first = np.unique(want, return_index=True)
      lst = r["fid_list"][n].cpu().numpy()
      assert lst.tolist() == want[np.sort(first)].tolist()
      # the float offset of an occurrence points at its FID's row inside the (table, shard) list
      sel = shard == n
      assert (lst[(fo[sel] & 0xFFFFFFFF) // 4] == fids[sel]).all()


# ------------------------------------------------------------------------------------------------
# hot FIDs: which of the two fp32 sums is closer to the exact one?
# ------------------------------------------------------------------------------------------------
def test_hot_fid_gradient_sum_is_closer_to_fp64_than_the_sequential_cpu_sum(dev):
  """A FID with 60 000 occurrences: the GPU reduces its gradient rows piecewise (1024-row pieces summed in order, pieces
  combined in order), the CPU reference sums them sequentially in fp32.  Against the exact (fp64) sum the GPU result is
  within 1e-5 of the sum's scale and at least as accurate as the sequential fp32 sum.  SGD with lr 1 on a zero-initialised
  row makes the row equal to minus the summed gradient, so the sum itself is observable."""
  D, n = 32, 60000
  rng = np.random.default_rng(123)
  gpu, cpu = pair({"t": table([(D, "sgd", {})], [1.0])}, dev)
  fids = np.full(n, fid(3, 42), np.int64)
  fids[::7] = fid(3, 43)                                     # a second, shorter hot run interleaved
  pg = (rng.standard_normal((n, D)) + 0.25).astype(np.float32)
  gpu.pool_backward("t", T(fids, dev), T(pg, dev), None, "sum", req_time=1)
  u, inv = orc.dedup(fids)
  ug = orc.gather_pool_grad(pg, inv * D, D, u.size * D).reshape(-1, D)
  cpu.apply_gradients({"t": (u, ug)}, req_time=1)
  got = -gpu_lookup(gpu, {"t": u}, dev)["t"].astype(np.float64)
  seq = -cpu.lookup({"t": u})["t"].astype(np.float64)
  exact = np.stack([pg[fids == k].astype(np.float64).sum(0) for k in u])
  scale = np.abs(pg.astype(np.float64)).sum(0).max()        # sum of |terms|: the natural error scale of a sum
  err_gpu, err_seq = np.abs(got - exact).max(), np.abs(seq - exact).max()
  assert err_gpu <= 1e-5 * np.abs(exact).max(), (err_gpu, np.abs(exact).max())
  assert err_gpu <= 5e-7 * scale
  assert err_gpu <= err_seq + 1e-12, (err_gpu, err_seq)


# ------------------------------------------------------------------------------------------------
# TMA-staged lookup (bulk row copies global -> shared -> global) == the register-path kernel == the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [16, 32, 64])
@pytest.mark.parametrize("n", [1, 31, 32, 33, 5000, 70001])
def test_lookup_tma_vs_register_path_and_oracle(dim, n, dev):
  import ctypes as C
  from monolith_b200 import _lib, entry
  lib = _lib.load()
  rng = np.random.default_rng(dim * 1000 + n)
  cfg = {"t": table([(dim, "sgd", {})], [0.1], capacity=64, init=entry.RandomUniformInitializer(-1.0, 1.0), init_seed=3)}
  gpu, cpu = pair(cfg, dev)
  vocab = np.unique(rand_fids(rng, 3000, 100000))
  vals = rng.standard_normal((vocab.size, dim)).astype(np.float32)
  gpu.assign({"t": (T(vocab, dev), T(vals, dev))})
  cpu.assign({"t": (vocab, vals)})
  ids = rng.choice(np.concatenate([vocab, vocab[:200] + 7]), size=n)          # ~6 % absent -> zero rows
  want = cpu.lookup({"t": ids})["t"]
  old = lib.mono_get_option(b"lookup_tma")
  try:
    outs = []
    for mode in (0, 1):
      assert lib.mono_set_option(b"lookup_tma", mode) == 0
      outs.append(gpu.lookup({"t": T(ids, dev)})["t"].cpu().numpy())
      pooled = gpu.lookup_pool("t", T(ids, dev), None, "sum").cpu().numpy()
      np.testing.assert_array_equal(pooled.view(np.uint32), want.view(np.uint32))
    np.testing.assert_array_equal(outs[0].view(np.uint32), want.view(np.uint32))
    np.testing.assert_array_equal(outs[1].view(np.uint32), want.view(np.uint32))
  finally:
    lib.mono_set_option(b"lookup_tma", old)
  assert lib.mono_set_option(b"no_such_option", 1) != 0


# ------------------------------------------------------------------------------------------------
# counting admission filter on the GPU (SURVEY §8(f) row 2) vs the oracle's HashFilter restatement
# ------------------------------------------------------------------------------------------------
def test_hash_filter_threshold_schedule_golden_cuda(dev):
  """The reference's test_gradients_with_hash_filter (NT/hash_table_ops_test.py:223-260) through the CUDA path: dim 1,
  SGD lr 0.1, occurrence_threshold 3, ids [0, 0, 1] with gradient -1 applied four times."""
  from monolith_b200 import MultiHashTable
  t = MultiHashTable({"t": sgd_table(1, 0.1)}, device=dev)
  t.set_hash_filter("t", capacity=1000, default_threshold=3)
  ids = T(np.array([0, 0, 1], np.int64), dev)
  g = T(-np.ones((3, 1), np.float32), dev)
  for want in ([[0.0], [0.0]], [[0.1], [0.0]], [[0.3], [0.0]], [[0.5], [0.1]]):
    t.apply_gradients({"t": (ids, g)})
    np.testing.assert_allclose(gpu_lookup(t, {"t": [0, 1]}, dev)["t"], want, rtol=1e-6, atol=1e-7)


def test_hash_filter_paths_vs_oracle(dev):
  """Per-slot thresholds, the dedup path (occurrence counts), assign (absent ids only), assign_add (every id, present or
  not: AssignAdd2 has no Contains check), the fused backward (one count per distinct FID and step) and threshold 0."""
  D = 4
  cfg = {"t": table([(D, "adagrad", {})], [0.1])}
  rng = np.random.default_rng(9)
  f = lambda slot, x: (np.int64(slot) << 48) | np.asarray(x, np.int64)

  def both():
    gpu, cpu = pair(cfg, dev)
    for t in (gpu, cpu):
      # a large filter: two FIDs with the same 12-bit signature and overlapping probe windows share a counter, and WHICH
      # ones do depends on the insertion order (sequential in the oracle, concurrent on the GPU) — unpinned in the
      # reference too (absl::Hash is salted per process); 3 M cells make that improbable for a few hundred FIDs
      t.set_hash_filter("t", capacity=2_000_000, default_threshold=2, slot_thresholds={7: 4, 9: 0})
    return gpu, cpu

  def same(gpu, cpu, ids):
    assert gpu.size("t") == cpu.size("t")
    got, want = gpu.lookup_entry("t", T(ids, dev))["raw"].cpu().numpy(), cpu.lookup_entry("t", ids)
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))

  # (1) optimize, unique ids per step, three slots with thresholds 2 (default), 4 and 0
  gpu, cpu = both()
  ids = np.concatenate([f(3, np.arange(200)), f(7, np.arange(200)), f(9, np.arange(50))])
  for step in range(6):
    sel = ids[rng.random(ids.size) < 0.7]
    g = rng.standard_normal((sel.size, D)).astype(np.float32)
    gpu.apply_gradients({"t": (T(sel, dev), T(g, dev))}, req_time=step, ids_unique=True)
    cpu.apply_gradients({"t": (sel, g)}, req_time=step)
    same(gpu, cpu, ids)
  # (2) dedup path: the filter is handed each id's occurrence count
  gpu, cpu = both()
  for step in range(3):
    sel = rng.choice(f(3, np.arange(60)), 400)
    g = rng.standard_normal((sel.size, D)).astype(np.float32)
    gpu.apply_gradients({"t": (T(sel, dev), T(g, dev))}, req_time=step, enable_dedup=True)
    cpu.apply_gradients({"t": (sel, g)}, req_time=step, enable_dedup=True)
    u = np.unique(sel)
    assert gpu.size("t") == cpu.size("t")
    np.testing.assert_allclose(gpu_lookup(gpu, {"t": u}, dev)["t"], cpu.lookup({"t": u})["t"], rtol=1e-5, atol=1e-6)
  # (3) duplicates without dedup: occurrence q of an absent id sees count c0 + q (sequential semantics)
  gpu, cpu = both()
  for step in range(4):
    sel = rng.choice(f(7, np.arange(30)), 100)
    g = rng.standard_normal((sel.size, D)).astype(np.float32)
    gpu.apply_gradients({"t": (T(sel, dev), T(g, dev))}, req_time=step)
    cpu.apply_gradients({"t": (sel, g)}, req_time=step)
    same(gpu, cpu, f(7, np.arange(30)))
  # (4) assign: absent ids consult the filter; assign_add: every id does
  gpu, cpu = both()
  ids4 = f(3, np.arange(40))
  for step in range(4):
    v = rng.standard_normal((ids4.size, D)).astype(np.float32)
    gpu.assign({"t": (T(ids4, dev), T(v, dev))}, req_time=step, ids_unique=True)
    cpu.assign({"t": (ids4, v)}, req_time=step)
    same(gpu, cpu, ids4)
  gpu, cpu = both()
  ids5 = f(7, np.arange(40))
  for step in range(7):
    v = rng.standard_normal((ids5.size, D)).astype(np.float32)
    gpu.assign_add({"t": (T(ids5, dev), T(v, dev))}, req_time=step, ids_unique=True)
    cpu.assign_add({"t": (ids5, v)}, req_time=step)
    same(gpu, cpu, ids5)
  # (5) fused backward: every distinct FID of the batch counts once per step
  gpu, cpu = both()
  vocab = np.concatenate([f(3, np.arange(300)), f(7, np.arange(100))])
  for step in range(6):
    fids = rng.choice(vocab, 2000)
    pg = rng.standard_normal((fids.size, D)).astype(np.float32)
    gpu.pool_backward("t", T(fids, dev), T(pg, dev), None, "sum", req_time=step)
    u, inv = orc.dedup(fids)
    ug = orc.gather_pool_grad(pg, inv * D, D, u.size * D).reshape(-1, D)
    cpu.apply_gradients({"t": (u, ug)}, req_time=step)
    same(gpu, cpu, vocab)


# ------------------------------------------------------------------------------------------------
# device-driven sharded step (csrc/xstep.cu) with world = 1: the whole flag / header / window protocol against itself
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["one_fid_per_row", "csr_mean"])
def test_sharded_direct_step_world1_vs_oracle(mode, dev):
  from monolith_b200 import MultiHashTable
  from monolith_b200.distributed_ps import ShardedStep
  D = 16
  cfg = {"t": table([(D, "adagrad", {})], [0.1])}
  gpu, cpu = pair(cfg, dev)
  st = ShardedStep(gpu, "t", D, 1, 0, dev, exchange="direct")
  rng = np.random.default_rng(31)
  hot = fid(5, 3)
  batches = []
  for step in range(5):
    n = 6000 + (500 * step if step < 3 else 1000)                # growing batches: the window is re-created once or twice
    ids = rng.integers(0, 900 + 50 * step, n)
    ids[rng.random(n) < 0.25] = 3                                # hot FID: a > 64-occurrence run (tree-reduced)
    fids = (np.int64(5) << 48) | ids.astype(np.int64)
    if mode == "csr_mean":
      lens = rng.integers(0, 5, n)
      ro = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
      ro = ro[ro <= n]
      ro[-1] = n
      R, pool = ro.size - 1, "mean"
    else:
      ro, R, pool = None, n, "sum"
    batches.append((fids, ro, R, pool, rng.standard_normal((R, D)).astype(np.float32), T(fids, dev)))
  try:
    for step, (fids, ro, R, pool, g, f_dev) in enumerate(batches):
      out = torch.empty(R, D, device=dev)
      st.step(f_dev, T(g, dev), out, 20 + step, None if ro is None else T(ro, dev), pool)
      if step + 1 < len(batches):
        st.prepare(batches[step + 1][5])                           # next batch's grouping on a side stream (same tensor object)
      want = cpu.lookup_pool("t", fids, ro, pool)
      got = out.cpu().numpy()
      if ro is None:
        cold = fids != hot
        np.testing.assert_array_equal(got[cold].view(np.uint32), want[cold].view(np.uint32))
        np.testing.assert_allclose(got[~cold], want[~cold], rtol=2e-3, atol=2e-3)
      else:
        np.testing.assert_allclose(got, want, rtol=2e-3, atol=2e-3)
      u, inv = orc.dedup(fids)
      ug = orc.gather_pool_grad(g, inv * D, D, u.size * D, ro, pool).reshape(-1, D)
      cpu.apply_gradients({"t": (u, ug)}, req_time=20 + step)
    keys = cpu.keys("t")
    assert gpu.size("t") == keys.size
    got = gpu.lookup_entry("t", T(keys, dev))["raw"].cpu().numpy()
    want = cpu.lookup_entry("t", keys)
    cold = keys != hot
    if mode == "one_fid_per_row":
      np.testing.assert_array_equal(got[cold].view(np.uint32), want[cold].view(np.uint32))
    else:
      np.testing.assert_allclose(got[cold][:, :-2], want[cold][:, :-2], rtol=2e-5, atol=1e-6)
    np.testing.assert_allclose(got[~cold][:, :-2], want[~cold][:, :-2], rtol=2e-3, atol=2e-3)
    np.testing.assert_array_equal(got[:, -2:].view(np.uint32), want[:, -2:].view(np.uint32))
  finally:
    st.close_direct()


# ------------------------------------------------------------------------------------------------
# the bench's batch shape (M = 2 097 152 occurrences, Zipf, dim 32, Adagrad) against the oracle
# ------------------------------------------------------------------------------------------------
def test_bench_shape_step_vs_oracle(dev):
  """One full sparse step at the benchmark's batch shape (C2: 1 048 576 samples x 2 slots, Zipf(1.05) ranks, dim 32,
  Adagrad) over a 1 M-key vocabulary: pooled rows bit for bit; after the fused backward every entry whose FID occurs
  <= 64 times bit for bit (reference summation order), the hot FIDs within 1e-5 of the row's scale (tree vs sequential
  fp32 sums; see the fp64 test above)."""
  import bench
  D = 32
  from monolith_b200 import entry
  cfg = {"t": table([(D, "adagrad", {"initial_accumulator_value": 0.1})], [0.05], capacity=1 << 20,
                    init=entry.RandomUniformInitializer(-0.05, 0.05), init_seed=1)}
  gpu, cpu = pair(cfg, dev)
  fids = bench.make_batches(1, 1 << 20, 500_000, seed=11)[0]
  M = fids.size
  rng = np.random.default_rng(3)
  vocab = np.unique(fids)
  pre = vocab[rng.random(vocab.size) < 0.9]                       # 10 % of the FIDs are new in this step (upserts)
  z = np.zeros((pre.size, D), np.float32)
  gpu.assign_add({"t": (T(pre, dev), T(z, dev))}, req_time=1, ids_unique=True)
  cpu.assign_add({"t": (pre, z)}, req_time=1)
  pooled = gpu.lookup_pool("t", T(fids, dev), None, "sum").cpu().numpy()
  np.testing.assert_array_equal(pooled.view(np.uint32), cpu.lookup_pool("t", fids, None, "sum").view(np.uint32))
  pg = rng.standard_normal((M, D)).astype(np.float32)
  gpu.pool_backward("t", T(fids, dev), T(pg, dev), None, "sum", req_time=7)
  u, inv = orc.dedup(fids)
  ug = orc.gather_pool_grad(pg, inv * D, D, u.size * D).reshape(-1, D)
  cpu.apply_gradients({"t": (u, ug)}, req_time=7)
  assert gpu.size("t") == cpu.size("t") == vocab.size
  got = gpu.lookup_entry("t", T(vocab, dev))["raw"].cpu().numpy()
  want = cpu.lookup_entry("t", vocab)
  cnt = np.bincount(np.searchsorted(vocab, fids), minlength=vocab.size)
  cold = cnt <= 64
  assert cold.sum() > 0.95 * vocab.size and (~cold).sum() > 100
  np.testing.assert_array_equal(got[cold].view(np.uint32), want[cold].view(np.uint32))
  np.testing.assert_array_equal(got[~cold][:, -2:].view(np.uint32), want[~cold][:, -2:].view(np.uint32))
  scale = np.abs(want[~cold][:, :-2]).max(axis=1, keepdims=True) + 1e-3
  assert float((np.abs(got[~cold][:, :-2] - want[~cold][:, :-2]) / scale).max()) < 2e-3


def test_bench_dump_outputs_follow_the_step_count(tmp_path):
  """bench.py --dump-outputs writes the last timed step's outputs as float32 arrays.  With one timed region the bench
  runs warmup + steps steps over 4 rotating batches: warmup 2 + 1 step dumps bit for bit what warmup 1 + 2 steps dumps
  (another process, same inputs), and warmup 1 + 6 steps ends on the same batch after four more Adagrad updates."""
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

  def run(name, steps, warmup):
    out = tmp_path / name
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--keys", "200000", "--batch", "8192",
                        "--steps", str(steps), "--warmup", str(warmup), "--repeats", "1", "--no-parity", "--no-e2e",
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    return {k: np.load(out / f"{k}.npy") for k in ("pooled", "embeddings", "adagrad_accumulators")}

  a, b, c = run("a", 2, 1), run("b", 1, 2), run("c", 6, 1)
  assert a["pooled"].shape == (8192 * 2, 32) and a["embeddings"].shape == a["adagrad_accumulators"].shape
  assert all(v.dtype == np.float32 for v in a.values()) and a["embeddings"].shape[0] > 1000
  for k in a:
    np.testing.assert_array_equal(a[k].view(np.uint32), b[k].view(np.uint32))
  assert (c["adagrad_accumulators"] >= a["adagrad_accumulators"]).all()
  assert (c["adagrad_accumulators"] > a["adagrad_accumulators"]).any()


def test_two_host_threads_share_one_handle(dev):
  """Two host threads drive ONE table handle concurrently (lookups against updates of disjoint FID sets, each on its
  own stream): the per-handle lock of the C ABI serialises them; results equal the sequential ones (ref: TF runs the
  ops of one resource from several inter-op threads)."""
  import threading
  D = 16
  cfg = {"t": table([(D, "adagrad", {})], [0.1])}
  gpu, cpu = pair(cfg, dev)
  rng = np.random.default_rng(5)
  a_ids, b_ids = fid(1, np.arange(20000)), fid(2, np.arange(20000))
  va = rng.standard_normal((a_ids.size, D)).astype(np.float32)
  gpu.assign({"t": (T(a_ids, dev), T(va, dev))}, ids_unique=True)
  cpu.assign({"t": (a_ids, va)})
  torch.cuda.synchronize()
  errs, looked = [], []
  grads = [rng.standard_normal((b_ids.size, D)).astype(np.float32) for _ in range(6)]

  def reader():
    try:
      with torch.cuda.stream(torch.cuda.Stream(device=dev)):
        for _ in range(30):
          looked.append(gpu.lookup({"t": T(a_ids, dev)})["t"].cpu().numpy())
    except Exception as e:  # pragma: no cover
      errs.append(e)

  def writer():
    try:
      with torch.cuda.stream(torch.cuda.Stream(device=dev)):
        for k, g in enumerate(grads):
          gpu.apply_gradients({"t": (T(b_ids, dev), T(g, dev))}, req_time=10 + k, ids_unique=True)
        torch.cuda.current_stream().synchronize()
    except Exception as e:  # pragma: no cover
      errs.append(e)

  ts = [threading.Thread(target=reader), threading.Thread(target=writer)]
  for t in ts:
    t.start()
  for t in ts:
    t.join()
  assert not errs, errs
  for k, g in enumerate(grads):
    cpu.apply_gradients({"t": (b_ids, g)}, req_time=10 + k)
  for x in looked:                                               # rows of set A never change: every lookup saw them all
    np.testing.assert_array_equal(x.view(np.uint32), va.view(np.uint32))
  both = np.concatenate([a_ids, b_ids])
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": both}, dev)["t"].view(np.uint32), cpu.lookup({"t": both})["t"].view(np.uint32))


# ------------------------------------------------------------------------------------------------
# the e2e bench's stand-in dense tower: the fused kernel (csrc/tower.cu) against torch.autograd
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch", [16, 5000, 65536 + 7])
def test_bench_tower_fused_vs_autograd(dev, batch):
  """floating point, bf16 operands: loss within 1e-3 relative, input gradient within 2 % in relative L2 norm (the two
  sides round to bf16 at the same points but accumulate in different orders, so a ReLU mask can flip on a unit whose
  pre-activation is ~0)."""
  import bench
  from monolith_b200 import _lib
  lib = _lib.load()
  torch.manual_seed(batch)
  fused = bench.Tower(dev, batch, seed=3, lib=lib)
  ref = bench.Tower(dev, batch, seed=3)
  pooled = torch.randn(batch * bench.SLOTS, bench.DIM, device=dev)
  labels = (torch.rand(batch, device=dev) < 0.3).float()
  g = torch.full((batch * bench.SLOTS, bench.DIM), 7.0, device=dev)
  loss = fused.grad(pooled, labels, g).clone()
  loss_ref, gx = ref.grad_autograd(pooled, labels)
  torch.cuda.synchronize()
  assert abs(float(loss) - float(loss_ref)) <= 1e-3 * abs(float(loss_ref))
  got = g.view(batch, bench.SLOTS * bench.DIM).double()
  want = gx.double()
  rel = float((got - want).norm() / want.norm())
  assert rel < 2e-2, rel
  # the torch formulation with the hand-written backward agrees with autograd too
  g2 = torch.empty_like(g)
  loss2 = ref.grad_torch(pooled, labels, g2)
  assert abs(float(loss2) - float(loss_ref)) <= 1e-3 * abs(float(loss_ref))
  assert float((g2.view(batch, -1).double() - want).norm() / want.norm()) < 2e-2


def test_lookup_never_misses_during_inserts_on_another_stream(dev):
  """Readers vs. structural change: one host thread looks up a resident FID set on its own stream while another thread
  INSERTS new FIDs (which displaces resident entries between their two buckets) on a second stream.  Every lookup must
  see every resident row: the cuckoo displacement copies a victim into its alternate bucket BEFORE its old slot is
  overwritten (csrc/common.cuh cuckoo_insert; the reference gives readers the same guarantee with bucket locks,
  cuckoohash_map.hpp find / uprase under lock).  Capacity is preallocated so that the table does not grow (growth
  swaps the bucket array and is stream-ordered by contract)."""
  import threading
  D = 8
  n_a, n_b = 300_000, 420_000
  cfg = {"t": sgd_table(D, capacity=n_a + n_b)}
  gpu, cpu = pair(cfg, dev)
  rng = np.random.default_rng(9)
  a_ids, b_ids = fid(1, np.arange(n_a)), fid(2, np.arange(n_b))
  va = rng.standard_normal((n_a, D)).astype(np.float32)
  vb = rng.standard_normal((n_b, D)).astype(np.float32)
  gpu.assign({"t": (T(a_ids, dev), T(va, dev))}, ids_unique=True)
  torch.cuda.synchronize()
  a_dev = T(a_ids, dev)
  va_dev = T(va, dev)
  errs, bad = [], []
  stop = threading.Event()

  def reader():
    try:
      with torch.cuda.stream(torch.cuda.Stream(device=dev)):
        n = 0
        while not stop.is_set() or n < 5:
          got = gpu.lookup({"t": a_dev})["t"]
          bad.append(int((got != va_dev).any(dim=1).sum().item()))
          n += 1
    except Exception as e:  # pragma: no cover
      errs.append(e)

  def writer():
    try:
      with torch.cuda.stream(torch.cuda.Stream(device=dev)):
        for lo in range(0, n_b, 20_000):
          sl = slice(lo, lo + 20_000)
          gpu.assign({"t": (T(b_ids[sl], dev), T(vb[sl], dev))}, ids_unique=True)
        torch.cuda.current_stream().synchronize()
    except Exception as e:  # pragma: no cover
      errs.append(e)
    finally:
      stop.set()

  ts = [threading.Thread(target=reader), threading.Thread(target=writer)]
  for t in ts:
    t.start()
  for t in ts:
    t.join()
  assert not errs, errs
  assert len(bad) >= 5 and sum(bad) == 0, (len(bad), sum(bad), max(bad))
  cpu.assign({"t": (a_ids, va)})
  cpu.assign({"t": (b_ids, vb)})
  both = np.concatenate([a_ids, b_ids])
  np.testing.assert_array_equal(gpu_lookup(gpu, {"t": both}, dev)["t"].view(np.uint32), cpu.lookup({"t": both})["t"].view(np.uint32))
  assert gpu.size("t") == n_a + n_b


def test_streaming_insert_evict_50_steps_vs_oracle(dev):
  """The C4 stream in miniature (bench.py --workload c4): 50 steps of fused lookup+pool / fused backward on a table that is
  small enough to GROW under load (capacity 1024 against ~30 K keys), every step 5 % never-seen FIDs, a TTL eviction scan
  every 8 steps (one-day window, ref: CuckooEmbeddingHashTable::Evict via the bridge's eviction thread,
  embedding_hash_table_tf_bridge.cc:73-104).  After every eviction and at the end: membership, rows, optimizer state and
  timestamps equal the oracle's — bit for bit for every FID that never had more than 64 occurrences in a step (freed rows
  are reused, the bucket array is rehashed several times), within the tree-sum tolerance for the hot ones."""
  from monolith_b200 import entry
  rng = np.random.default_rng(50)
  D, M = 8, 4200
  DAY, dt = 86400, 86400 // 20                       # the window is 20 steps
  cfg = {"t": table([(D, "adagrad", {"initial_accumulator_value": 0.1})], [0.05], capacity=1024, default_expire_time=1,
                    init=entry.RandomUniformInitializer(-0.05, 0.05), init_seed=4)}
  gpu, cpu = pair(cfg, dev)
  resident = 20_000
  base = fid(1, np.arange(resident))
  for c in range(20):                                 # prefill with last-update times spread over the window
    sl = slice(c * resident // 20, (c + 1) * resident // 20)
    z = np.zeros((base[sl].size, D), np.float32)
    gpu.assign_add({"t": (T(base[sl], dev), T(z, dev))}, req_time=c * dt, ids_unique=True)
    cpu.assign_add({"t": (base[sl], z)}, req_time=c * dt)
  fresh = resident
  hot_fids = set()
  for step in range(50):
    now = DAY + (step + 1) * dt
    ranks = np.minimum((rng.pareto(1.05, M) * 50).astype(np.int64), resident - 1)
    ids = fid(1, ranks)
    n_new = M // 20
    pos = rng.choice(M, n_new, replace=False)
    ids[pos] = fid(1, fresh + np.arange(n_new))
    fresh += n_new
    u, inv = orc.dedup(ids)
    cnt = np.bincount(inv, minlength=u.size)
    hot_fids.update(u[cnt > 64].tolist())
    cold = ~np.isin(ids, np.fromiter(hot_fids, np.int64, len(hot_fids)))
    pooled = gpu.lookup_pool("t", T(ids, dev), None, "sum").cpu().numpy()
    np.testing.assert_array_equal(pooled[cold].view(np.uint32), cpu.lookup({"t": ids})["t"][cold].view(np.uint32))
    g = rng.standard_normal((M, D)).astype(np.float32)
    gpu.pool_backward("t", T(ids, dev), T(g, dev), None, "sum", req_time=now)
    ug = orc.gather_pool_grad(g, inv * D, D, u.size * D).reshape(-1, D)
    cpu.apply_gradients({"t": (u, ug)}, req_time=now)
    if (step + 1) % 8 == 0:
      gpu.evict("t", now)
      cpu.evict("t", now)
      assert gpu.size("t") == cpu.size("t")
  keys = cpu.keys("t")
  assert gpu.size("t") == keys.size and 5_000 < keys.size < 15_000       # steady state: the window holds ~8 K live keys
  probe = np.concatenate([keys, base])                             # live keys + every prefilled key (many evicted)
  np.testing.assert_array_equal(gpu.contains("t", T(probe, dev)).cpu().numpy(), cpu.contains("t", probe))
  eg = gpu.lookup_entry("t", T(keys, dev))["raw"].cpu().numpy()
  ec = cpu.lookup_entry("t", keys)
  hot = np.isin(keys, np.fromiter(hot_fids, np.int64, len(hot_fids)))
  assert 0 < hot.sum() < 200
  np.testing.assert_array_equal(eg[~hot].view(np.uint32), ec[~hot].view(np.uint32))
  np.testing.assert_allclose(eg[hot][:, :-2], ec[hot][:, :-2], rtol=2e-3, atol=2e-4)
  np.testing.assert_array_equal(eg[hot][:, -2:].view(np.uint32), ec[hot][:, -2:].view(np.uint32))
