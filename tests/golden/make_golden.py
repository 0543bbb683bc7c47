"""Generates the committed golden fixtures for the oracle tests.

Two kinds of vectors:
 1. TRANSCRIBED: known-answer tests copied by hand from the reference's own test files
    (bytedance/monolith @ 135c491; paths relative to monolith/native_training/).  TensorFlow/bazel
    are not available, so the reference tests cannot be executed; each case cites file:line.
    -> tests/golden/reference_known_answers.json
 2. GENERATED from the REAL reference code: the two header-only pieces that compile here
    (oracle/_ref/libmonoref.so, built by oracle/Makefile from /root/reference in place):
    runtime/hash_table/optimizer/avx_utils.h (Adagrad) and
    data/kernels/internal/uniq_hashtable.h (first-occurrence dedup ordinals).
    -> tests/golden/ref_adagrad.npz, tests/golden/ref_adagrad_avx_lanes.npz, tests/golden/ref_uniq_fid.npz

Run from the repo root in the build container (needs /root/reference):
    make -C oracle && python tests/golden/make_golden.py
"""
import ctypes as C
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

KNOWN = {
    "optimizers": [
        # runtime/hash_table/optimizer/adagrad_optimizer_test.cc:32-42
        {"name": "adagrad_basic", "opt": "adagrad", "dim": 2, "params": {"initial_accumulator_value": 1.0},
         "steps": [{"grad": [1.0, 2.0], "lr": [0.1], "expect": [-0.07071067, -0.08944272]}], "tol": 1e-6},
        # adagrad_optimizer_test.cc:56-72
        {"name": "adagrad_weight_decay", "opt": "adagrad", "dim": 2,
         "params": {"initial_accumulator_value": 1.0, "weight_decay_factor": 0.1},
         "steps": [{"grad": [1.0, 2.0], "lr": [0.1], "expect": [-0.07071067, -0.08944272]},
                   {"grad": [1.0, 2.0], "lr": [0.1], "expect": [-0.128173, -0.155943]}], "tol": 1e-6},
        # ftrl_optimizer_test.cc:32-51 (proto defaults: beta 0, init_acc 0.1, l1 0, l2 0)
        {"name": "ftrl_basic", "opt": "ftrl", "dim": 1, "params": {},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [-0.009995]},
                   {"grad": [10.0], "lr": [0.01], "expect": [-0.0170643]}], "tol": 1e-6},
        # ftrl_optimizer_test.cc:53-73
        {"name": "ftrl_list", "opt": "ftrl", "dim": 2, "params": {},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.009995, -0.00953463]},
                   {"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.0170643, -0.0164353]}], "tol": 1e-6},
        # adam_optimizer_test.cc:32-51 (proto defaults: beta1 .9, beta2 .99, eps .01)
        {"name": "adam_basic", "opt": "adam", "dim": 1, "params": {},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [-0.00990099]},
                   {"grad": [10.0], "lr": [0.01], "expect": [-0.01983060]}], "tol": 1e-6},
        # adam_optimizer_test.cc:53-73
        {"name": "adam_list", "opt": "adam", "dim": 2, "params": {},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.00990099, -0.00909091]},
                   {"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.01983060, -0.01842895]}], "tol": 1e-6},
        # sgd_optimizer_test.cc:32-41
        {"name": "sgd_basic", "opt": "sgd", "dim": 1, "params": {},
         "steps": [{"grad": [1.0], "lr": [0.1], "expect": [-0.1]}], "tol": 1e-6},
        # momentum_optimizer_test.cc:32-49,51-72 (proto defaults: momentum .9, no nesterov, wd 0)
        {"name": "momentum_basic", "opt": "momentum", "dim": 1, "params": {},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [-0.1]},
                   {"grad": [10.0], "lr": [0.01], "expect": [-0.29]}], "tol": 1e-6},
        {"name": "momentum_list", "opt": "momentum", "dim": 2, "params": {},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.1, -0.01]},
                   {"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.29, -0.029]}], "tol": 1e-6},
        # rmsprop_optimizer_test.cc:32-49 (v1: the CONFIG's learning rate .01, momentum .9) and :51-72 (v2)
        {"name": "rmsprop_basic", "opt": "rmsprop", "dim": 1, "params": {"learning_rate": 0.01},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [-0.024025]},
                   {"grad": [10.0], "lr": [0.01], "expect": [-0.042686]}], "tol": 1e-6},
        {"name": "rmspropv2_list", "opt": "rmspropv2", "dim": 2, "params": {},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.0090909, -0.005]},
                   {"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.0158549, -0.0092045]}], "tol": 1e-6},
        # adadelta_optimizer_test.cc:32-51 (proto defaults: averaging_ratio .9, epsilon .01)
        {"name": "adadelta_basic", "opt": "adadelta", "dim": 1, "params": {},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [-0.0031607]},
                   {"grad": [10.0], "lr": [0.01], "expect": [-0.0064035]}], "tol": 1e-6},
        # amsgrad_optimizer_test.cc:32-51,53-73 (proto defaults as Adam)
        {"name": "amsgrad_basic", "opt": "amsgrad", "dim": 1, "params": {},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [-0.00990099]},
                   {"grad": [10.0], "lr": [0.01], "expect": [-0.01983060]}], "tol": 1e-6},
        {"name": "amsgrad_list", "opt": "amsgrad", "dim": 2, "params": {},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.00990099, -0.00909091]},
                   {"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.01983060, -0.01842895]}], "tol": 1e-6},
        # moving_average_optimizer_test.cc:32-49,51-74 (proto default momentum .9; the learning rate is ignored)
        {"name": "moving_average_basic", "opt": "moving_average", "dim": 1, "params": {},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [1.0]},
                   {"grad": [10.0], "lr": [0.01], "expect": [1.9]}], "tol": 1e-6},
        {"name": "moving_average_list", "opt": "moving_average", "dim": 2, "params": {},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [1.0, 0.1]},
                   {"grad": [10.0, 1.0], "lr": [0.01], "expect": [1.9, 0.19]}], "tol": 1e-6},
        # group_adagrad_optimizer_test.cc:32-54 (Basic), :56-80 (ListUpdate), :82-96 (ZeroLambda), :98-112 (SetZero)
        {"name": "group_adagrad_basic", "opt": "group_adagrad", "dim": 1,
         "params": {"l2": 1.0, "beta": 1.0, "initial_accumulator_value": 0.0},
         "steps": [{"grad": [10.0], "lr": [0.01], "expect": [-0.008182]},
                   {"grad": [10.0], "lr": [0.01], "expect": [-0.014125]}], "tol": 1e-6},
        {"name": "group_adagrad_list", "opt": "group_adagrad", "dim": 2,
         "params": {"l2": 0.5, "beta": 1.0, "initial_accumulator_value": 0.0},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.008639, -0.000864]},
                   {"grad": [1.0, 5.0], "lr": [0.01], "expect": [-0.009096, -0.004778]}], "tol": 1e-6},
        {"name": "group_adagrad_zero_lambda", "opt": "group_adagrad", "dim": 2,
         "params": {"l2": 0.0, "beta": 1.0, "initial_accumulator_value": 0.0},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [-0.009091, -0.000909]}], "tol": 1e-6},
        {"name": "group_adagrad_set_zero", "opt": "group_adagrad", "dim": 2,
         "params": {"l2": 1000.0, "beta": 1.0, "initial_accumulator_value": 0.0},
         "steps": [{"grad": [10.0, 1.0], "lr": [0.01], "expect": [0.0, 0.0]}], "tol": 1e-6},
    ],
    # optimizer_combination_test.cc:30-60: adagrad(dim 1, acc 1) | adagrad(dim 2, acc 2), lrs {1, 2}
    "combination": {
        "segments": [{"dim": 1, "opt": "adagrad", "params": {"initial_accumulator_value": 1.0}},
                     {"dim": 2, "opt": "adagrad", "params": {"initial_accumulator_value": 2.0}}],
        "grad": [1.0, 2.0, 3.0], "lr": [1.0, 2.0],
        "expect_step1": [-0.70710677, -1.6329931, -1.8090681],
        # second Optimize on the restored state continues from step 1 (the test restores the dump into
        # a fresh entry whose num is zero again):
        "expect_step2_from_zero_num": [-0.57735026, -1.264911, -1.3416407], "tol": 1e-6},
    # distribution_ops_fused_test.py:59-127 (+ docstring distribution_ops.py:235-243)
    "fused_reorder_by_indices": [
        {"ids": [[0, 1, 2, 2, 3, 5]], "N": 3, "output": [0, 3, 1, 2, 5], "shard_sizes": [2, 1, 2],
         "sharded_slot_sizes": [2, 1, 2]},
        {"ids": [[0, 1, 2, 2, 3, 5], []], "N": 3, "output": [0, 3, 1, 2, 5], "shard_sizes": [2, 1, 2],
         "sharded_slot_sizes": [2, 0, 1, 0, 2, 0]},
        {"ids": [[0, 1, 2, 2, 3, 5], [6, 7, 8, 8, 9, 11]], "N": 3,
         "output": [0, 3, 6, 9, 1, 7, 2, 5, 8, 11], "shard_sizes": [4, 2, 4],
         "sharded_slot_sizes": [2, 2, 1, 1, 2, 2]},
        {"ids": [[], []], "N": 2, "output": [], "shard_sizes": [0, 0], "sharded_slot_sizes": [0, 0, 0, 0]},
        {"ids": [[0, 1, 4, 5], [2, 3, 6, 7]], "N": 2, "output": [0, 4, 2, 6, 1, 5, 3, 7],
         "shard_sizes": [4, 4], "sharded_slot_sizes": [2, 2, 2, 2]},
        {"ids": [[0, 1, 0], [3, 2, 3], [5, 6, 7]], "N": 2, "dims": [1, 2, 3],
         "output": [0, 2, 6, 1, 3, 5, 7], "shard_sizes": [3, 4], "sharded_slot_sizes": [1, 1, 1, 1, 1, 2],
         "offsets": [0, 6, 0, 7, 1, 7, 9, 3, 12]},
        {"ids": [[2, 3, 1, 2, 7, 2], [5, 8, 4, 4, 5, 11, 6]], "N": 3, "dims": [3, 2],
         "output": [3, 6, 1, 7, 4, 2, 5, 8, 11], "shard_sizes": [2, 3, 4],
         "sharded_slot_sizes": [1, 1, 2, 1, 1, 3],
         "offsets": [13, 0, 5, 13, 8, 13, 16, 18, 11, 11, 16, 20, 3]},
    ],
    # hash_table_ops_test.py:1086-1108 test_fused_lookup: three SGD/zeros tables dims [1,1,2];
    # table x assigned ids {3x, 3x+1} = ones (x even) / zeros (x odd)
    "fused_lookup": {
        "dims": [1, 1, 2],
        "assign": [{"ids": [0, 1], "value": 1.0}, {"ids": [3, 4], "value": 0.0}, {"ids": [6, 7], "value": 1.0}],
        "ids": [0, 4, 6, 1, 3, 7], "fused_slot_size": [1, 1, 1, 1, 1, 1], "N": 2,
        "embeddings": [1, 0, 1, 1, 1, 0, 1, 1], "recv_splits": [4, 4],
        "id_offsets": [0, 1, 2, 3, 4, 5, 6], "emb_offsets": [0, 1, 2, 4, 5, 6, 8]},
    # hash_table_ops_test.py:1110-1150 test_fused_optimize: SGD tables dims [1,2], lr 0.1 each
    "fused_optimize": {
        "dims": [1, 2], "lr": [0.1, 0.1],
        "assign": [{"ids": [0, 1], "value": 1.0}, {"ids": [3, 4], "value": 0.0}],
        "ids": [0, 4, 1, 3], "fused_slot_size": [1, 1, 1, 1], "N": 2,
        "grads": [-1, -2, -2, -1, -2, -2],
        "embeddings_after": [1.1, 0.2, 0.2, 1.1, 0.2, 0.2], "recv_splits": [3, 3],
        "id_offsets": [0, 1, 2, 3, 4], "emb_offsets": [0, 1, 3, 4, 6]},
    # hash_table_ops_test.py:68-99 (vocab_hash_table = SGD, zeros init, lr 1.0)
    "basic": {
        "assign_add": {"ids": [0, 1], "lookup": [0, 1, 2], "expect": [[1], [1], [0]], "size": 2},
        "assign_overwrite": {"first": [[1], [1], [0]], "second": [[1], [5], [0]]}},
    # hash_table_ops_test.py:132-147 (dup ids applied sequentially), :183-203, :205-219
    "gradients": [
        {"name": "dup_ids", "dim": 1, "lr": 0.1, "ids": [0, 0, 1], "grads": [[-1], [-1], [-1]],
         "lookup": [0, 1], "expect": [[0.2], [0.1]], "dedup": False},
        {"name": "dedup", "dim": 10, "lr": 0.1, "ids": [0, 1, 0, 1, 0], "grads": "minus_ones",
         "lookup": [0, 1], "expect_scalar": [0.3, 0.2], "dedup": True},
        {"name": "different_ids", "dim": 1, "lr": 0.1, "ids": [1, 0, 1], "grads": [[-1], [-1], [-1]],
         "lookup": [0, 1], "expect": [[0.1], [0.2]], "dedup": False}],
    # runtime/hash_table/embedding_hash_table_test.h:41-94 (SingleThread; SGD lr 0.01, zeros init, dim 1)
    "single_thread": {
        "miss": {"id": 5, "expect": [0.0]},
        "assign_add": {"id": -10, "value": [2.5], "ts": 100, "expect": [2.5]},
        "optimize_fresh": {"id": 13, "grad": [1.0], "lr": 0.01, "expect": [-0.01]}},
    # embedding_hash_table_test.h:282-327 (OneTimeEvict): default TTL 14 d, slot1 5 d, slot2 6 d
    "evict": {
        "default_expire_days": 14, "slot_expire": {"0": 0, "1": 5, "2": 6}, "write_ts": 1234,
        "rows": [{"slot": 1, "sig": 123, "value": 2.0}, {"slot": 2, "sig": 234, "value": 5.0},
                 {"slot": 3, "sig": 456, "value": 7.0}],
        "evict_at": 1234 + 5 * 86400 + 60, "expect_after": [0.0, 5.0, 7.0]},
    # multi_hash_table_ops_test.py:52-140
    "multi_hash_table": {
        "reinitialize": {"known_status": [0, 1, 1], "unknown_status": [-1, -1, -1]},
        "apply_gradients_sgd": {"slot0": [[-2.0]], "slot1": [[-1.0, -3.0], [-2.0, -4.0]]}},
}


def main():
  with open(os.path.join(HERE, "reference_known_answers.json"), "w") as f:
    json.dump(KNOWN, f, indent=1, sort_keys=True)
  so = os.path.join(ROOT, "oracle", "_ref", "libmonoref.so")
  if not os.path.exists(so):
    raise SystemExit("oracle/_ref/libmonoref.so missing: run `make -C oracle` where /root/reference exists")
  ref = C.CDLL(so)
  rng = np.random.default_rng(20260922)
  cases = {}
  for ci, (dim, wd) in enumerate([(1, 0.0), (7, 0.0), (8, 0.0), (16, 0.0), (32, 0.0), (37, 0.0), (32, 0.1), (13, 0.05)]):
    num = (rng.standard_normal(dim) * 0.1).astype(np.float32)
    norm = np.full(dim, 0.1, np.float32)
    num0 = num.copy()
    seq_num, seq_norm, grads = [], [], []
    for step in range(4):
      g = (rng.standard_normal(dim) * (0.01 if step % 2 else 1.0)).astype(np.float32)
      ref.ref_adagrad(num.ctypes.data_as(C.c_void_p), norm.ctypes.data_as(C.c_void_p),
                      g.ctypes.data_as(C.c_void_p), C.c_int64(dim), C.c_float(0.05), C.c_float(wd))
      grads.append(g.copy()); seq_num.append(num.copy()); seq_norm.append(norm.copy())
    cases[f"c{ci}_dim"] = np.int64(dim)
    cases[f"c{ci}_wd"] = np.float32(wd)
    cases[f"c{ci}_num0"] = num0
    cases[f"c{ci}_grads"] = np.stack(grads)
    cases[f"c{ci}_num"] = np.stack(seq_num)
    cases[f"c{ci}_norm"] = np.stack(seq_norm)
  cases["n_cases"] = np.int64(8)
  np.savez(os.path.join(HERE, "ref_adagrad.npz"), **cases)

  # rows whose every lane takes the AVX path (dim % 8 == 0): the oracle must match these bit for bit over the whole row
  rng = np.random.default_rng(1)
  lr = np.float32(0.01)
  lanes = {"lr": lr}
  for ci, dim in enumerate((8, 24, 64)):
    num, norm = rng.standard_normal(dim).astype(np.float32), np.full(dim, 0.1, np.float32)
    lanes[f"c{ci}_num0"], lanes[f"c{ci}_norm0"] = num.copy(), norm.copy()
    seq_num, seq_norm, grads = [], [], []
    for step in range(5):
      g = rng.standard_normal(dim).astype(np.float32)
      ref.ref_adagrad(num.ctypes.data_as(C.c_void_p), norm.ctypes.data_as(C.c_void_p),
                      g.ctypes.data_as(C.c_void_p), C.c_int64(dim), C.c_float(lr), C.c_float(0.0))
      grads.append(g.copy()); seq_num.append(num.copy()); seq_norm.append(norm.copy())
    lanes[f"c{ci}_grads"] = np.stack(grads)
    lanes[f"c{ci}_num"] = np.stack(seq_num)
    lanes[f"c{ci}_norm"] = np.stack(seq_norm)
  lanes["n_cases"] = np.int64(3)
  np.savez(os.path.join(HERE, "ref_adagrad_avx_lanes.npz"), **lanes)

  # first-occurrence ordinals from the reference's MultiShardUniqHashTable
  u = {}
  rng = np.random.default_rng(7)
  for ci, (n, vocab, shards) in enumerate([(50, 10, 1), (1000, 100, 4), (5000, 3000, 8), (20000, 500, 5)]):
    fids = ((rng.integers(1, 30, size=n).astype(np.uint64) << np.uint64(48)) |
            rng.integers(0, vocab, size=n).astype(np.uint64))
    idx = np.zeros(n, np.int64)
    sizes = np.zeros(shards, np.int64)
    ref.ref_uniq_fid(fids.ctypes.data_as(C.c_void_p), C.c_int64(n), shards, idx.ctypes.data_as(C.c_void_p),
                     sizes.ctypes.data_as(C.c_void_p))
    u[f"c{ci}_fids"] = fids.view(np.int64)
    u[f"c{ci}_shards"] = np.int64(shards)
    u[f"c{ci}_uniq_idx"] = idx
    u[f"c{ci}_sizes"] = sizes
  u["n_cases"] = np.int64(4)
  np.savez(os.path.join(HERE, "ref_uniq_fid.npz"), **u)
  print("wrote golden fixtures")


if __name__ == "__main__":
  main()
