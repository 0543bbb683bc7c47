"""ctypes/numpy binding of the CPU oracle (oracle/liboracle.so) — test infrastructure only."""
import ctypes as C
import os

import numpy as np

from monolith_b200 import _lib as plib
from monolith_b200.entry import to_c_table_cfgs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_so = None


def lib():
  global _so
  if _so is None:
    _so = C.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
    _so.orc_mtable_size.restype = C.c_int64
    _so.orc_mtable_max_update_ts.restype = C.c_int64
    _so.orc_mtable_keys.restype = C.c_int64
    _so.orc_reorder_by_indices.restype = C.c_int64
    _so.orc_dedup.restype = C.c_int64
    _so.orc_uniform_init.restype = C.c_float
    _so.orc_uniform_init.argtypes = [C.c_uint64, C.c_int64, C.c_int, C.c_float, C.c_float]
    _so.orc_ps_size.restype = C.c_int64
  return _so


def p(a):
  return None if a is None else a.ctypes.data_as(C.c_void_p)


def i64(x):
  return np.ascontiguousarray(np.asarray(x, dtype=np.int64))


def f32(x):
  return np.ascontiguousarray(np.asarray(x, dtype=np.float32))


def i32(x):
  return np.ascontiguousarray(np.asarray(x, dtype=np.int32))


class OracleMultiHashTable:
  """Same surface as monolith_b200.MultiHashTable, numpy in / numpy out."""

  def __init__(self, configs):
    self.names = tuple(sorted(configs.keys()))
    self.configs = {k: configs[k] for k in self.names}
    arr, keep = to_c_table_cfgs(self.configs)
    self._keep = keep
    h = C.c_void_p()
    assert lib().orc_mtable_create(arr, len(self.names), C.byref(h)) == 0
    self.h = h
    self.dims = [lib().orc_mtable_dim(h, k) for k in range(len(self.names))]
    self.state = [lib().orc_mtable_state_floats(h, k) for k in range(len(self.names))]

  def __del__(self):
    try:
      lib().orc_mtable_destroy(self.h)
    except Exception:
      pass

  def set_hash_filter(self, slot, capacity, default_threshold, slot_thresholds=None):
    """Counting admission filter on table `slot` (oracle only so far: SURVEY §8(f) row 2)."""
    st = slot_thresholds or {}
    ks = np.ascontiguousarray(np.array(list(st.keys()), np.uint32))
    vs = np.ascontiguousarray(np.array(list(st.values()), np.uint32))
    assert lib().orc_mtable_set_hash_filter(self.h, self.names.index(slot), C.c_int64(capacity),
                                            C.c_uint32(default_threshold), p(ks), p(vs), len(st)) == 0

  def lrs(self):
    out = []
    for n in self.names:
      out += self.configs[n].call_learning_rate_fns()
    return f32(out)

  def pack(self, d):
    ids, splits = [], [0]
    for n in self.names:
      v = i64(d[n]).reshape(-1) if n in d else np.zeros(0, np.int64)
      ids.append(v)
      splits.append(splits[-1] + v.size)
    return i64(np.concatenate(ids)), i64(splits)

  def pack_vals(self, d):
    return f32(np.concatenate([f32(d[n]).reshape(-1) for n in self.names if n in d] or [np.zeros(0, np.float32)]))

  def unpack(self, splits, flat):
    out, off = {}, 0
    for k, n in enumerate(self.names):
      c = int(splits[k + 1] - splits[k])
      out[n] = flat[off:off + c * self.dims[k]].reshape(c, self.dims[k])
      off += c * self.dims[k]
    return out

  def raw_lookup(self, ids, splits):
    ids, splits = i64(ids), i64(splits)
    total = sum(int(splits[k + 1] - splits[k]) * self.dims[k] for k in range(len(self.dims)))
    out = np.zeros(total, np.float32)
    lib().orc_mtable_lookup(self.h, p(ids), p(splits), p(out))
    return out

  def lookup(self, d):
    ids, splits = self.pack(d)
    emb = self.unpack(splits, self.raw_lookup(ids, splits))
    return {k: v for k, v in emb.items() if k in d}

  def assign(self, d, req_time=0):
    ids, splits = self.pack({k: v[0] for k, v in d.items()})
    vals = self.pack_vals({k: v[1] for k, v in d.items()})
    lib().orc_mtable_assign(self.h, p(ids), p(splits), p(vals), C.c_int64(req_time))

  def assign_add(self, d, req_time=0):
    ids, splits = self.pack({k: v[0] for k, v in d.items()})
    vals = self.pack_vals({k: v[1] for k, v in d.items()})
    lib().orc_mtable_assign_add(self.h, p(ids), p(splits), p(vals), C.c_int64(req_time))

  def apply_gradients(self, d, global_step=0, req_time=0, enable_dedup=False):
    ids, splits = self.pack({k: v[0] for k, v in d.items()})
    vals = self.pack_vals({k: v[1] for k, v in d.items()})
    self.raw_apply_gradients(ids, splits, vals, global_step, req_time, enable_dedup)

  def raw_apply_gradients(self, ids, splits, grads, global_step=0, req_time=0, enable_dedup=False):
    ids, splits, grads, lr = i64(ids), i64(splits), f32(grads), self.lrs()
    lib().orc_mtable_optimize(self.h, p(ids), p(splits), p(grads), p(lr), C.c_int64(req_time),
                              C.c_int64(global_step), int(enable_dedup))

  def reinitialize(self, slot, ids, update_time=0):
    ids = i64(ids)
    st = np.zeros(ids.size, np.int32)
    k = self.names.index(slot) if slot in self.names else -1
    lib().orc_mtable_reinitialize(self.h, k, p(ids), C.c_int64(ids.size), p(st), C.c_int64(update_time))
    return st

  def fused_offsets(self, slot_size, N):
    ss = i32(slot_size)
    K = len(self.dims)
    es, ko, eo = np.zeros(N, np.int32), np.zeros(N * K + 1, np.int32), np.zeros(N * K + 1, np.int32)
    lib().orc_mtable_fused_offsets(self.h, p(ss), N, p(es), p(ko), p(eo))
    return es, ko, eo

  def fused_lookup(self, ids, slot_size, N):
    ids, ss = i64(ids), i32(slot_size)
    es, ko, eo = self.fused_offsets(ss, N)
    out = np.zeros(int(eo[-1]), np.float32)
    lib().orc_mtable_fused_lookup(self.h, p(ids), p(ss), N, p(out))
    return out, es, ko, eo

  def fused_apply_gradient(self, ids, slot_size, grads, N, req_time=0, enable_grad_accumulation=False):
    ids, ss, grads, lr = i64(ids), i32(slot_size), f32(grads), self.lrs()
    es, ko, eo = self.fused_offsets(ss, N)
    lib().orc_mtable_fused_optimize(self.h, p(ids), p(ss), p(grads), p(ko), p(eo), p(lr), C.c_int64(req_time),
                                    C.c_int64(0), N, int(enable_grad_accumulation))

  def evict(self, slot, max_update_time):
    lib().orc_mtable_evict(self.h, self.names.index(slot), C.c_int64(max_update_time))

  def size(self, slot):
    return lib().orc_mtable_size(self.h, self.names.index(slot))

  def contains(self, slot, ids):
    ids = i64(ids)
    out = np.zeros(ids.size, np.uint8)
    lib().orc_mtable_contains(self.h, self.names.index(slot), p(ids), C.c_int64(ids.size), p(out))
    return out.astype(bool)

  def lookup_entry(self, slot, ids):
    k = self.names.index(slot)
    ids = i64(ids)
    W = self.dims[k] + self.state[k] + 2
    out = np.zeros((ids.size, W), np.float32)
    lib().orc_mtable_lookup_entry(self.h, k, p(ids), C.c_int64(ids.size), p(out))
    return out

  def keys(self, slot):
    k = self.names.index(slot)
    n = self.size(slot)
    out = np.zeros(max(n, 1), np.int64)
    lib().orc_mtable_keys(self.h, k, p(out), C.c_int64(out.size))
    return np.sort(out[:n])

  def lookup_pool(self, slot, fids, row_offsets=None, pooling="sum"):
    k = self.names.index(slot)
    fids = i64(fids)
    ro = None if row_offsets is None else i32(row_offsets)
    n_rows = fids.size if ro is None else ro.size - 1
    out = np.zeros((n_rows, self.dims[k]), np.float32)
    lib().orc_mtable_lookup_pool(self.h, k, p(fids), p(ro), C.c_int64(n_rows), {"sum": 0, "mean": 1}[pooling],
                                 p(out), C.c_int64(self.dims[k]), 0)
    return out


def reorder_by_indices(inputs, N, dims, rank0_empty=False):
  K = len(inputs)
  ids = i64(np.concatenate([i64(x).reshape(-1) for x in inputs] or [np.zeros(0, np.int64)]))
  splits = i64(np.cumsum([0] + [np.asarray(x).size for x in inputs]))
  M = ids.size
  out = np.zeros(max(M, 1), np.int64)
  shard_sizes, slot_sizes = np.zeros(N, np.int32), np.zeros(N * K, np.int32)
  sz, offs = np.zeros(K, np.int32), np.zeros(max(M, 1), np.int32)
  u = lib().orc_reorder_by_indices(p(ids), p(splits), K, N, p(i32(dims)), int(rank0_empty), p(out),
                                   p(shard_sizes), p(slot_sizes), p(sz), p(offs))
  return out[:u], shard_sizes, slot_sizes, sz, offs[:M]


def dedup(ids):
  ids = i64(ids)
  u, inv = np.zeros(max(ids.size, 1), np.int64), np.zeros(max(ids.size, 1), np.int32)
  n = lib().orc_dedup(p(ids), C.c_int64(ids.size), p(u), p(inv))
  return u[:n], inv[:ids.size]


def gather_pool(fused, offsets, dim, row_offsets=None, pooling="sum"):
  fused, offsets = f32(fused), i32(offsets)
  ro = None if row_offsets is None else i32(row_offsets)
  n_rows = offsets.size if ro is None else ro.size - 1
  out = np.zeros((n_rows, dim), np.float32)
  lib().orc_gather_pool(p(fused), p(offsets), p(ro), C.c_int64(n_rows), dim, {"sum": 0, "mean": 1}[pooling],
                        p(out), C.c_int64(dim), 0)
  return out


def gather_pool_grad(pooled_grad, offsets, dim, total, row_offsets=None, pooling="sum"):
  g, offsets = f32(pooled_grad), i32(offsets)
  ro = None if row_offsets is None else i32(row_offsets)
  n_rows = offsets.size if ro is None else ro.size - 1
  out = np.zeros(total, np.float32)
  lib().orc_gather_pool_grad(p(g), C.c_int64(dim), 0, p(offsets), p(ro), C.c_int64(n_rows), dim,
                             {"sum": 0, "mean": 1}[pooling], p(out))
  return out


def _task_arr(tasks):
  arr = (plib.SliceTask * len(tasks))()
  for i, t in enumerate(tasks):
    for f, _ in plib.SliceTask._fields_:
      setattr(arr[i], f, int(getattr(t, f)))
  return arr


def embedding_to_layout(embs, strides, fid_offset, feature_offset, nfl_offset, batch_size, tasks, out_shapes):
  embs = [f32(e).reshape(-1) for e in embs]
  outs = [np.zeros(s, np.float32) for s in out_shapes]
  ep = (C.c_void_p * len(embs))(*[e.ctypes.data for e in embs])
  op = (C.c_void_p * len(outs))(*[o.ctypes.data for o in outs])
  sizes = i64([o.size for o in outs])
  fo = np.ascontiguousarray(np.asarray(fid_offset, dtype=np.uint64))
  fe, nf = i32(feature_offset), np.ascontiguousarray(np.asarray(nfl_offset, dtype=np.uint32))
  lib().orc_embedding_to_layout(ep, p(i32(strides)), len(embs), p(fo), C.c_int64(fo.size), p(fe), fe.size, p(nf),
                                nf.size, batch_size, _task_arr(tasks), len(tasks), op, p(sizes), len(outs))
  return outs


def embedding_to_layout_grad(emb_sizes, strides, fid_offset, feature_offset, nfl_offset, batch_size, tasks,
                             out_grads):
  grads = [np.zeros(n, np.float32) for n in emb_sizes]
  og = [f32(g) for g in out_grads]
  gp = (C.c_void_p * len(grads))(*[g.ctypes.data for g in grads])
  op = (C.c_void_p * len(og))(*[g.ctypes.data for g in og])
  fo = np.ascontiguousarray(np.asarray(fid_offset, dtype=np.uint64))
  fe, nf = i32(feature_offset), np.ascontiguousarray(np.asarray(nfl_offset, dtype=np.uint32))
  lib().orc_embedding_to_layout_grad(gp, p(i32(strides)), p(i64(emb_sizes)), len(grads), p(fo), C.c_int64(fo.size),
                                     p(fe), fe.size, p(nf), nf.size, batch_size, _task_arr(tasks), len(tasks), op)
  return grads
