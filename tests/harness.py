"""Shared helpers for the parity tests: run the CUDA path through the C ABI on (values, valid) columns
and compare with the oracle.  Columns are (np.ndarray, bool ndarray | None)."""
from __future__ import annotations

import json
import os
import shutil
from typing import List, Optional, Sequence

import numpy as np

from datafusion_b200 import capi as D

HERE = os.path.dirname(os.path.abspath(__file__))
NP_TYPE = {"int32": np.int32, "int64": np.int64, "uint32": np.uint32, "float64": np.float64}


def load_golden(name: str):
    return json.load(open(os.path.join(HERE, "golden", name)))


def cuda_tool(name: str) -> str:
    """a CUDA toolkit binary (cuobjdump, ...): from PATH, else from the toolkit the Makefile's nvcc comes from, so the build-evidence
    tests do not depend on the toolkit's bin/ being on PATH"""
    return shutil.which(name) or os.path.join("/usr/local/cuda", "bin", name)


def col_from_list(values: Sequence, dtype=np.int32):
    """python list with None -> (values, valid)"""
    valid = np.array([v is not None for v in values], bool)
    vals = np.array([0 if v is None else v for v in values], dtype=dtype)
    return vals, (None if valid.all() else valid)


def host_cols(cols, start=0, stop=None, types=None):
    out = []
    for i, (v, val) in enumerate(cols):
        t = None if types is None else types[i]
        out.append(D.HostColumn(v[start:stop], None if val is None else val[start:stop], t))
    return out


def type_ids(cols, types=None):
    if types is not None:
        return list(types)
    return [D.TYPE_OF_NP[np.asarray(v).dtype] for v, _ in cols]


def batches_to_cols(batches, ncols) -> List:
    """concatenate output dfgpu batches into (values, valid) columns"""
    out = []
    for c in range(ncols):
        vals, valids, anyv = [], [], False
        for b in batches:
            v, val = b.column_numpy(c)
            vals.append(v)
            valids.append(np.ones(len(v), bool) if val is None else val)
            anyv |= val is not None
        if not vals:
            out.append((np.zeros(0, np.int64), None))
            continue
        v = np.concatenate(vals)
        val = np.concatenate(valids)
        out.append((v, None if (not anyv or val.all()) else val))
    return out


def split_points(n: int, batch_rows: Optional[int]):
    if not batch_rows or batch_rows >= n:
        return [(0, n)]
    return [(s, min(n, s + batch_rows)) for s in range(0, n, batch_rows)]


def gpu_hash_join(ctx, build, probe, on_build, on_probe, out_side, out_index, join_type=D.JOIN_INNER, null_equality=D.NULL_EQUALS_NOTHING,
                  batch_size=8192, phj=(1024, 0.15), force_collisions=False, build_batch_rows=None, probe_batch_rows=None, device=False,
                  build_types=None, probe_types=None, return_handle=False, filter=None, null_aware=False, ordered_output=True, membership_filter=False):
    bt, pt = type_ids(build, build_types), type_ids(probe, probe_types)
    j = D.HashJoinHandle(ctx, bt, pt, on_build, on_probe, out_side, out_index, join_type, null_equality, batch_size, phj[0], phj[1], force_collisions, null_aware, ordered_output, membership_filter)
    if filter is not None:
        j.set_filter(*filter)
    nb, npr = len(build[0][0]), len(probe[0][0])
    keep = []
    for s, e in split_points(nb, build_batch_rows):
        hc = host_cols(build, s, e, build_types)
        if device:
            dc = [D.DeviceColumn.from_host(ctx, h) for h in hc]
            keep.append(dc)
            j.push_build_device(dc)
        else:
            j.push_build_host(hc)
    j.finish_build()
    outs = []
    for s, e in split_points(npr, probe_batch_rows):
        hc = host_cols(probe, s, e, probe_types)
        if device:
            dc = [D.DeviceColumn.from_host(ctx, h) for h in hc]
            keep.append(dc)
            j.push_probe_device(dc)
        else:
            j.push_probe_host(hc)
        outs += j.drain(host=not device)
    j.finish_probe()
    outs += j.drain(host=not device)
    cols = batches_to_cols(outs, len(out_side))
    if return_handle:
        return cols, j
    j.close()
    return cols


def gpu_group_by(ctx, cols, group_cols, aggs, mode=D.AGG_SINGLE, batch_rows=None, device=False, types=None, capacity_hint=0, return_handle=False, skip_partial=None):
    t = type_ids(cols, types)
    a = D.AggHandle(ctx, t, group_cols, aggs, mode, 8192, capacity_hint)
    if skip_partial is not None:
        a.set_skip_partial(*skip_partial)
    n = len(cols[0][0])
    keep = []
    for s, e in split_points(n, batch_rows):
        hc = host_cols(cols, s, e, types)
        if device:
            dc = [D.DeviceColumn.from_host(ctx, h) for h in hc]
            keep.append(dc)
            a.push_device(dc)
        else:
            a.push_host(hc)
    a.finish()
    outs = a.drain(host=not device)
    ncols = outs[0].num_columns if outs else 0
    res = batches_to_cols(outs, ncols)
    if return_handle:
        return res, a
    a.close()
    return res


def gpu_filter(ctx, cols, nodes, projection=None, batch_rows=8192, batch_size=8192, fetch=-1, device=False, types=None):
    t = type_ids(cols, types)
    f = D.FilterHandle(ctx, t, nodes, projection, batch_size, fetch)
    n = len(cols[0][0])
    outs, keep = [], []
    for s, e in split_points(n, batch_rows):
        hc = host_cols(cols, s, e, types)
        if device:
            dc = [D.DeviceColumn.from_host(ctx, h) for h in hc]
            keep.append(dc)
            f.push_device(dc)
        else:
            f.push_host(hc)
        outs += f.drain(host=not device)
    f.finish()
    outs += f.drain(host=not device)
    nout = len(cols) if projection is None else len(projection)
    sizes = [o.num_rows for o in outs]
    res = batches_to_cols(outs, nout)
    f.close()
    return res, sizes


# ---- comparison ---------------------------------------------------------------------------
def _norm(col):
    v, val = col
    v = np.asarray(v)
    if val is None:
        val = np.ones(len(v), bool)
    val = np.asarray(val, bool)
    if v.dtype == np.bool_:
        v = v.astype(np.int8)
    v = np.where(val, v, np.zeros((), v.dtype))
    return v, val


def rows_matrix(cols):
    """structured view: each column contributes (valid, value-bits) so NULLs compare equal only to NULLs"""
    parts = []
    for c in cols:
        v, val = _norm(c)
        bits = v.view(np.int64) if v.dtype.itemsize == 8 else v.astype(np.int64) if v.dtype.kind in "iub" else v.astype(np.float64).view(np.int64)
        parts.append(val.astype(np.int64))
        parts.append(bits)
    return np.stack(parts, axis=1) if parts else np.zeros((0, 0), np.int64)


def assert_cols_equal(got, exp, ordered=True, what=""):
    assert len(got) == len(exp), f"{what}: column count {len(got)} != {len(exp)}"
    g, e = rows_matrix(got), rows_matrix(exp)
    assert g.shape == e.shape, f"{what}: shape {g.shape} != {e.shape}"
    if not ordered and len(g):
        g = g[np.lexsort(g.T[::-1])]
        e = e[np.lexsort(e.T[::-1])]
    if not np.array_equal(g, e):
        bad = np.nonzero((g != e).any(axis=1))[0][:5]
        raise AssertionError(f"{what}: rows differ at {bad.tolist()}:\n got {g[bad].tolist()}\n exp {e[bad].tolist()}")
